"""GPU tests of extract_kmer_pairs from the strand-symmetric scan (Scan.extract(pix, "symm"),
hm_scan_extract_path): the candidates the scan leaves on the device are judged again and the isolated pairs of
labelled pixels written as records -- the pair and its mirror image (csrc/hm_symm.cu, RecordSink).  Compared with
the golden pair lists the reference wrote, with the direct route (hm_scan_extract), with the digests of the
reference's output on seeded tables and with the oracle, on replicas and on sharded tables."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
import oracle_util as ou
from smudgeplot_b200 import _lib, fastk, hetmers
from tools import synth
from test_gpu_parity import EXTRACT_CASES, _golden_pairs, label_sma, reference_run
from test_symm_extract_identity import symmetric_table

pytestmark = pytest.mark.gpu

DNA = "acgt"
REC_BYTES = 24                                   # sizeof(hm_pair_rec)


@pytest.fixture(scope="module", autouse=True)
def _need_gpu(built):
    assert _lib.lib().hm_device_count() >= 1, "these tests need a CUDA device (no CPU fallback exists)"


def _golden(name):
    return os.path.join(GOLDEN, name, name)


def read_sma(path):
    """pixmap + label names in order of first appearance, as extract_kmer_pairs reads a .sma (hetmers_main.c)"""
    pix = np.zeros((_lib.SMAX + 1, _lib.PLOT_W), dtype=np.uint16)
    order = []
    with open(path) as f:
        f.readline()
        for ln in f:
            covb, cova, _, lab = ln.split()
            if lab not in order:
                order.append(lab)
            pix[int(covb) + int(cova), int(covb)] = order.index(lab) + 1
    return pix, order


def fmt(r, k):
    bases = [((int(r["key_hi"]) if p < 32 else int(r["key_lo"])) >> (62 - 2 * (p & 31))) & 3 for p in range(k)]
    return "".join(f"({DNA[b]}/{DNA[int(r['alt'])]})" if p == int(r["pos"]) else DNA[b] for p, b in enumerate(bases))


def pair_lines(rec, k, order):
    """{label: sorted lines} of a record array (every label of the .sma, empty ones included)"""
    out = {lab: [] for lab in order}
    for r in rec:
        out[order[int(r["smudge"]) - 1]].append(fmt(r, k))
    return {lab: sorted(v) for lab, v in out.items()}


def placements():
    return [None, 2, 3, 5]


def open_scan(kt, S):
    return hetmers.Scan(kt) if S is None else hetmers.Scan(kt, shards=[0] * S)


def oracle_lines(tmp_path, k, keys, cnt, plot, tag):
    """the oracle's extract_kmer_pairs on the table written as a file and a .sma labelling `plot`"""
    table = str(tmp_path / f"o{tag}")
    fastk.write_ktab(table, k, keys, cnt, ibyte=1 if k < 8 else 2)
    sma = str(tmp_path / f"o{tag}.sma")
    pix, order = label_sma(plot, sma)
    out = str(tmp_path / f"okp{tag}")
    assert ou.oracle_extract(table, 1, sma, out) == 0
    return pix, order, ou.sorted_pair_files(out)


# ------------------------------------------------------------------ 1. goldens with a .sma -----

SMA_GOLDENS = [n for n in golden_cases() if os.path.exists(os.path.join(GOLDEN, n, n + ".sma"))]


@pytest.mark.parametrize("S", placements())
@pytest.mark.parametrize("name", SMA_GOLDENS)
def test_golden_pair_lists_from_the_symmetric_scan(name, S):
    kt = fastk.read_ktab(_golden(name))
    pix, order = read_sma(_golden(name) + ".sma")
    with open_scan(kt, S) as sc:
        plot, _ = sc.run()
        rec, st = sc.extract(pix, "symm", stats=True)
    assert st["path"] == 2 and st["n_records"] == len(rec) == int(plot[pix > 0].sum())
    want = {lab: sorted(v) for lab, v in _golden_pairs(name).items()}
    assert pair_lines(rec, kt.kmer, order) == want


# ------------------------------------------------------------------ 2. every golden table ------

@pytest.mark.parametrize("name", golden_cases())
def test_symmetric_records_equal_direct_records_on_every_golden(name, tmp_path):
    kt = fastk.read_ktab(_golden(name))
    with hetmers.Scan(kt) as sc:
        plot, _ = sc.run()
        pix, _ = label_sma(plot, str(tmp_path / "a.sma"))
        sym, st = sc.extract(pix, "symm", stats=True)
        direct = sc.extract(pix, "direct")
    assert st["path"] == 2
    assert len(sym) == int(plot[pix > 0].sum())
    assert np.array_equal(sym, direct)
    with hetmers.Scan(kt) as sc:
        assert np.array_equal(sc.extract(pix), direct)                  # hm_scan_extract, as before
    with hetmers.Scan(kt, shards=[0] * 3) as sc:
        sc.run()
        shd = sc.extract(pix, "symm")
    assert np.array_equal(shd, direct)


# ------------------------------------------------------------------ 3. seeded, vs the reference's digests

def expected_slices(keys, cnt, k, ranges):
    """slices an extraction takes: per scan range, its candidates over the records' room in the range's
    run-head region (hm_symm_extract_slice: 8 * runs_cap bytes, 2 records per candidate)"""
    import ctypes as C
    import torch
    from smudgeplot_b200.device import DeviceTable
    khi = keys[:, 0].contiguous() if k > 32 else keys
    klo = keys[:, 1].contiguous() if k > 32 else None
    t = DeviceTable(k, khi, cnt.to(torch.int16), keys_lo=klo).build_index(direct=False)
    total = 0
    for lo, hi in ranges:
        t.alloc_symm(lo, hi)
        t.runscan()
        nc, st = t.symm_status()
        assert st == 0
        lay = _lib.SymmLayout()
        _lib.check(_lib.lib().hm_symm_plan(t.n, hi - lo, k, 1, C.byref(lay)))
        per = (8 * lay.runs_cap // REC_BYTES) // 2
        total += -(-nc // per)
    return total


@pytest.mark.parametrize("S", [None, 3])
@pytest.mark.parametrize("k,G,ploidy,seed,L", EXTRACT_CASES)
def test_seeded_extraction_matches_reference_digests(k, G, ploidy, seed, L, S, tmp_path):
    want = reference_run("extract", k, G, ploidy, seed, L)
    keys, cnt = synth.synth_table(k, G, ploidy, 0.02, 20 * ploidy, L, seed, device="cuda")
    kt = synth.write_table(str(tmp_path / "t"), k, keys, cnt, ibyte=3, nparts=3)
    assert kt.nels == want["nels"]
    with open_scan(kt, S) as sc:
        plot, _ = sc.run()
        pix, order = label_sma(plot, str(tmp_path / "ann.sma"))
        rec, st = sc.extract(pix, "symm", stats=True)
        info = sc.shard_info()
    ranges = [(0, kt.nels)] if S is None else [(s["first_index"], s["first_index"] + s["n"]) for s in info]
    lines = pair_lines(rec, k, order)
    assert {lab: len(v) for lab, v in lines.items()} == {lab: w["lines"] for lab, w in want["pairs"].items()}
    assert {lab: ou.sha256_lines(v) for lab, v in lines.items()} == {lab: w["sha256"] for lab, w in want["pairs"].items()}
    assert st["slices"] >= 2
    assert st["slices"] == expected_slices(keys, cnt, k, ranges)


# ------------------------------------------------------------------ 4. seeded tables vs the oracle

def _check_vs_oracle(tmp_path, k, keys, cnt, tag, nparts=1):
    kt = fastk.write_ktab(str(tmp_path / f"t{tag}"), k, keys, cnt, ibyte=1 if k < 8 else 2, nparts=nparts)
    with hetmers.Scan(kt) as sc:
        plot, _ = sc.run()
        pix, order, want = oracle_lines(tmp_path, k, keys, cnt, plot, tag)
        sym = sc.extract(pix, "symm")
        direct = sc.extract(pix, "direct")
    assert np.array_equal(sym, direct)
    assert pair_lines(sym, k, order) == want
    return len(sym)


@pytest.mark.parametrize("k,G,ploidy,seed", [(33, 40000, 2, 61), (47, 40000, 3, 62), (64, 30000, 2, 63),
                                             (9, 3000, 2, 64), (5, 400, 2, 65)])
def test_seeded_symmetric_tables_equal_direct_and_oracle(k, G, ploidy, seed, tmp_path):
    keys, cnt = synth.synth_table(k, G, ploidy, 0.03, 20 * ploidy, 1, seed, extra_hom_repeats=1)
    ku = synth.keys_to_u64_numpy(keys)
    n = _check_vs_oracle(tmp_path, k, ku, cnt.numpy().astype(np.uint16), "s")
    assert n > 0 or k <= 7                                             # (crowded tiny-k tables may have no isolated pair)


@pytest.mark.parametrize("k,n0,cmin,cmax,seed,middle", [(31, 1500, 1, 40, 2, 40), (25, 1500, 7, 8, 5, 30),
                                                        (5, 300, 3, 4, 8, 5), (7, 2000, 1, 6, 9, 10)])
def test_middle_base_tables_equal_direct_and_oracle(k, n0, cmin, cmax, seed, middle, tmp_path):
    keys, cnt = symmetric_table(k, n0, cmin, cmax, seed, dense=(k <= 7), middle=middle)
    _check_vs_oracle(tmp_path, k, keys, cnt, "m")


# ------------------------------------------------------------------ 5. paths and refusals ------

def test_paths_and_refusals(golden_meta, tmp_path):
    # a table that passes the reference's one-k-mer probe without being symmetric: AUTO takes the direct route
    k = 31
    keys, cnt = synth.synth_table(k, 60000, 2, 0.02, 40, 4, 321)
    ku = synth.keys_to_u64_numpy(keys)
    cu = cnt.numpy().astype(np.uint16)
    keep = np.ones(len(ku), dtype=bool)
    keep[len(ku) // 3] = False
    ku, cu = ku[keep], cu[keep]
    akt = fastk.write_ktab(str(tmp_path / "asym"), k, ku, cu, ibyte=3, nparts=2)
    with hetmers.Scan(akt) as sc:
        assert sc.examine(4) == (True, True)                            # the probe is fooled
        plot, st = sc.run()
        assert st["path"] == 1
        pix, order, want = oracle_lines(tmp_path, k, ku, cu, plot, "a")
        rec, xs = sc.extract(pix, "auto", stats=True)
        assert xs["path"] == 1 and pair_lines(rec, k, order) == want
        with pytest.raises(_lib.HetmersError) as e:
            sc.extract(pix, "symm")
        assert e.value.code == _lib.EINVAL
        plot2, _ = sc.run()                                             # still usable after the refusal
        assert np.array_equal(plot2, plot)
        assert np.array_equal(sc.extract(pix, "auto"), rec)
    # extraction before any run scans first; so does extraction after a conditioning
    name = "dip_k21"
    pix, order = read_sma(_golden(name) + ".sma")
    want = {lab: sorted(v) for lab, v in _golden_pairs(name).items()}
    with hetmers.Scan(fastk.read_ktab(_golden(name))) as sc:
        rec, xs = sc.extract(pix, "symm", stats=True)
        assert xs["path"] == 2 and pair_lines(rec, 21, order) == want
        rec2, xs = sc.extract(pix, "auto", stats=True)
        assert xs["path"] == 2 and np.array_equal(rec2, rec)
    c = golden_meta["_conditioning"]["asymmetric"]
    ckt = fastk.read_ktab(os.path.join(GOLDEN, "conditioning", "asymmetric"))
    with hetmers.Scan(ckt) as sc:
        sc.condition(c["e"], False, True)
        plot, _ = sc.run()
        pix, _ = label_sma(plot, str(tmp_path / "c.sma"))
        direct = sc.extract(pix, "direct")
        sc.condition(c["e"], True, False)                               # the same table, conditioned again
        assert np.array_equal(sc.extract(pix, "symm"), direct)
    with hetmers.Scan(ckt) as sc:
        sc.condition(c["e"], False, True)
        rec, xs = sc.extract(pix, "symm", stats=True)                   # no run since the conditioning
        assert xs["path"] == 2 and np.array_equal(rec, direct) and len(rec) == int(plot[pix > 0].sum())
    with hetmers.Scan(ckt) as sc:                                       # not symmetrised: no symmetric route
        with pytest.raises(_lib.HetmersError) as e:
            sc.extract(pix, "symm")
        assert e.value.code == _lib.EINVAL


def test_sharded_table_refuses_the_direct_route():
    kt = fastk.read_ktab(_golden("dip_k21"))
    pix, _ = read_sma(_golden("dip_k21") + ".sma")
    with hetmers.Scan(kt, shards=[0, 0]) as sc:
        with pytest.raises(_lib.HetmersError) as e:
            sc.extract(pix, "direct")
        assert e.value.code == _lib.EUNSUPPORTED
        rec, xs = sc.extract(pix, "auto", stats=True)
        assert xs["path"] == 2 and len(rec) > 0


# ------------------------------------------------------------------ 6. several GPUs ------------

def test_several_gpus_equal_one_gpu_direct(tmp_path):
    ngpu = _lib.lib().hm_device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    keys, cnt = synth.synth_table(31, 400000, 3, 0.01, 60, 12, 4, device="cuda")
    kt = synth.write_table(str(tmp_path / "t"), 31, keys, cnt, ibyte=3, nparts=3)
    with hetmers.Scan(kt) as sc:
        plot, _ = sc.run("direct")
        pix, _ = label_sma(plot, str(tmp_path / "a.sma"))
        want = sc.extract(pix, "direct")
    for g in (2, 4, 8):
        if g > ngpu:
            continue
        with hetmers.Scan(kt, gpus=g) as sc:
            sc.run()
            assert np.array_equal(sc.extract(pix, "symm"), want)
        with hetmers.Scan(kt, shards=list(range(g))) as sc:
            sc.run()
            assert np.array_equal(sc.extract(pix, "symm"), want)


# ------------------------------------------------------------------ 7. the executable ----------

def _run_extract(table, sma, out, L, gpus=1):
    env = dict(os.environ, HETMERS_STATS="1", HETMERS_GPUS=str(gpus))
    r = subprocess.run([hetmers.get_binary_path("extract_kmer_pairs"), f"-e{L}", "-T4", f"-o{out}", table,
                        sma[:-4] if sma.endswith(".sma") else sma], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    return json.loads([ln for ln in r.stderr.splitlines() if ln.startswith("{")][-1])


@pytest.mark.parametrize("name", SMA_GOLDENS)
def test_executable_extracts_from_the_symmetric_scan(name, golden_meta, tmp_path):
    out = str(tmp_path / "kp")
    st = _run_extract(_golden(name), _golden(name) + ".sma", out, golden_meta[name]["e"])
    assert ou.sorted_pair_files(out) == {lab: sorted(v) for lab, v in _golden_pairs(name).items()}
    assert st["path"] == "symmetric" and st["extract"]["path"] == "symmetric"
    assert st["extract"]["pairs"] == sum(len(v) for v in _golden_pairs(name).values())
    assert st["extract"]["slices"] >= 1


def test_executable_extracts_pairs_of_a_sharded_table(tmp_path):
    """the ballast setup of test_executable_shards_a_table_its_gpus_cannot_hold_as_replicas: the executable
    places the table as sharded and writes the pair files of an in-process replica extraction"""
    import torch
    ngpu = _lib.lib().hm_device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    g = min(ngpu, 8)
    k, L = 31, 12
    G = synth.calibrate_G(k, 200_000_000, 2, 0.01, 40, L)
    keys, cnt = synth.synth_table(k, G, 2, 0.01, 40, 1, 21, device="cuda")
    rc = synth.revcomp_left(keys, k)
    canon = (keys.view(torch.int64) ^ (1 << 63)) <= (rc.view(torch.int64) ^ (1 << 63))
    raw = str(tmp_path / "raw")
    kt = synth.write_table(raw, k, keys[canon].contiguous(), cnt[canon].contiguous(), ibyte=3, nparts=4)
    del keys, cnt, rc, canon
    sma = str(tmp_path / "ann.sma")
    with hetmers.Scan(fastk.read_ktab(raw)) as sc:
        sc.condition(L, True, True)
        plot, _ = sc.run()
        pix, order = label_sma(plot, sma)
        want = pair_lines(sc.extract(pix, "symm"), k, order)
    torch.cuda.empty_cache()
    _, rep, shd = _lib.plan_placement(k, kt.nels, [1 << 50] * g, True)
    target = (rep + shd) // 2 + (512 << 20)
    ballast = []
    try:
        for d in range(g):
            free, _ = torch.cuda.mem_get_info(d)
            if free <= target:
                pytest.skip(f"GPU {d} has only {free} bytes free")
            ballast.append(torch.empty(free - target, dtype=torch.uint8, device=f"cuda:{d}"))
        out = str(tmp_path / "kp")
        st = _run_extract(raw, sma, out, L, g)
    finally:
        del ballast
        torch.cuda.empty_cache()
    assert st["placement"] == "sharded" and st["extract"]["path"] == "symmetric"
    assert ou.sorted_pair_files(out) == want
