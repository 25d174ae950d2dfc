"""GPU parity tests (run with -m gpu on the B200 box).  Everything goes through the C ABI of
libhetmers_b200.so (in-process via ctypes, or through the drop-in `hetmers` executable) and is
compared bit for bit with (a) the golden .smu files written by the unmodified reference binary,
(b) the oracle on seeded tables, (c) what the reference binaries wrote for larger seeded tables
(digests in golden/reference_runs.json), and (d) size-independent properties at BASELINE.json's full size."""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
import oracle_util as ou
from smudgeplot_b200 import _lib, fastk, hetmers
from tools import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu(built):
    assert _lib.lib().hm_device_count() >= 1, "these tests need a CUDA device (no CPU fallback exists)"


def _golden(name):
    return os.path.join(GOLDEN, name, name)


# ------------------------------------------------------------------ (a) golden vectors ------

@pytest.mark.parametrize("name", golden_cases())
def test_executable_reproduces_reference_smu(name, golden_meta, tmp_path):
    c = golden_meta[name]
    out = str(tmp_path / "out")
    r = subprocess.run([_lib.BIN_PATH, "-v", f"-e{c['e']}", "-T4", f"-o{out}", _golden(name)],
                       input="n\n", capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout == ""
    assert r.stderr == ("\n  The input table is trimmed and symmetric\n"
                        "\n  Starting to count covariant pairs\n"
                        "\n  Count complete, outputting table\n")       # the reference's -v lines
    assert open(out + ".smu").read() == open(_golden(name) + ".smu").read()


@pytest.mark.parametrize("name", golden_cases())
def test_inprocess_scan_reproduces_reference_smu_and_oracle_deg(name, golden_meta):
    c = golden_meta[name]
    kt = fastk.read_ktab(_golden(name))
    kb, cn = fastk.unpack_host(kt)
    with hetmers.Scan(kt) as sc:
        assert sc.examine(c["e"]) == (True, True)
        plot, stats = sc.run()
        keys, cnt, deg = sc.download()
    assert hetmers.smu_text(plot) == open(_golden(name) + ".smu").read()
    assert np.array_equal(keys, fastk.keys_bytes_to_u64(kb))            # GPU unpack == host unpack
    assert np.array_equal(cnt, cn)
    want_plot, want_deg = ou.oracle_scan(kb, cn, kt.kmer)
    assert np.array_equal(deg, want_deg)                                # pass-1 incidence array
    assert np.array_equal(plot, want_plot)                              # incl. the dropped m=500 column
    assert stats["nels"] == c["nels"] and stats["kernel_launches"] >= 4


def test_default_output_root_and_ktab_suffix(tmp_path):
    d = tmp_path / "g"
    shutil.copytree(os.path.join(GOLDEN, "dip_k21"), d)
    r = subprocess.run([_lib.BIN_PATH, str(d / "dip_k21.KTAB")], input="n\n", capture_output=True, text=True)
    assert r.returncode == 0, r.stderr                                  # default -e4, -T4
    assert (d / "dip_k21.smu").read_text() == open(_golden("dip_k21") + ".smu").read()
    # second run: file exists -> prompt; "n" recomputes, "y" leaves it
    r = subprocess.run([_lib.BIN_PATH, str(d / "dip_k21")], input="n\n", capture_output=True, text=True)
    assert r.returncode == 0 and "Found het-table" in r.stdout


# ------------------------------------------------------------------ extract_kmer_pairs -------

def _golden_pairs(name):
    d = os.path.join(GOLDEN, name)
    pre = name + ".pairs."
    return {f[len(pre):-4]: open(os.path.join(d, f)).read().splitlines()
            for f in sorted(os.listdir(d)) if f.startswith(pre)}


@pytest.mark.parametrize("name", [n for n in golden_cases() if os.path.exists(os.path.join(GOLDEN, n, n + ".sma"))])
def test_extract_executable_reproduces_reference_pair_lists(name, golden_meta, tmp_path):
    c = golden_meta[name]
    out = str(tmp_path / "kp")
    hetmers.run_extract(_golden(name), _golden(name) + ".sma", o=out, t=4, e=c["e"])
    assert ou.sorted_pair_files(out) == _golden_pairs(name)


def reference_run(kind, *params):
    """what the reference binaries wrote for the seeded table of one parameter set (golden/reference_runs.json,
    recorded by golden/make_golden.py; keyed like the pytest id)"""
    with open(os.path.join(GOLDEN, "reference_runs.json")) as f:
        return json.load(f)[kind]["-".join(str(p) for p in params)]


def label_sma(plot, sma):
    """write <sma> labelling every plotted pixel by (sum + min) % 4 (three smudges, a quarter unlabelled)
    -> (pixmap uint16[1001,501] of smudge numbers in order of first appearance, label names in that order)"""
    s_idx, m_idx = np.nonzero(plot[:, :_lib.FMAX] > 0)
    pix = np.zeros((_lib.SMAX + 1, _lib.PLOT_W), dtype=np.uint16)
    labels = ["1A1B", "2A1B", "2A2B"]
    order = []
    with open(sma, "w") as f:
        f.write("covB\tcovA\tfreq\tsmudge\n")
        for s, m in zip(s_idx.tolist(), m_idx.tolist()):
            lab = (s + m) % 4
            if lab < 3:
                if labels[lab] not in order:
                    order.append(labels[lab])
                pix[s, m] = order.index(labels[lab]) + 1
                f.write(f"{m}\t{s - m}\t{plot[s, m]}\t{labels[lab]}\n")
    return pix, order


EXTRACT_CASES = [(31, 400000, 3, 41, 12), (40, 150000, 2, 42, 4)]


@pytest.mark.parametrize("k,G,ploidy,seed,L", EXTRACT_CASES)
def test_extract_matches_reference_binary_and_inprocess_list(k, G, ploidy, seed, L, tmp_path):
    """bigger seeded table: our extract_kmer_pairs vs the reference's (sorted lines, as digests), and the
    in-process pair list (hm_scan_extract) vs the files"""
    want = reference_run("extract", k, G, ploidy, seed, L)
    keys, cnt = synth.synth_table(k, G, ploidy, 0.02, 20 * ploidy, L, seed, device="cuda")
    name = str(tmp_path / "t")
    kt = synth.write_table(name, k, keys, cnt, ibyte=3, nparts=3)
    assert kt.nels == want["nels"]                                    # the table the reference read
    sma = str(tmp_path / "ann.sma")
    with hetmers.Scan(kt) as sc:
        plot, _ = sc.run()
        pix, order = label_sma(plot, sma)
        rec = sc.extract(pix)
    assert len(rec) == int(plot[pix > 0].sum())                       # one record per labelled isolated pair
    out = str(tmp_path / "kp")
    hetmers.run_extract(name, sma, o=out, t=4, e=L)
    ours = ou.sorted_pair_files(out)
    assert sum(len(v) for v in ours.values()) == len(rec)
    assert {lab: len(v) for lab, v in ours.items()} == {lab: w["lines"] for lab, w in want["pairs"].items()}
    assert {lab: ou.sha256_lines(v) for lab, v in ours.items()} == {lab: w["sha256"] for lab, w in want["pairs"].items()}
    dna = "acgt"
    def fmt(r):
        bases = [((int(r["key_hi"]) if p < 32 else int(r["key_lo"])) >> (62 - 2 * (p & 31))) & 3 for p in range(k)]
        return "".join(f"({dna[b]}/{dna[int(r['alt'])]})" if p == int(r["pos"]) else dna[b] for p, b in enumerate(bases))
    mine = {}
    for r in rec[:: max(1, len(rec) // 2000)]:                        # spot-check the in-process records
        assert fmt(r) in ours[order[int(r["smudge"]) - 1]]
    del mine


# ------------------------------------------------------------------ conditioning verdicts ----

@pytest.mark.parametrize("name,verdict,tool", [("untrimmed", (False, True), "Logex"),
                                               ("asymmetric", (True, False), "Symmex")])
def test_examine_table_decisions(name, verdict, tool, golden_meta, tmp_path):
    c = golden_meta["_conditioning"][name]
    table = os.path.join(GOLDEN, "conditioning", name)
    with hetmers.Scan(fastk.read_ktab(table)) as sc:
        assert sc.examine(c["e"]) == verdict
    # with HETMERS_EXTERNAL_CONDITIONING the executable prints the reference's verdict and then
    # shells out to the same FastK tool with the same command line as the reference
    env = dict(os.environ, HETMERS_EXTERNAL_CONDITIONING="1")
    r = subprocess.run([_lib.BIN_PATH, "-v", f"-e{c['e']}", "-T4", f"-o{tmp_path}/o", table],
                       input="n\n", capture_output=True, text=True, cwd=tmp_path, env=env)
    assert r.returncode == 1
    assert c["verbose"][0] in r.stderr
    if shutil.which(tool) is None:
        want = c["stderr_tail"][0].replace("/root/repo/tests/golden", GOLDEN)
        assert want in r.stderr                                         # "hetmers: Command '...' failed"


def _condition_numpy(ku, cn, k, L, trim, symm):
    """test-side restatement of Logex 'A[L-]' + Symmex (documented effect): keep count >= L, add
    the reverse complement of every k-mer with the same count, originals win on duplicates."""
    import torch
    two = ku.ndim == 2
    if trim:
        keep = cn >= L
        ku, cn = ku[keep], cn[keep]
    if symm:
        t = torch.from_numpy(ku.view(np.int64))
        if two:
            rh, rl = synth.revcomp_long(t[:, 0].contiguous(), t[:, 1].contiguous(), k)
            rc = torch.stack([rh, rl], dim=1).numpy().view(np.uint64)
        else:
            rc = synth.revcomp_left(t, k).numpy().view(np.uint64)
        allk = np.concatenate([ku, rc])
        allc = np.concatenate([cn, cn])
        kb = fastk.keys_u64_to_bytes(allk, k)
        order = np.lexsort(tuple(kb[:, j] for j in range(kb.shape[1] - 1, -1, -1)))   # stable
        kb, allc, allk = kb[order], allc[order], allk[order]
        first = np.ones(len(kb), dtype=bool)
        first[1:] = (kb[1:] != kb[:-1]).any(axis=1)
        ku, cn = allk[first], allc[first]
    return ku, cn


def canonical_untrimmed_table(k, G, ploidy, seed):
    """seeded FastK-style table: canonical k-mers only, every count >= 1 -> (keys uint64, counts uint16)"""
    import torch
    keys, cnt = synth.synth_table(k, G, ploidy, 0.02, 40, 1, seed)          # untrimmed: counts from 1
    ku = synth.keys_to_u64_numpy(keys)
    cn = cnt.numpy().astype(np.uint16)
    if k > 32:
        rh, rl = synth.revcomp_long(keys[:, 0].contiguous(), keys[:, 1].contiguous(), k)
        rcb = fastk.keys_u64_to_bytes(torch.stack([rh, rl], 1).numpy().view(np.uint64), k)
    else:
        rcb = fastk.keys_u64_to_bytes(synth.revcomp_left(keys, k).numpy().view(np.uint64), k)
    kb = fastk.keys_u64_to_bytes(ku, k)
    w = kb.shape[1]
    canon = kb.view(f"S{w}").reshape(-1) <= rcb.view(f"S{w}").reshape(-1)   # x <= rc(x)
    return ku[canon], cn[canon]


CONDITIONING_CASES = [(21, 60000, 2, 31, 6), (31, 80000, 3, 32, 12), (32, 50000, 2, 33, 5),
                      (40, 50000, 2, 34, 6), (12, 30000, 2, 35, 12)]


@pytest.mark.parametrize("k,G,ploidy,seed,L", CONDITIONING_CASES)
def test_gpu_conditioning_of_canonical_untrimmed_table(k, G, ploidy, seed, L, tmp_path):
    """a FastK-style table (canonical k-mers only, every count >= 1) is trimmed and symmetrised on
    the GPU; the .smu must equal what the REFERENCE binary wrote for the table conditioned by the
    numpy restatement (recorded as a digest), and the -v lines must be the reference's"""
    want = reference_run("conditioning", k, G, ploidy, seed, L)
    ku, cn = canonical_untrimmed_table(k, G, ploidy, seed)
    raw = str(tmp_path / "raw")
    fastk.write_ktab(raw, k, ku, cn, ibyte=3, nparts=3)
    out = str(tmp_path / "gpu")
    r = subprocess.run([_lib.BIN_PATH, "-v", f"-e{L}", "-T4", f"-o{out}", raw], input="n\n",
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stderr == ("\n  The input table is untrimmed and not symmetric\n"
                        f"\n  Trimming k-mers in table with count < {L}\n"
                        "\n  Making trimmed table symmetric\n"
                        "\n  Starting to count covariant pairs\n"
                        "\n  Count complete, outputting table\n")
    ck, cc = _condition_numpy(ku, cn, k, L, True, True)
    assert len(cc) == want["nels"]                                          # the table the reference read
    got = open(out + ".smu").read()
    assert len(got) > 0 and len(got.splitlines()) == want["smu_rows"]
    assert ou.sha256_text(got) == want["smu_sha256"]
    # in-process route + the conditioned table itself
    with hetmers.Scan(fastk.read_ktab(raw)) as sc:
        assert sc.examine(L) == (False, False)
        n2 = sc.condition(L, True, True)
        assert n2 == len(cc)
        assert sc.examine(L) == (True, True)
        k2, c2, _ = sc.download(deg=False)
        plot, _ = sc.run()
    assert np.array_equal(k2, ck) and np.array_equal(c2, cc)
    assert hetmers.smu_text(plot) == got


def test_gpu_conditioning_trim_only_and_symm_only(golden_meta, tmp_path):
    # golden "untrimmed" (symmetric, -e9 above its smallest count) and "asymmetric" (one rc missing)
    for name, (trim, symm) in (("untrimmed", (True, False)), ("asymmetric", (False, True))):
        c = golden_meta["_conditioning"][name]
        kt = fastk.read_ktab(os.path.join(GOLDEN, "conditioning", name))
        kb, cn = fastk.unpack_host(kt)
        ck, cc = _condition_numpy(fastk.keys_bytes_to_u64(kb), cn, 21, c["e"], trim, symm)
        want_plot, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(ck, 21), cc, 21)
        with hetmers.Scan(kt) as sc:
            assert sc.condition(c["e"], trim, symm) == len(cc)
            plot, _ = sc.run()
        assert np.array_equal(plot, want_plot)


# ------------------------------------------------------------------ (b) seeded tables vs oracle

CASES = [  # k, G, ploidy, het, cov, L, seed, ibyte, nparts
    (13, 60000, 2, 0.02, 40, 4, 101, 3, 1),
    (21, 80000, 2, 0.01, 40, 4, 1, 3, 2),
    (27, 50000, 4, 0.02, 80, 10, 102, 2, 3),
    (31, 100000, 3, 0.01, 60, 12, 4, 3, 4),
    (32, 40000, 2, 0.03, 40, 4, 103, 3, 1),
    (12, 200000, 2, 0.02, 30, 4, 104, 3, 2),      # kbyte == ibyte: records are counts only
    (4, 300, 2, 0.2, 30, 1, 105, 1, 1),           # tiny k, saturated neighbourhoods
    (33, 60000, 2, 0.02, 40, 4, 106, 3, 2),       # two 64-bit words per k-mer from here on
    (40, 80000, 3, 0.02, 60, 8, 107, 3, 3),       # FastK's default k
    (47, 50000, 2, 0.03, 40, 4, 108, 2, 1),
    (64, 40000, 4, 0.02, 80, 10, 109, 3, 2),
]


@pytest.mark.parametrize("k,G,ploidy,het,cov,L,seed,ibyte,nparts", CASES)
def test_seeded_table_matches_oracle(k, G, ploidy, het, cov, L, seed, ibyte, nparts, tmp_path):
    keys, cnt = synth.synth_table(k, G, ploidy, het, cov, L, seed, extra_hom_repeats=1)
    name = str(tmp_path / "t")
    kt = synth.write_table(name, k, keys, cnt, ibyte=ibyte, nparts=nparts)
    kb, cn = fastk.unpack_host(kt)
    want_plot, want_deg = ou.oracle_scan(kb, cn, k)
    with hetmers.Scan(fastk.read_ktab(name)) as sc:
        plot, _ = sc.run()
        _, _, deg = sc.download()
    assert np.array_equal(deg, want_deg)
    assert np.array_equal(plot, want_plot)
    plot2, _ = hetmers.scan_table(kt)                                   # one-call route
    assert np.array_equal(plot2, want_plot)


def test_two_entry_and_pairless_tables(tmp_path):
    # smallest legal table (nels >= 2) and a table without any one-away pair
    k = 21
    keys = np.array([0x0123456789AB << 16, (0x0123456789AB << 16) + (1 << 22)], dtype=np.uint64)
    for cn, rows in (([5, 9], "5\t9\t1\n"), ([600, 500], "")):
        name = str(tmp_path / f"t{cn[0]}")
        kt = fastk.write_ktab(name, k, keys, np.array(cn, dtype=np.uint16), ibyte=3)
        plot, _ = hetmers.scan_table(kt)
        assert hetmers.smu_text(plot) == rows
    far = np.array([1 << 30, 7 << 40, 9 << 50], dtype=np.uint64)
    kt = fastk.write_ktab(str(tmp_path / "far"), k, far, np.array([9, 9, 9], dtype=np.uint16), ibyte=2)
    plot, _ = hetmers.scan_table(kt)
    assert plot.sum() == 0


def test_result_independent_of_bucket_bits_and_work_split():
    """layer A on torch tensors: any bucket width, any prefix-filter width and any split of the index range into work
    ranges (the multi-GPU sharding, DESIGN.md §6) gives the same plot."""
    import torch
    from smudgeplot_b200.device import DeviceTable
    keys, cnt = synth.synth_table(25, 60000, 3, 0.02, 60, 8, 77, device="cuda")
    c16 = cnt.to(torch.int16)
    ref = None
    for bits, fbits in ((2, 22), (9, 23), (15, 26), (20, 29), (17, 31), (17, 32), (12, 33), (17, 34), (16, 35), (17, 36), (17, 37)):
        t = DeviceTable(25, keys, c16, bits=bits, fbits=fbits).build_index()
        p = t.scan("direct").clone()
        ref = p if ref is None else ref
        assert torch.equal(p, ref), (bits, fbits)
        del t
    n = keys.numel()
    t = DeviceTable(25, keys, c16).build_index()
    cuts = [0, n // 7, n // 2, n - 3, n]
    deg = torch.zeros((n + 4) & ~3, dtype=torch.uint8, device="cuda")
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        w = DeviceTable(25, keys, c16)
        w.bucket, w.filter = t.bucket, t.filter
        w.alloc_work(lo, hi)
        w.deg = deg                       # shared incidence array == result of the all-reduce
        w.pass1()
        parts.append(w)
    plot = torch.zeros_like(ref).view(-1)
    for w in parts:
        w.plot = plot
        w.pass2()
    torch.cuda.synchronize()
    assert torch.equal(plot.view_as(ref), ref)


# ------------------------------------------------------------------ (c) vs the reference binary

@pytest.mark.parametrize("k", [31, 40])
def test_64bit_offset_kernels_match_32bit(k):
    """tables with >= 2^32 entries (BASELINE configs[4]: 5e9) use uint64 bucket offsets / partner
    indices; force those kernel instantiations on a small table and compare with the uint32 ones"""
    import torch
    from smudgeplot_b200.device import DeviceTable
    keys, cnt = synth.synth_table(k, 120000, 3, 0.02, 60, 8, 91, device="cuda")
    khi = keys[:, 0].contiguous() if k > 32 else keys
    klo = keys[:, 1].contiguous() if k > 32 else None
    c16 = cnt.to(torch.int16)
    a = DeviceTable(k, khi, c16, keys_lo=klo).build_index()
    b = DeviceTable(k, khi, c16, keys_lo=klo, force_idx64=True).build_index()
    pa, pb = a.scan("direct").clone(), b.scan("direct").clone()
    assert b.up.dtype == torch.int64 and b.bucket.dtype == torch.int64
    assert torch.equal(pa, pb) and int(pa.sum()) > 0
    assert torch.equal(a.deg[:a.n], b.deg[:b.n])
    one = a.deg[:a.n] == 1                   # (with several partners the recorded one is arbitrary and unused)
    assert torch.equal(a.up.long()[one], b.up[one])
    q = khi[:1000].contiguous()
    assert torch.equal(a.find(q, klo[:1000].contiguous() if klo is not None else None),
                       b.find(q, klo[:1000].contiguous() if klo is not None else None))


def test_long_kmer_work_split_and_filter_widths():
    """k = 40 (two key words): plot independent of bucket / filter width and of the work split"""
    import torch
    from smudgeplot_b200.device import DeviceTable
    keys, cnt = synth.synth_table(40, 50000, 3, 0.02, 60, 8, 55, device="cuda")
    khi, klo, c16 = keys[:, 0].contiguous(), keys[:, 1].contiguous(), cnt.to(torch.int16)
    ref = None
    for bits, fbits in ((3, 22), (14, 27), (16, 32), (15, 35), (16, 37)):
        t = DeviceTable(40, khi, c16, bits=bits, fbits=fbits, keys_lo=klo).build_index()
        p = t.scan("direct").clone()
        ref = p if ref is None else ref
        assert torch.equal(p, ref), (bits, fbits)
    n = khi.numel()
    deg = torch.zeros((n + 4) & ~3, dtype=torch.uint8, device="cuda")
    plot = torch.zeros_like(ref).view(-1)
    parts = []
    for lo, hi in ((0, n // 3), (n // 3, n - 5), (n - 5, n)):
        w = DeviceTable(40, khi, c16, keys_lo=klo)
        w.bucket, w.filter = t.bucket, t.filter
        w.bits, w.fbits = t.bits, t.fbits
        w.alloc_work(lo, hi)
        w.deg = deg
        w.pass1()
        parts.append(w)
    for w in parts:
        w.plot = plot
        w.pass2()
    torch.cuda.synchronize()
    assert torch.equal(plot.view_as(ref), ref)
    rhi, rlo = synth.revcomp_long(khi, klo, 40)
    pos = t.find(rhi, rlo)
    assert bool((pos >= 0).all())                       # symmetric table: every reverse complement is found


MEDIUM_CASES = [  # ref_threads: the reference's -T when its output was recorded (0: min(cores, 64))
    (21, 1_000_000, 2, 0.01, 40, 4, 1, 1),        # BASELINE configs[0]: reference C hetmers on 1 CPU thread
    (31, 20_000_000, 2, 0.01, 40, 12, 2, 0),      # configs[1] at 1/10 of the bench size
    (31, 30_000_000, 4, 0.01, 40, 12, 3, 0),      # stand-in for configs[2] (the real S. cerevisiae table needs
                                                  #   network + FastK): synthetic tetraploid ~3e7, clearly not real data
    (31, 12_000_000, 3, 0.01, 60, 12, 4, 0),      # configs[3] parameters (triploid cov 60) at reduced size
    (31, 12_000_000, 4, 0.02, 80, 10, 5, 0),      # configs[4] parameters (tetraploid het 2% cov 80, L=10), reduced
    (40, 5_000_000, 2, 0.01, 40, 4, 6, 0),        # FastK's default k=40: two-word keys against the reference
]


@pytest.mark.parametrize("k,target,ploidy,het,cov,L,seed,ref_threads", MEDIUM_CASES)
def test_medium_table_matches_reference_binary(k, target, ploidy, het, cov, L, seed, ref_threads, tmp_path):
    """our executable's .smu == the reference binary's on the same seeded table (recorded as a digest)"""
    want = reference_run("medium", k, target, ploidy, het, cov, L, seed, ref_threads)
    G = synth.calibrate_G(k, target, ploidy, het, cov, L)
    keys, cnt = synth.synth_table(k, G, ploidy, het, cov, L, seed, device="cuda")
    name = str(tmp_path / "t")
    kt = synth.write_table(name, k, keys, cnt, ibyte=3, nparts=4)
    assert abs(kt.nels - target) < 0.25 * target          # calibrate_G is a coarse model for ploidy > 2
    assert kt.nels == want["nels"]                         # the table the reference read
    out = str(tmp_path / "gpu")
    hetmers.run_hetmers(name, o=out, L=L, t=4)
    got = open(out + ".smu").read()
    assert len(got) > 0 and len(got.splitlines()) == want["smu_rows"]
    assert ou.sha256_text(got) == want["smu_sha256"]


# ------------------------------------------------------------------ (d) full-size properties --

def test_full_size_properties_config2():
    """BASELINE config 2 (k=31, ~2e8 k-mers, diploid het 1%, cov 40, L=12) on one GPU.
    Size-independent properties of a symmetric table with symmetric counts:
      * deg[rc(x)] == deg[x]  (a neighbour at base p of x is a neighbour at base k-1-p of rc(x):
        ties the low-position search, whose partners are ~n/4^p entries away, to the
        high-position search, whose partners are adjacent)
      * sum(plot) == #{x : deg[x]==1 and deg[partner(x)]==1} / 2, recounted with torch ops
      * the plot does not change when the scan is repeated (idempotence / no stale state)"""
    import torch
    from smudgeplot_b200.device import DeviceTable
    k, L = 31, 12
    G = synth.calibrate_G(k, 200_000_000, 2, 0.01, 40, L)
    keys, cnt = synth.synth_table(k, G, 2, 0.01, 40, L, 2, device="cuda")
    n = keys.numel()
    assert abs(n - 2e8) < 2e7
    t = DeviceTable(k, keys, cnt.to(torch.int16)).build_index()
    plot = t.scan("direct").clone()
    deg = t.deg[:n].clone()
    plot_again = t.scan("direct")
    assert torch.equal(plot, plot_again)
    assert t.check_symmetric()
    assert torch.equal(t.scan("symm"), plot)          # the strand-symmetric scan: same plot, twice
    assert torch.equal(t.scan("symm"), plot)
    rc = synth.revcomp_left(keys, k)
    pos = t.find(rc)
    assert bool((pos >= 0).all())
    assert torch.equal(deg[pos], deg)
    up = t.up.long()
    has = (deg == 1) & (up >= 0)            # -1 == the all-ones 'none' marker
    idx = torch.nonzero(has).squeeze(1)
    iso = deg[up[idx]] == 1
    assert int(iso.sum()) == int(plot.sum())
    # every isolated pair has an isolated mirror pair (rc), so hom/het structure is strand-symmetric
    assert int(plot.sum()) > 0.1 * n * 0.5 * 0.2


# ------------------------------------------------------------------ multi-GPU (one process) ---

@pytest.mark.parametrize("path", ["symm", "direct"])
@pytest.mark.parametrize("ngpu", [2, 4, 8])
def test_multi_gpu_single_process_matches_single_gpu(ngpu, path, tmp_path, monkeypatch):
    """HETMERS_GPUS=n: shards unpacked per GPU (one host thread each), gathered by peer copies; symmetric
    scan: Bloom segments exchanged by peer copies; direct passes: degree bytes reached through the owner's
    array (csrc/hm_peer.cu for the dense fall-back); plots reduced onto GPU 0 -- same .smu as one GPU."""
    if _lib.lib().hm_device_count() < ngpu:
        pytest.skip(f"needs {ngpu} GPUs")
    monkeypatch.setenv("HETMERS_PATH", path)
    keys, cnt = synth.synth_table(31, 400000, 3, 0.01, 60, 12, 4, device="cuda")
    name = str(tmp_path / "t")
    kt = synth.write_table(name, 31, keys, cnt, ibyte=3, nparts=3)
    one, _ = hetmers.scan_table(kt, gpus=1)
    many, st = hetmers.scan_table(kt, gpus=ngpu)
    assert st["n_gpus"] == ngpu and st["path"] == (2 if path == "symm" else 1)
    assert np.array_equal(one, many)
    out = str(tmp_path / "o")
    hetmers.run_hetmers(name, o=out, L=12, t=4, gpus=ngpu)
    assert open(out + ".smu").read() == hetmers.smu_text(one)
    # extract_kmer_pairs' pair list is the same set whichever GPU found the pair
    pix = (one > 0).astype(np.uint16)
    recs = []
    for g in (1, ngpu):
        with hetmers.Scan(kt, gpus=g) as sc:
            sc.run()
            recs.append(sc.extract(pix))
    assert len(recs[0]) == int(one.sum()) and np.array_equal(recs[0], recs[1])


def test_multi_gpu_dense_exchange_fallback(tmp_path, monkeypatch):
    """same as above through the dense route (partial arrays summed by the peer-memory kernel),
    which is what runs when the GPUs have no native NVLink atomics"""
    if _lib.lib().hm_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    keys, cnt = synth.synth_table(27, 300000, 2, 0.02, 40, 6, 9, device="cuda")
    kt = synth.write_table(str(tmp_path / "t"), 27, keys, cnt, ibyte=3, nparts=2)
    one, _ = hetmers.scan_table(kt, gpus=1)
    monkeypatch.setenv("HETMERS_PATH", "direct")
    monkeypatch.setenv("HETMERS_DENSE_EXCHANGE", "1")
    many, _ = hetmers.scan_table(kt, gpus=2)
    assert np.array_equal(one, many)


def _dist_worker(rank, world, port, q, dense, path="direct"):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), HETMERS_PATH=path)
    if dense:
        os.environ["HETMERS_DENSE_EXCHANGE"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from smudgeplot_b200 import dist as hd
        job = hd.ShardedScan.from_synthetic(31, 500000, 3, 0.01, 60, 12, 4, torch.device("cuda", rank))
        plots = [job.scan().clone().cpu().numpy() for _ in range(3)]       # repeated: double buffering
        assert job.symm_ok()
        q.put((rank, job.exchange, plots, job.n_total))
    finally:
        dist.barrier()
        dist.destroy_process_group()


@pytest.mark.parametrize("dense,path", [(False, "direct"), (True, "direct"), (False, "symm")])
def test_one_process_per_gpu_nccl_matches_single_gpu(dense, path):
    """torch.distributed/NCCL route (bench.py --gpus N): the sharded symmetric scan (Bloom segments
    all-gathered), the direct passes over peer-mapped incidence arrays (CUDA IPC) and their dense
    all-reduce fallback, against a single-GPU scan of the same seeded table"""
    import torch
    import torch.multiprocessing as mp
    from smudgeplot_b200.device import DeviceTable
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 1000) + int(dense) + 2 * int(path == "symm")
    procs = [ctx.Process(target=_dist_worker, args=(r, world, port, q, dense, path)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    keys, cnt = synth.synth_table(31, 500000, 3, 0.01, 60, 12, 4, device="cuda")
    want = DeviceTable(31, keys, cnt.to(torch.int16)).build_index().scan("direct").cpu().numpy().reshape(-1)
    for rank, exchange, plots, n_total in res:
        assert n_total == keys.numel()
        if path == "symm":
            assert "Bloom" in exchange, exchange
        else:
            assert ("all-reduce" in exchange) == dense, exchange
        for p in plots:
            assert np.array_equal(p.reshape(-1), want)


@pytest.mark.parametrize("seed", range(8))
def test_random_dense_asymmetric_tables_match_oracle(seed, tmp_path):
    """arbitrary tables (not genome-like, NOT symmetric, tiny k, counts around the SMAX/FMAX gates):
    nothing in the CUDA path may rely on strand symmetry or on sparse neighbourhoods"""
    rng = np.random.default_rng(2000 + seed)
    k = int(rng.integers(2, 10))
    n = int(min(rng.integers(2, 3000), 4 ** k))
    cmax = int(rng.choice([6, 40, 520, 700]))
    vals = np.sort(rng.choice(4 ** k, size=n, replace=False).astype(np.uint64))
    keys = vals << np.uint64(64 - 2 * k)
    cnt = rng.integers(1, cmax + 1, size=n).astype(np.uint16)
    ibyte = 1 if k < 8 else int(rng.integers(1, 3))
    kt = fastk.write_ktab(str(tmp_path / "t"), k, keys, cnt, ibyte=ibyte, nparts=int(rng.integers(1, 4)))
    want_plot, want_deg = ou.oracle_scan(fastk.keys_u64_to_bytes(keys, k), cnt, k)
    with hetmers.Scan(kt) as sc:
        plot, _ = sc.run()
        got_keys, got_cnt, deg = sc.download()
    assert np.array_equal(got_keys, keys) and np.array_equal(got_cnt, cnt)
    assert np.array_equal(deg, want_deg)
    assert np.array_equal(plot, want_plot)
