"""GPU tests of sharded placement (hetmers.Scan(kt, shards=[...]), hm_scan_create_sharded): every shard holds
only its own run-aligned key range.  Logical shards on device 0 exercise every code path on one GPU; the
result must be the replica's -- the golden .smu, the replica's conditioned table entry for entry, the
oracle's plot on degenerate tables -- and what a sharded table cannot do must be refused, not guessed."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
import oracle_util as ou
from smudgeplot_b200 import _lib, fastk, hetmers
from tools import synth

pytestmark = pytest.mark.gpu

BALANCE = 0.10          # shard sizes within 10 % of n/S on tables of >= 1e6 entries


@pytest.fixture(scope="module", autouse=True)
def _need_gpu(built):
    assert _lib.lib().hm_device_count() >= 1, "these tests need a CUDA device (no CPU fallback exists)"


def _golden(name):
    return os.path.join(GOLDEN, name, name)


def check_shards(sc, k, balance=None):
    """shards contiguous and in order, sum n_r == n, no run split by a cut (and balance when asked);
    returns the concatenated keys"""
    info = sc.shard_info()
    keys, cnt, _ = sc.download()
    n = len(cnt)
    assert sum(s["n"] for s in info) == n
    at = 0
    for s in info:
        assert s["first_index"] == at
        at += s["n"]
    hi = keys[:, 0] if keys.ndim == 2 else keys
    psh = np.uint64(64 - 2 * (k // 2))
    for s in info[1:]:
        f = s["first_index"]
        if 0 < f < n:
            assert (hi[f - 1] >> psh) != (hi[f] >> psh), "a run crosses a shard cut"
    if balance is not None:
        S = len(info)
        for s in info:
            assert abs(s["n"] - n / S) <= balance * n / S, [s["n"] for s in info]
    return keys, cnt


# ------------------------------------------------------------------ 1. goldens -----------------

@pytest.mark.parametrize("S", [2, 3, 5])
@pytest.mark.parametrize("name", golden_cases())
def test_sharded_scan_reproduces_reference_smu(name, S):
    kt = fastk.read_ktab(_golden(name))
    with hetmers.Scan(kt, shards=[0] * S) as sc:
        trim, symm = sc.examine(1)
        plot, st = sc.run()
        assert sc.is_symmetric()
        keys, cnt = check_shards(sc, kt.kmer)
    assert st["path"] == 2 and st["n_gpus"] == S
    assert hetmers.smu_text(plot) == open(_golden(name) + ".smu").read()
    kb, cn = fastk.unpack_host(kt)                                  # the table itself, unchanged
    assert np.array_equal(cnt, cn)
    assert np.array_equal(fastk.keys_u64_to_bytes(keys, kt.kmer), kb)
    with hetmers.Scan(kt) as rp:
        assert rp.examine(1) == (trim, symm)                           # examine on raw shards == replica


# ------------------------------------------------------------------ 2. conditioning ------------

from test_gpu_parity import CONDITIONING_CASES, canonical_untrimmed_table, reference_run  # noqa: E402


@pytest.mark.parametrize("k,G,ploidy,seed,L", CONDITIONING_CASES)
def test_sharded_conditioning_equals_replica(k, G, ploidy, seed, L, tmp_path):
    want = reference_run("conditioning", k, G, ploidy, seed, L)
    ku, cn = canonical_untrimmed_table(k, G, ploidy, seed)
    raw = str(tmp_path / "raw")
    kt = fastk.write_ktab(raw, k, ku, cn, ibyte=3, nparts=3)
    with hetmers.Scan(kt) as rp:
        assert rp.examine(L) == (False, False)
        n_rep = rp.condition(L, True, True)
        k_rep, c_rep, _ = rp.download(deg=False)
        plot_rep, _ = rp.run()
    for S in (2, 3):
        with hetmers.Scan(fastk.read_ktab(raw), shards=[0] * S) as sc:
            assert sc.examine(L) == (False, False)
            assert sc.condition(L, True, True) == n_rep == want["nels"]
            assert sc.examine(L) == (True, True)
            k_sh, c_sh = check_shards(sc, k)
            plot, st = sc.run()
        assert np.array_equal(k_sh, k_rep) and np.array_equal(c_sh, c_rep)
        assert np.array_equal(plot, plot_rep)
        got = hetmers.smu_text(plot)
        assert len(got.splitlines()) == want["smu_rows"] and ou.sha256_text(got) == want["smu_sha256"]


def test_sharded_trim_only_and_symm_only(golden_meta):
    from test_gpu_parity import _condition_numpy
    for name, (trim, symm) in (("untrimmed", (True, False)), ("asymmetric", (False, True))):
        c = golden_meta["_conditioning"][name]
        kt = fastk.read_ktab(os.path.join(GOLDEN, "conditioning", name))
        kb, cn = fastk.unpack_host(kt)
        ck, cc = _condition_numpy(fastk.keys_bytes_to_u64(kb), cn, 21, c["e"], trim, symm)
        want_plot, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(ck, 21), cc, 21)
        with hetmers.Scan(kt, shards=[0, 0, 0]) as sc:
            assert sc.condition(c["e"], trim, symm) == len(cc)
            keys, cnt = check_shards(sc, 21)
            plot, _ = sc.run()
        assert np.array_equal(keys, ck) and np.array_equal(cnt, cc)
        assert np.array_equal(plot, want_plot)


# ------------------------------------------------------------------ 3./5. size, balance, memory -

def test_sharded_memory_and_balance_on_2e7_entries(tmp_path):
    """S = 4 on ~2e7 entries: balance within BALANCE, and every shard's device bytes at most 1/S of the
    replica's table-dependent bytes x 1.1 plus the fixed per-device part (bucket index of the table's
    width, 4 MB plot, Bloom filter of S segments sized for the largest shard)"""
    k, S = 31, 4
    G = synth.calibrate_G(k, 20_000_000, 2, 0.01, 40, 4)
    keys, cnt = synth.synth_table(k, G, 2, 0.01, 40, 4, 11, device="cuda")
    kt = synth.write_table(str(tmp_path / "big"), k, keys, cnt, ibyte=3, nparts=4)
    n = kt.nels
    assert n >= 15_000_000
    with hetmers.Scan(kt) as rp:
        plot_rep, _ = rp.run()
        rep_bytes = rp.shard_info()[0]["device_bytes"]
    with hetmers.Scan(fastk.read_ktab(str(tmp_path / "big")), shards=[0] * S) as sc:
        plot, _ = sc.run()
        info = sc.shard_info()
        check_shards(sc, k, balance=BALANCE)
    assert np.array_equal(plot, plot_rep)
    bits = _lib.lib().hm_pick_bucket_bits(n)
    fixed = 4 * ((1 << bits) + 1) + 8 * _lib.PLOT_CELLS + (1 << 20) + S * (n // S + 1) // 8 * 1.2
    for s in info:
        assert s["device_bytes"] <= (rep_bytes - fixed) / S * 1.1 + fixed, (s, rep_bytes)


# ------------------------------------------------------------------ 4. degenerate tables -------

def _sym(vals, k, rng, cmax=40):
    from test_gpu_symm import _symmetric_closure
    return _symmetric_closure(vals, k, rng, cmax)


def _scan_vs_oracle(tmp_path, k, keys, cnt, S, nparts=1):
    kt = fastk.write_ktab(str(tmp_path / f"t{S}"), k, keys, cnt, ibyte=1 if k < 8 else 2, nparts=nparts)
    want, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(keys, k), cnt, k)
    with hetmers.Scan(kt, shards=[0] * S) as sc:
        plot, _ = sc.run()
        check_shards(sc, k)
    assert np.array_equal(plot, want)
    return want


def test_degenerate_tables(tmp_path):
    rng = np.random.default_rng(99)
    k = 21
    sh = np.uint64(64 - 2 * k)
    # two entries: one k-mer and its reverse complement
    x = np.array([int(rng.integers(0, 4 ** k))], dtype=np.uint64) << sh
    keys, cnt = _sym(x, k, rng)
    assert len(keys) == 2
    for S in (2, 8):
        _scan_vs_oracle(tmp_path, k, keys, cnt, S)
    # no pairs at all (spread-out k-mers)
    vals = rng.choice(4 ** k, size=300, replace=False).astype(np.uint64) << sh
    keys, cnt = _sym(vals, k, rng)
    assert _scan_vs_oracle(tmp_path, k, keys, cnt, 3).sum() == 0
    # S = 8 on under 100 entries: empty shards
    vals = rng.choice(4 ** k, size=20, replace=False).astype(np.uint64) << sh
    vals = np.concatenate([vals, vals ^ (np.uint64(1) << (sh + np.uint64(4)))])        # some pairs
    keys, cnt = _sym(vals, k, rng)
    assert len(keys) < 100
    _scan_vs_oracle(tmp_path, k, keys, cnt, 8, nparts=2)
    # dense k = 11: long runs, S larger than the number of runs in places
    k = 11
    vals = rng.choice(4 ** k, size=int(4 ** k * 0.2), replace=False).astype(np.uint64) << np.uint64(64 - 2 * k)
    keys, cnt = _sym(vals, k, rng, 700)
    _scan_vs_oracle(tmp_path, k, keys, cnt, 5, nparts=3)
    # the golden dense k = 11 table over 8 shards
    kt = fastk.read_ktab(_golden("dense_k11"))
    with hetmers.Scan(kt, shards=[0] * 8) as sc:
        plot, _ = sc.run()
    assert hetmers.smu_text(plot) == open(_golden("dense_k11") + ".smu").read()


# ------------------------------------------------------------------ 6. errors ------------------

def test_sharded_refuses_what_it_cannot_do(tmp_path):
    kt = fastk.read_ktab(_golden("dip_k21"))
    with hetmers.Scan(kt, shards=[0, 0]) as sc:
        with pytest.raises(_lib.HetmersError) as e:
            sc.run("direct")
        assert e.value.code == _lib.EUNSUPPORTED
        plot, _ = sc.run()
        with pytest.raises(_lib.HetmersError) as e:
            sc.extract(np.ones((_lib.SMAX + 1, _lib.PLOT_W), dtype=np.uint16))
        assert e.value.code == _lib.EUNSUPPORTED
        plot2, _ = sc.run()                                             # still usable
    assert np.array_equal(plot, plot2)
    # a table that passes the reference's one-k-mer probe without being symmetric (one entry missing)
    k = 31
    keys, cnt = synth.synth_table(k, 60000, 2, 0.02, 40, 4, 321)
    ku = synth.keys_to_u64_numpy(keys)
    cu = cnt.numpy().astype(np.uint16)
    drop = np.ones(len(ku), dtype=bool)
    drop[len(ku) // 3] = False
    akt = fastk.write_ktab(str(tmp_path / "asym"), k, ku[drop], cu[drop], ibyte=3, nparts=2)
    with hetmers.Scan(akt, shards=[0, 0, 0]) as sc:
        assert sc.examine(4) == (True, True)                            # the probe is fooled
        with pytest.raises(_lib.HetmersError) as e:
            sc.run()
        assert e.value.code == _lib.EUNSUPPORTED
    want, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(ku[drop], k), cu[drop], k)
    with hetmers.Scan(akt) as rp:                                       # the replica is not affected
        plot, st = rp.run()
    assert st["path"] == 1 and np.array_equal(plot, want)


# ------------------------------------------------------------------ 7. several physical GPUs ---

def test_sharded_over_physical_gpus(tmp_path):
    ngpu = _lib.lib().hm_device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    k = 31
    G = synth.calibrate_G(k, 20_000_000, 2, 0.01, 40, 4)
    keys, cnt = synth.synth_table(k, G, 2, 0.01, 40, 4, 12, device="cuda")
    name = str(tmp_path / "big")
    kt = synth.write_table(name, k, keys, cnt, ibyte=3, nparts=4)
    with hetmers.Scan(kt) as rp:
        want, _ = rp.run()
    for g in (2, 4, 8):
        if g > ngpu:
            continue
        with hetmers.Scan(fastk.read_ktab(name), shards=list(range(g))) as sc:
            plot, _ = sc.run()
            check_shards(sc, k, balance=BALANCE)
        assert np.array_equal(plot, want)


# ------------------------------------------------------------------ the executable -------------

def _exec(table, out, L, gpus, env_extra=None):
    import json
    import subprocess
    env = dict(os.environ, HETMERS_STATS="1", HETMERS_GPUS=str(gpus), **(env_extra or {}))
    r = subprocess.run([_lib.BIN_PATH, f"-e{L}", "-T4", f"-o{out}", table], input="n\n",
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    stats = json.loads([ln for ln in r.stderr.splitlines() if ln.startswith("{")][-1])
    return open(out + ".smu").read(), stats


def test_executable_reports_its_placement(tmp_path):
    """HETMERS_STATS: a table that fits one GPU is placed as a replica; the device bytes are the library's"""
    name = _golden("trip_k31")
    got, st = _exec(name, str(tmp_path / "o"), 4, 1)
    assert got == open(name + ".smu").read()
    assert st["placement"] == "replica" and len(st["device_bytes"]) == 1 and st["device_bytes"][0] > 0


def test_executable_shards_a_table_its_gpus_cannot_hold_as_replicas(tmp_path):
    """several GPUs whose free memory holds the shards of a canonical table symmetrised but not a replica
    conditioning it (the rest is taken by a ballast allocation): the executable loads a replica, re-plans
    for symmetrising, shards, and writes the replica's .smu; with HETMERS_GPUS=n on a table that fits it
    keeps the replicas and writes the golden .smu"""
    import torch
    ngpu = _lib.lib().hm_device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    from test_gpu_parity import canonical_untrimmed_table
    g = min(ngpu, 8)
    name = _golden("dip_k21")
    got, st = _exec(name, str(tmp_path / "r"), 4, g)
    assert got == open(name + ".smu").read()
    assert st["placement"] == "replica" and len(st["device_bytes"]) == g
    # ~1e8 canonical entries of k = 31, trimmed at L and symmetrised by the executable
    k, L = 31, 12
    G = synth.calibrate_G(k, 200_000_000, 2, 0.01, 40, L)
    keys, cnt = synth.synth_table(k, G, 2, 0.01, 40, 1, 21, device="cuda")
    rc = synth.revcomp_left(keys, k)
    canon = (keys.view(torch.int64) ^ (1 << 63)) <= (rc.view(torch.int64) ^ (1 << 63))
    raw = str(tmp_path / "raw")
    kt = synth.write_table(raw, k, keys[canon].contiguous(), cnt[canon].contiguous(), ibyte=3, nparts=4)
    del keys, cnt, rc, canon
    with hetmers.Scan(fastk.read_ktab(raw)) as sc:
        sc.condition(L, True, True)
        want = hetmers.smu_text(sc.run()[0])
    torch.cuda.empty_cache()
    r1, _, _ = _lib.plan_placement(k, kt.nels, [1 << 50] * g, False)
    _, rep, shd = _lib.plan_placement(k, kt.nels, [1 << 50] * g, True)
    assert r1 == _lib.PLACE_REPLICA and shd < rep
    target = (rep + shd) // 2 + (512 << 20)           # + the executable's own CUDA context
    ballast = []
    try:
        for d in range(g):
            free, _ = torch.cuda.mem_get_info(d)
            if free <= target:
                pytest.skip(f"GPU {d} has only {free} bytes free")
            ballast.append(torch.empty(free - target, dtype=torch.uint8, device=f"cuda:{d}"))
        got, st = _exec(raw, str(tmp_path / "s"), L, g)
    finally:
        del ballast
        torch.cuda.empty_cache()
    assert st["placement"] == "sharded" and len(st["device_bytes"]) == g
    assert got == want
