"""CPU tests of the host side of sharded placement: the placement planner (hm_plan_placement) on made-up
free-memory figures around each of its boundaries, and the shard cuts (hm_shard_cuts) on synthetic key
sets: run-aligned, one owner per entry, balanced."""
import numpy as np
import pytest

from smudgeplot_b200 import _lib
from tools import synth

GB = 1 << 30


@pytest.mark.parametrize("k,nels,symm", [(31, 2_000_000_000, False), (31, 8_000_000_000, True),
                                          (40, 1_000_000_000, False), (21, 123_456_789, True)])
def test_placement_planner_boundaries(built, k, nels, symm):
    _, rep, shd = _lib.plan_placement(k, nels, [1 << 50], symm)
    for g in (2, 4, 8):
        _, rep_g, shd_g = _lib.plan_placement(k, nels, [1 << 50] * g, symm)
        if g >= 4:
            assert shd_g < rep_g
        if shd_g >= rep_g:                                          # (sorting a shard's inbox needs room too)
            continue
        # replica when every device has room for one
        assert _lib.plan_placement(k, nels, [rep_g] * g, symm)[0] == _lib.PLACE_REPLICA
        # one byte short on ONE device: sharded if the shards fit
        free = [rep_g] * g
        free[g - 1] = rep_g - 1
        assert _lib.plan_placement(k, nels, free, symm)[0] == _lib.PLACE_SHARDED
        assert _lib.plan_placement(k, nels, [shd_g] * g, symm)[0] == _lib.PLACE_SHARDED
        # one byte short of a shard: does not fit
        assert _lib.plan_placement(k, nels, [shd_g - 1] * g, symm)[0] == _lib.PLACE_NOFIT
        # a shard needs about 1/g of the table: its peak is the redistribution (the received entries, their
        # sort buffers and flags, ~3 copies), plus the per-device index and plot
        tb = 8 * (2 if k > 32 else 1) + 2
        n2 = nels * (2 if symm else 1)
        assert shd_g <= (3 * tb + 9) * (n2 / g * 1.05 + 1024) + 9 * GB
    # one device: never sharded
    assert _lib.plan_placement(k, nels, [rep - 1], symm)[0] == _lib.PLACE_NOFIT


def test_placement_planner_counts_the_conditioning_peak(built):
    n = 4_000_000_000
    _, plain, _ = _lib.plan_placement(31, n, [1 << 50] * 8, False)
    _, cond, _ = _lib.plan_placement(31, n, [1 << 50] * 8, True)
    assert cond > 2 * plain                                           # 2 x the entries + the sort buffers
    # the example of the project's scope: a 2e10-entry symmetrised table needs 8 B200s, sharded
    r, rep, shd = _lib.plan_placement(31, 10_000_000_000, [178 * GB] * 8, True)
    assert r == _lib.PLACE_SHARDED and rep > 178 * GB >= shd


def test_placement_planner_rejects_bad_arguments(built):
    with pytest.raises(_lib.HetmersError):
        _lib.plan_placement(31, -1, [GB])
    with pytest.raises(_lib.HetmersError):
        _lib.plan_placement(31, 10, [GB] * 17)


def _owners(keys, cuts):
    return np.searchsorted(cuts[1:], keys, side="right")             # ties to the higher shard


@pytest.mark.parametrize("k,S", [(31, 2), (31, 8), (21, 5), (32, 16), (17, 3)])
def test_shard_cuts_are_run_aligned_and_balanced(built, k, S):
    """1e6 entries: every cut is the prefix of a run (first k/2 bases, rest zero), so every run has one
    owner; shard sizes within 5 % of n/S (the sample here is the whole key set)"""
    rng = np.random.default_rng(k * 100 + S)
    n = 1_000_000
    keys = np.unique(rng.integers(0, 1 << 63, size=n, dtype=np.int64).astype(np.uint64) << np.uint64(1))
    if k < 32:
        keys = np.unique(keys >> np.uint64(64 - 2 * k) << np.uint64(64 - 2 * k))
    cuts = _lib.shard_cuts(keys, None, None, k, S)
    assert cuts[0] == 0 and np.all(np.diff(cuts.astype(object)) >= 0)
    psh = np.uint64(64 - 2 * (k // 2))
    assert np.all((cuts >> psh) << psh == cuts)                       # on a run boundary
    own = _owners(keys, cuts)
    run = keys >> psh
    same = run[1:] == run[:-1]
    assert np.all(own[1:][same] == own[:-1][same])                    # no run crosses a cut
    sizes = np.bincount(own, minlength=S)
    assert sizes.sum() == len(keys)
    assert np.all(np.abs(sizes - len(keys) / S) <= 0.05 * len(keys) / S), sizes


def test_shard_cuts_with_reverse_complements_and_trim(built):
    """symmetrising: the cuts balance the table WITH the reverse complements; trimming leaves low counts out"""
    import torch
    k, S = 31, 4
    rng = np.random.default_rng(5)
    keys = np.unique(rng.integers(0, 1 << 62, size=400_000, dtype=np.int64).astype(np.uint64) << np.uint64(2))
    cnt = rng.integers(1, 30, size=len(keys)).astype(np.uint16)
    rc = synth.revcomp_left(torch.from_numpy(keys.view(np.int64)), k).numpy().view(np.uint64)
    cuts = _lib.shard_cuts(keys, None, cnt, k, S, min_count=5, add_rc=True)
    keep = cnt >= 5
    full = np.concatenate([keys[keep], rc[keep]])
    sizes = np.bincount(_owners(full, cuts), minlength=S)
    assert np.all(np.abs(sizes - len(full) / S) <= 0.05 * len(full) / S), sizes
    # degenerate samples: nothing kept -> every cut 0 (all entries with the last shard)
    assert np.all(_lib.shard_cuts(keys[:10], None, cnt[:10] * 0, k, S, min_count=1) == 0)
    assert np.all(_lib.shard_cuts(keys[:0], None, None, k, S) == 0)


def test_planner_keeps_tables_that_fit_a_multi_gpu_replica_on_the_replica_path(built):
    """a multi-GPU replica scans only its run-aligned 1/G of the table: its work area is planned for that
    share, so every table today's replica layout holds stays a replica (within 2 % of the library's own
    allocation sizes: table arrays + bucket index + plot + hm_symm_plan(n, n/G))"""
    import ctypes as C
    L = _lib.lib()
    free = 178_000_000_000
    for n, g in ((10_000_000_000, 8), (12_000_000_000, 8), (5_000_000_000, 4), (3_000_000_000, 2)):
        lay = _lib.SymmLayout()
        _lib.check(L.hm_symm_plan(n, n // g, 31, g, C.byref(lay)))
        ib = 8 if n >= 0xFFFFFFF0 else 4                               # 64-bit bucket offsets from 2^32 entries
        real = 10 * n + ib * ((1 << L.hm_pick_bucket_bits(n)) + 1) + 8 * _lib.PLOT_CELLS + lay.bytes
        r, rep, _ = _lib.plan_placement(31, n, [free] * g)
        assert real <= rep <= real * 1.02, (n, g, rep, real)
        assert (r == _lib.PLACE_REPLICA) == (real * 1.02 <= free), (n, g, r)
    assert _lib.plan_placement(31, 10_000_000_000, [free] * 8)[0] == _lib.PLACE_REPLICA
    assert _lib.plan_placement(31, 16_000_000_000, [free] * 8)[0] == _lib.PLACE_SHARDED


def test_planner_respects_the_shard_sort_limit_for_long_kmers(built):
    """for k > 32 a shard's sort carries 32-bit indices: no shard may receive 2^32 - 16 entries"""
    r, _, shd = _lib.plan_placement(40, 10_000_000_000, [1 << 60] * 2)
    assert shd == (1 << 63) - 1 and r == _lib.PLACE_REPLICA
    r, _, shd = _lib.plan_placement(40, 10_000_000_000, [1 << 60] * 4)
    assert shd < (1 << 63) - 1
    r, rep, shd = _lib.plan_placement(40, 5_000_000_000, [1 << 60] * 2, True)     # 1e10 after symmetrising
    assert rep == (1 << 63) - 1 and shd == (1 << 63) - 1 and r == _lib.PLACE_NOFIT
