"""CPU pin of extraction from the strand-symmetric scan (RecordSink in csrc/hm_symm.cu), against the oracle's
extract_kmer_pairs.  Restated on top of oracle_util.partial_runscan / partial_resolve: every isolated candidate
x < y (differing at position p >= k/2, counts cx / cy, bases bx < by there) whose pixel carries a label gives

    the pair itself      cx < cy: y with alt bx, else (a tie too) x with alt by                       pos p
    its mirror image     (rc y, rc x), left out when 2p == k-1:
                         cy < cx: rc x with alt 3-by, else (a tie too) rc y with alt 3-bx            pos k-1-p

and the formatted, sorted lines must be the oracle's files.  Ties go to the OTHER member in the mirror; tables
with forced ties (cx == cy) catch a sink that gets that wrong.  No GPU needed; the GPU tests run the kernel."""

import numpy as np
import pytest

import oracle_util as ou
from smudgeplot_b200 import fastk

DNA = "acgt"


def _rc(x, k):
    return ou._rc(int(x), k)


def _middle_pairs(k, m, rng):
    """odd k: pairs that differ at the middle base -- m pairs (x, x with another middle base) and m k-mers whose
    reverse complement differs from them only there (first half h, middle b, then rc(h))"""
    mid = (k - 1) // 2
    out = []
    for _ in range(m):
        v = [int(b) for b in rng.integers(0, 4, size=k)]
        x = 0
        for b in v:
            x = (x << 2) | b
        x <<= 64 - 2 * k
        sh = 62 - 2 * mid
        out += [x, (x & ~(3 << sh)) | (((((x >> sh) & 3) + int(rng.integers(1, 4))) & 3) << sh)]
        h = v[:mid]
        pal = h + [int(rng.integers(0, 4))] + [3 - b for b in reversed(h)]
        y = 0
        for b in pal:
            y = (y << 2) | b
        out.append(y << (64 - 2 * k))
    return out


def symmetric_table(k, n0, cmin, cmax, seed, dense=False, middle=0):
    """-> (keys uint64 left aligned, counts uint16): a table holding rc(x) with count(x) for every x, with planted
    one-substitution partners; counts uniform in [cmin, cmax] per canonical k-mer (cmin == cmax: every pair a tie)"""
    rng = np.random.default_rng(seed)
    space = 4 ** k
    if dense or space < (1 << 40):
        pick = rng.choice(space, size=min(n0, space), replace=False).astype(np.uint64)
    elif k < 32:
        pick = rng.integers(0, space, size=n0, dtype=np.int64).astype(np.uint64)
    else:                                                                # 4^32 does not fit an int64 bound
        pick = (rng.integers(0, 1 << 62, size=n0, dtype=np.int64).astype(np.uint64) << np.uint64(2)) | \
               rng.integers(0, 4, size=n0).astype(np.uint64)
    vals = pick << np.uint64(64 - 2 * k)
    pos = rng.integers(k // 2, k, size=vals.size)
    mate = vals ^ (rng.integers(1, 4, size=vals.size).astype(np.uint64) << (np.uint64(62) - np.uint64(2) * pos.astype(np.uint64)))
    allv = np.concatenate([vals, mate[: vals.size // 2],
                           np.array(_middle_pairs(k, middle, rng) if middle else [], dtype=np.uint64)])
    rc = np.array([_rc(x, k) for x in allv.tolist()], dtype=np.uint64)
    keys = np.unique(np.concatenate([allv, rc]))
    canon = np.minimum(keys, np.array([_rc(x, k) for x in keys.tolist()], dtype=np.uint64))
    _, inv = np.unique(canon, return_inverse=True)
    cnt = rng.integers(cmin, cmax + 1, size=inv.max() + 1).astype(np.uint16)[inv]
    return keys, cnt


def label_pixels(plot, sma):
    """write <sma> labelling every plotted pixel by (sum + min) % 4 (three smudges, a quarter unlabelled)
    -> (pixmap uint16[1001,501] of smudge numbers in order of first appearance, label names in that order)"""
    s_idx, m_idx = np.nonzero(plot[:, :ou.FMAX] > 0)
    pix = np.zeros((ou.SMAX + 1, ou.PLOT_W), dtype=np.uint16)
    names, order = ["1A1B", "2A1B", "2A2B"], []
    with open(sma, "w") as f:
        f.write("covB\tcovA\tfreq\tsmudge\n")
        for s, m in zip(s_idx.tolist(), m_idx.tolist()):
            lab = (s + m) % 4
            if lab < 3:
                if names[lab] not in order:
                    order.append(names[lab])
                pix[s, m] = order.index(names[lab]) + 1
                f.write(f"{m}\t{s - m}\t{plot[s, m]}\t{names[lab]}\n")
    return pix, order


def symm_records(keys, cnt, k, pix, seg_bits):
    """the record sink restated: (label, key, pos, alt) of every record extraction from the symmetric scan writes"""
    n = len(keys)
    seg, cand = ou.partial_runscan(keys, cnt, k, 0, n, seg_bits)
    recs = []
    for c in cand:
        if ou.partial_resolve(keys, cnt, k, [c], [seg], [int(keys[0])]).sum() == 0:
            continue                                                   # not isolated
        x, cx, cy, p, by = c
        lab = int(pix[cx + cy, min(cx, cy)])
        if lab == 0:
            continue
        sh = 62 - 2 * p
        bx = (x >> sh) & 3
        y = (x & ~(3 << sh)) | (by << sh)
        recs.append((lab, y, p, bx) if cx < cy else (lab, x, p, by))
        if 2 * p != k - 1:
            q = k - 1 - p
            shq = 62 - 2 * q
            rx = _rc(x, k)
            ry = (rx & ~(3 << shq)) | ((3 - by) << shq)
            recs.append((lab, rx, q, 3 - by) if cy < cx else (lab, ry, q, 3 - bx))
    return recs


def fmt(key, k, pos, alt):
    """one line of print_het (PloidyList.c:128-165)"""
    bases = [(key >> (62 - 2 * i)) & 3 for i in range(k)]
    return "".join(f"({DNA[b]}/{DNA[alt]})" if i == pos else DNA[b] for i, b in enumerate(bases))


CASES = [  # k, n0, cmin, cmax, seed, dense, middle pairs
    (21, 1500, 1, 40, 1, False, 0),
    (31, 1500, 1, 40, 2, False, 40),      # odd k: middle-base pairs, rc-of-each-other pairs among them
    (32, 1000, 1, 40, 3, False, 0),
    (16, 1200, 6, 6, 4, False, 0),        # every count equal: every pair is a tie
    (25, 1500, 7, 8, 5, False, 30),       # mostly ties, odd k with middle-base pairs
    (17, 1500, 480, 520, 6, False, 20),   # count sums around SMAX
    (4, 100, 1, 520, 7, True, 0),         # tiny crowded k
    (5, 300, 3, 4, 8, True, 5),
    (7, 2000, 1, 6, 9, True, 10),
]


@pytest.mark.parametrize("k,n0,cmin,cmax,seed,dense,middle", CASES)
def test_symmetric_extraction_records_equal_the_oracle_pair_files(k, n0, cmin, cmax, seed, dense, middle, tmp_path):
    keys, cnt = symmetric_table(k, n0, cmin, cmax, seed, dense=dense, middle=middle)
    want_plot, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(keys, k), cnt, k)
    sma = str(tmp_path / "ann.sma")
    pix, order = label_pixels(want_plot, sma)
    table = str(tmp_path / "t")
    fastk.write_ktab(table, k, keys, cnt, ibyte=1 if k < 8 else 2)
    out = str(tmp_path / "kp")
    assert ou.oracle_extract(table, 1, sma, out) == 0
    want = ou.sorted_pair_files(out)
    for seg_bits in (1 << 20, 61):                                     # a roomy filter and one full of false hits
        recs = symm_records(keys, cnt, k, pix, seg_bits)
        assert len(recs) == int(want_plot[pix > 0].sum())
        got = {lab: [] for lab in order}
        for lab, key, pos, alt in recs:
            got[order[lab - 1]].append(fmt(key, k, pos, alt))
        assert {lab: sorted(v) for lab, v in got.items()} == want
    if cmin == cmax or (k, seed) == (25, 5):
        assert len(recs) > 0 or k <= 7                                 # the ties were exercised


def test_mirror_rule_gives_ties_to_the_other_member():
    """a tie (cx == cy): the pair prints its LOWER member x, the mirror image its lower member rc y -- which is
    the reverse complement of y, not of x; printing rc x there would repeat x's strand"""
    k = 21
    x = 0x123456789AB << 22
    p = 15
    sh = 62 - 2 * p
    bx = (x >> sh) & 3
    by = (bx + 1) & 3
    if by < bx:
        bx, by = by, bx
        x = (x & ~(3 << sh)) | (bx << sh)
    y = (x & ~(3 << sh)) | (by << sh)
    keys = np.unique(np.array([x, y, _rc(x, k), _rc(y, k)], dtype=np.uint64))
    cnt = np.full(len(keys), 9, dtype=np.uint16)
    pix = np.zeros((ou.SMAX + 1, ou.PLOT_W), dtype=np.uint16)
    pix[18, 9] = 1
    recs = sorted(symm_records(keys, cnt, k, pix, 1 << 20))
    want = sorted([(1, x, p, by), (1, _rc(y, k), k - 1 - p, 3 - bx)])
    assert recs == want
