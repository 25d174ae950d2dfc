"""Test-side access to the CPU checkers (oracle/ is test infrastructure only):
  * liboracle.so  -- oracle/hetmers_oracle.c, the C restatement of the reference algorithm
  * oracle/_ref/hetmers -- the unmodified reference binary, when it has been built
  * brute_force() -- SURVEY.md Appendix B, an independent 15-line definition (tiny inputs only)
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "hetmers")
SMAX, FMAX, PLOT_W = 1000, 500, 501
PLOT_CELLS = 1001 * 501

_lib = None


def oracle_lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so", "hetmers_oracle"], check=True)
        L = C.CDLL(ORACLE_SO)
        L.oracle_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
        L.oracle_hetmers_file.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int),
                                          C.POINTER(C.c_int), C.POINTER(C.c_int64)]
        L.oracle_extract_file.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_char_p]
        _lib = L
    return _lib


def oracle_extract(table: str, ethresh: int, sma: str, out_root: str) -> int:
    """oracle restatement of extract_kmer_pairs; 0 ok / 1 cannot open / 2 needs conditioning / 3 bad .sma"""
    return oracle_lib().oracle_extract_file(table.encode(), ethresh, sma.encode(), out_root.encode())


def sha256_text(text: str) -> str:
    """digest of an output file's text (golden/reference_runs.json holds these for outputs too large to store)"""
    return hashlib.sha256(text.encode()).hexdigest()


def sha256_lines(lines) -> str:
    return sha256_text("".join(ln + "\n" for ln in lines))


def sorted_pair_files(out_root: str):
    """{label: sorted lines} of every <out_root>.<a>A<b>B.txt (the reference's line order depends on its
    thread schedule, so pair lists are compared as sorted multisets)"""
    d, base = os.path.split(out_root)
    res = {}
    for f in sorted(os.listdir(d or ".")):
        if f.startswith(base + ".") and f.endswith(".txt"):
            res[f[len(base) + 1:-4]] = sorted(open(os.path.join(d or ".", f)).read().splitlines())
    return res


def oracle_scan(keys_bytes: np.ndarray, cnt: np.ndarray, kmer: int):
    """keys_bytes uint8[n,kbyte] sorted; -> (plot int64[1001,501], deg uint8[n])"""
    L = oracle_lib()
    keys_bytes = np.ascontiguousarray(keys_bytes, dtype=np.uint8)
    cnt = np.ascontiguousarray(cnt, dtype=np.uint16)
    n = keys_bytes.shape[0]
    plot = np.zeros(PLOT_CELLS, dtype=np.int64)
    deg = np.zeros(max(n, 1), dtype=np.uint8)
    rc = L.oracle_scan(keys_bytes.ctypes.data, cnt.ctypes.data, n, kmer, plot.ctypes.data, deg.ctypes.data)
    assert rc == 0
    return plot.reshape(SMAX + 1, PLOT_W), deg[:n]


def oracle_file(table: str, ethresh: int, smu_path: str):
    """-> (rc, trim, symm, nels); rc 0 ok / 1 cannot open / 2 needs conditioning"""
    L = oracle_lib()
    trim, symm, nels = C.c_int(-1), C.c_int(-1), C.c_int64(0)
    rc = L.oracle_hetmers_file(table.encode(), ethresh, smu_path.encode(), C.byref(trim), C.byref(symm), C.byref(nels))
    return rc, trim.value, symm.value, nels.value


def have_ref():
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def run_ref(table: str, out: str, ethresh: int, threads: int = 4, verbose=False):
    """run the unmodified reference binary; returns CompletedProcess (output in out + '.smu')"""
    if os.path.exists(out + ".smu"):
        os.remove(out + ".smu")
    cmd = [REF_BIN, f"-e{ethresh}", f"-T{threads}", f"-o{out}", table]
    if verbose:
        cmd.insert(1, "-v")
    return subprocess.run(cmd, input="n\n", capture_output=True, text=True)


def smu_text(plot) -> str:
    p = np.asarray(plot).reshape(SMAX + 1, PLOT_W)[:, :FMAX]
    s, m = np.nonzero(p > 0)
    return "".join(f"{mi}\t{si - mi}\t{p[si, mi]}\n" for si, mi in zip(s.tolist(), m.tolist()))


def brute_force(keys_u64: np.ndarray, cnt: np.ndarray, k: int):
    """SURVEY.md Appendix B on left-aligned uint64 keys (python ints; n <~ 2e4)."""
    tab = {int(x): int(c) for x, c in zip(keys_u64.tolist(), cnt.tolist())}
    deg = {x: 0 for x in tab}
    pairs = []
    for x, cx in tab.items():
        for p in range(k):
            sh = 62 - 2 * p
            b = (x >> sh) & 3
            for alt in range(b + 1, 4):
                y = x + ((alt - b) << sh)
                cy = tab.get(y)
                if cy is not None and cx + cy <= SMAX:
                    deg[x] = (deg[x] + 1) & 0xFF
                    deg[y] = (deg[y] + 1) & 0xFF
                    pairs.append((x, y))
    plot = np.zeros((SMAX + 1, PLOT_W), dtype=np.int64)
    for x, y in pairs:
        if deg[x] <= 1 and deg[y] <= 1:
            plot[tab[x] + tab[y], min(tab[x], tab[y])] += 1
    return plot, np.array([deg[int(x)] for x in keys_u64.tolist()], dtype=np.uint8)


# ---- range-restricted restatement of the two kernels' contracts (multi-GPU host-logic tests) ----

def partial_pass1(keys_u64: np.ndarray, cnt: np.ndarray, k: int, lo: int, hi: int):
    """what hm_k_pass1_degree contributes for the work range [lo,hi): partial incidence array over
    the WHOLE table (lower pair member books both ends) and up[x-lo] = index of the upper partner."""
    pos = {int(x): i for i, x in enumerate(keys_u64.tolist())}
    deg = np.zeros(len(keys_u64), dtype=np.uint8)
    up = np.full(hi - lo, -1, dtype=np.int64)
    for i in range(lo, hi):
        x, cx = int(keys_u64[i]), int(cnt[i])
        for p in range(k):
            sh = 62 - 2 * p
            b = (x >> sh) & 3
            for alt in range(b + 1, 4):
                j = pos.get(x + ((alt - b) << sh))
                if j is not None and cx + int(cnt[j]) <= SMAX:
                    deg[i] += 1
                    deg[j] += 1
                    up[i - lo] = j
    return deg, up


def partial_pass2(cnt: np.ndarray, deg: np.ndarray, up: np.ndarray, lo: int, hi: int):
    """what hm_k_pass2_plot adds for [lo,hi) given the SUMMED incidence array"""
    plot = np.zeros((SMAX + 1, PLOT_W), dtype=np.int64)
    for i in range(lo, hi):
        j = int(up[i - lo])
        if deg[i] <= 1 and j >= 0 and deg[j] <= 1:
            ci, cj = int(cnt[i]), int(cnt[j])
            plot[ci + cj, min(ci, cj)] += 1
    return plot


# ---- the strand-symmetric scan's two kernels, restated (multi-GPU host-logic tests; k <= 32) ----

def _rc(x: int, k: int) -> int:
    r = 0
    v = x >> (64 - 2 * k)
    for _ in range(k):
        r = (r << 2) | (3 - (v & 3))
        v >>= 2
    return r << (64 - 2 * k)


def partial_runscan(keys_u64: np.ndarray, cnt: np.ndarray, k: int, lo: int, hi: int, seg_bits: int):
    """what hm_k_symm_runscan leaves for the run-aligned range [lo,hi): a membership segment over the
    entries with a partner at a position >= k - k/2 (here an exact bitmap hashed by key % seg_bits, so
    that false positives exist as in the Bloom filter) and the candidate records (x, cx, cy, pos, yb)."""
    pos_of = {int(x): i for i, x in enumerate(keys_u64.tolist())}
    Pr, pup = k // 2, k - k // 2
    seg = np.zeros(seg_bits, dtype=np.uint8)

    def partners(i, p0):
        x, cx, out = int(keys_u64[i]), int(cnt[i]), []
        for p in range(p0, k):
            sh = 62 - 2 * p
            b = (x >> sh) & 3
            for alt in range(4):
                if alt != b:
                    j = pos_of.get((x & ~(3 << sh)) | (alt << sh))
                    if j is not None and cx + int(cnt[j]) <= SMAX:
                        out.append((j, p))
        return out

    cand = []
    for i in range(lo, hi):
        pr = partners(i, Pr)
        if any(p >= pup for _, p in pr):
            seg[int(keys_u64[i]) % seg_bits] = 1
        if len(pr) == 1 and pr[0][0] > i and len(partners(pr[0][0], Pr)) == 1:
            j, p = pr[0]
            cand.append((int(keys_u64[i]), int(cnt[i]), int(cnt[j]), p, (int(keys_u64[j]) >> (62 - 2 * p)) & 3))
    return seg, cand


def partial_resolve(keys_u64: np.ndarray, cnt: np.ndarray, k: int, cand, segs, first_keys):
    """what hm_k_symm_resolve adds for one shard's candidates given ALL shards' segments: a Bloom hit is
    settled exactly on the replica; isolated pairs count once, or twice when the mirror pair is another"""
    pos_of = {int(x): i for i, x in enumerate(keys_u64.tolist())}
    pup = k - k // 2
    plot = np.zeros((SMAX + 1, PLOT_W), dtype=np.int64)

    def in_S(q):
        owner = sum(1 for f in first_keys[1:] if q >= f)
        if not segs[owner][q % len(segs[owner])]:
            return False
        i = pos_of[q]
        cq = int(cnt[i])
        for p in range(pup, k):
            sh = 62 - 2 * p
            b = (q >> sh) & 3
            for alt in range(4):
                if alt != b:
                    j = pos_of.get((q & ~(3 << sh)) | (alt << sh))
                    if j is not None and cq + int(cnt[j]) <= SMAX:
                        return True
        return False

    for x, cx, cy, p, yb in cand:
        rx = _rc(x, k)
        sh = 62 - 2 * (k - 1 - p)
        ry = (rx & ~(3 << sh)) | ((3 - yb) << sh)
        if in_S(rx) or in_S(ry):
            continue
        plot[cx + cy, min(cx, cy)] += 1 if 2 * p == k - 1 else 2
    return plot
