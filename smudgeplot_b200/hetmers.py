"""Host-side mirror of the reference's `hetmers` task.

Reference interface (the only one this path has): ``smudgeplot hetmers -L <cutoff> -t <threads>
-o <prefix> [--verbose] [-tmp <dir>] <FastK_Table>`` builds ``["-o<o>", "-e<L>", "-T<t>", ("-v"),
("-P<tmp>" iff tmp != "."), infile]`` and spawns the ``hetmers`` binary
(/root/reference/src/smudgeplot/cli.py:57-72, 348-361).  `hetmers_args` + `run_hetmers` reproduce
exactly that against OUR executable (smudgeplot_b200/bin/hetmers); `scan_table` / `Scan` are the
in-process route through the same C ABI (include/hetmers_b200.h layer B) for callers that already
hold the table in host memory.  Everything computes on the GPU; there is no fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import shlex
import subprocess
import sys

import numpy as np

from . import _lib
from .fastk import KtabFiles, read_ktab


def get_binary_path(name: str = "hetmers") -> str:
    """bundled binary first, then PATH -- the lookup order of cli.py:18-54"""
    import shutil
    bundled = os.path.join(os.path.dirname(_lib.BIN_PATH), name)
    if os.path.exists(bundled) and os.access(bundled, os.X_OK):
        return bundled
    found = shutil.which(name)
    if found:
        return found
    raise FileNotFoundError(f"Binary '{name}' not found (looked in {os.path.dirname(bundled)} and PATH); run `make`")


def hetmers_args(infile, o="smudgeplot", L=None, t=4, verbose=False, tmp="."):
    """argv tail exactly as cli.py:350-359 builds it (L is required there via argparse)."""
    if L is None:
        raise ValueError("-L (count threshold) is required, as in `smudgeplot hetmers`")
    args = [f"-o{o}", f"-e{L}", f"-T{t}"]
    if verbose:
        args.append("-v")
    if tmp != ".":
        args.append(f"-P{tmp}")
    args.append(str(infile))
    return args


def run_hetmers(infile, o="smudgeplot", L=None, t=4, verbose=False, tmp=".", gpus=None, stdin_text="n\n"):
    """Spawn the drop-in executable like run_binary (cli.py:57-72): raises CalledProcessError on a
    non-zero exit.  Returns the path of the .smu written."""
    cmd = [get_binary_path("hetmers")] + hetmers_args(infile, o, L, t, verbose, tmp)
    sys.stderr.write(f"Calling: {shlex.join(cmd)}\n")
    env = dict(os.environ)
    if gpus is not None:
        env["HETMERS_GPUS"] = str(gpus)
    subprocess.run(cmd, check=True, input=stdin_text, text=True, env=env)
    return f"{o}.smu"


def extract_args(infile, sma, o="kmerpairs", t=4, verbose=False, tmp="."):
    """argv tail of `smudgeplot extract` exactly as cli.py:368-378 builds it"""
    args = [f"-o{o}", f"-T{t}"]
    if verbose:
        args.append("-v")
    if tmp != ".":
        args.append(f"-P{tmp}")
    args.append(str(infile))
    s = str(sma)
    args.append(s[:-4] if s.endswith(".sma") else s)
    return args


def run_extract(infile, sma, o="kmerpairs", t=4, verbose=False, tmp=".", gpus=None, e=None):
    """Spawn our `extract_kmer_pairs` (same boundary as the reference's second binary,
    src/lib/PloidyList.c; cli.py:368-382).  Writes <o>.<a>A<b>B.txt per smudge of the .sma."""
    cmd = [get_binary_path("extract_kmer_pairs")] + extract_args(infile, sma, o, t, verbose, tmp)
    if e is not None:
        cmd.insert(1, f"-e{e}")
    sys.stderr.write(f"Calling: {shlex.join(cmd)}\n")
    env = dict(os.environ)
    if gpus is not None:
        env["HETMERS_GPUS"] = str(gpus)
    subprocess.run(cmd, check=True, env=env)


# ------------------------------------------------------------------ in-process (C ABI layer B) --

def _host_table(kt: KtabFiles):
    """hm_host_table view over a KtabFiles (keeps the numpy buffers alive via the returned refs)."""
    index = np.ascontiguousarray(kt.index, dtype=np.int64)
    recs = [np.ascontiguousarray(r) if not isinstance(r, np.memmap) else r for r in kt.records]
    nparts = len(recs)
    part_nels = (C.c_int64 * max(nparts, 1))(*[int(x) for x in kt.part_nels])
    part_rec = (C.c_void_p * max(nparts, 1))(*[r.ctypes.data if r.size else None for r in recs])
    ht = _lib.HostTable(kt.kmer, kt.ibyte, nparts, kt.minval, kt.nels,
                        index.ctypes.data_as(C.POINTER(C.c_int64)), part_nels, part_rec, None, None)
    return ht, (index, recs, part_nels, part_rec)


class Scan:
    """Device-resident table + both passes (hm_scan_*).  shards=[d0, d1, ...]: sharded placement, shard r
    on device d_r (a device may carry several shards): each holds only its own key range, so the table
    may exceed one GPU's memory; only the strand-symmetric scan runs on such a table."""

    def __init__(self, kt: KtabFiles, gpus: int = 1, devices=None, shards=None):
        L = _lib.lib()
        self._L = L
        self._h = None
        self.kt = kt
        ht, self._keep = _host_table(kt)
        self.sharded = shards is not None
        devs = list(shards) if shards is not None else (list(devices) if devices is not None else list(range(gpus)))
        arr = (C.c_int * len(devs))(*devs)
        h = C.c_void_p()
        create = L.hm_scan_create_sharded if self.sharded else L.hm_scan_create
        _lib.check(create(C.byref(ht), arr, len(devs), C.byref(h)))
        self._h = h
        self.n_dev = len(devs)

    def shard_info(self):
        """per shard (or replica): dict(dev, first_index, n, device_bytes) -- hm_scan_shard_info"""
        out = []
        for r in range(self.n_dev):
            d, f, n, b = C.c_int(), C.c_int64(), C.c_int64(), C.c_int64()
            _lib.check(self._L.hm_scan_shard_info(self._h, r, C.byref(d), C.byref(f), C.byref(n), C.byref(b)))
            out.append({"dev": d.value, "first_index": f.value, "n": n.value, "device_bytes": b.value})
        return out

    def examine(self, ethresh: int):
        """(trimmed?, symmetric?) as examine_table decides them (PloidyPlot.c:1167-1230)."""
        trim, symm = C.c_int(), C.c_int()
        _lib.check(self._L.hm_scan_examine(self._h, ethresh, C.byref(trim), C.byref(symm)))
        return bool(trim.value), bool(symm.value)

    def condition(self, ethresh: int, trim: bool, symm: bool) -> int:
        """trim (count >= ethresh) and / or symmetrise the device table in place (what the reference
        gets from FastK's Logex / Symmex, PloidyPlot.c:1381-1426); returns the new entry count"""
        n = C.c_int64()
        _lib.check(self._L.hm_scan_condition(self._h, ethresh, int(trim), int(symm), C.byref(n)))
        self.nels = n.value
        return n.value

    PATHS = {"auto": 0, "direct": 1, "symm": 2}

    def is_symmetric(self) -> bool:
        """whole-table verdict of the symmetry fingerprint (hm_scan_create / hm_scan_condition)"""
        return bool(self._L.hm_scan_is_symmetric(self._h))

    def run(self, path: str = "auto"):
        """-> (plot int64[1001,501], stats dict).  path "auto": the strand-symmetric scan when the table
        is symmetric, else the direct passes; "direct" / "symm" force one (stats["path"]: 1 / 2)"""
        plot = np.zeros(_lib.PLOT_CELLS, dtype=np.int64)
        st = _lib.ScanStats()
        _lib.check(self._L.hm_scan_run_path(self._h, self.PATHS[path], plot.ctypes.data, C.byref(st)))
        return plot.reshape(_lib.SMAX + 1, _lib.PLOT_W), st.as_dict()

    def extract(self, pixmap: np.ndarray, path: str | None = None, stats: bool = False):
        """pair list of extract_kmer_pairs: pixmap uint16[1001,501], label 0 = none; -> structured array
        (key_hi, key_lo, smudge, pos, alt) sorted by (smudge, k-mer).  path=None: hm_scan_extract (the
        direct passes, run first if the last run was not theirs); "auto" / "direct" / "symm":
        hm_scan_extract_path ("symm" re-judges the symmetric scan's candidates and works on sharded
        tables; "auto" takes the route run() takes).  stats=True: -> (records, stats dict)"""
        pm = np.ascontiguousarray(pixmap, dtype=np.uint16).reshape(-1)
        assert pm.size == _lib.PLOT_CELLS
        out = C.POINTER(_lib.PairRec)()
        n = C.c_int64()
        st = _lib.ExtractStats()
        if path is None:
            _lib.check(self._L.hm_scan_extract(self._h, pm.ctypes.data, C.byref(out), C.byref(n)))
            st.path, st.slices, st.n_records = 1, 1, n.value
        else:
            _lib.check(self._L.hm_scan_extract_path(self._h, self.PATHS[path], pm.ctypes.data, C.byref(out),
                                                    C.byref(n), C.byref(st)))
        dt = np.dtype([("key_hi", "<u8"), ("key_lo", "<u8"), ("smudge", "<u4"), ("pos", "u1"), ("alt", "u1"),
                       ("pad", "<u2")])
        arr = np.empty(n.value, dtype=dt)
        if n.value:
            C.memmove(arr.ctypes.data, out, n.value * dt.itemsize)
        libc = C.CDLL(None)
        libc.free.argtypes = [C.c_void_p]
        libc.free(out)
        return (arr, st.as_dict()) if stats else arr

    def download(self, deg: bool = True):
        """-> (keys, cnt, deg) of the device table; a sharded table gives the concatenation of its shards
        (run a scan or condition() first: that fixes the shards' key ranges) and no deg"""
        if self.sharded:
            deg = False
            n = sum(s["n"] for s in self.shard_info())
        else:
            n = getattr(self, "nels", self.kt.nels)
        keys = np.empty(n, dtype=np.uint64)
        klo = np.empty(n, dtype=np.uint64) if self.kt.kmer > 32 else None
        cnt = np.empty(n, dtype=np.uint16)
        d = np.empty(n, dtype=np.uint8) if deg else None
        _lib.check(self._L.hm_scan_download(self._h, keys.ctypes.data, klo.ctypes.data if klo is not None else None,
                                            cnt.ctypes.data, d.ctypes.data if deg else None))
        if klo is not None:
            keys = np.stack([keys, klo], axis=1)          # [n, 2] (hi, lo) words
        return keys, cnt, d

    def close(self):
        if self._h:
            self._L.hm_scan_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scan_table(kt: KtabFiles, gpus: int = 1):
    """one call: H2D + unpack + index + pass 1 + pass 2 + plot D2H (hm_hetmers_host)."""
    L = _lib.lib()
    ht, keep = _host_table(kt)
    devs = (C.c_int * gpus)(*range(gpus))
    plot = np.zeros(_lib.PLOT_CELLS, dtype=np.int64)
    st = _lib.ScanStats()
    _lib.check(L.hm_hetmers_host(C.byref(ht), devs, gpus, plot.ctypes.data, C.byref(st)))
    del keep
    return plot.reshape(_lib.SMAX + 1, _lib.PLOT_W), st.as_dict()


def smu_text(plot: np.ndarray) -> str:
    """the .smu rows: "min\\t(sum-min)\\tcount", sum-major, min < 500 (PloidyPlot.c:1612-1615)"""
    p = np.asarray(plot).reshape(_lib.SMAX + 1, _lib.PLOT_W)[:, :_lib.FMAX]
    s, m = np.nonzero(p > 0)
    return "".join(f"{mi}\t{si - mi}\t{p[si, mi]}\n" for si, mi in zip(s.tolist(), m.tolist()))


def write_smu(path: str, plot: np.ndarray) -> None:
    L = _lib.lib()
    a = np.ascontiguousarray(np.asarray(plot, dtype=np.int64).reshape(-1))
    _lib.check(L.hm_write_smu(path.encode(), a.ctypes.data))


def hetmers(infile, o="smudgeplot", L=None, t=4, verbose=False, tmp=".", gpus: int = 1):
    """In-process equivalent of the `hetmers` task: returns the path of the .smu.  Tables that need
    trimming / symmetrising are conditioned on the GPU (hm_scan_condition)."""
    if L is None:
        raise ValueError("-L (count threshold) is required")
    kt = read_ktab(infile, mmap=True)
    with Scan(kt, gpus=gpus) as sc:
        trim, symm = sc.examine(int(L))
        if verbose:
            sys.stderr.write("\n  The input table is %s\n" % (
                ("trimmed and symmetric" if symm else "trimmed but not symmetric") if trim else
                ("untrimmed yet symmetric" if symm else "untrimmed and not symmetric")))
        if not (trim and symm):
            sc.condition(int(L), not trim, not symm)          # on the GPU (the reference: Logex / Symmex)
        plot, _ = sc.run()
    write_smu(f"{o}.smu", plot)
    return f"{o}.smu"
