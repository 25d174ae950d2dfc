"""Time extract_kmer_pairs' two routes on the bench table (BASELINE configs[1]: k = 31, diploid, ~2e8 k-mers,
tools/synth.py, seeded) in one process, alternating:

  direct     the direct passes (the scan extract_kmer_pairs needs them for) + the two extract passes of
             hm_scan_extract (Scan.run("direct") + Scan.extract(pix, "direct"))
  symmetric  the candidates the symmetric scan left on the device judged again (Scan.extract(pix, "symm"),
             after the Scan.run() that made the plot)

Reported per route: the extraction kernels, the copy of the records to the host, the host sort, end to end
(wall clock of the calls), and the device bytes the route adds to the loaded table.  Those are measured as
the drop in free device memory over the route's first run on a fresh scan (allocations the route keeps),
plus the records' device buffer of hm_scan_extract, which it frees before returning (computed: 24 B per
record, and the 1 MB label map).  Every pair of record arrays is checked equal.  The label map marks every
plotted pixel by (sum + min) % 4 < 3, as the tests do.

    python tools/time_extract.py OUT.json [nels=2e8] [reps=5]
"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from smudgeplot_b200 import _lib, fastk, hetmers  # noqa: E402
from tools import synth  # noqa: E402

K, P, HET, COV, L, SEED = 31, 2, 0.01, 40.0, 12, 2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def free_bytes():
    import ctypes as C
    f = C.c_int64()
    _lib.check(_lib.lib().hm_device_free_bytes(0, C.byref(f)))
    return f.value


def labels(plot):
    s, m = np.nonzero(plot[:, :_lib.FMAX] > 0)
    pix = np.zeros((_lib.SMAX + 1, _lib.PLOT_W), dtype=np.uint16)
    lab = (s + m) % 4
    keep = lab < 3
    pix[s[keep], m[keep]] = lab[keep] + 1
    return pix


def route(sc, pix, kind):
    t0 = time.perf_counter()
    if kind == "direct":
        _, st = sc.run("direct")
        scan_ms = st["ms_scan"]
    else:
        scan_ms = 0.0
    rec, xs = sc.extract(pix, "direct" if kind == "direct" else "symm", stats=True)
    e2e = (time.perf_counter() - t0) * 1e3
    return rec, {"e2e_ms": e2e, "direct_scan_ms": scan_ms, "kernel_ms": xs["ms_kernel"], "copy_ms": xs["ms_copy"],
                 "sort_ms": xs["ms_sort"], "slices": xs["slices"], "records": xs["n_records"]}


def main():
    out = sys.argv[1]
    nels = float(sys.argv[2]) if len(sys.argv) > 2 else 2e8
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    res = {"card": card(), "workload": f"configs[1]: k={K}, ploidy {P}, het {HET}, cov {COV}, L {L}, seed {SEED}"}
    with tempfile.TemporaryDirectory() as td:
        G = synth.calibrate_G(K, int(nels), P, HET, COV, L)
        keys, cnt = synth.synth_table(K, G, P, HET, COV, L, SEED, device="cuda")
        name = os.path.join(td, "bench")
        kt = synth.write_table(name, K, keys, cnt, ibyte=3, nparts=4)
        del keys, cnt
        import torch
        torch.cuda.empty_cache()
        res["nels"] = kt.nels
        kt = fastk.read_ktab(name)
        # device bytes each route adds, on fresh scans (the symmetric scan's work area is the scan's own)
        added = {}
        for kind in ("symmetric", "direct"):
            with hetmers.Scan(kt) as sc:
                plot, _ = sc.run()
                pix = labels(plot)
                f0 = free_bytes()
                rec, m = route(sc, pix, kind)
                kept = f0 - free_bytes()
            transient = 0 if kind == "symmetric" else _lib.PLOT_CELLS * 2 + 24 * len(rec)
            added[kind] = {"kept_measured": kept, "freed_buffers_computed": transient, "peak": kept + transient}
        res["device_bytes_added"] = added
        with hetmers.Scan(kt) as sc:
            plot, st = sc.run()
            res["symmetric_scan_ms"] = st["ms_scan"]
            pix = labels(plot)
            res["labelled_isolated_pairs"] = int(plot[pix > 0].sum())
            runs = {"direct": [], "symmetric": []}
            ref = None
            for i in range(reps + 1):
                for kind in (("direct", "symmetric") if i % 2 == 0 else ("symmetric", "direct")):
                    rec, m = route(sc, pix, kind)
                    if ref is None:
                        ref = rec
                    assert np.array_equal(rec, ref), f"{kind} records differ"
                    if i > 0:                                   # the first round warms up
                        runs[kind].append(m)
        res["records_equal"] = True
        res["records"] = len(ref)
        res["median"] = {k: {f: float(np.median([r[f] for r in v])) for f in v[0]} for k, v in runs.items()}
        res["runs"] = runs
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "nels", "records", "records_equal", "median", "device_bytes_added")},
                     indent=1))


if __name__ == "__main__":
    main()
