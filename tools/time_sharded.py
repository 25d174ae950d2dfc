"""Time replica against sharded placement on the bench workload (BASELINE configs[1]: k = 31, diploid, ~2e8
k-mers) through the C ABI: load (hm_scan_create / hm_scan_create_sharded), the first scan (which, on a
sharded table, first gives every shard its run-aligned key range: the redistribution step that
conditioning also runs), steady-state scans, conditioning of a canonical untrimmed table of the same
genome, and the device bytes each shard keeps.  Sharded over S = 1/2/4/8 logical shards on GPU 0 and over
2/4/8 physical GPUs when the box has them.  Every sharded plot is checked against the replica's.

    python tools/time_sharded.py OUT.json [nels=2e8] [reps=5]
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


def one(name, shards, reps, cond=None):
    t0 = time.perf_counter()
    sc = hetmers.Scan(fastk.read_ktab(name), shards=shards) if shards is not None else hetmers.Scan(fastk.read_ktab(name))
    t1 = time.perf_counter()
    r = {}
    if cond is not None:
        sc.condition(cond, True, True)
        r["condition_ms"] = (time.perf_counter() - t1) * 1e3
        t1 = time.perf_counter()
    plot, _ = sc.run()
    t2 = time.perf_counter()
    scans = []
    for _ in range(reps):
        _, st = sc.run()
        scans.append(st["ms_scan"])
    info = sc.shard_info()
    sc.close()
    r.update({"load_ms": (t1 - t0) * 1e3, "first_scan_ms": (t2 - t1) * 1e3, "scan_ms": float(np.median(scans)),
              "n": [s["n"] for s in info], "device_bytes": [s["device_bytes"] for s in info]})
    return r, plot


def main():
    out = sys.argv[1]
    nels = float(sys.argv[2]) if len(sys.argv) > 2 else 2e8
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    ngpu = _lib.lib().hm_device_count()
    res = {"card": card(), "gpus": ngpu, "workload": f"configs[1]: k={K}, ploidy {P}, het {HET}, cov {COV}, L {L}"}
    G = synth.calibrate_G(K, int(nels), P, HET, COV, L)
    with tempfile.TemporaryDirectory() as d:
        name = os.path.join(d, "t")
        keys, cnt = synth.synth_table(K, G, P, HET, COV, L, SEED, device="cuda")
        kt = synth.write_table(name, K, keys, cnt, ibyte=3, nparts=4)
        del keys, cnt
        res["nels"] = kt.nels
        rep, want = one(name, None, reps)
        res["replica"] = rep
        runs = [("logical", [0] * s) for s in (1, 2, 4, 8)]
        runs += [("physical", list(range(g))) for g in (2, 4, 8) if g <= ngpu]
        for kind, sh in runs:
            r, plot = one(name, sh, reps)
            r["plot_equals_replica"] = bool(np.array_equal(plot, want))
            res[f"sharded_{kind}_{len(sh)}"] = r
            print(kind, len(sh), json.dumps(r), flush=True)
        # conditioning: the same genome as a canonical untrimmed table (what FastK writes)
        import torch
        keys, cnt = synth.synth_table(K, G, P, HET, COV, 1, SEED, device="cuda")
        rc = synth.revcomp_left(keys, K)
        canon = (keys.view(torch.int64) ^ (1 << 63)) <= (rc.view(torch.int64) ^ (1 << 63))     # unsigned x <= rc x
        craw = os.path.join(d, "raw")
        ckt = synth.write_table(craw, K, keys[canon].contiguous(), cnt[canon].contiguous(), ibyte=3, nparts=4)
        del keys, cnt, rc
        res["canonical_nels"] = ckt.nels
        crep, cwant = one(craw, None, reps, cond=L)
        res["condition_replica"] = crep
        for s in (2, 4, 8):
            r, plot = one(craw, [0] * s, reps, cond=L)
            r["plot_equals_replica"] = bool(np.array_equal(plot, cwant))
            res[f"condition_sharded_logical_{s}"] = r
            print("condition", s, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    bad = [k for k, v in res.items() if isinstance(v, dict) and v.get("plot_equals_replica") is False]
    if bad:
        sys.exit(f"sharded plots differ from the replica's: {bad}")


if __name__ == "__main__":
    main()
