#!/usr/bin/env python3
"""bench.py -- k-mers/s scanned by the hetmers hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our CUDA path
  python bench.py --impl reference ...                     the reference's own C hetmers on host cores
  python bench.py ... --dump-outputs DIR                   also writes the last timed step's plot to DIR/plot.npy

A "step" is one full scan (pass 1 + degree exchange + pass 2 + plot reduce = T_scan of SURVEY.md
§8d) of one synthetic FastK table.  Workload = BASELINE.json configs[1]: synthetic diploid k=31
table, het 1 %, coverage 40x, L=12, ~2e8 k-mers per GPU (weak scaling: with N GPUs the table has
N x 2e8 k-mers, every rank holds a replica and scans a contiguous 1/N index range).

  value  k-mers/s with the table already unpacked in HBM (CUDA events, max over ranks).  The table is
         strand-symmetric (as the reference requires of its input), so the scan is the symmetric one
         of csrc/hm_symm.cu: runscan_kernel + resolve_kernel (HETMERS_PATH=direct: the direct passes)
  e2e    k-mers/s through the public C-ABI call hm_hetmers_host() on HOST buffers holding the raw
         FastK part payloads in pinned memory: H2D + unpack + bucket index + symmetry fingerprint +
         both kernels + plot D2H
  roofline   dominant kernel (runscan_kernel): it reads every entry once, TBYTE = 10 B/k-mer at k=31
             (the official whole-scan figure of SURVEY §8d, A = 2*TBYTE+2 = 22 B/k-mer over T_scan, is
             reported next to it as roofline.whole_scan), against MEASURED_PEAKS.json hbm_gbs
  parity     hard gates (non-zero exit): the timed table's plot == the plot of the independent direct
             passes; N > 1: the sharded plot == a one-GPU scan of the same table on rank 0; the .smu
             of our executable == the reference binary's on the same files
  cpu_baseline  the reference C hetmers (oracle/_ref/hetmers; else the oracle port) on the host
             cores, on the SAME table files our executable reads (e2e_exec)
Inputs (1.9 GB table + 0.27 GB bucket index per 2e8 k-mers) exceed the 126 MB L2, so no flush is
needed between timed iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, PLOIDY, HET, COV, LCUT, SEED = 31, 2, 0.01, 40.0, 12, 2
TBYTE = (K + 3) // 4 + 2                                   # packed k-mer + uint16 count: 10 B at k=31
ALGO_BYTES_PER_KMER = 2 * TBYTE + 2                        # 22 B at k=31 (SURVEY.md §8d): two passes + deg byte
UNIT = "k-mers/s"


def _baseline_metric():
    """the metric string of BASELINE.json (the driver compares against it), else a local default"""
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "k-mers/sec scanned (hetmers)"


METRIC = _baseline_metric()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nels", type=float, default=2e8, help="target k-mers per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the plot the last timed step computed to DIR/plot.npy (our arm only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs: only our arm returns a plot (the reference arm writes a .smu of a sample table)")
    return args


def workload_name(n_gpus):
    return (f"BASELINE configs[1]: synthetic diploid k={K} FastK table, het={HET:.0%}, cov={COV:g}x, L={LCUT}, "
            f"~2e8 k-mers per GPU x {n_gpus} GPU(s)")


# ------------------------------------------------------------------------------ clocks ------

class ClockSampler:
    """SM clock + throttle reasons during the timed region (pynvml; B200_PROFILING.md recipe)."""

    def __init__(self, index=0, period=0.05):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.index, self.period = index, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------- reference arm -------

def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def scratch_dir():
    for d in ("/dev/shm", tempfile.gettempdir()):
        if os.path.isdir(d) and os.access(d, os.W_OK):
            return tempfile.mkdtemp(prefix="hetmers_bench_", dir=d)
    return tempfile.mkdtemp(prefix="hetmers_bench_")


def make_sample_table(dirname, n_target, device):
    """seeded table of ~n_target k-mers with the bench workload's parameters, written as FastK files"""
    from tools import synth
    G = synth.calibrate_G(K, int(n_target), PLOIDY, HET, COV, LCUT)
    keys, cnt = synth.synth_table(K, G, PLOIDY, HET, COV, LCUT, SEED, device=device)
    name = os.path.join(dirname, "sample")
    synth.write_table(name, K, keys, cnt, ibyte=3, nparts=4)
    return name, int(keys.numel())


def time_reference(table, nels, threads, runs=1):
    """wall clock of the CPU implementation on `table`; -> (seconds list, kind)"""
    ref = os.path.join(ROOT, "oracle", "_ref", "hetmers")
    ora = os.path.join(ROOT, "oracle", "hetmers_oracle")
    out = os.path.join(os.path.dirname(table), "cpu_out")
    times = []
    if os.path.exists(ref):
        cmd, kind = [ref, f"-e{LCUT}", f"-T{threads}", f"-o{out}", table], "reference"
    else:
        cmd, kind = [ora, f"-e{LCUT}", f"-o{out}", table], "port"
    for _ in range(runs):
        if os.path.exists(out + ".smu"):
            os.remove(out + ".smu")
        t0 = time.perf_counter()
        r = subprocess.run(cmd, input="n\n", capture_output=True, text=True)
        times.append(time.perf_counter() - t0)
        if r.returncode != 0:
            raise RuntimeError(f"CPU baseline failed: {r.stderr[-500:]}")
    return times, kind, out + ".smu"


def cpu_sample_size(args, threads):
    # reference arm: survey anchor ~0.45e6 k-mers/s per thread at k=31 (SURVEY.md §6), but the reference stops
    # scaling near 8-9e6 k-mers/s (measured: 7.8e6/s at -T64 on a B200 host); bounded by the GPU workload
    n = min(0.45e6 * threads, 9e6) * args.cpu_seconds
    return int(max(2e6, min(n, args.nels)))


def bench_config(world):
    """the `config` object BOTH arms print: the workload and nothing run-specific (what a run did with it is
    in the line's `run` object; the reference arm's bounded sample in `cpu_baseline.sample`)"""
    return {"workload": workload_name(world), "k": K, "ploidy": PLOIDY, "het": HET, "cov": COV, "L": LCUT, "seed": SEED,
            "target_nels_per_gpu": 2e8,
            "l2": "inputs (>= 1.9 GB table + bucket index per GPU) exceed the 126 MB L2; no flush between iterations"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = min(host_cores(), 64)
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "hetmers")):
        threads = 1
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    d = scratch_dir()
    try:
        n_s = cpu_sample_size(args, threads)
        table, nels = make_sample_table(d, n_s, dev)
        warm, kind, _ = time_reference(table, nels, threads, runs=max(args.warmup, 0))
        secs, kind, _ = time_reference(table, nels, threads, runs=args.steps)
        total = sum(secs)
        value = nels * args.steps / total
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
                "data": "synthetic", "gpu_launches": 0,
                "config": bench_config(args.gpus),
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                                 "sample": f"per step one pass of the {'reference C hetmers' if kind == 'reference' else 'oracle port'} "
                                           f"-T{threads} over a seeded {nels}-k-mer table of this workload (same generator, "
                                           f"parameters and seed as the GPU arm's table; the reference is linear in the "
                                           f"table size, BASELINE.md §2)", "nels_sample": nels},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


# -------------------------------------------------------------------------- our arm ---------

def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel, nels, grid):
    """dram bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json),
    scaled per k-mer.  The record names the launch shape it was captured with: a record of another shape
    (entries per CTA) is refused rather than quoted."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        j = json.load(open(p))[kernel]
        if grid is not None and j.get("entries_per_cta") is not None and \
                abs(nels / grid - j["entries_per_cta"]) > 0.02 * j["entries_per_cta"]:
            return None
        return float(j["dram_bytes_per_kmer"]) * nels
    except Exception:
        return None


def dump_outputs(dirname, plot):
    """DIR/plot.npy: what a caller of the scan receives, the (count sum, min count) histogram of isolated pairs,
    as float64 [1001, 501] (exact: a cell counts at most one pair per table entry, far below 2^53).  The table is
    generated from a fixed seed, so two builds given the same arguments can be compared cell for cell."""
    import numpy as np
    from smudgeplot_b200 import _lib
    os.makedirs(dirname, exist_ok=True)
    a = plot.cpu().numpy().reshape(_lib.SMAX + 1, _lib.PLOT_W).astype(np.float64)
    np.save(os.path.join(dirname, "plot.npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hetmers path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    multi = world > 1
    if multi:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from smudgeplot_b200 import _lib
    from smudgeplot_b200.device import DeviceTable
    from tools import synth
    if multi:
        from smudgeplot_b200 import dist as hdist

    # ---- synthetic table (setup, untimed) ---------------------------------------------------
    n_target = int(args.nels) * world
    G = synth.calibrate_G(K, n_target, PLOIDY, HET, COV, LCUT)
    want_direct = os.environ.get("HETMERS_PATH") == "direct"
    if multi:
        job = hdist.ShardedScan.from_synthetic(K, G, PLOIDY, HET, COV, LCUT, SEED, dev)
        nels, my_n = job.n_total, job.hi - job.lo
        path = job.path
        table = job.table
    else:
        keys, cnt = synth.synth_table(K, G, PLOIDY, HET, COV, LCUT, SEED, device=dev)
        table = DeviceTable(K, keys, cnt.to(torch.int16)).build_index(direct=False)
        path = "symm" if (table.check_symmetric() and not want_direct) else "direct"
        if path == "symm":
            table.alloc_symm()
        else:
            table.build_filter()
            table.alloc_work()
        nels = my_n = table.n
    torch.cuda.synchronize()

    def one_scan(events=None):
        if multi:
            return job.scan(events)
        table.plot.zero_()
        if path == "symm":
            if events is not None:
                events[0].record()
            table.runscan(mid_event=events[1] if events is not None else None)   # [0],[1] bracket runscan_kernel alone
            table.resolve()
            return table.plot
        table.deg.zero_()
        if events is not None:
            events[0].record()
        table.pass1()
        if events is not None:
            events[1].record()
        table.pass2()
        return table.plot

    for _ in range(max(args.warmup, 3)):
        one_scan()
    torch.cuda.synchronize()
    if multi:
        job.profile_phases = True
    if multi:
        dist.barrier()
    # ---- timed region: exactly K steps ------------------------------------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p1 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local) as clk:
        torch.cuda.synchronize()
        ev0.record()
        for s in range(args.steps):
            plot = one_scan(p1[s])
        ev1.record()
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
        ms_total = ev0.elapsed_time(ev1)
        ms_p1 = sum(a.elapsed_time(b) for a, b in p1) / args.steps
        timed_plot = plot.clone()
        # keep the sampler alive over the e2e region too (more samples under load)
        e2e = None
        if multi:
            job.profile_phases = False
        if not args.no_e2e:
            e2e = measure_e2e(args, torch, dist, dev, multi, world, rank,
                              job if multi else None, (keys, cnt) if not multi else None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, timed_plot)
    if multi:
        t = torch.tensor([ms_total, ms_p1], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_p1 = t.tolist()
    ms_step = ms_total / args.steps
    value = nels / (ms_step * 1e-3)
    # kernels of ours per scan: runscan + runs + resolve (symmetric) / pass 1 + pass 2 (+ deferred look-ups, N > 1)
    launches = (3 if (path == "symm" or multi) else 2) * args.steps

    # ---- parity gates (untimed): the timed plot against independent computations of the same table ----
    parity = {"path": path}
    ok = True
    if path == "symm":
        clean = job.symm_ok() if multi else (table.symm_status()[1] == 0)
        parity["symmetric_scan_status_clean"] = bool(clean)
        ok &= bool(clean)
    if rank == 0:
        ref_t = DeviceTable(K, table.keys, table.cnt, bits=table.bits)
        ref_t.bucket = table.bucket
        ref_t.build_filter()
        ref_t.alloc_work()
        direct_plot = ref_t.scan("direct").reshape(-1).clone()          # the direct passes: another algorithm
        parity["vs_direct_passes_one_gpu"] = bool(torch.equal(direct_plot, timed_plot.reshape(-1)))
        ok &= parity["vs_direct_passes_one_gpu"]
        if multi:
            one = DeviceTable(K, table.keys, table.cnt, bits=table.bits)
            one.bucket = table.bucket
            one_plot = one.scan("symm" if path == "symm" else "direct").reshape(-1).clone()
            parity["vs_single_gpu"] = bool(torch.equal(one_plot, timed_plot.reshape(-1)))
            ok &= parity["vs_single_gpu"]
            del one
        parity["pairs_counted"] = int(timed_plot.sum())
        del ref_t, direct_plot
        torch.cuda.empty_cache()

    peak, peak_src = peaks()
    per_launch = my_n
    # pass 1 of the symmetric scan has two kernels: the launcher takes the all-pairs-in-the-run one when an entry
    # has more than 0.6 run mates on average (n / 4^(k/2): from N = 4 on in this weak-scaling series)
    dense = os.environ.get("HETMERS_RUNSCAN", "dense" if nels / float(4 ** (K // 2)) > 0.6 else "sparse") == "dense"
    kname = ("runscan_dense_kernel" if dense else "runscan_kernel") if path == "symm" else "pass1_filter_kernel"
    kbytes = TBYTE if path == "symm" else ALGO_BYTES_PER_KMER
    achieved = kbytes * per_launch / (ms_p1 * 1e-3) / 1e9
    whole = ALGO_BYTES_PER_KMER * nels / world / (ms_step * 1e-3) / 1e9
    grid = (per_launch + 2047) // 2048 if path == "symm" else None
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": bench_config(world),
            "run": {"nels": nels, "nels_per_gpu": my_n, "bucket_bits": table.bits, "scan": path,
                    "parallelism": (f"table replica per GPU, {world} contiguous run-aligned index shards; exchange: {job.exchange}"
                                    if multi else "1 GPU")},
            "clocks": clk.summary(), "gpu_launches": launches, "parity": parity,
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_kmer": kbytes, "ms_per_launch": ms_p1,
                         "traffic": measured_traffic(kname, per_launch, grid),
                         "note": (kname + " reads every entry (8 B key + 2 B count) exactly once; the second kernel "
                                  "reads candidate records only.  whole_scan = SURVEY §8d's official 22 B/k-mer over T_scan"
                                  if path == "symm" else "22 B/k-mer = SURVEY §8d (two passes)"),
                         "whole_scan": {"algorithmic_bytes_per_kmer": ALGO_BYTES_PER_KMER, "achieved": whole,
                                        "frac": whole / peak, "ms": ms_step}}}
    if multi and job.phase_ms():
        allp = [None] * world
        dist.all_gather_object(allp, {k: round(v, 3) for k, v in job.phase_ms().items()})
        names = list(allp[0].keys())                                   # one compact list per phase, all ranks
        line["run"]["phases_ms_by_rank"] = {nm: [a[nm] for a in allp] for nm in names if nm != "-"}
    if e2e is not None:
        line["e2e"] = e2e
        if multi and "plot_matches_resident_scan" in e2e:
            parity["e2e_vs_resident"] = bool(e2e["plot_matches_resident_scan"])
            ok &= parity["e2e_vs_resident"]
    if rank == 0:
        if not args.no_cpu and world == 1:
            cb = cpu_baseline(args, dev, keys, cnt, timed_plot)
            line["cpu_baseline"] = cb["cpu_baseline"]
            line["e2e_exec"] = cb["e2e_exec"]
            parity.update(cb["parity"])
            ok &= all(bool(v) for v in cb["parity"].values())
        parity["ok"] = bool(ok)
        print(json.dumps(line), flush=True)
    if multi:
        job.close()
        flag = torch.tensor([int(ok)], dtype=torch.int32, device=dev)
        dist.broadcast(flag, src=0)
        ok = bool(flag.item())
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        sys.stderr.write("bench.py: PARITY GATE FAILED -- see the \"parity\" object of the JSON line\n")
        sys.exit(3)


def cpu_baseline(args, dev, keys, cnt, timed_plot):
    """The timed table itself as FastK files in /dev/shm: the unmodified reference binary (-T min(cores,64)) and
    our drop-in executable read the same files.  -> cpu_baseline, e2e_exec (process wall clock of the executable
    with its own phase breakdown) and the .smu parity flags."""
    import numpy as np
    from smudgeplot_b200 import hetmers
    from tools import synth
    threads = min(host_cores(), 64)
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "hetmers"))
    d = scratch_dir()
    try:
        full = have_ref and not os.environ.get("BENCH_CPU_SAMPLE")
        if full:                                                   # the GPU arm's table, all of it
            table = os.path.join(d, "table")
            synth.write_table(table, K, keys, cnt, ibyte=3, nparts=4)
            nels = int(keys.numel())
        else:                                                      # scalar port: a bounded sample
            threads = threads if have_ref else 1
            table, nels = make_sample_table(d, cpu_sample_size(args, threads), dev)
        secs, kind, smu = time_reference(table, nels, threads, runs=1)
        # our executable on the same files: wall clock of the process (files -> .smu), best of 3
        out = os.path.join(d, "gpu_out")
        env = dict(os.environ, HETMERS_STATS="1")
        runs = []
        for _ in range(3):
            if os.path.exists(out + ".smu"):
                os.remove(out + ".smu")
            t0 = time.perf_counter()
            r = subprocess.run([hetmers.get_binary_path("hetmers"), f"-e{LCUT}", f"-T{threads}", f"-o{out}", table],
                               input="n\n", capture_output=True, text=True, env=env)
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                raise RuntimeError(f"our hetmers executable failed: {r.stderr[-500:]}")
            st = None
            for ln in r.stderr.splitlines():
                if ln.startswith("{"):
                    try:
                        st = json.loads(ln)
                    except Exception:
                        pass
            runs.append((dt, st))
        best = min(runs, key=lambda x: x[0])
        same = open(out + ".smu").read() == open(smu).read()
        par = {"exec_smu_vs_reference_smu": bool(same)}
        if full:                                                   # and the timed in-process plot says the same
            par["timed_plot_vs_reference_smu"] = bool(hetmers.smu_text(timed_plot.cpu().numpy()) == open(smu).read())
        ref_name = "oracle/_ref/hetmers (unmodified reference C)" if kind == "reference" else "the oracle port"
        return {"cpu_baseline": {"value": nels / secs[0], "unit": UNIT, "cores": threads, "kind": kind,
                                 "sample": f"one run of {ref_name} -e{LCUT} -T{threads} on "
                                           f"{'the timed table itself' if full else 'a seeded sample table of the same workload'}: "
                                           f"{nels} k-mers, 4 part files in {os.path.dirname(table)} (warm page cache), "
                                           f"wall clock {secs[0]:.2f} s",
                                 "seconds": secs[0], "nels": nels},
                "e2e_exec": {"value": nels / best[0], "unit": UNIT, "seconds_wall": best[0],
                             "all_runs_s": [round(x[0], 3) for x in runs], "nels": nels, "threads": threads,
                             "speedup_vs_reference_wall": secs[0] / best[0],
                             "what": "process wall clock of smudgeplot_b200/bin/hetmers: FastK files in /dev/shm -> .smu "
                                     "(CUDA start-up, file reads, H2D, unpack, index, scan, .smu write), same files and "
                                     "-T as the reference run beside it",
                             "stats": best[1]},
                "parity": par}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def measure_e2e(args, torch, dist, dev, multi, world, rank, job, tabl):
    """the same scan through the public host-buffer API, copies inside the timed region"""
    import ctypes as C
    from smudgeplot_b200 import _lib
    if multi:
        return job.measure_e2e(args.steps, max(args.warmup, 1))
    keys, cnt = tabl
    n = keys.numel()
    kbyte, ibyte = (K + 3) // 4, 3
    pbyte = kbyte - ibyte + 2
    # FastK records + stub index built on the GPU (setup), then parked in pinned host memory
    rec = torch.empty((n, pbyte), dtype=torch.uint8, device=dev)
    for j in range(ibyte, kbyte):
        rec[:, j - ibyte] = ((keys >> (56 - 8 * j)) & 0xFF).to(torch.uint8)
    rec[:, pbyte - 2] = (cnt & 0xFF).to(torch.uint8)
    rec[:, pbyte - 1] = ((cnt >> 8) & 0xFF).to(torch.uint8)
    pre = (keys >> 40) & 0xFFFFFF
    index = torch.cumsum(torch.bincount(pre, minlength=1 << 24), 0)
    h_rec = torch.empty(rec.numel(), dtype=torch.uint8, pin_memory=True)
    h_rec.copy_(rec.view(-1))
    h_idx = torch.empty(1 << 24, dtype=torch.int64, pin_memory=True)
    h_idx.copy_(index)
    del rec, pre, index
    torch.cuda.synchronize()
    L = _lib.lib()
    part_nels = (C.c_int64 * 1)(n)
    part_rec = (C.c_void_p * 1)(h_rec.data_ptr())
    ht = _lib.HostTable(K, ibyte, 1, LCUT, n, C.cast(h_idx.data_ptr(), C.POINTER(C.c_int64)), part_nels, part_rec, None, None)
    devs = (C.c_int * 1)(dev.index or 0)
    plot = torch.empty(_lib.PLOT_CELLS, dtype=torch.int64, pin_memory=True)
    st = _lib.ScanStats()

    def call():
        _lib.check(L.hm_hetmers_host(C.byref(ht), devs, 1, plot.data_ptr(), C.byref(st)))

    for _ in range(max(args.warmup, 1)):
        call()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        call()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    return {"value": n / dt, "unit": UNIT, "ms_per_step": dt * 1e3,
            "h2d_bytes_per_step": int(h_rec.numel() + h_idx.numel() * 8),
            "d2h_bytes_per_step": int(_lib.PLOT_CELLS * 8),
            "api": "hm_hetmers_host(hm_host_table in pinned host memory) -> int64 plot[1001*501]",
            "last_call_ms": {"load": st.ms_h2d_unpack, "load_alloc": st.ms_alloc, "load_records": st.ms_records,
                             "load_index": st.ms_index, "pass1": st.ms_pass1, "pass2": st.ms_pass2, "scan": st.ms_scan,
                             "total_in_call": st.ms_total},
            "kernel_launches_per_call": int(st.kernel_launches)}


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
