#!/usr/bin/env python3
"""Regenerate tests/golden/: seeded synthetic FastK tables + the .smu the UNMODIFIED reference
`hetmers` (oracle/_ref/hetmers, built from /root/reference by oracle/Makefile) writes for them.

The reference ships no golden vectors for this path (SURVEY.md §4), so these files ARE the pin:
tests/test_oracle.py requires oracle/hetmers_oracle.c to reproduce each .smu byte for byte, and
the -m gpu tests require the CUDA path to do the same.  Run from the repo root, in the build
container (needs /root/reference):   python tests/golden/make_golden.py
Only reference_runs.json (digests of the reference's outputs on the larger seeded tables of the GPU
tests):   python tests/golden/make_golden.py --reference-runs
"""
import json
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from smudgeplot_b200 import fastk  # noqa: E402
from tools import synth  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "hetmers")
REF_EXTRACT = os.path.join(ROOT, "oracle", "_ref", "extract_kmer_pairs")
EXTRACT_CASES = ("dip_k21", "dip_k40", "tet_k32")      # golden pair lists (extract_kmer_pairs)


def write_sma(path, smu_text):
    """label the pixels of a .smu the way `smudgeplot all` writes <o>.sma (cli.py:451-456):
    header + "covB covA freq <a>A<b>B"; labels here are synthetic (by sum mod 3), one third unlabelled"""
    with open(path, "w") as f:
        f.write("covB\tcovA\tfreq\tsmudge\n")
        for ln in smu_text.splitlines():
            m, rest, cnt = (int(v) for v in ln.split("\t"))
            lab = {0: "1A1B", 1: "2A1B"}.get((m + rest) % 3)
            if lab:
                f.write(f"{m}\t{rest}\t{cnt}\t{lab}\n")


def run_ref_extract(table, sma, out, e, threads=1):
    return subprocess.run([REF_EXTRACT, f"-e{e}", f"-T{threads}", f"-o{out}", table, sma],
                          capture_output=True, text=True)

# name -> generator parameters (+ file layout, -e threshold handed to the reference)
CASES = {
    "dip_k21":   dict(k=21, G=4000,  ploidy=2, het=0.01, cov=40,  L=4,  seed=1, ibyte=1, nparts=1, e=4),
    "trip_k31":  dict(k=31, G=4500,  ploidy=3, het=0.02, cov=60,  L=12, seed=4, ibyte=1, nparts=4, e=12, rep=2),
    "tet_k32":   dict(k=32, G=2500,  ploidy=4, het=0.02, cov=80,  L=10, seed=5, ibyte=2, nparts=2, e=10),
    "dense_k11": dict(k=11, G=40000, ploidy=2, het=0.05, cov=30,  L=4,  seed=7, ibyte=1, nparts=3, e=4),
    "smax_k17":  dict(k=17, G=5000,  ploidy=2, het=0.03, cov=985, L=4,  seed=9, ibyte=1, nparts=1, e=4),
    "dip_k40":   dict(k=40, G=3000,  ploidy=2, het=0.02, cov=40,  L=4,  seed=13, ibyte=1, nparts=2, e=4),
    "midcut_k21": dict(k=21, G=5000, ploidy=2, het=0.02, cov=40,  L=4,  seed=11, ibyte=1, nparts=4, e=4, midcut=True),
}


def run_ref(table, out, e, threads=4):
    smu = out + ".smu"
    if os.path.exists(smu):
        os.remove(smu)
    r = subprocess.run([REF, "-v", f"-e{e}", f"-T{threads}", f"-o{out}", table],
                       input="n\n", capture_output=True, text=True)
    return r


def main():
    if not os.path.exists(REF):
        sys.exit("oracle/_ref/hetmers missing: run `make -C oracle` where /root/reference exists")
    meta = {}
    for name, c in CASES.items():
        d = os.path.join(HERE, name)
        shutil.rmtree(d, ignore_errors=True)
        os.makedirs(d)
        keys, cnt = synth.synth_table(c["k"], c["G"], c["ploidy"], c["het"], c["cov"], c["L"], c["seed"],
                                      extra_hom_repeats=c.get("rep", 0))
        table = os.path.join(d, name)
        synth.write_table(table, c["k"], keys, cnt, ibyte=c["ibyte"], nparts=c["nparts"],
                          cut_on_buckets=not c.get("midcut", False))
        outs = []
        for T in (1, 4):
            r = run_ref(table, os.path.join(d, f"ref_T{T}"), c["e"], T)
            assert r.returncode == 0, r.stderr
            outs.append(open(os.path.join(d, f"ref_T{T}.smu")).read())
        assert outs[0] == outs[1], f"{name}: reference output depends on -T ?"
        os.rename(os.path.join(d, "ref_T1.smu"), os.path.join(d, name + ".smu"))
        os.remove(os.path.join(d, "ref_T4.smu"))
        meta[name] = dict(c, nels=int(keys.shape[0]), smu_rows=len(outs[0].splitlines()),
                          verbose=[ln.strip() for ln in r.stderr.splitlines() if "input table" in ln])
        print(name, meta[name]["nels"], "entries,", meta[name]["smu_rows"], "rows")
        if name in EXTRACT_CASES:
            # extract_kmer_pairs: the reference's line order depends on its thread schedule, so the
            # golden files hold the SORTED lines of each <out>.<a>A<b>B.txt (-T1 and -T4 must agree)
            sma = os.path.join(d, name + ".sma")
            write_sma(sma, outs[0])
            lists = []
            for T in (1, 4):
                for old in os.listdir(d):
                    if old.startswith("refx."):
                        os.remove(os.path.join(d, old))
                r = run_ref_extract(table, sma, os.path.join(d, "refx"), c["e"], T)
                assert r.returncode == 0, r.stderr
                lists.append({f: sorted(open(os.path.join(d, f)).read().splitlines())
                              for f in sorted(os.listdir(d)) if f.startswith("refx.")})
            assert lists[0] == lists[1] and lists[0], f"{name}: extract output depends on -T ?"
            npairs = {}
            for f, lines in lists[0].items():
                os.remove(os.path.join(d, f))
                lab = f[len("refx."):-len(".txt")]
                with open(os.path.join(d, f"{name}.pairs.{lab}.txt"), "w") as g:
                    g.write("".join(ln + "\n" for ln in lines))
                npairs[lab] = len(lines)
            meta[name]["pairs"] = npairs
            print("   extract:", npairs)

    # conditioning decisions (examine_table, PloidyPlot.c:1167-1230): the reference prints its
    # verdict with -v and then dies trying to run the absent FastK tools Logex / Symmex.
    keys, cnt = synth.synth_table(21, 3000, 2, 0.01, 40, 4, 21)
    ku = synth.keys_to_u64_numpy(keys)
    cn = cnt.numpy().astype(np.uint16)
    d = os.path.join(HERE, "conditioning")
    shutil.rmtree(d, ignore_errors=True)
    os.makedirs(d)
    # (a) untrimmed: threshold above the smallest count
    fastk.write_ktab(os.path.join(d, "untrimmed"), 21, ku, cn, ibyte=1)
    # (b) not symmetric: drop the reverse complement of entry 1
    rc1 = synth.keys_to_u64_numpy(synth.revcomp_left(keys[1:2], 21))[0]
    keep = ku != rc1
    fastk.write_ktab(os.path.join(d, "asymmetric"), 21, ku[keep], cn[keep], ibyte=1)
    cond = {}
    for nm, e in (("untrimmed", 9), ("asymmetric", 4)):
        r = run_ref(os.path.join(d, nm), os.path.join(d, nm + "_out"), e)
        cond[nm] = dict(e=e, returncode=r.returncode,
                        verbose=[ln.strip() for ln in r.stderr.splitlines() if "input table" in ln],
                        stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith("hetmers:")])
        print(nm, cond[nm])
        for junk in (".trim", ".symx"):
            pass
    meta["_conditioning"] = cond
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    reference_runs()


def reference_runs():
    """reference_runs.json: what the reference binaries write for the seeded tables of the GPU tests that
    compare with them (tests/test_gpu_parity.py MEDIUM_CASES, CONDITIONING_CASES, EXTRACT_CASES), keyed like
    the pytest ids.  The tests regenerate the tables from their seeds (synth gives the same table on CPU and
    GPU); the outputs, megabytes of text, are kept as entry count, line count and sha256."""
    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    import oracle_util as ou
    import test_gpu_parity as tp
    if not (os.path.exists(REF) and os.path.exists(REF_EXTRACT)):
        sys.exit("oracle/_ref/ missing: run `make -C oracle` where the reference sources exist")
    threads = min(os.cpu_count() or 4, 64)
    key = lambda params: "-".join(str(p) for p in params)          # noqa: E731
    runs = {"medium": {}, "conditioning": {}, "extract": {}}
    d = tempfile.mkdtemp(prefix="reference_runs_")
    try:
        for c in tp.MEDIUM_CASES:
            k, target, ploidy, het, cov, L, seed, ref_threads = c
            G = synth.calibrate_G(k, target, ploidy, het, cov, L)
            keys, cnt = synth.synth_table(k, G, ploidy, het, cov, L, seed)
            table = os.path.join(d, "medium")
            kt = synth.write_table(table, k, keys, cnt, ibyte=3, nparts=4)
            del keys, cnt
            r = run_ref(table, os.path.join(d, "medium"), L, ref_threads or threads)
            assert r.returncode == 0, r.stderr
            smu = open(os.path.join(d, "medium.smu")).read()
            runs["medium"][key(c)] = dict(nels=kt.nels, smu_rows=len(smu.splitlines()), smu_sha256=ou.sha256_text(smu))
            fastk.remove_ktab(table)
            print("medium", key(c), runs["medium"][key(c)])
        for c in tp.CONDITIONING_CASES:
            k, G, ploidy, seed, L = c
            ku, cn = tp.canonical_untrimmed_table(k, G, ploidy, seed)
            ck, cc = tp._condition_numpy(ku, cn, k, L, True, True)
            table = os.path.join(d, "cond")
            fastk.write_ktab(table, k, ck, cc, ibyte=3, nparts=2)
            r = run_ref(table, os.path.join(d, "cond"), L, 4)
            assert r.returncode == 0 and "trimmed and symmetric" in r.stderr, r.stderr
            smu = open(os.path.join(d, "cond.smu")).read()
            runs["conditioning"][key(c)] = dict(nels=len(cc), smu_rows=len(smu.splitlines()),
                                                smu_sha256=ou.sha256_text(smu))
            print("conditioning", key(c), runs["conditioning"][key(c)])
        for c in tp.EXTRACT_CASES:
            k, G, ploidy, seed, L = c
            keys, cnt = synth.synth_table(k, G, ploidy, 0.02, 20 * ploidy, L, seed)
            table = os.path.join(d, "ex")
            kt = synth.write_table(table, k, keys, cnt, ibyte=3, nparts=3)
            r = run_ref(table, os.path.join(d, "ex"), L, threads)
            assert r.returncode == 0, r.stderr
            plot = np.zeros((ou.SMAX + 1, ou.PLOT_W), dtype=np.int64)
            for ln in open(os.path.join(d, "ex.smu")).read().splitlines():
                m, rest, n = (int(v) for v in ln.split("\t"))
                plot[m + rest, m] = n
            sma = os.path.join(d, "ex.sma")
            tp.label_sma(plot, sma)                                # the .sma the test writes from its plot
            out = os.path.join(d, "pairs", "refx")
            shutil.rmtree(os.path.dirname(out), ignore_errors=True)
            os.makedirs(os.path.dirname(out))
            r = run_ref_extract(table, sma, out, L, threads)
            assert r.returncode == 0, r.stderr
            lists = ou.sorted_pair_files(out)
            assert lists
            runs["extract"][key(c)] = dict(nels=kt.nels, pairs={lab: dict(lines=len(v), sha256=ou.sha256_lines(v))
                                                                for lab, v in lists.items()})
            print("extract", key(c), runs["extract"][key(c)])
    finally:
        shutil.rmtree(d, ignore_errors=True)
    with open(os.path.join(HERE, "reference_runs.json"), "w") as f:
        json.dump(runs, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    if sys.argv[1:] == ["--reference-runs"]:
        reference_runs()
    else:
        main()
