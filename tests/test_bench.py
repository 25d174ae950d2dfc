"""bench.py end to end at a small size (run with -m gpu): the JSON line honours --steps, and --dump-outputs
writes the plot of the last timed step, which must be the oracle's plot of the same seeded table."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
import oracle_util as ou
from smudgeplot_b200 import fastk
from tools import synth

pytestmark = pytest.mark.gpu


def test_bench_dumps_the_plot_of_its_seeded_table(built, tmp_path):
    import bench
    nels, steps = 300_000, 2
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "1", "--nels", str(nels), "--no-e2e", "--no-cpu", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["parity"]["ok"]
    got = np.load(out / "plot.npy")
    assert got.dtype == np.float64 and got.shape == (ou.SMAX + 1, ou.PLOT_W)
    G = synth.calibrate_G(bench.K, nels, bench.PLOIDY, bench.HET, bench.COV, bench.LCUT)
    keys, cnt = synth.synth_table(bench.K, G, bench.PLOIDY, bench.HET, bench.COV, bench.LCUT, bench.SEED)
    assert keys.numel() == line["run"]["nels"]
    want, _ = ou.oracle_scan(fastk.keys_u64_to_bytes(synth.keys_to_u64_numpy(keys), bench.K),
                             cnt.numpy().astype(np.uint16), bench.K)
    assert want.sum() > 0
    assert np.array_equal(got, want.astype(np.float64))
