"""bench.py --steps / --dump-outputs: --steps sets how many steps the timed loop runs, and the dumped files are
what its last step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import ROOT

pytestmark = pytest.mark.gpu

WARMUP, FRAMES = 3, 5


def run_bench(tmp_path, steps):
    out = tmp_path / ("outputs_%d" % steps)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(WARMUP),
                          "--frames", str(FRAMES), "--e2e-steps", "3", "--no-cpu", "--no-extras", "--no-sweep", "--no-resent",
                          "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip())
    assert sorted(os.listdir(out)) == ["iou_counts.npy", "mask.npy"]
    return line, np.load(out / "mask.npy"), np.load(out / "iou_counts.npy")


def test_steps_and_dump_outputs(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from pcm.synthetic import SyntheticSequence
    seq = SyntheticSequence(bench.WIDTH, bench.HEIGHT, bench.SEQ_FRAMES, seed=0)
    launches = {}
    for steps in (4, 8):
        line, mask, counts = run_bench(tmp_path, steps)
        assert line["steps"] == steps and line["warmup"] == WARMUP
        launches[steps] = line["gpu_launches"]
        assert mask.dtype == np.float32 and mask.shape == (bench.HEIGHT, bench.WIDTH)
        assert counts.dtype == np.float64 and counts.shape == (2,)
        assert set(np.unique(mask).tolist()) <= {0.0, 255.0} and mask.any()
        # the last timed step is step WARMUP + steps - 1, on frame (WARMUP + steps - 1) % FRAMES (1 and 0 here)
        truth = seq.truth((WARMUP + steps - 1) % FRAMES) != 0
        fg = mask != 0
        assert counts.tolist() == [float(np.sum(fg & truth)), float(np.sum(fg | truth))]
    # every step of the timed loop launches the same kernels: twice the steps, twice the launches
    assert launches[4] > 0 and launches[8] == 2 * launches[4], launches
