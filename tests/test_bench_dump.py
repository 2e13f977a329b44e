"""bench.py --dump-outputs: what the timed path computed in its last step, sampled by input-set index and written as
float64 limbs, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from tests import util
from tests.util import po

BENCH = os.path.join(util.ROOT, "bench.py")


def test_bench_rejects_zero_steps_and_dump_without_the_gpu_arm(tmp_path):
    r = subprocess.run([sys.executable, BENCH, "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
    r = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_witnesses_of_the_last_timed_step(tmp_path):
    """three launches per step (4736 + 4736 + 1128 sets; the sample holds rows of each, the first row of the last launch
    among them), each dumped row equal to the C oracle's witness of the same synthetic input set"""
    from oracle import cref
    name, batch, steps = "circuit9_authV2", 10600, 2
    r = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--batch", str(batch),
                        "--chunk", "4736", "--no-e2e", "--no-cpu", "--no-configs", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == steps * 3 and line["extra"]["verified_against_oracle"]
    assert line["extra"]["dump_copy_ms_excluded"] > 0
    assert sorted(os.listdir(tmp_path)) == ["input_set.npy", "witness.npy"]
    w, idx = np.load(tmp_path / "witness.npy"), np.load(tmp_path / "input_set.npy")
    assert w.dtype == np.float64 and idx.dtype == np.float64
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    data = util.golden_graph(name)
    cg = cref.CGraph(data)
    assert w.shape == (len(idx), cg.n_witness, 8) and len(idx) >= 8
    rows = idx.astype(np.int64)
    assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < batch
    plan = bench.launch_plan(batch, 4736, 148)
    assert len(plan) == 3 and all(((rows >= lo) & (rows < hi)).any() for lo, hi in plan) and plan[2][0] in rows
    _, _, imap = po.deserialize_graph(data)
    inp = bench.synth_inputs(name, 0, batch, cg.n_inputs, imap, seed=9)[rows]
    want = cg.evaluate_batch(inp, min(len(rows), os.cpu_count() or 1)).view("<u4")
    assert (w == want.astype(np.float64)).all()
    # a second run with another step count and launch plan (one launch) dumps the same input sets and the same values
    r = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "1", "--warmup", "1", "--batch", str(batch),
                        "--no-e2e", "--no-cpu", "--no-configs", "--dump-outputs", str(tmp_path / "again")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert (np.load(tmp_path / "again" / "input_set.npy") == idx).all()
    assert (np.load(tmp_path / "again" / "witness.npy") == w).all()
