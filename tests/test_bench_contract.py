"""bench.py contract pieces: without a GPU, the reference arm prints exactly one JSON line on stdout (library chatter goes
to stderr) with the keys a harness reads, and ranks other than 0 stay silent; on the GPU, --dump-outputs writes the last
timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, timeout=600)


# what a torchrun worker inherits when --nproc-per-node > 1: the agent-store switch (turns every TCP rendezvous into a client
# of the agent's store -- the reference's private 1-rank group must not depend on it) and one OpenMP thread per worker
TORCHRUN_ENV = {"TORCHELASTIC_USE_AGENT_STORE": "True", "TORCHELASTIC_RESTART_COUNT": "0", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "1",
                "LOCAL_RANK": "0", "OMP_NUM_THREADS": "1"}


def test_reference_arm_prints_one_json_line():
    r = _run(dict(TORCHRUN_ENV, RANK="0", WORLD_SIZE="2"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["n_gpus"] == 2
    # "reference": the unmodified class staged in baseline/_ref (or /root/reference) ran; "port": those files are absent
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "1000000 classes" in d["cpu_baseline"]["sample"] and "full size" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "c3" in d["config"]["workload"] and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)          # rank 0 has the box to itself: OMP_NUM_THREADS=1 is overridden


def test_reference_arm_other_ranks_are_silent():
    r = _run(dict(TORCHRUN_ENV, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: x_grad, the loss and a fixed sample of sub_weight.grad rows of the last timed step, as float .npy files."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "c2", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    out = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["loss", "sub_weight_grad", "sub_weight_grad_rows", "x_grad"]
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in out.values())
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    rows = out["sub_weight_grad_rows"]
    assert out["x_grad"].shape == (512, 512) and out["sub_weight_grad"].shape == (len(rows), 512) and len(rows) == 8192
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < 100_000 and float(out["loss"]) > 0
