"""bench.py --dump-outputs (GPU): the last timed training step's loss and parameters as float32 .npy files, the same
arrays from a second run with the same arguments (seeded inputs, deterministic kernels), and other arrays when --steps
adds a timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "0", "--no-extras",
           "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {n: np.load(os.path.join(out_dir, n)) for n in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
@pytest.mark.timeout(1800)
def test_dump_outputs_are_the_timed_step_and_repeat(tmp_path):
    import bench
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    a = _bench(tmp_path / "a", steps=2)
    params = dict(GraphSAGEModel(10, bench.HIDDEN, 1, bench.LAYERS).named_parameters())
    assert sorted(a) == sorted(["loss.npy"] + [f"param.{k}.npy" for k in params])
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for n, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), n
        if n != "loss.npy":
            assert v.shape == tuple(params[n[len("param."):-len(".npy")]].shape), n
    assert a["loss.npy"].shape == (1,) and a["loss.npy"][0] > 0
    b = _bench(tmp_path / "b", steps=2)
    for n, v in a.items():
        assert np.array_equal(b[n], v), n
    # the state before the timed region is the same for both step counts: the arrays differ only if they were taken after
    # the timed steps, and a third timed step really ran
    c = _bench(tmp_path / "c", steps=3)
    assert sorted(c) == sorted(a)
    assert not np.array_equal(c["loss.npy"], a["loss.npy"])
    assert all(not np.array_equal(c[n], a[n]) for n in a if n.startswith("param.") and n.endswith(".weight.npy"))
