"""The tensor-core linear has two kernels behind one entry point: the persistent one (default) and the classic one-tile-per-CTA
kernel (shapes the persistent kernel does not take; DFW_TC_PERSIST=0 forces it); DFW_FORCE_SIMT=1 sends every linear to the
SIMT kernels.  The environment switches are read once per process, so the linear
parity tests, the element-wise bounds of test_gpu_linear_bounds.py and the layer replay of test_gpu_layer_replay.py are
re-run in a subprocess per variant."""
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DFW_TC_PERSIST": "0"}, {"DFW_FORCE_SIMT": "1"}], ids=["classic", "simt"])
def test_linear_parity_suite_on_kernel_variant(env):
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(REPO, "tests", "test_gpu_kernels.py"),
                        os.path.join(REPO, "tests", "test_gpu_linear_bounds.py"), "-m", "gpu", "-q", "-x", "-k", "linear or mlp or sage_layer",
                        "-p", "no:cacheprovider"], cwd=REPO, env=e, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DFW_TC_PERSIST": "0"}, {"DFW_FORCE_SIMT": "1"}], ids=["classic", "simt"])
def test_layer_replay_on_kernel_variant(env):
    """The per-stage replay of the model and the one-call entry points (test_gpu_layer_replay.py) on the same variants."""
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(REPO, "tests", "test_gpu_layer_replay.py"), "-m", "gpu", "-q", "-x",
                        "-p", "no:cacheprovider"], cwd=REPO, env=e, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
