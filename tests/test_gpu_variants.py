"""Environment knobs that select another kernel or schedule (read once per process) must stay correct: the conv /
update-block / encoder parity tests are re-run in a subprocess with each knob set."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernel_parity(env):
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_kernels.py"), "-q", "-x",
                        "-k", "(conv2d or update_block or encoder) and tc", "--timeout", "300", "-p", "no:cacheprovider"],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-1000:]


@pytest.mark.parametrize("knob", ["RAFT_B200_NO_HOIST", "RAFT_B200_NO_STASH", "RAFT_B200_NO_PDL", "RAFT_B200_NO_SPLITK",
                                  "RAFT_B200_NO_SPLITK_CLUSTER"])
def test_variant_passes_conv_and_update_parity(cuda, knob):
    _kernel_parity(dict(os.environ, **{knob: "1"}))


def test_warp_per_pixel_lookup_kernel_bit_exact(cuda):
    """RAFT_B200_LOOKUP_V5=1 selects the warp-per-pixel lookup kernel (the one the volume-free path instantiates) for the
    materialised volume: same bit-exact results."""
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_kernels.py"), "-q", "-x",
                        "-k", "lookup", "--timeout", "300", "-p", "no:cacheprovider"],
                       env=dict(os.environ, RAFT_B200_LOOKUP_V5="1"), cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-1000:]
