"""Parity of the alternative tensor-core kernels that the library's switches select (DESIGN.md compares against them):

    DDN_TC_PAIR=0   single-CTA conv_tc_kernel everywhere, no CTA pairs (tcgen05.mma.cta_group::2) for the 256-channel layers
    DDN_TC_TAIL=0   no N-split of the tiles of the last, partial wave
    DDN_TC_HALO=0   layer 1 through conv_tc_kernel / wgrad_tc_kernel instead of the halo-tile kernels

The library reads each switch once per process, so every setting runs the tensor-core operator cases, the whole-network
gradient and inference matrix and the fused-loss steps in a SUBPROCESS, under a hard timeout so that a hang cannot take the
machine with it.  The fp32 CUDA-core parametrizations are deselected: the switches do not reach them.
"""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUITES = ["tests/test_gpu_ops.py::test_conv2d_tcgen05",
          "tests/test_gpu_network.py::test_whole_network_gradients_over_shapes_descriptor_sizes_and_groups",
          "tests/test_gpu_network.py::test_inference_forward_over_shapes_descriptor_sizes_and_groups",
          "tests/test_gpu_network.py::test_fused_loss_step_at_the_shape_matrix"]


@pytest.mark.parametrize("switch", ["DDN_TC_PAIR", "DDN_TC_TAIL", "DDN_TC_HALO"])
def test_alternative_kernels_pass_the_parity_suites(switch):
    env = dict(os.environ, **{switch: "0"})
    cmd = ["timeout", "600", sys.executable, "-m", "pytest", *SUITES, "-m", "gpu", "-k", "not fp32", "-x", "-q", "-p", "no:cacheprovider"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, "%s=0: rc=%d (124 = hang)\n%s\n%s" % (switch, r.returncode, r.stdout[-3000:], r.stderr[-2000:])
