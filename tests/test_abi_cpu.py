"""CPU: libddn_b200.so loads without a GPU, exports every function include/ddn_b200.h declares, describes the
parameter layout of the reference state dict, and rejects contract violations before touching the device."""
import ctypes
import os
import re

import pytest
import torch

import pdc_b200
from pdc_b200 import _native as N
from oracle.resnet34_8s_oracle import seeded_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "ddn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ddn_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    names = _declared_functions()
    assert len(names) >= 20
    lib = ctypes.CDLL(N.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "declared in ddn_b200.h but not exported: " + n
    assert set(names) == set(N.EXPORTED_SYMBOLS), set(names) ^ set(N.EXPORTED_SYMBOLS)
    assert N.lib.ddn_abi_version() == 3


@pytest.mark.parametrize("D", [3, 8, 16])
def test_param_table_is_reference_state_dict(D):
    sd = seeded_oracle(D).state_dict()
    learn = [(k, tuple(v.shape)) for k, v in seeded_oracle(D).named_parameters()]
    tab = N.param_table(D)
    assert [("resnet34_8s." + n, s) for n, s, _, _ in tab] == learn
    assert len(tab) == 110
    # offsets: in order, non-overlapping, 16-byte aligned
    end = 0
    for _, s, off, n in tab:
        assert off >= end and off % 4 == 0
        end = off + n
    assert N.lib.ddn_resnet34_8s_param_count(D) >= end
    assert sum(n for _, _, _, n in tab) == sum(v.numel() for k, v in seeded_oracle(D).named_parameters())
    btab = N.buffer_table()
    assert len(btab) == 72
    for name, shape, _, _ in btab:
        assert tuple(sd["resnet34_8s." + name].shape) == shape
    m = pdc_b200.Resnet34_8s(num_classes=D)
    assert list(m.state_dict().keys()) == list(sd.keys()) and len(sd) == 218
    m.load_state_dict(sd)
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    # every parameter aliases the flat array at the advertised offset
    for (name, shape, off, n), p in zip(tab, m._params):
        assert p.data_ptr() == m._flat.data_ptr() + 4 * off


def test_workspace_and_argument_checks():
    wb = N.lib.ddn_resnet34_8s_workspace_bytes(1, 480, 640, 3, 1, N.PRECISION_FP32_SIMT)
    assert 3e8 < wb < 2e9
    assert N.lib.ddn_resnet34_8s_workspace_bytes(2, 480, 640, 3, 1, 0) > 1.9 * wb - 5e7
    assert N.lib.ddn_resnet34_8s_workspace_bytes(1, 481, 640, 3, 1, 0) == 0          # H not a multiple of 8
    assert N.lib.ddn_resnet34_8s_workspace_bytes(1, 480, 640, 33, 1, 0) == 0         # D out of range
    assert b"multiple" in N.lib.ddn_last_error() or b"dimension" in N.lib.ddn_last_error()
    # null pointers / bad sizes are refused with DDN_EINVAL and never reach a kernel launch
    before = N.launch_count()
    assert N.lib.ddn_resnet34_8s_forward(None, None, None, None, None, 0, 1, 480, 640, 3, 1, 1, 0.1, 1e-5, 0, None, None) == -1
    assert N.lib.ddn_contrastive_terms_forward(None, None, 0, 0, 0, 1, 10, 3, 4, None, 0, None, None, None) == -1
    assert N.lib.ddn_upsample_bilinear_forward(None, None, 1, 1, 1, 1, 1, None) == -1
    assert N.lib.ddn_conv2d_workspace_bytes(1, 60, 80, 64, 64, 3, 1, 1, 1, 0) >= 3 * 9 * 64 * 64 * 4
    assert N.lib.ddn_batchnorm_workspace_bytes(4800, 6) == 0 and N.lib.ddn_batchnorm_workspace_bytes(4800, 512) > 0
    assert N.launch_count() == before
    with pytest.raises(N.DdnError):
        N.check(-1)


def test_product_refuses_cpu_tensors():
    m = pdc_b200.Resnet34_8s(num_classes=3)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 3, 64, 64))
    pcl = pdc_b200.PixelwiseContrastiveLoss([8, 8], {"M_pixel": 50})
    with pytest.raises(RuntimeError, match="CUDA"):
        pcl.match_loss(torch.zeros(1, 64, 3), torch.zeros(1, 64, 3), torch.tensor([1]), torch.tensor([2]))
    with pytest.raises(ValueError):
        pdc_b200.DenseCorrespondenceNetwork.get_fcn({"backbone": {"model_class": "Resnet", "resnet_name": "Resnet101_8s"},
                                                     "descriptor_dimension": 3})
    with pytest.raises(ValueError):
        pdc_b200.DenseCorrespondenceNetwork.get_fcn({"backbone": {"model_class": "Foo"}, "descriptor_dimension": 3})


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "pytorch-dense-correspondence_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "oracle/" not in text, f
