"""CPU: the oracle restatements are pinned against the EXECUTED reference source.  oracle/make_golden.py runs the
reference's own files (made importable by oracle/build_ref.py with documented line-anchored py2->py3 patches) on seeded
inputs, checks that the restatement agrees bit-for-bit there, and stores the inputs and the reference's results under
tests/golden/; these tests run the restatement on the stored inputs and compare:

  * loss: values, hard-negative counts and autograd gradients of PixelwiseContrastiveLoss.* and loss_composer.*
    (dense_correspondence/loss_functions/pixelwise_contrastive_loss.py:35-411, loss_composer.py:7-218)
  * non-match sampler: create_non_correspondences + create_non_matches + flatten_uv_tensor
    (correspondence_tools/correspondence_finder.py:276-405, dataset/spartan_dataset_masked.py:841-858,1255-1264)
  * reprojection match finder: batch_find_pixel_correspondences (correspondence_finder.py:409-619)

Integer results must be equal.  Floating-point results are compared to 1e-5 relative: the stored values were computed
on one CPU, and torch may vectorise a sum differently on another."""
import os

import numpy as np
import pytest
import torch

from oracle import loss_oracle as LO
from oracle import ref_cases

RTOL, ATOL = 1e-5, 1e-8


def _golden(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=True)


def same(x, y, what="result"):
    """x (the restatement's result) equals y (the reference's stored result)."""
    if isinstance(x, torch.Tensor):
        assert isinstance(y, torch.Tensor) and x.shape == y.shape and x.dtype == y.dtype, what
        if x.is_floating_point():
            torch.testing.assert_close(x, y, rtol=RTOL, atol=ATOL, msg=what)
        else:
            assert torch.equal(x, y), what
    elif isinstance(x, (tuple, list)):
        assert isinstance(y, (tuple, list)) and len(x) == len(y), what
        for i, (a, b) in enumerate(zip(x, y)):
            same(a, b, "%s[%d]" % (what, i))
    elif isinstance(x, dict):
        assert sorted(x) == sorted(y), what
        for k in x:
            same(x[k], y[k], "%s/%s" % (what, k))
    elif isinstance(x, float):
        assert x == pytest.approx(y, rel=RTOL, abs=ATOL), what
    else:
        assert x == y, what


def _golden_case(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    cfg = dict(LO.DEFAULT_LOSS_CONFIG)
    for k, v in zip(g["cfg_keys"], g["cfg_vals"]):
        k = str(k)
        cfg[k] = bool(v) if isinstance(LO.DEFAULT_LOSS_CONFIG[k], bool) else float(v)
    idx = {k: torch.tensor(g[k]) for k in ("matches_a", "matches_b", "masked_a", "masked_b", "background_a", "background_b",
                                           "blind_a", "blind_b")}
    return g, cfg, idx


@pytest.mark.parametrize("name", ["loss_default_d3", "loss_pixelw_blind_d8", "loss_noscale_d16"])
def test_composed_loss_restatement_equals_executed_reference(golden_dir, name):
    g, cfg, idx = _golden_case(golden_dir, name)
    A, B = torch.tensor(g["A"]), torch.tensor(g["B"])
    _, D, H, W = A.shape
    five_o, dA_o, dB_o = ref_cases.run_get_loss(LO.TorchPixelwiseContrastiveLoss([H, W], dict(cfg)), LO.get_loss, A, B, idx)
    np.testing.assert_allclose(five_o, g["five"], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(dA_o.numpy(), g["dA"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(dB_o.numpy(), g["dB"], rtol=RTOL, atol=ATOL)


def test_every_loss_method_equals_executed_reference(golden_dir):
    g = _golden(golden_dir, "ref_loss_methods")
    same(ref_cases.loss_methods(LO.TorchPixelwiseContrastiveLoss, g["inputs"]), g["outputs"], "loss methods")


def test_composer_branches_equal_executed_reference(golden_dir):
    g = _golden(golden_dir, "ref_composer_branches")
    ref = dict(g["outputs"])
    empty, data_types = ref.pop("empty_tensor"), ref.pop("data_types")
    out = ref_cases.composer_branches(LO.TorchPixelwiseContrastiveLoss, LO.get_loss, LO.empty_tensor, g["inputs"])
    same(out, ref, "composer")
    # blind sentinel [-1]: not entered; across-scene: the reference's own NameError; unknown type: ValueError
    assert out["empty_blind"][4] == 0.0
    assert out["raises/type1"] in ("NameError", "UnboundLocalError") and out["raises/type9"] == "ValueError"
    assert torch.equal(LO.empty_tensor(), empty)
    T = LO.SpartanDatasetDataType
    assert data_types and all(getattr(T, k) == v for k, v in data_types.items())


def test_non_match_sampler_restatement_equals_executed_reference(golden_dir):
    """The reference draws its uniforms from torch.rand; the restatement takes them as arguments.  The stored results
    are the reference's for the stored uniforms, with an object mask, without one, and with an empty one."""
    g = _golden(golden_dir, "ref_non_match_sampler")
    i = g["inputs"]
    H, W = i["H"], i["W"]
    for m, (na_r, nb_r) in zip(i["masks"], g["outputs"]):
        na_o, nb_o = LO.create_non_correspondences_flat(i["matches_a"], (H, W), i["k"], m, i["rand_u"], i["rand_v"])
        assert torch.equal(na_o, na_r) and torch.equal(nb_o, nb_r)
        if m is not None and bool(m.any()):
            assert bool((m.view(-1)[nb_r] == 1).all())


def test_reprojection_restatement_equals_executed_reference(golden_dir):
    """A rendered tilted plane with no-return pixels (depth 0) in image a and an occluder in image b."""
    g = _golden(golden_dir, "ref_reprojection")
    i = g["inputs"]
    da, db = i["depth_a"].numpy().astype(np.uint16), i["depth_b"].numpy().astype(np.uint16)
    pa, pb, K, mask, ru = i["pose_a"].numpy(), i["pose_b"].numpy(), i["K"].numpy(), i["mask_a"], i["rand"]
    n = len(ru)
    # the candidates random_sample_from_masked_image_torch drew (correspondence_finder.py:92-121)
    nz = torch.nonzero(mask.view(-1))
    cand = torch.index_select(nz, 0, torch.floor(ru * len(nz)).long()).squeeze(1)
    uv_a_o, uv_b_o = LO.batch_find_pixel_correspondences(da, pa, db, pb, cand, K)
    uv_a_r = g["outputs"][0]
    assert len(uv_a_r) > 0.3 * n and len(uv_a_r) < n                   # some pruned by every rule
    same(list(uv_a_o) + list(uv_b_o), g["outputs"], "reprojection")
