"""Loss-code cases that tests/test_oracle_ref_cpu.py checks the oracle restatement on, shared with oracle/make_golden.py.

make_golden.py runs each case on the executed reference source (oracle/build_ref.py) and stores the inputs and the
results under tests/golden/; the test runs the same case on the restatement (oracle/loss_oracle.py) with the stored
inputs and compares.  A case takes the implementation's PixelwiseContrastiveLoss class (and get_loss) plus the inputs and
returns a dict of results: tensors, numbers and tuples / lists of them.
"""
import torch

from oracle import loss_oracle as LO
from oracle.resnet34_8s_oracle import process_network_output


def run_get_loss(pcl, get_loss, A, B, idx, match_type=0):
    """get_loss on [1,D,H,W] descriptor maps -> (five loss values as floats, dloss/dA, dloss/dB)."""
    A = A.clone().requires_grad_(); B = B.clone().requires_grad_()
    _, D, H, W = A.shape
    pa = process_network_output(A, 1, D, H, W); pb = process_network_output(B, 1, D, H, W)
    five = get_loss(pcl, torch.tensor([match_type]), pa, pb, idx["matches_a"], idx["matches_b"], idx["masked_a"], idx["masked_b"],
                    idx["background_a"], idx["background_b"], idx["blind_a"], idx["blind_b"])
    five[0].reshape(()).backward()
    return [float(t) for t in five], A.grad, B.grad


def loss_methods(pcl_cls, inp):
    """Every method of PixelwiseContrastiveLoss, including its single-index and zero-distance branches."""
    A, B, ma, mb, na, nb = (inp[k] for k in ("A", "B", "ma", "mb", "na", "nb"))
    p = pcl_cls([inp["H"], inp["W"]], dict(LO.DEFAULT_LOSS_CONFIG, M_descriptor=0.6))
    out = {"match_loss": p.match_loss(A, B, ma, mb)}
    for inv in (False, True):
        out["non_match_descriptor_loss/invert=%s" % inv] = p.non_match_descriptor_loss(A, B, na, nb, M=0.6, invert=inv)
        out["non_match_loss_descriptor_only/invert=%s" % inv] = p.non_match_loss_descriptor_only(A, B, na, nb, M_descriptor=0.6,
                                                                                                 invert=inv)
    out["non_match_loss_with_l2_pixel_norm"] = p.non_match_loss_with_l2_pixel_norm(A, B, mb, na, nb, M_descriptor=0.6, M_pixel=7)
    out["l2_pixel_loss"] = p.l2_pixel_loss(mb, nb, M_pixel=7)
    out["flattened_pixel_locations_to_u_v"] = p.flattened_pixel_locations_to_u_v(nb.unsqueeze(1))
    for l2 in (False, True):
        out["get_loss_matched_and_non_matched_with_l2/l2=%s" % l2] = p.get_loss_matched_and_non_matched_with_l2(
            A, B, ma, mb, na, nb, use_l2_pixel_loss=l2)
    out["get_triplet_loss"] = p.get_triplet_loss(A, B, ma, mb, na, nb, 0.1)
    out["get_loss_original"] = p.get_loss_original(A, B, ma, mb, na, nb)
    # single-element index tensors (the unsqueeze branch, pcl.py:161-163,199-201) and identical descriptors (d = 0)
    one, two = torch.tensor([7]), torch.tensor([11])
    out["match_loss/one"] = p.match_loss(A, B, one, two)
    out["non_match_descriptor_loss/one"] = p.non_match_descriptor_loss(A, B, one, two, M=100.0)
    Z = torch.zeros_like(A)
    out["non_match_loss_descriptor_only/zero"] = p.non_match_loss_descriptor_only(Z, Z, na, nb, M_descriptor=0.5)
    return out


# configuration overrides x match types of the composer case; the last override leaves zero hard negatives -> max(h, 1)
COMPOSER_OVERRIDES = ({}, {"scale_by_hard_negatives": False}, {"scale_by_hard_negatives_DIFFERENT_OBJECT": False},
                      {"M_masked": 1e-6, "M_background": 1e-6})
COMPOSER_MATCH_TYPES = (0, 2, 3, 4)          # within-scene, different-object, multi-object, synthetic multi-object


def composer_branches(pcl_cls, get_loss, empty_tensor, inp):
    """loss_composer.get_loss over COMPOSER_OVERRIDES x COMPOSER_MATCH_TYPES, the empty blind sentinel, and the names of the
    exceptions raised for the across-scene type (the reference's own NameError) and for an unknown type."""
    A, B, idx = inp["A"], inp["B"], inp["idx"]
    H, W = A.shape[2:]
    out = {}
    for i, over in enumerate(COMPOSER_OVERRIDES):
        cfg = dict(LO.DEFAULT_LOSS_CONFIG); cfg.update(over)
        for mt in COMPOSER_MATCH_TYPES:
            out["cfg%d/type%d" % (i, mt)] = run_get_loss(pcl_cls([H, W], dict(cfg)), get_loss, A, B, idx, mt)
    cfg = dict(LO.DEFAULT_LOSS_CONFIG)
    idx_e = dict(idx, blind_a=empty_tensor(), blind_b=empty_tensor())
    out["empty_blind"] = run_get_loss(pcl_cls([H, W], dict(cfg)), get_loss, A, B, idx_e, 0)[0]
    for mt in (1, 9):
        try:
            run_get_loss(pcl_cls([H, W], dict(cfg)), get_loss, A, B, idx, mt)
            out["raises/type%d" % mt] = None
        except Exception as e:       # the class name is the result
            out["raises/type%d" % mt] = type(e).__name__
    return out
