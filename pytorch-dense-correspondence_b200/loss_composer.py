"""loss_composer -- same functions and 5-tuples as the reference's
dense_correspondence/loss_functions/loss_composer.py, evaluated without host synchronisation.

``get_loss`` (reference :7-67) is what ``DenseCorrespondenceTraining.run`` calls every step
(dense_correspondence/training/training.py:336-342).  For the within-scene pair types it runs ONE
gather/hinge/reduce kernel over all terms, ONE compose kernel that applies the hard-negative scaling of
loss_composer.py:107-141 on the device, and the backward is ONE scatter kernel.

Batch extension (the reference is batch-1 only, training.py:314-323): descriptor images may be
``[B, W*H, D]`` with ``[B, n]`` index tensors; the loss is then the mean over the B pairs of the reference's
per-pair loss (SURVEY.md 8a).
"""
import torch

from . import _native as N
from .contrastive_ops import Term, within_scene_loss, contrastive_terms
from .resnet_dilated import lowres_of


def _fused_lowres(image_a_pred, image_b_pred, image_width):
    """When both descriptor images are untouched outputs of Resnet34_8s (they carry the low-resolution map they were upsampled
    from), the loss is evaluated THROUGH the upsample: (low_a, low_b, (h, w, H, W)), else None (the generic gather from the
    full-resolution images)."""
    ta, tb = lowres_of(image_a_pred), lowres_of(image_b_pred)
    if ta is None or tb is None or ta[1:3] != tb[1:3] or ta[2] != image_width or ta[0].shape != tb[0].shape:
        return None
    H, W = ta[1], ta[2]
    if ta[0].dim() != 3 or ta[0].shape[1] != (H // 8) * (W // 8) or image_a_pred.shape[-2] != H * W:
        return None
    return ta[0], tb[0], (H // 8, W // 8, H, W)


class SpartanDatasetDataType:
    """dense_correspondence/dataset/spartan_dataset_masked.py:31-36."""
    SINGLE_OBJECT_WITHIN_SCENE = 0
    SINGLE_OBJECT_ACROSS_SCENE = 1
    DIFFERENT_OBJECT = 2
    MULTI_OBJECT = 3
    SYNTHETIC_MULTI_OBJECT = 4


def empty_tensor():
    """DenseCorrespondenceDataset.empty_tensor (dataset/dense_correspondence_dataset_masked.py:209-216)."""
    return torch.LongTensor([-1])


def is_empty(tensor):
    """DenseCorrespondenceDataset.is_empty (:218-223).  NB: on a CUDA tensor of length 1 this reads the value
    back (a sync) -- the fused within-scene path below never calls it."""
    return (len(tensor) == 1) and bool(tensor[0] == -1)


def pad_index_lists(lists, device=None, pad=-1):
    """Per-pair index lists of DIFFERENT lengths (what SpartanDataset really returns: num_matching_attempts is only an upper
    bound on the matches found, dataset/spartan_dataset_masked.py:652-660) -> (``[B, n_max]`` int64 padded with -1, ``[B]``
    int64 true lengths) for the ``num_valid`` argument of ``get_loss`` / ``get_within_scene_loss``."""
    B = len(lists)
    n_max = max(1, max(int(t.numel()) for t in lists))
    dev = device if device is not None else lists[0].device
    out = torch.full((B, n_max), pad, dtype=torch.int64, device=dev)
    lens = torch.empty(B, dtype=torch.int64)
    for i, t in enumerate(lists):
        t = t.reshape(-1)
        out[i, :t.numel()] = t.to(dev)
        lens[i] = t.numel()
    return out, lens.to(dev)


def get_loss(pixelwise_contrastive_loss, match_type,
             image_a_pred, image_b_pred,
             matches_a, matches_b,
             masked_non_matches_a, masked_non_matches_b,
             background_non_matches_a, background_non_matches_b,
             blind_non_matches_a, blind_non_matches_b, num_valid=None):
    """loss_composer.py:7-67 -> (loss, match_loss, masked_non_match_loss, background_non_match_loss,
    blind_non_match_loss).  ``num_valid`` (batch extension, optional): dict of ``[B]`` int64 CUDA tensors with the true
    per-pair counts of ``"matches"``, ``"masked"``, ``"background"`` (and ``"blind"``) when the ``[B, n_max]`` index tensors
    are padded with -1 (see ``pad_index_lists``)."""
    T = SpartanDatasetDataType
    mt = torch.as_tensor(match_type)
    if mt.is_cuda:
        mt = mt.cpu()
    within = (T.SINGLE_OBJECT_WITHIN_SCENE, T.MULTI_OBJECT, T.SYNTHETIC_MULTI_OBJECT)
    if any(bool((mt == k).all()) for k in within):
        return get_within_scene_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                                     matches_a, matches_b,
                                     masked_non_matches_a, masked_non_matches_b,
                                     background_non_matches_a, background_non_matches_b,
                                     blind_non_matches_a, blind_non_matches_b, num_valid=num_valid)
    if bool((mt == T.SINGLE_OBJECT_ACROSS_SCENE).all()):
        return get_same_object_across_scene_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                                                 blind_non_matches_a, blind_non_matches_b)
    if bool((mt == T.DIFFERENT_OBJECT).all()):
        return get_different_object_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                                         blind_non_matches_a, blind_non_matches_b)
    raise ValueError("Should only have above scenes?")


def get_within_scene_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                          matches_a, matches_b,
                          masked_non_matches_a, masked_non_matches_b,
                          background_non_matches_a, background_non_matches_b,
                          blind_non_matches_a, blind_non_matches_b, num_valid=None):
    """loss_composer.py:70-143.

    The ``[-1]`` sentinel for "no blind non-matches" needs no host-side test here: index -1 is skipped by
    the kernel, giving sum 0 / count 0, and max(count, 1) = 1 reproduces the reference's
    ``zero_loss()`` / ``num_blind_hard_negatives = 1`` branch exactly (loss_composer.py:99-105)."""
    pcl = pixelwise_contrastive_loss
    cfg = pcl._config
    gt_m = matches_b if cfg["use_l2_pixel_loss_on_masked_non_matches"] else None
    gt_b = matches_b if cfg["use_l2_pixel_loss_on_background_non_matches"] else None
    nv = num_valid or {}
    terms = [
        Term(matches_a, matches_b, N.TERM_MATCH, lengths=nv.get("matches")),
        Term(masked_non_matches_a, masked_non_matches_b, N.TERM_HINGE, cfg["M_masked"], gt_b=gt_m,
             m_pixel=cfg["M_pixel"], lengths=nv.get("masked"), gt_lengths=nv.get("matches")),
        Term(background_non_matches_a, background_non_matches_b, N.TERM_HINGE, cfg["M_background"], gt_b=gt_b,
             m_pixel=cfg["M_pixel"], lengths=nv.get("background"), gt_lengths=nv.get("matches")),
    ]
    has_blind = blind_non_matches_a is not None
    if has_blind:
        terms.append(Term(blind_non_matches_a, blind_non_matches_b, N.TERM_HINGE, cfg["M_masked"], lengths=nv.get("blind")))
    lengths = (nv.get("matches"), nv.get("masked"), nv.get("background"), nv.get("blind")) if num_valid else None
    loss, rest, counts = within_scene_loss(image_a_pred, image_b_pred, pcl.image_width, terms,
                                           cfg["match_loss_weight"], cfg["non_match_loss_weight"],
                                           cfg["scale_by_hard_negatives"], has_blind, lengths=lengths,
                                           lowres=_fused_lowres(image_a_pred, image_b_pred, pcl.image_width))
    if pcl.debug:
        pcl.debug_data["num_hard_negatives_device"] = counts
    return loss, rest[0:1], rest[1:2], rest[2:3], rest[3:4]


def get_within_scene_loss_triplet(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                                  matches_a, matches_b,
                                  masked_non_matches_a, masked_non_matches_b,
                                  background_non_matches_a, background_non_matches_b,
                                  blind_non_matches_a, blind_non_matches_b):
    """loss_composer.py:145-166 (not reachable from get_loss)."""
    pcl = pixelwise_contrastive_loss
    masked = pcl.get_triplet_loss(image_a_pred, image_b_pred, matches_a, matches_b, masked_non_matches_a,
                                  masked_non_matches_b, pcl._config["alpha_triplet"])
    background = pcl.get_triplet_loss(image_a_pred, image_b_pred, matches_a, matches_b, background_non_matches_a,
                                      background_non_matches_b, pcl._config["alpha_triplet"])
    z = zero_loss(image_a_pred.device)
    return masked + background, z, z.clone(), z.clone(), z.clone()


def get_different_object_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                              blind_non_matches_a, blind_non_matches_b):
    """loss_composer.py:168-191: blind non-matches only, margin M_background, scaled by #hard negatives (kept on the
    device) or by their number."""
    pcl = pixelwise_contrastive_loss
    z = zero_loss(image_a_pred.device)
    if blind_non_matches_a.numel() == 1 and is_empty(blind_non_matches_a.reshape(-1)):
        return z, z.clone(), z.clone(), z.clone(), z.clone()
    sums, counts = contrastive_terms(image_a_pred, image_b_pred, pcl.image_width,
                                     [Term(blind_non_matches_a, blind_non_matches_b, N.TERM_HINGE,
                                           pcl.config["M_background"])])
    if pcl.config["scale_by_hard_negatives_DIFFERENT_OBJECT"]:
        scale = counts[:, 0].clamp(min=1).to(torch.float64)
    else:
        scale = float(max(blind_non_matches_a.shape[-1], 1))
    blind = (sums[:, 0] / scale).mean().to(torch.float32).reshape(1)
    return blind, z, z.clone(), z.clone(), blind


def get_same_object_across_scene_loss(pixelwise_contrastive_loss, image_a_pred, image_b_pred,
                                      blind_non_matches_a, blind_non_matches_b):
    """loss_composer.py:193-212.  Upstream this branch cannot run: it reads an undefined global ``pcl`` (:203) when
    the blind set is non-empty and an unbound ``num_hard_negatives`` (:205-206) when it is empty.  The same two
    exceptions are raised here rather than inventing semantics the reference never had."""
    if not (blind_non_matches_a.numel() == 1 and is_empty(blind_non_matches_a.reshape(-1))):
        raise NameError("name 'pcl' is not defined")
    raise UnboundLocalError("local variable 'num_hard_negatives' referenced before assignment")


def zero_loss(device="cuda"):
    """loss_composer.py:214-215."""
    return torch.zeros(1, dtype=torch.float32, device=device)


def is_zero_loss(loss):
    """loss_composer.py:217-218."""
    return loss.item() < 1e-20
