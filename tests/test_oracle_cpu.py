"""CPU: the oracle reproduces the committed golden vectors (which were written from the REAL reference by
oracle/make_golden.py), the numpy and torch loss restatements agree, and the oracle equals the reference modules on the
inputs stored with their outputs."""
import os

import numpy as np
import pytest
import torch

from oracle import loss_oracle as LO
from oracle import well_conditioned as WC
from oracle.resnet34_8s_oracle import GOLDEN_CPU_THREADS, seeded_oracle, process_network_output
import pdc_b200
from pdc_b200 import synthetic


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name,D,B,H,W", [("backbone_small_d3", 3, 2, 64, 96), ("backbone_small_d16", 16, 1, 48, 64)])
def test_backbone_oracle_matches_golden(golden_dir, golden_threads, name, D, B, H, W):
    g = _load(golden_dir, name)
    net = seeded_oracle(D=D, seed=0)
    x = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(int(g["x_seed"])))
    net.train()
    y = net(x)
    # same torch build -> bit equal; a different CPU/torch build may reorder fp32 sums
    np.testing.assert_allclose(y.detach().numpy(), g["y_train"], rtol=1e-4, atol=1e-5)
    sd = net.state_dict()
    for k in g.files:
        if k.startswith("rs:"):
            np.testing.assert_allclose(sd[k[3:]].numpy(), g[k], rtol=1e-4, atol=1e-6)
    # the golden cotangent is drawn right after x from the same generator
    gen = torch.Generator().manual_seed(int(g["x_seed"]))
    _ = torch.randn(B, 3, H, W, generator=gen)
    cot = torch.randn(y.shape, generator=gen)
    (y * cot).sum().backward()
    params = dict(net.named_parameters())
    for k in g.files:
        if k.startswith("grad:"):
            ref = g[k]
            got = params[k[5:]].grad.numpy()
            assert np.linalg.norm(got - ref) <= 2e-3 * np.linalg.norm(ref) + 1e-7, k
    net.eval()
    with torch.no_grad():
        ye = net(x)
    np.testing.assert_allclose(ye.numpy(), g["y_eval"], rtol=1e-4, atol=1e-5)


def _loss_inputs(g):
    A = torch.tensor(g["A"]).requires_grad_()
    B = torch.tensor(g["B"]).requires_grad_()
    idx = {k: torch.tensor(g[k]) for k in ("matches_a", "matches_b", "masked_a", "masked_b", "background_a",
                                           "background_b", "blind_a", "blind_b")}
    cfg = dict(LO.DEFAULT_LOSS_CONFIG)
    for k, v in zip(g["cfg_keys"], g["cfg_vals"]):
        k = str(k)
        cfg[k] = bool(v) if isinstance(LO.DEFAULT_LOSS_CONFIG[k], bool) else float(v)
    return A, B, idx, cfg


@pytest.mark.parametrize("name", ["loss_default_d3", "loss_pixelw_blind_d8", "loss_noscale_d16"])
def test_loss_oracles_match_golden(golden_dir, name):
    g = _load(golden_dir, name)
    A, B, idx, cfg = _loss_inputs(g)
    _, D, H, W = A.shape
    pcl = LO.TorchPixelwiseContrastiveLoss([H, W], cfg)
    pa = process_network_output(A, 1, D, H, W); pb = process_network_output(B, 1, D, H, W)
    five = LO.get_loss(pcl, torch.tensor([0]), pa, pb, idx["matches_a"], idx["matches_b"], idx["masked_a"],
                       idx["masked_b"], idx["background_a"], idx["background_b"], idx["blind_a"], idx["blind_b"])
    np.testing.assert_allclose([float(t) for t in five], g["five"], rtol=1e-6, atol=1e-8)
    five[0].reshape(()).backward()
    np.testing.assert_allclose(A.grad.numpy(), g["dA"], rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(B.grad.numpy(), g["dB"], rtol=1e-5, atol=1e-8)
    An = g["A"][0].reshape(D, H * W).T; Bn = g["B"][0].reshape(D, H * W).T
    five_np, counts = LO.np_within_scene_loss(An, Bn, {k: v.numpy() for k, v in idx.items()}, cfg, W)
    np.testing.assert_allclose(five_np, g["five"], rtol=1e-6, atol=1e-8)
    assert tuple(counts) == tuple(int(c) for c in g["counts"])


def test_loss_oracle_edge_cases():
    H, W, D = 8, 10, 3
    g = torch.Generator().manual_seed(5)
    A = torch.randn(1, H * W, D, generator=g); B = torch.randn(1, H * W, D, generator=g)
    pcl = LO.TorchPixelwiseContrastiveLoss([H, W], dict(LO.DEFAULT_LOSS_CONFIG))
    one = torch.tensor([7]); two = torch.tensor([11])
    # single-element index tensors take the unsqueeze branch (pcl.py:161-163,199-201)
    ml, a, b = pcl.match_loss(A, B, one, two)
    assert abs(float(ml) - float(((A[0, 7] - B[0, 11]) ** 2).sum())) < 1e-6
    vec, hard, _, _ = pcl.non_match_descriptor_loss(A, B, one, two, M=100.0)
    assert hard == 1 and vec.shape == (1,)
    # identical descriptors: d = 0 -> hinge = M^2, counted as hard, zero gradient from the norm
    Az = torch.zeros(1, H * W, D, requires_grad=True); Bz = torch.zeros(1, H * W, D)
    s, hard = pcl.non_match_loss_descriptor_only(Az, Bz, torch.tensor([1, 2]), torch.tensor([3, 4]), M_descriptor=0.5)
    assert hard == 2 and abs(float(s) - 0.5) < 1e-7
    s.backward()
    assert float(Az.grad.abs().sum()) == 0.0
    # sentinel handling + unknown pair type
    assert LO.is_empty(LO.empty_tensor()) and not LO.is_empty(torch.tensor([3]))
    with pytest.raises(ValueError):
        LO.get_loss(pcl, torch.tensor([9]), A, B, one, two, one, two, one, two, one, two)
    with pytest.raises((NameError, UnboundLocalError)):
        LO.get_loss(pcl, torch.tensor([1]), A, B, one, two, one, two, one, two, one, two)


def test_train_step_oracle_matches_golden(golden_dir, golden_threads):
    g = _load(golden_dir, "train_step_small_d3")
    D, B, H, W = 3, 2, 64, 96
    net = seeded_oracle(D=D, seed=0).train()
    data = synthetic.make_pair_batch(B, H, W, 40, 120, 120, 0, seed=int(g["seed"]))
    pcl = LO.TorchPixelwiseContrastiveLoss([H, W], dict(LO.DEFAULT_LOSS_CONFIG))
    ya = net(data["img_a"]); yb = net(data["img_b"])
    five = LO.batched_within_scene_loss(pcl, process_network_output(ya, B, D, H, W),
                                        process_network_output(yb, B, D, H, W), data)
    np.testing.assert_allclose([float(t) for t in five], g["five"], rtol=2e-4, atol=1e-6)
    five[0].backward()
    params = dict(net.named_parameters())
    for k in g.files:
        if k.startswith("grad:"):
            ref = g[k]; got = params[k[5:]].grad.numpy()
            assert np.linalg.norm(got - ref) <= 5e-3 * np.linalg.norm(ref) + 1e-7, k


def test_synthetic_structure():
    d = synthetic.make_pair_batch(2, 16, 24, num_matches=5, num_masked=15, num_background=10, num_blind=0, seed=3)
    assert d["img_a"].shape == (2, 3, 16, 24) and d["masked_a"].shape == (2, 15)
    # non_matches_a repeats each match k times consecutively (spartan_dataset_masked.py:853-854)
    assert torch.equal(d["masked_a"], d["matches_a"].repeat_interleave(3, dim=1))
    assert torch.equal(d["background_a"], d["matches_a"].repeat_interleave(2, dim=1))
    assert d["blind_a"] is None
    assert int(d["masked_b"].max()) < 16 * 24 and int(d["masked_b"].min()) >= 0
    d2 = synthetic.make_pair_batch(2, 16, 24, 5, 15, 10, 0, seed=3)
    assert all(torch.equal(d[k], d2[k]) for k in d if d[k] is not None)


def test_oracle_bit_equal_to_reference_modules(golden_dir, golden_threads):
    """The reference's own Resnet34_8s (D = 8) was loaded with this oracle's seeded weights by oracle/make_golden.py, which
    checked bit-equality there and stored the reference's parameter names, dilation bookkeeping and outputs."""
    g = _load(golden_dir, "ref_backbone_modules_d8")
    oracle = seeded_oracle(D=8, seed=0)
    assert list(oracle.state_dict().keys()) == [str(k) for k in g["state_dict_keys"]]
    assert len(g["state_dict_keys"]) == 218
    x = torch.tensor(g["x"])
    for mode in ("train", "eval"):
        getattr(oracle, mode)()
        # same torch build -> bit equal; a different CPU/torch build may reorder fp32 sums
        np.testing.assert_allclose(oracle(x).detach().numpy(), g["y_" + mode], rtol=1e-4, atol=1e-5, err_msg=mode)
    # the dilation bookkeeping the modern torchvision API gets differently (SURVEY.md 3.2)
    r = oracle.resnet34_8s
    for name, got, want in (("layer3.0.conv1.dilation", r.layer3[0].conv1.dilation, (2, 2)),
                            ("layer3.0.conv1.padding", r.layer3[0].conv1.padding, (2, 2)),
                            ("layer4.0.conv1.dilation", r.layer4[0].conv1.dilation, (4, 4)),
                            ("layer4.0.downsample.0.stride", r.layer4[0].downsample[0].stride, (1, 1)),
                            ("layer2.0.conv1.stride", r.layer2[0].conv1.stride, (2, 2)),
                            ("layer2.0.downsample.0.stride", r.layer2[0].downsample[0].stride, (2, 2))):
        assert tuple(g["attr:" + name]) == want and tuple(got) == want, name


def test_reprojection_oracle_against_ray_cast_ground_truth():
    """The restated batch_find_pixel_correspondences must send a pixel of A to the pixel of B that sees the same 3-D point:
    checked against an independent float64 ray-cast of a known plane (no reference code involved)."""
    import numpy
    H, W, n = 240, 320, 1500
    K = numpy.array([[266.8, 0, 159.7], [0, 267.4, 118.2], [0, 0, 1.0]])
    def pose(rx, ry, t):
        cx, sx, cy, sy = numpy.cos(rx), numpy.sin(rx), numpy.cos(ry), numpy.sin(ry)
        Rx = numpy.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]); Ry = numpy.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        T = numpy.eye(4); T[:3, :3] = Ry.dot(Rx); T[:3, 3] = t
        return T
    pa, pb = pose(0.01, -0.02, [0, 0, 0]), pose(-0.04, 0.1, [0.15, -0.03, 0.04])
    nrm, d0 = numpy.array([-0.1, 0.05, 1.0]), 1.2
    def render(T):
        us, vs = numpy.meshgrid(numpy.arange(W), numpy.arange(H))
        rays = numpy.linalg.inv(K).dot(numpy.stack([us.ravel(), vs.ravel(), numpy.ones(H * W)]))
        s = (d0 - nrm.dot(T[:3, 3])) / nrm.dot(T[:3, :3].dot(rays))
        return (s * 1000.0).reshape(H, W)
    da, db = render(pa).astype(numpy.float32), render(pb).astype(numpy.float32)     # unrounded depth: exact geometry
    cand = torch.randint(0, H * W, (n,), generator=torch.Generator().manual_seed(1))
    uv_a, uv_b = LO.batch_find_pixel_correspondences(da, pa, db, pb, cand, K)
    assert uv_a is not None and len(uv_a[0]) > 0.5 * n
    # ground truth in float64
    u, v = uv_a[0].numpy().astype(numpy.float64), uv_a[1].numpy().astype(numpy.float64)
    z = render(pa)[uv_a[1].numpy(), uv_a[0].numpy()] / 1000.0
    pc = numpy.linalg.inv(K).dot(numpy.stack([u * z, v * z, z]))
    pw = pa[:3, :3].dot(pc) + pa[:3, 3:4]
    p2 = pb[:3, :3].T.dot(pw - pb[:3, 3:4])
    q = K.dot(p2)
    assert numpy.abs(q[0] / q[2] - uv_b[0].numpy()).max() < 2e-2 and numpy.abs(q[1] / q[2] - uv_b[1].numpy()).max() < 2e-2
    # and the restated sampler: every sample on the mask, A side = matches repeated k times
    mask = torch.zeros(H, W); mask[50:90, 60:200] = 1.0
    ru, rv = torch.rand(40 * 7, generator=torch.Generator().manual_seed(2)), torch.rand(40 * 7, generator=torch.Generator().manual_seed(3))
    ma = torch.randint(0, H * W, (40,), generator=torch.Generator().manual_seed(5))
    na, nb = LO.create_non_correspondences_flat(ma, (H, W), 7, mask, ru, rv)
    assert torch.equal(na, ma.repeat_interleave(7)) and bool((mask.view(-1)[nb] == 1).all())


@pytest.mark.parametrize("case", WC.CASES, ids=WC.case_id)
def test_well_conditioned_fixtures_have_their_certificate(case):
    """Every input the whole-network fp64 gradient gate of the GPU suite may try (oracle/well_conditioned.py): the fp32 oracle's
    parameter gradients lie within 1e-4 (relative, per tensor) of fp64 -- so a failure of that gate is the network's, not the
    inputs'."""
    D, B, groups, H, W, mode, seeds = case
    for seed in seeds:
        x, cot, oracle = WC.build(mode, D, B, H, W, seed, groups)
        _, _, big, _, cert = WC.reference(oracle, mode, x, cot, groups)
        assert cert < 1e-4, (seed, cert)
        assert len(big) > 100          # of ~110 parameter tensors: only the cancelling fc.bias gradient is negligible
