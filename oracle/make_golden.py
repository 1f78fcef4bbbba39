"""Pins the oracle against the real reference and writes tests/golden/*.npz.

Run in the BUILD CONTAINER only (needs /root/reference):   python oracle/make_golden.py

For every backbone case the REAL reference module (loaded unmodified by oracle/ref_loader.py)
and the oracle restatement are run on the same seeded weights and inputs and must agree
bit-for-bit (forward, running statistics, parameter gradients); the reference's outputs are what
is stored.  For the loss the reference's OWN source is executed (oracle/build_ref.py: the Python-2 files with a short
list of line-anchored py2->py3 patches, written to the git-ignored oracle/_ref/): its outputs and autograd gradients
are what is stored, and the torch restatement must equal them bit-for-bit and the numpy one to 1e-6.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "pytorch-dense-correspondence_b200"))

from oracle import loss_oracle as LO            # noqa: E402
from oracle import build_ref                    # noqa: E402
from oracle import ref_loader                   # noqa: E402
from oracle import ref_cases                    # noqa: E402
from oracle.resnet34_8s_oracle import GOLDEN_CPU_THREADS, seeded_oracle, process_network_output  # noqa: E402
import synthetic                                # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
torch.set_num_threads(GOLDEN_CPU_THREADS)


def bit_equal(a, b, what):
    assert a.shape == b.shape, what
    assert torch.equal(a, b), "%s: oracle != reference (max abs diff %g)" % (what, (a - b).abs().max().item())


def backbone_case(name, D, B, H, W, seed_data):
    oracle = seeded_oracle(D=D, seed=0)
    ref = ref_loader.reference_resnet34_8s(D, oracle.state_dict())
    assert list(ref.state_dict().keys()) == list(oracle.state_dict().keys())
    g = torch.Generator().manual_seed(seed_data)
    x = torch.randn(B, 3, H, W, generator=g)
    out = {}
    ref.train(); oracle.train()
    y_ref = ref(x); y_or = oracle(x)
    bit_equal(y_ref, y_or, name + " train fwd")
    for k in ("resnet34_8s.bn1.running_mean", "resnet34_8s.bn1.running_var",
              "resnet34_8s.layer4.2.bn2.running_mean", "resnet34_8s.layer4.2.bn2.running_var",
              "resnet34_8s.layer3.0.downsample.1.running_var"):
        bit_equal(ref.state_dict()[k], oracle.state_dict()[k], name + " " + k)
        out["rs:" + k] = ref.state_dict()[k].numpy().copy()
    # a backward through a fixed random cotangent
    cot = torch.randn(y_ref.shape, generator=g)
    (y_ref * cot).sum().backward(); (y_or * cot).sum().backward()
    gr = dict(ref.named_parameters()); go = dict(oracle.named_parameters())
    for k in gr:
        bit_equal(gr[k].grad, go[k].grad, name + " grad " + k)
    out["x_seed"] = np.int64(seed_data)
    out["y_train"] = y_ref.detach().numpy() if H * W <= 96 * 96 else y_ref.detach()[:, :, ::16, ::16].numpy()
    for k in ("resnet34_8s.conv1.weight", "resnet34_8s.bn1.weight", "resnet34_8s.bn1.bias",
              "resnet34_8s.layer1.0.conv1.weight", "resnet34_8s.layer2.0.downsample.0.weight",
              "resnet34_8s.layer2.0.conv1.weight", "resnet34_8s.layer3.0.bn1.weight",
              "resnet34_8s.layer4.2.bn2.bias", "resnet34_8s.fc.weight", "resnet34_8s.fc.bias"):
        out["grad:" + k] = gr[k].grad.numpy().copy()
    out["gradnorm:all"] = np.array([gr[k].grad.double().norm().item() for k in gr])
    ref.eval(); oracle.eval()
    with torch.no_grad():
        ye_ref = ref(x); ye_or = oracle(x)
    bit_equal(ye_ref, ye_or, name + " eval fwd")
    out["y_eval"] = ye_ref.numpy() if H * W <= 96 * 96 else ye_ref[:, :, ::16, ::16].numpy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


def loss_case(name, D, H, W, Nm, k_masked, k_bg, n_blind, cfg_over, seed):
    cfg = dict(LO.DEFAULT_LOSS_CONFIG); cfg.update(cfg_over)
    g = torch.Generator().manual_seed(seed)
    P = H * W
    # descriptors with the scale the network produces (|.| ~ 0.19, SURVEY 8d) so both hinge branches fire
    A = (0.25 * torch.randn(1, D, H, W, generator=g)).requires_grad_()
    Bt = (0.25 * torch.randn(1, D, H, W, generator=g)).requires_grad_()
    pa = process_network_output(A, 1, D, H, W); pb = process_network_output(Bt, 1, D, H, W)
    ma = torch.randint(0, P, (Nm,), generator=g); mb = torch.randint(0, P, (Nm,), generator=g)
    na_m = ma.repeat_interleave(k_masked); nb_m = torch.randint(0, P, (Nm * k_masked,), generator=g)
    na_b = ma.repeat_interleave(k_bg); nb_b = torch.randint(0, P, (Nm * k_bg,), generator=g)
    if n_blind:
        xa = torch.randint(0, P, (n_blind,), generator=g); xb = torch.randint(0, P, (n_blind,), generator=g)
    else:
        xa = xb = LO.empty_tensor()
    # the executed reference (oracle/_ref) produces the stored values ...
    ref = build_ref.load()
    mt = torch.tensor([ref.dataset.SpartanDatasetDataType.SINGLE_OBJECT_WITHIN_SCENE])
    five = ref.composer.get_loss(ref.pcl.PixelwiseContrastiveLoss([H, W], dict(cfg)), mt, pa, pb, ma, mb, na_m, nb_m, na_b, nb_b, xa, xb)
    five[0].reshape(()).backward()
    # ... and the torch restatement must reproduce them bit-for-bit (same ops, same order)
    A2 = A.detach().clone().requires_grad_(); B2 = Bt.detach().clone().requires_grad_()
    five_o = LO.get_loss(LO.TorchPixelwiseContrastiveLoss([H, W], dict(cfg)), mt, process_network_output(A2, 1, D, H, W),
                         process_network_output(B2, 1, D, H, W), ma, mb, na_m, nb_m, na_b, nb_b, xa, xb)
    five_o[0].reshape(()).backward()
    assert [float(t) for t in five_o] == [float(t) for t in five], name
    assert torch.equal(A2.grad, A.grad) and torch.equal(B2.grad, Bt.grad), name
    idx = dict(matches_a=ma.numpy(), matches_b=mb.numpy(), masked_a=na_m.numpy(), masked_b=nb_m.numpy(),
               background_a=na_b.numpy(), background_b=nb_b.numpy(),
               blind_a=xa.numpy(), blind_b=xb.numpy())
    An = A.detach().numpy()[0].reshape(D, P).T; Bn = Bt.detach().numpy()[0].reshape(D, P).T
    five_np, counts = LO.np_within_scene_loss(An, Bn, idx, cfg, W)
    for t, n_ in zip(five, five_np):
        assert abs(float(t) - n_) <= 1e-6 * max(1.0, abs(n_)), (name, float(t), n_)
    out = dict(idx)
    out.update(A=A.detach().numpy(), B=Bt.detach().numpy(), five=np.array([float(t) for t in five]),
               counts=np.array(counts), dA=A.grad.numpy(), dB=Bt.grad.numpy(),
               cfg_keys=np.array(sorted(cfg_over.keys())), cfg_vals=np.array([float(cfg_over[k]) for k in sorted(cfg_over)]))
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, "five", out["five"], "counts", counts)


def train_step_case(name, D, B, H, W, Nm, Nn, seed):
    """fwd(A), fwd(B), within-scene loss (mean over pairs), backward -- reference backbone + the loss restatement (which the
    loss cases above and tests/test_oracle_ref_cpu.py pin bit-for-bit to the executed reference loss)."""
    oracle = seeded_oracle(D=D, seed=0)
    ref = ref_loader.reference_resnet34_8s(D, oracle.state_dict())
    ref.train()
    data = synthetic.make_pair_batch(B, H, W, Nm, Nn, Nn, 0, seed=seed)
    pcl = LO.TorchPixelwiseContrastiveLoss([H, W], dict(LO.DEFAULT_LOSS_CONFIG))
    ya = ref(data["img_a"]); yb = ref(data["img_b"])
    pa = process_network_output(ya, B, D, H, W); pb = process_network_output(yb, B, D, H, W)
    five = LO.batched_within_scene_loss(pcl, pa, pb, data)
    five[0].backward()
    gr = dict(ref.named_parameters())
    out = dict(five=np.array([float(t) for t in five]), seed=np.int64(seed),
               gradnorm=np.array([gr[k].grad.double().norm().item() for k in gr]))
    for k in ("resnet34_8s.conv1.weight", "resnet34_8s.fc.weight", "resnet34_8s.fc.bias",
              "resnet34_8s.layer4.0.downsample.1.weight", "resnet34_8s.layer1.2.bn2.bias"):
        out["grad:" + k] = gr[k].grad.numpy().copy()
    out["rs:resnet34_8s.bn1.running_mean"] = ref.state_dict()["resnet34_8s.bn1.running_mean"].numpy().copy()
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, "five", out["five"])


def assert_same(x, y, what):
    """Bit-equal results (tensors, numbers, strings, None, and tuples / lists / dicts of them)."""
    if isinstance(x, torch.Tensor):
        assert isinstance(y, torch.Tensor) and x.dtype == y.dtype, what
        bit_equal(x, y, what)
    elif isinstance(x, (tuple, list)):
        assert isinstance(y, (tuple, list)) and len(x) == len(y), what
        for i, (a, b) in enumerate(zip(x, y)):
            assert_same(a, b, "%s[%d]" % (what, i))
    elif isinstance(x, dict):
        assert sorted(x) == sorted(y), what
        for k in x:
            assert_same(x[k], y[k], "%s/%s" % (what, k))
    else:
        assert x == y, (what, x, y)


def ref_loss_cases():
    """Every PixelwiseContrastiveLoss method and every loss_composer branch (oracle/ref_cases.py), run on the executed
    reference; the torch restatement must agree bit-for-bit."""
    ref = build_ref.load()
    H, W, D, P = 12, 20, 5, 240
    gen = torch.Generator().manual_seed(3)
    A = 0.3 * torch.randn(1, P, D, generator=gen); B = 0.3 * torch.randn(1, P, D, generator=gen)
    ma = torch.randint(0, P, (7,), generator=gen); mb = torch.randint(0, P, (7,), generator=gen)
    inp = dict(H=H, W=W, A=A, B=B, ma=ma, mb=mb, na=ma.repeat_interleave(4), nb=torch.randint(0, P, (28,), generator=gen))
    out = ref_cases.loss_methods(ref.pcl.PixelwiseContrastiveLoss, inp)
    assert_same(ref_cases.loss_methods(LO.TorchPixelwiseContrastiveLoss, inp), out, "loss methods")
    torch.save({"inputs": inp, "outputs": out}, os.path.join(GOLD, "ref_loss_methods.pt"))

    H, W, D, P = 10, 16, 3, 160
    gen = torch.Generator().manual_seed(9)
    A = 0.3 * torch.randn(1, D, H, W, generator=gen); B = 0.3 * torch.randn(1, D, H, W, generator=gen)
    ma = torch.randint(0, P, (6,), generator=gen); mb = torch.randint(0, P, (6,), generator=gen)
    idx = dict(matches_a=ma, matches_b=mb, masked_a=ma.repeat_interleave(3), masked_b=torch.randint(0, P, (18,), generator=gen),
               background_a=ma.repeat_interleave(2), background_b=torch.randint(0, P, (12,), generator=gen),
               blind_a=torch.randint(0, P, (9,), generator=gen), blind_b=torch.randint(0, P, (9,), generator=gen))
    inp = dict(A=A, B=B, idx=idx)
    SD = ref.dataset.SpartanDataset
    out = ref_cases.composer_branches(ref.pcl.PixelwiseContrastiveLoss, ref.composer.get_loss, SD.empty_tensor, inp)
    assert_same(ref_cases.composer_branches(LO.TorchPixelwiseContrastiveLoss, LO.get_loss, LO.empty_tensor, inp), out, "composer")
    out["empty_tensor"] = SD.empty_tensor()
    T = ref.dataset.SpartanDatasetDataType
    out["data_types"] = {k: getattr(T, k) for k in dir(T) if k.isupper()}
    torch.save({"inputs": inp, "outputs": out}, os.path.join(GOLD, "ref_composer_branches.pt"))
    print("wrote ref_loss_methods, ref_composer_branches")


def _with_rand(fn, fake):
    """fn() with torch.rand replaced by fake (the reference samplers draw their uniforms from it)."""
    real = torch.rand
    torch.rand = fake
    try:
        return fn()
    finally:
        torch.rand = real


def ref_non_match_sampler_case():
    """create_non_correspondences draws torch.rand(n) (mask branch) or torch.rand(2, n) (no mask), then two more draws for the
    no-op perturbation; the restatement takes the uniforms as arguments -- feed both the same numbers."""
    ref = build_ref.load()
    H, W, k = 30, 40, 5
    gen = torch.Generator().manual_seed(4)
    ma = torch.randint(0, H * W, (11,), generator=gen)
    uv_a = (ma % W, ma // W)
    uv_b = ((ma % W).float(), (ma // W).float())
    n = len(ma) * k
    ru, rv = torch.rand(n, generator=gen), torch.rand(n, generator=gen)
    mask = torch.zeros(H, W); mask[5:20, 8:30] = 1.0
    masks, outs = [mask, None, torch.zeros(H, W)], []
    SD = ref.dataset.SpartanDataset
    for m in masks:
        calls = []

        def fake_rand(*shape):
            calls.append(shape)
            if len(calls) == 1:
                return ru.clone() if shape == (n,) else torch.stack((ru, rv)).clone()
            return torch.zeros(*shape)
        uv_b_non = _with_rand(lambda: ref.finder.create_non_correspondences(uv_b, (H, W), num_non_matches_per_match=k, img_b_mask=m),
                              fake_rand)
        uv_a_long, uv_b_long = SD.create_non_matches(None, uv_a, uv_b_non, k)
        na_r = SD.flatten_uv_tensor(uv_a_long, W).squeeze(1); nb_r = SD.flatten_uv_tensor(uv_b_long, W).squeeze(1)
        assert_same(list(LO.create_non_correspondences_flat(ma, (H, W), k, m, ru, rv)), [na_r, nb_r], "sampler")
        outs.append((na_r, nb_r))
    torch.save({"inputs": dict(H=H, W=W, k=k, matches_a=ma, rand_u=ru, rand_v=rv, masks=masks), "outputs": outs},
               os.path.join(GOLD, "ref_non_match_sampler.pt"))
    print("wrote ref_non_match_sampler", [len(o[1]) for o in outs])


def ref_reprojection_case():
    """batch_find_pixel_correspondences on a rendered tilted plane with no-return pixels and an occluder."""
    ref = build_ref.load()
    H, W, n = 120, 160, 900
    K = np.array([[133.4, 0, 79.8], [0, 133.7, 59.1], [0, 0, 1.0]])

    def pose(rx, ry, t):
        cx, sx, cy, sy = np.cos(rx), np.sin(rx), np.cos(ry), np.sin(ry)
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]); Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        T = np.eye(4); T[:3, :3] = Ry.dot(Rx); T[:3, 3] = t
        return T
    pa, pb = pose(0.01, -0.02, [0, 0, 0]), pose(-0.04, 0.1, [0.15, -0.03, 0.04])
    nrm, d0 = np.array([-0.1, 0.05, 1.0]), 1.2

    def render(T):
        us, vs = np.meshgrid(np.arange(W), np.arange(H))
        rays = np.linalg.inv(K).dot(np.stack([us.ravel(), vs.ravel(), np.ones(H * W)]))
        s = (d0 - nrm.dot(T[:3, 3])) / nrm.dot(T[:3, :3].dot(rays))
        return (s * 1000.0).reshape(H, W)
    da = np.round(render(pa)).astype(np.uint16); db = np.round(render(pb)).astype(np.uint16)
    da[10:30, 20:50] = 0                                               # no-return pixels (depth 0) are pruned
    db[60:80, 100:130] = 300                                           # an occluder in front of the plane in image b
    mask = np.zeros((H, W), dtype=np.float32); mask[5:110, 10:150] = 1.0
    ru = torch.rand(n, generator=torch.Generator().manual_seed(8))
    # the reference first draws (and discards) rand(2, n) for unmasked candidates, then rand(n) for the masked sample
    uv_a, uv_b = _with_rand(lambda: ref.finder.batch_find_pixel_correspondences(da, pa, db, pb, num_attempts=n, img_a_mask=mask, K=K),
                            lambda *s: ru.clone() if s == (n,) else torch.zeros(*s))
    nz = torch.nonzero(torch.from_numpy(mask).view(-1))
    cand = torch.index_select(nz, 0, torch.floor(ru * len(nz)).long()).squeeze(1)
    uv_a_o, uv_b_o = LO.batch_find_pixel_correspondences(da, pa, db, pb, cand, K)
    assert_same(list(uv_a_o) + list(uv_b_o), list(uv_a) + list(uv_b), "reprojection")
    inp = {k: torch.from_numpy(v.astype(np.int32) if v.dtype == np.uint16 else v)
           for k, v in dict(depth_a=da, pose_a=pa, depth_b=db, pose_b=pb, K=K, mask_a=mask).items()}
    inp["rand"] = ru
    torch.save({"inputs": inp, "outputs": list(uv_a) + list(uv_b)}, os.path.join(GOLD, "ref_reprojection.pt"))
    print("wrote ref_reprojection", len(uv_a[0]), "of", n)


def ref_backbone_modules_case():
    """The reference modules themselves at D = 8: parameter names, the dilation bookkeeping, train- and eval-mode outputs."""
    D = 8
    oracle = seeded_oracle(D=D, seed=0)
    ref = ref_loader.reference_resnet34_8s(D, oracle.state_dict())
    x = torch.randn(1, 3, 40, 56, generator=torch.Generator().manual_seed(2))
    out = {"x": x.numpy(), "state_dict_keys": np.array(list(ref.state_dict().keys()))}
    for mode in ("train", "eval"):
        getattr(ref, mode)(); getattr(oracle, mode)()
        y = ref(x).detach()
        bit_equal(y, oracle(x).detach(), "backbone modules " + mode)
        out["y_" + mode] = y.numpy()
    r = ref.resnet34_8s
    for name, v in (("layer3.0.conv1.dilation", r.layer3[0].conv1.dilation), ("layer3.0.conv1.padding", r.layer3[0].conv1.padding),
                    ("layer4.0.conv1.dilation", r.layer4[0].conv1.dilation), ("layer4.0.downsample.0.stride", r.layer4[0].downsample[0].stride),
                    ("layer2.0.conv1.stride", r.layer2[0].conv1.stride), ("layer2.0.downsample.0.stride", r.layer2[0].downsample[0].stride)):
        out["attr:" + name] = np.array(v)
    np.savez_compressed(os.path.join(GOLD, "ref_backbone_modules_d8.npz"), **out)
    print("wrote ref_backbone_modules_d8")


if __name__ == "__main__":
    assert ref_loader.reference_available() and build_ref.reference_available(), "needs the reference checkout"
    build_ref.build()
    os.makedirs(GOLD, exist_ok=True)
    backbone_case("backbone_small_d3", D=3, B=2, H=64, W=96, seed_data=11)
    backbone_case("backbone_small_d16", D=16, B=1, H=48, W=64, seed_data=12)
    backbone_case("backbone_full_d3", D=3, B=1, H=480, W=640, seed_data=13)
    loss_case("loss_default_d3", 3, 48, 64, 50, 3, 2, 0, {}, 21)
    loss_case("loss_pixelw_blind_d8", 8, 48, 64, 40, 4, 4, 37,
              {"use_l2_pixel_loss_on_masked_non_matches": True, "use_l2_pixel_loss_on_background_non_matches": True,
               "M_pixel": 25, "M_masked": 0.7, "M_background": 0.4, "non_match_loss_weight": 2.0}, 22)
    loss_case("loss_noscale_d16", 16, 48, 64, 64, 2, 1, 5, {"scale_by_hard_negatives": False, "M_masked": 1.5,
                                                             "M_background": 1.2}, 23)
    train_step_case("train_step_small_d3", D=3, B=2, H=64, W=96, Nm=40, Nn=120, seed=31)
    ref_loss_cases()
    ref_non_match_sampler_case()
    ref_reprojection_case()
    ref_backbone_modules_case()
