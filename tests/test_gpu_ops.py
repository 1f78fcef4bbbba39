"""GPU: every single-operator C-ABI entry point against a plain PyTorch fp32 CPU reference of the same op
(tolerances written per test), and the loss kernels against the oracle / golden vectors."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import pdc_b200
from pdc_b200 import ops, loss_composer, _native as N
from pdc_b200.contrastive_ops import Term, contrastive_terms
from oracle import loss_oracle as LO
from oracle.resnet34_8s_oracle import process_network_output

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    a = a.double().cpu(); b = b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


CONV_CASES = [
    # N, H, W, Cin, Cout, k, stride, pad, dil
    (2, 30, 40, 64, 64, 3, 1, 1, 1),      # layer1
    (1, 30, 40, 64, 128, 3, 2, 1, 1),     # layer2.0.conv1
    (1, 30, 40, 64, 128, 1, 2, 0, 1),     # layer2.0.downsample
    (1, 15, 20, 128, 256, 3, 1, 2, 2),    # layer3.0.conv1 (dilation 2)
    (2, 15, 20, 256, 256, 3, 1, 2, 2),
    (1, 15, 20, 256, 512, 3, 1, 4, 4),    # layer4.0.conv1 (dilation 4)
    (1, 15, 20, 256, 512, 1, 1, 0, 1),    # layer4.0.downsample
    (1, 13, 9, 512, 512, 3, 1, 4, 4),     # odd sizes, M not a tile multiple
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv2d_forward_backward_fp32(case):
    n, h, w, cin, cout, k, s, p, d = case
    g = torch.Generator().manual_seed(hash(case) % 1000)
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (k * k * cin)) ** 0.5
    xr = x.clone().requires_grad_(); wr = wt.clone().requires_grad_()
    y_ref = F.conv2d(xr, wr, None, s, p, d)
    dy = torch.randn(y_ref.shape, generator=g)
    y_ref.backward(dy)
    y = ops.conv2d_forward(nhwc(x).to(DEV), wt.to(DEV), s, p, d)
    assert rel(y, nhwc(y_ref.detach())) < 2e-6          # fp32 FFMA vs fp32 CPU: summation order only
    dx, dw = ops.conv2d_backward(nhwc(x).to(DEV), wt.to(DEV), nhwc(dy).to(DEV), s, p, d)
    assert rel(dx, nhwc(xr.grad)) < 2e-6
    assert rel(dw, wr.grad) < 5e-6                       # split-K fp32 atomics


TC_CASES = [c for c in CONV_CASES if c[6] == 1] + [
    (1, 60, 80, 64, 64, 3, 1, 1, 1),       # exact tiles (W = 5 x 16), Cout = 64 path
    (2, 60, 80, 512, 512, 3, 1, 4, 4),     # the dominant GEMM: 72 k-blocks, 4 N-tiles
    (1, 8, 12, 512, 512, 3, 1, 4, 4),      # feature map smaller than one 8x16 tile
    (1, 60, 80, 128, 256, 1, 1, 0, 1),     # 1x1 downsample (layer3.0)
    (2, 30, 40, 64, 128, 3, 2, 1, 1),      # layer2.0.conv1: stride 2 through TMA element strides; dgrad by zero insertion
    (1, 30, 40, 64, 128, 1, 2, 0, 1),      # layer2.0.downsample: 1x1 stride 2
    (1, 120, 160, 64, 128, 3, 2, 1, 1),    # the real layer2.0.conv1 size
    (2, 24, 32, 64, 64, 3, 1, 1, 1),       # 64 -> 64 on a map of whole 8x16 tiles: the halo-tile kernel (resident weights), 2 images
    (1, 120, 160, 64, 64, 3, 1, 1, 1),     # the real layer1 size through the halo-tile kernel: 150 tiles
]


@pytest.mark.parametrize("precision,tol", [("bf16x3", 2e-5), ("bf16", 8e-3)])
@pytest.mark.parametrize("case", TC_CASES)
def test_conv2d_tcgen05(case, precision, tol):
    """tcgen05 implicit GEMM vs the fp32 CPU reference: bf16x3 split must be fp32-class (<= 2e-5 relative Frobenius
    error, ~2^-16 per product), single-pass bf16 within bf16 rounding."""
    prec = {"bf16x3": N.PRECISION_BF16X3, "bf16": N.PRECISION_BF16}[precision]
    if N.lib.ddn_resnet34_8s_workspace_bytes(1, 64, 64, 3, 1, prec) == 0:
        pytest.skip("tcgen05 path not in this build")
    n, h, w, cin, cout, k, s, p, d = case
    g = torch.Generator().manual_seed(hash(case) % 1000 + 1)
    x = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (k * k * cin)) ** 0.5
    xr = x.clone().requires_grad_(); wr = wt.clone().requires_grad_()
    y_ref = F.conv2d(xr, wr, None, s, p, d)
    dy = torch.randn(y_ref.shape, generator=g)
    y_ref.backward(dy)
    y = ops.conv2d_forward(nhwc(x).to(DEV), wt.to(DEV), s, p, d, precision=prec)
    torch.cuda.synchronize()
    assert rel(y, nhwc(y_ref.detach())) < tol
    dx, dw = ops.conv2d_backward(nhwc(x).to(DEV), wt.to(DEV), nhwc(dy).to(DEV), s, p, d, precision=prec)
    assert rel(dx, nhwc(xr.grad)) < tol
    assert rel(dw, wr.grad) < max(tol, 5e-6)


@pytest.mark.parametrize("C,relu,residual", [(64, True, False), (128, True, True), (256, False, False), (512, True, True)])
def test_batchnorm_forward_backward(C, relu, residual):
    g = torch.Generator().manual_seed(C)
    M = 2 * 15 * 20
    x = torch.randn(M, C, generator=g) * 2 + 0.5
    gamma = torch.rand(C, generator=g) + 0.5; beta = torch.randn(C, generator=g)
    res = torch.randn(M, C, generator=g) if residual else None
    rm = torch.zeros(C); rv = torch.ones(C)
    xr = x.clone().requires_grad_(); gr = gamma.clone().requires_grad_(); br = beta.clone().requires_grad_()
    rr = res.clone().requires_grad_() if residual else None
    y_ref = F.batch_norm(xr, rm, rv, gr, br, True, 0.1, 1e-5)
    if residual:
        y_ref = y_ref + rr
    if relu:
        y_ref = F.relu(y_ref)
    dy = torch.randn(M, C, generator=g)
    y_ref.backward(dy)
    rmg = torch.zeros(C, device=DEV); rvg = torch.ones(C, device=DEV)
    y, mean, invstd = ops.batchnorm_forward(x.to(DEV), gamma.to(DEV), beta.to(DEV), res.to(DEV) if residual else None,
                                            relu=relu, training=True, running_mean=rmg, running_var=rvg)
    assert rel(y, y_ref.detach()) < 2e-6
    assert rel(rmg, rm) < 1e-6 and rel(rvg, rv) < 1e-6     # momentum 0.1, unbiased variance
    dx, dgamma, dbeta, dres = ops.batchnorm_backward(dy.to(DEV), x.to(DEV), y, gamma.to(DEV), mean, invstd, relu=relu,
                                                     need_residual_grad=residual)
    assert rel(dx, xr.grad) < 1e-5
    assert rel(dgamma, gr.grad) < 1e-5 and rel(dbeta, br.grad) < 1e-5
    if residual:
        assert rel(dres, rr.grad) < 1e-6
    # eval mode uses the running statistics
    ye, _, _ = ops.batchnorm_forward(x.to(DEV), gamma.to(DEV), beta.to(DEV), None, relu=False, training=False,
                                     running_mean=rmg, running_var=rvg)
    assert rel(ye, F.batch_norm(x, rm, rv, gamma, beta, False, 0.1, 1e-5)) < 2e-6


@pytest.mark.parametrize("shape", [(2, 3, 8, 12, 64, 96), (1, 16, 60, 80, 480, 640), (1, 3, 6, 8, 48, 64)])
def test_upsample_bilinear(shape):
    n, c, h, w, H, W = shape
    g = torch.Generator().manual_seed(7)
    x = torch.randn(n, c, h, w, generator=g, requires_grad=True)
    y_ref = F.interpolate(x, size=(H, W), mode="bilinear", align_corners=True)
    dy = torch.randn(y_ref.shape, generator=g)
    y_ref.backward(dy)
    y = ops.upsample_bilinear_forward(x.detach().to(DEV), H, W)
    assert float((y.cpu() - y_ref.detach()).abs().max()) < 2e-5
    dx = ops.upsample_bilinear_backward(dy.to(DEV), h, w)
    assert rel(dx, x.grad) < 1e-5


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


@pytest.mark.parametrize("name", ["loss_default_d3", "loss_pixelw_blind_d8", "loss_noscale_d16"])
def test_fused_within_scene_loss_matches_golden(golden_dir, name):
    g = _golden(golden_dir, name)
    cfg = dict(LO.DEFAULT_LOSS_CONFIG)
    for k, v in zip(g["cfg_keys"], g["cfg_vals"]):
        k = str(k)
        cfg[k] = bool(v) if isinstance(LO.DEFAULT_LOSS_CONFIG[k], bool) else float(v)
    A = torch.tensor(g["A"], device=DEV).requires_grad_(); B = torch.tensor(g["B"], device=DEV).requires_grad_()
    _, D, H, W = A.shape
    pcl = pdc_b200.PixelwiseContrastiveLoss([H, W], cfg)
    pa = A.view(1, D, H * W).permute(0, 2, 1); pb = B.view(1, D, H * W).permute(0, 2, 1)
    idx = {k: torch.tensor(g[k], device=DEV) for k in ("matches_a", "matches_b", "masked_a", "masked_b",
                                                       "background_a", "background_b", "blind_a", "blind_b")}
    five = loss_composer.get_loss(pcl, torch.tensor([0]), pa, pb, idx["matches_a"], idx["matches_b"], idx["masked_a"],
                                  idx["masked_b"], idx["background_a"], idx["background_b"], idx["blind_a"], idx["blind_b"])
    got = np.array([float(t) for t in five])
    np.testing.assert_allclose(got, g["five"], rtol=2e-6, atol=1e-7)        # north_star gate: 1e-4 on the scalar loss
    five[0].backward()
    assert rel(A.grad, torch.tensor(g["dA"])) < 1e-5 and rel(B.grad, torch.tensor(g["dB"])) < 1e-5
    assert pcl.debug is False
    pcl.debug = True
    loss_composer.get_loss(pcl, torch.tensor([0]), pa, pb, idx["matches_a"], idx["matches_b"], idx["masked_a"],
                           idx["masked_b"], idx["background_a"], idx["background_b"], idx["blind_a"], idx["blind_b"])
    counts = pcl.debug_data["num_hard_negatives_device"][0].tolist()
    assert counts[1] == int(g["counts"][0]) and counts[2] == int(g["counts"][1])     # hard negatives: exact
    if not (len(g["blind_a"]) == 1 and g["blind_a"][0] == -1):
        assert counts[3] == int(g["counts"][2])


def test_loss_methods_match_oracle_and_edge_cases():
    H, W, D = 24, 32, 5
    gen = torch.Generator().manual_seed(3)
    A = (0.3 * torch.randn(1, D, H, W, generator=gen)); B = (0.3 * torch.randn(1, D, H, W, generator=gen))
    P = H * W
    ma = torch.randint(0, P, (37,), generator=gen); mb = torch.randint(0, P, (37,), generator=gen)
    na = ma.repeat_interleave(3); nb = torch.randint(0, P, (111,), generator=gen)
    cfg = dict(LO.DEFAULT_LOSS_CONFIG); cfg["M_descriptor"] = 0.6
    ref = LO.TorchPixelwiseContrastiveLoss([H, W], cfg)
    ours = pdc_b200.PixelwiseContrastiveLoss([H, W], cfg)
    Ar = A.clone().requires_grad_(); Br = B.clone().requires_grad_()
    Ag = A.to(DEV).requires_grad_(); Bg = B.to(DEV).requires_grad_()
    par, pbr = process_network_output(Ar, 1, D, H, W), process_network_output(Br, 1, D, H, W)
    pag, pbg = process_network_output(Ag, 1, D, H, W), process_network_output(Bg, 1, D, H, W)
    c = lambda t: t.to(DEV)
    # match_loss
    r = ref.match_loss(par, pbr, ma, mb)[0]; o = ours.match_loss(pag, pbg, c(ma), c(mb))[0]
    assert abs(float(r) - float(o)) < 1e-6 * abs(float(r))
    # descriptor-only, inverted, pixel-weighted
    for fn, args_r, args_o, kw in [
        ("non_match_loss_descriptor_only", (par, pbr, na, nb), (pag, pbg, c(na), c(nb)), dict(M_descriptor=0.6)),
        ("non_match_loss_descriptor_only", (par, pbr, na, nb), (pag, pbg, c(na), c(nb)), dict(M_descriptor=0.3, invert=True)),
        ("non_match_loss_with_l2_pixel_norm", (par, pbr, mb, na, nb), (pag, pbg, c(mb), c(na), c(nb)), dict(M_descriptor=0.6, M_pixel=9)),
    ]:
        rs, rh = getattr(ref, fn)(*args_r, **kw); os_, oh = getattr(ours, fn)(*args_o, **kw)
        assert rh == oh, fn
        assert abs(float(rs) - float(os_)) < 2e-6 * max(1.0, abs(float(rs))), fn
    # combined + gradients through the generic autograd path
    rm, rn, rh = ref.get_loss_matched_and_non_matched_with_l2(par, pbr, ma, mb, na, nb, M_descriptor=0.6)
    om, on, oh = ours.get_loss_matched_and_non_matched_with_l2(pag, pbg, c(ma), c(mb), c(na), c(nb), M_descriptor=0.6)
    assert rh == oh
    (rm + 0.5 * rn).backward(); (om + 0.5 * on).backward()
    assert rel(Ag.grad, Ar.grad) < 1e-5 and rel(Bg.grad, Br.grad) < 1e-5
    # vector-returning method + legacy loss keep the reference's values
    rv = ref.non_match_descriptor_loss(par, pbr, na, nb, M=0.6); ov = ours.non_match_descriptor_loss(pag, pbg, c(na), c(nb), M=0.6)
    assert rv[1] == ov[1] and rel(ov[0], rv[0]) < 1e-6
    rl = ref.get_loss_original(par, pbr, ma, mb, na, nb); ol = ours.get_loss_original(pag, pbg, c(ma), c(mb), c(na), c(nb))
    assert abs(float(rl[0]) - float(ol[0])) < 1e-5
    # single index pair, identical descriptors (d = 0 -> counted hard, zero gradient), contiguous [1,P,D] input
    Z = torch.zeros(1, P, D, device=DEV, requires_grad=True)
    s, h = ours.non_match_loss_descriptor_only(Z, Z.detach().clone(), c(torch.tensor([5])), c(torch.tensor([9])), M_descriptor=0.5)
    assert h == 1 and abs(float(s) - 0.25) < 1e-7
    s.backward()
    assert float(Z.grad.abs().sum()) == 0.0
    # different-object composition and the two pair types the reference cannot run
    xa = torch.randint(0, P, (50,), generator=gen); xb = torch.randint(0, P, (50,), generator=gen)
    rfive = LO.get_loss(ref, torch.tensor([2]), par, pbr, ma, mb, na, nb, na, nb, xa, xb)
    ofive = loss_composer.get_loss(ours, torch.tensor([2]), pag, pbg, c(ma), c(mb), c(na), c(nb), c(na), c(nb), c(xa), c(xb))
    assert abs(float(rfive[0]) - float(ofive[0])) < 1e-6 and abs(float(rfive[4]) - float(ofive[4])) < 1e-6
    with pytest.raises((NameError, UnboundLocalError)):
        loss_composer.get_loss(ours, torch.tensor([1]), pag, pbg, c(ma), c(mb), c(na), c(nb), c(na), c(nb), c(xa), c(xb))
    with pytest.raises(ValueError):
        loss_composer.get_loss(ours, torch.tensor([7]), pag, pbg, c(ma), c(mb), c(na), c(nb), c(na), c(nb), c(xa), c(xb))


@pytest.mark.parametrize("D,n_nm", [(3, 150_000), (16, 5_000)])
def test_loss_large_properties(D, n_nm):
    """Full-size (640x480) size-independent properties: permutation invariance of the sums, linearity of the
    backward in the upstream gradient, and duplicate-heavy A-side indices scatter exactly like index_add_."""
    H, W, B = 480, 640, 2
    P = H * W
    gen = torch.Generator().manual_seed(9)
    A = (0.2 * torch.randn(B, D, H, W, generator=gen)).to(DEV); Bt = (0.2 * torch.randn(B, D, H, W, generator=gen)).to(DEV)
    pa = A.view(B, D, P).permute(0, 2, 1); pb = Bt.view(B, D, P).permute(0, 2, 1)
    ma = torch.randint(0, P, (B, 1000), generator=gen).to(DEV); mb = torch.randint(0, P, (B, 1000), generator=gen).to(DEV)
    na = ma.repeat_interleave(n_nm // 1000, dim=1); nb = torch.randint(0, P, (B, n_nm), generator=gen).to(DEV)
    terms = lambda a, b: [Term(ma, mb, N.TERM_MATCH), Term(a, b, N.TERM_HINGE, 0.5)]
    s1, c1 = contrastive_terms(pa, pb, W, terms(na, nb))
    perm = torch.randperm(n_nm, generator=gen).to(DEV)
    s2, c2 = contrastive_terms(pa, pb, W, terms(na[:, perm], nb[:, perm]))
    assert torch.equal(c1, c2)
    assert float(((s1 - s2).abs() / s1.abs().clamp(min=1e-12)).max()) < 1e-9
    # against a torch (CUDA, fp32) composition of the same math
    ga = torch.gather(pa, 1, na.unsqueeze(-1).expand(-1, -1, D)); gb = torch.gather(pb, 1, nb.unsqueeze(-1).expand(-1, -1, D))
    dist = (ga - gb).norm(2, 2)
    hinge = torch.clamp(0.5 - dist, min=0).pow(2)
    assert float(((hinge.double().sum(1) - s1[:, 1]).abs() / s1[:, 1]).max()) < 1e-5
    assert torch.equal((hinge != 0).sum(1), c1[:, 1])
    # backward: linear in upstream, equals autograd of the torch composition
    Ar = A.clone().requires_grad_(); Br = Bt.clone().requires_grad_()
    par = Ar.view(B, D, P).permute(0, 2, 1); pbr = Br.view(B, D, P).permute(0, 2, 1)
    ga = torch.gather(par, 1, na.unsqueeze(-1).expand(-1, -1, D)); gb = torch.gather(pbr, 1, nb.unsqueeze(-1).expand(-1, -1, D))
    torch.clamp(0.5 - (ga - gb).norm(2, 2), min=0).pow(2).sum().backward()
    Ag = A.clone().requires_grad_(); Bg = Bt.clone().requires_grad_()
    s, _ = contrastive_terms(Ag.view(B, D, P).permute(0, 2, 1), Bg.view(B, D, P).permute(0, 2, 1), W, terms(na, nb))
    (3.0 * s[:, 1].sum()).backward()
    assert rel(Ag.grad, 3.0 * Ar.grad) < 1e-5 and rel(Bg.grad, 3.0 * Br.grad) < 1e-5


def test_host_buffer_entry_point(golden_dir):
    import ctypes
    g = _golden(golden_dir, "loss_default_d3")
    A = np.ascontiguousarray(g["A"]); B = np.ascontiguousarray(g["B"])
    _, D, H, W = A.shape
    five = np.zeros(5, dtype=np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    idx = [np.ascontiguousarray(g[k]) for k in ("matches_a", "matches_b", "masked_a", "masked_b", "background_a", "background_b")]
    rc = N.lib.ddn_within_scene_loss_host(p(A), p(B), 1, H, W, D, p(idx[0]), p(idx[1]), len(idx[0]), p(idx[2]), p(idx[3]),
                                          len(idx[2]), p(idx[4]), p(idx[5]), len(idx[4]), 0.5, 0.5, 1.0, 1.0, 1, p(five))
    N.check(rc)
    np.testing.assert_allclose(five[:4], g["five"][:4], rtol=2e-6, atol=1e-7)


def test_find_best_matches_cuda_vs_numpy_reference():
    """Batched device-side best match vs the reference's numpy scan (net.py:488-525), on the strided [H,W,D] view that
    forward_single_image_tensor returns; includes an exact tie (first minimum wins, like numpy.argmin)."""
    H, W, D, Q = 120, 160, 3, 37
    gen = torch.Generator().manual_seed(12)
    a = torch.randn(1, D, H, W, generator=gen); b = torch.randn(1, D, H, W, generator=gen)
    b[0, :, 50, 60] = b[0, :, 10, 20]                                  # duplicate descriptor -> tie
    res_a = a[0].permute(1, 2, 0); res_b = b[0].permute(1, 2, 0)        # strided views, like the network output
    px = torch.stack([torch.randint(0, W, (Q,), generator=gen), torch.randint(0, H, (Q,), generator=gen)], 1)
    with torch.no_grad():
        a[0, :, px[0, 1], px[0, 0]] = b[0, :, 10, 20]                   # query 0 matches the duplicated pixel exactly
    uv, diff, nd = pdc_b200.DenseCorrespondenceNetwork.find_best_matches_cuda(px, res_a.to(DEV), res_b.to(DEV), return_norm_diffs=True)
    ra, rb = res_a.numpy(), res_b.numpy()
    for i in range(Q):
        ref_uv, ref_diff, ref_nd = pdc_b200.DenseCorrespondenceNetwork.find_best_match((int(px[i, 0]), int(px[i, 1])), ra, rb)
        got_uv = (int(uv[i, 0]), int(uv[i, 1]))
        if got_uv != ref_uv:        # only allowed when the two candidates are numerically tied
            assert abs(ref_nd[got_uv[1], got_uv[0]] - ref_diff) < 1e-6, (i, got_uv, ref_uv)
        assert abs(float(diff[i]) - float(ref_diff)) < 1e-5
        if i < 3:
            np.testing.assert_allclose(nd[i].cpu().numpy(), ref_nd, rtol=1e-5, atol=1e-6)
    assert (int(uv[0, 0]), int(uv[0, 1])) == (20, 10) and float(diff[0]) == 0.0     # first of the two exact matches
    # masked variant (evaluation.py:1052-1059): best match restricted to the object mask of image b, same pass
    mask = torch.zeros(H, W); mask[30:90, 40:130] = 1.0
    out = pdc_b200.DenseCorrespondenceNetwork.find_best_matches_cuda(px, res_a.to(DEV), res_b.to(DEV), mask_b=mask)
    assert len(out) == 4 and torch.equal(out[0], uv)
    mnp = mask.numpy()
    for i in range(Q):
        _, _, ref_nd = pdc_b200.DenseCorrespondenceNetwork.find_best_match((int(px[i, 0]), int(px[i, 1])), ra, rb)
        masked = ref_nd + (1 - mnp) * 1e6
        idx = np.unravel_index(np.argmin(masked), masked.shape)
        got = (int(out[2][i, 1]), int(out[2][i, 0]))
        assert got == (int(idx[0]), int(idx[1])) or abs(masked[got] - masked[idx]) < 1e-6, i
        assert mnp[got] == 1.0 and abs(float(out[3][i]) - float(masked[idx])) < 1e-5


@pytest.mark.parametrize("mask_kind", ["blob", "none", "empty", "full", "single"])
def test_device_non_match_sampling_matches_restated_reference(mask_kind):
    """ddn_sample_non_matches vs the restated create_non_correspondences + create_non_matches + flatten_uv_tensor on the same
    uniform numbers: bit-identical indices (the reference draws them with torch.rand on the CPU)."""
    from pdc_b200 import sampling
    H, W, Nm, k = 480, 640, 300, 150
    gen = torch.Generator().manual_seed(31)
    matches_a = torch.randint(0, H * W, (Nm,), generator=gen)
    if mask_kind == "none":
        mask = None
    else:
        mask = torch.zeros(H, W)
        if mask_kind == "blob":
            mask[100:333, 217:505] = (torch.rand(233, 288, generator=gen) > 0.3).float()
            mask[0, 0] = 1.0; mask[H - 1, W - 1] = 2.5
        elif mask_kind == "full":
            mask.fill_(1.0)
        elif mask_kind == "single":
            mask[77, 123] = 1.0
    ru = torch.rand(Nm * k, generator=gen); rv = torch.rand(Nm * k, generator=gen)
    ref_a, ref_b = LO.create_non_correspondences_flat(matches_a, (H, W), k, mask, ru, rv)
    got_a, got_b = sampling.sample_non_matches(matches_a.to(DEV), None if mask is None else mask.to(DEV), (H, W), k,
                                               rand=(ru.to(DEV), rv.to(DEV)))
    assert torch.equal(got_a.cpu(), ref_a) and torch.equal(got_b.cpu(), ref_b)
    if mask is not None and mask_kind != "empty":
        assert bool((mask.view(-1)[got_b.cpu()] != 0).all())           # every sample lies on the mask
    # without explicit numbers: right structure and range, and the loss kernels accept the result directly
    a2, b2 = sampling.sample_non_matches(matches_a.to(DEV), None if mask is None else mask.to(DEV), (H, W), k)
    assert torch.equal(a2.cpu(), matches_a.repeat_interleave(k)) and int(b2.min()) >= 0 and int(b2.max()) < H * W


def test_device_reprojection_match_finder_vs_restated_reference():
    """ddn_find_pixel_correspondences vs the restated batch_find_pixel_correspondences on a synthetic scene: a tilted plane
    seen from two poses, with a depth hole, an occluder in view B and candidates partly outside B's frustum."""
    from pdc_b200 import sampling
    import numpy
    H, W, n = 480, 640, 10000
    K = numpy.array([[533.6422696034836, 0, 319.4091030774892], [0, 534.7824445233571, 236.4374299691866], [0, 0, 1.0]])
    def pose(rx, ry, t):
        cx, sx, cy, sy = numpy.cos(rx), numpy.sin(rx), numpy.cos(ry), numpy.sin(ry)
        Rx = numpy.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]); Ry = numpy.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        T = numpy.eye(4); T[:3, :3] = Ry.dot(Rx); T[:3, 3] = t
        return T
    pose_a = pose(0.02, -0.03, [0.0, 0.0, 0.0]); pose_b = pose(-0.05, 0.12, [0.18, -0.04, 0.05])
    # scene: plane z_world = 1.2 + 0.1 x - 0.05 y; render both depth images by ray casting (exact)
    def render(T):
        us, vs = numpy.meshgrid(numpy.arange(W), numpy.arange(H))
        rays = numpy.linalg.inv(K).dot(numpy.stack([us.ravel(), vs.ravel(), numpy.ones(H * W)]))
        rw = T[:3, :3].dot(rays); o = T[:3, 3]
        nrm = numpy.array([-0.1, 0.05, 1.0]); d0 = 1.2
        s = (d0 - nrm.dot(o)) / nrm.dot(rw)
        return (s * 1000.0).reshape(H, W)        # depth along the optical axis = s (rays have z = 1), millimetres
    depth_a = numpy.round(render(pose_a)).astype(numpy.float32); depth_b = numpy.round(render(pose_b)).astype(numpy.float32)
    depth_a[200:230, 300:340] = 0.0                   # sensor hole in A
    depth_b[100:260, 380:470] = 600.0                 # an occluder close to camera B
    gen = torch.Generator().manual_seed(4)
    cand = torch.randint(0, H * W, (n,), generator=gen)
    ref_a, ref_b = LO.batch_find_pixel_correspondences(depth_a, pose_a, depth_b, pose_b, cand, K)
    ga, gb, gu2, gv2 = sampling.find_pixel_correspondences(torch.from_numpy(depth_a).to(DEV), pose_a, torch.from_numpy(depth_b).to(DEV),
                                                         pose_b, cand.to(DEV), K)
    ref_a_flat = ref_a[1] * W + ref_a[0]; ref_b_flat = ref_b[1].long() * W + ref_b[0].long()
    assert 0.3 * n < len(ref_a_flat) < 0.95 * n        # all pruning branches are exercised
    ga, gb = ga.cpu(), gb.cpu()
    # fp32 mat-mul rounding order (MKL vs FFMA) may flip a borderline candidate or move a match by one pixel: allow 0.2 %
    ra = {int(a): int(b) for a, b in zip(ref_a_flat.tolist(), ref_b_flat.tolist())}
    same = sum(1 for a, b in zip(ga.tolist(), gb.tolist()) if ra.get(a) == b)
    assert abs(len(ga) - len(ref_a_flat)) <= 0.002 * n and same >= 0.998 * len(ref_a_flat), (len(ga), len(ref_a_flat), same)
    if len(ga) == len(ref_a_flat) and torch.equal(ga, ref_a_flat):
        assert float((gu2.cpu() - ref_b[0]).abs().max()) < 2e-2 and float((gv2.cpu() - ref_b[1]).abs().max()) < 2e-2


# ---------------------------------------------------------------------------------------------------- round 2
@pytest.mark.parametrize("over", [{}, {"scale_by_hard_negatives": False},
                                  {"use_l2_pixel_loss_on_masked_non_matches": True, "use_l2_pixel_loss_on_background_non_matches": True, "M_pixel": 9}])
@pytest.mark.parametrize("path", ["generic", "fused"])
def test_ragged_batch_matches_the_reference_loop(path, over):
    """Real SpartanDataset samples have a different number of matches per pair (num_matching_attempts is only an upper bound,
    dataset/spartan_dataset_masked.py:652-660), so a batch is ragged: rows padded with -1 + per-pair counts.  The fused loss
    must equal the mean over the pairs of the reference's per-pair loss on the un-padded lists (values, all five outputs,
    gradients).  generic: gathered from full-resolution descriptor images.  fused: the images are bilinear upsamples of
    low-resolution maps they are tagged with (what Resnet34_8s returns), so the loss runs through csrc/loss_lowres.cu and the
    gradient w.r.t. the low-resolution maps is compared."""
    H, W, D, B = 24, 32, 4, 3
    P = H * W
    gen = torch.Generator().manual_seed(11)
    if path == "generic":
        A = 0.3 * torch.randn(B, D, H, W, generator=gen); Bt = 0.3 * torch.randn(B, D, H, W, generator=gen)
    else:
        lows = [(0.3 * torch.randn(B, D, H // 8, W // 8, generator=gen)).requires_grad_() for _ in range(2)]
        A, Bt = [F.interpolate(t, size=(H, W), mode="bilinear", align_corners=True) for t in lows]
    n_match, k_m, k_b, n_blind = [41, 7, 23], 3, 2, [5, 0, 9]
    lists = {k: [] for k in ("matches_a", "matches_b", "masked_a", "masked_b", "background_a", "background_b", "blind_a", "blind_b")}
    for b in range(B):
        ma = torch.randint(0, P, (n_match[b],), generator=gen); mb = torch.randint(0, P, (n_match[b],), generator=gen)
        lists["matches_a"].append(ma); lists["matches_b"].append(mb)
        lists["masked_a"].append(ma.repeat_interleave(k_m)); lists["masked_b"].append(torch.randint(0, P, (n_match[b] * k_m,), generator=gen))
        lists["background_a"].append(ma.repeat_interleave(k_b)); lists["background_b"].append(torch.randint(0, P, (n_match[b] * k_b,), generator=gen))
        if n_blind[b]:
            lists["blind_a"].append(torch.randint(0, P, (n_blind[b],), generator=gen)); lists["blind_b"].append(torch.randint(0, P, (n_blind[b],), generator=gen))
        else:       # this pair has no blind non-matches: the reference's [-1] sentinel
            lists["blind_a"].append(LO.empty_tensor()); lists["blind_b"].append(LO.empty_tensor())
    cfg = dict(LO.DEFAULT_LOSS_CONFIG); cfg.update(over)
    # reference: per-pair loop over the un-padded lists, mean over pairs
    Ar = A.detach().clone().requires_grad_(); Br = Bt.detach().clone().requires_grad_()
    ref = LO.TorchPixelwiseContrastiveLoss([H, W], dict(cfg))
    par, pbr = process_network_output(Ar, B, D, H, W), process_network_output(Br, B, D, H, W)
    outs = [LO.get_within_scene_loss(ref, par[b:b + 1], pbr[b:b + 1], *[lists[k][b] for k in
            ("matches_a", "matches_b", "masked_a", "masked_b", "background_a", "background_b", "blind_a", "blind_b")]) for b in range(B)]
    five_r = [sum(o[i].reshape(()) for o in outs) / B for i in range(5)]
    five_r[0].backward()
    # ours: padded [B, n_max] + per-pair counts
    Ag = A.detach().to(DEV).requires_grad_(); Bg = Bt.detach().to(DEV).requires_grad_()
    pag, pbg = process_network_output(Ag, B, D, H, W), process_network_output(Bg, B, D, H, W)
    if path == "fused":
        low_g = [nhwc(t.detach()).reshape(B, (H // 8) * (W // 8), D).to(DEV).requires_grad_() for t in lows]
        from pdc_b200 import resnet_dilated
        resnet_dilated.attach_lowres(pag, low_g[0], H, W); resnet_dilated.attach_lowres(pbg, low_g[1], H, W)
    pad = {k: loss_composer.pad_index_lists(v, device=DEV) for k, v in lists.items()}
    blind_len = torch.tensor([n if n else 0 for n in n_blind], dtype=torch.int64, device=DEV)
    nv = {"matches": pad["matches_a"][1], "masked": pad["masked_a"][1], "background": pad["background_a"][1], "blind": blind_len}
    ours = pdc_b200.PixelwiseContrastiveLoss([H, W], dict(cfg))
    five = loss_composer.get_loss(ours, torch.zeros(B, dtype=torch.int64), pag, pbg, pad["matches_a"][0], pad["matches_b"][0],
                                  pad["masked_a"][0], pad["masked_b"][0], pad["background_a"][0], pad["background_b"][0],
                                  pad["blind_a"][0], pad["blind_b"][0], num_valid=nv)
    for i in range(5):
        assert abs(float(five[i]) - float(five_r[i])) <= 2e-6 * max(1.0, abs(float(five_r[i]))), (i, float(five[i]), float(five_r[i]))
    five[0].backward()
    if path == "generic":
        assert rel(Ag.grad, Ar.grad) < 1e-5 and rel(Bg.grad, Br.grad) < 1e-5
    else:                   # the full-resolution images were never differentiated; upsample^T of the reference gradient
        assert Ag.grad is None and Bg.grad is None
        A.backward(Ar.grad); Bt.backward(Br.grad)
        for t_g, t_r in zip(low_g, lows):
            assert rel(t_g.grad, nhwc(t_r.grad).reshape(B, -1, D)) < 1e-5


def test_triplet_loss_matches_the_oracle():
    """PixelwiseContrastiveLoss.get_triplet_loss / loss_composer.get_within_scene_loss_triplet
    (pixelwise_contrastive_loss.py:103-129, loss_composer.py:145-166): values and gradients."""
    H, W, D = 24, 32, 5
    P = H * W
    gen = torch.Generator().manual_seed(4)
    A = 0.3 * torch.randn(1, D, H, W, generator=gen); Bt = 0.3 * torch.randn(1, D, H, W, generator=gen)
    ma = torch.randint(0, P, (29,), generator=gen); mb = torch.randint(0, P, (29,), generator=gen)
    na = ma.repeat_interleave(4); nb = torch.randint(0, P, (116,), generator=gen)
    ga = ma.repeat_interleave(2); gb = torch.randint(0, P, (58,), generator=gen)
    cfg = dict(LO.DEFAULT_LOSS_CONFIG)
    ref = LO.TorchPixelwiseContrastiveLoss([H, W], cfg); ours = pdc_b200.PixelwiseContrastiveLoss([H, W], cfg)
    Ar = A.clone().requires_grad_(); Br = Bt.clone().requires_grad_()
    Ag = A.to(DEV).requires_grad_(); Bg = Bt.to(DEV).requires_grad_()
    par, pbr = process_network_output(Ar, 1, D, H, W), process_network_output(Br, 1, D, H, W)
    pag, pbg = process_network_output(Ag, 1, D, H, W), process_network_output(Bg, 1, D, H, W)
    c = lambda t: t.to(DEV)
    r = ref.get_triplet_loss(par, pbr, ma, mb, na, nb, 0.1)
    o = ours.get_triplet_loss(pag, pbg, c(ma), c(mb), c(na), c(nb), 0.1)
    assert abs(float(r) - float(o)) <= 1e-6 * max(1.0, abs(float(r)))
    r5 = (ref.get_triplet_loss(par, pbr, ma, mb, na, nb, cfg["alpha_triplet"]) + ref.get_triplet_loss(par, pbr, ma, mb, ga, gb, cfg["alpha_triplet"]))
    o5 = loss_composer.get_within_scene_loss_triplet(ours, pag, pbg, c(ma), c(mb), c(na), c(nb), c(ga), c(gb), None, None)
    assert abs(float(r5) - float(o5[0])) <= 1e-6 * max(1.0, abs(float(r5)))
    assert all(float(t) == 0.0 for t in o5[1:])
    r5.backward(); o5[0].backward()
    assert rel(Ag.grad, Ar.grad) < 1e-5 and rel(Bg.grad, Br.grad) < 1e-5


@pytest.mark.parametrize("D,over", [(3, {}), (16, {}), (8, {"use_l2_pixel_loss_on_masked_non_matches": True, "M_pixel": 9,
                                                        "scale_by_hard_negatives": False}),
                                    (32, {}), (5, {}), (16, {"use_l2_pixel_loss_on_masked_non_matches": True, "M_pixel": 25}),
                                    (1, {}), (4, {}), (4, {"use_l2_pixel_loss_on_background_non_matches": True, "M_pixel": 9}),
                                    (12, {}), (24, {})])
def test_loss_fused_with_the_upsample_equals_the_generic_loss(D, over):
    """csrc/loss_lowres.cu: the loss evaluated through the bilinear upsample (4 low-resolution cells per sampled pixel) must equal
    the loss gathered from the upsampled image -- all five outputs, hard-negative counts -- and its gradient w.r.t. the
    low-resolution map must equal upsample^T of the generic path's full-resolution gradient.  D = 4 is the float4 / red.v4
    instantiation, 8 / 16 / 32 the channel-quad kernels, every other D the run-time-D scalar kernel."""
    _check_fused_loss_equals_generic(D, over, 64, 96)


@pytest.mark.parametrize("D", [1, 3, 4, 8, 12, 32])
def test_loss_fused_with_the_upsample_on_an_odd_low_resolution_map(D):
    """40x56 images: a 5x7 low-resolution map (35 cells per image, neither even nor a multiple of 4)."""
    _check_fused_loss_equals_generic(D, {}, 40, 56)


def _check_fused_loss_equals_generic(D, over, H, W):
    B = 2
    h, w, P = H // 8, W // 8, H * W
    gen = torch.Generator().manual_seed(21)
    low = [(0.3 * torch.randn(B, h * w, D, generator=gen)).to(DEV) for _ in range(2)]
    nchw = lambda t: t.view(B, h, w, D).permute(0, 3, 1, 2).contiguous()
    ma = torch.randint(0, P, (B, 40), generator=gen).to(DEV); mb = torch.randint(0, P, (B, 40), generator=gen).to(DEV)
    ma[:, 0] = 0; mb[:, 0] = P - 1; ma[:, 1] = W - 1; mb[:, 1] = P - W         # image corners: the clamped edge cells of the blend
    na = ma.repeat_interleave(3, dim=1); nb = torch.randint(0, P, (B, 120), generator=gen).to(DEV)
    ga = ma.repeat_interleave(2, dim=1); gb = torch.randint(0, P, (B, 80), generator=gen).to(DEV)
    xa = torch.randint(0, P, (B, 17), generator=gen).to(DEV); xb = torch.randint(0, P, (B, 17), generator=gen).to(DEV)
    cfg = dict(LO.DEFAULT_LOSS_CONFIG); cfg.update(over)
    pcl = pdc_b200.PixelwiseContrastiveLoss([H, W], cfg)
    pcl.debug = True
    mt = torch.zeros(B, dtype=torch.int64)
    from pdc_b200 import resnet_dilated
    res = {}
    for path in ("generic", "fused"):
        lows = [t.clone().requires_grad_() for t in low]
        imgs = [ops.upsample_bilinear_forward(nchw(t.detach()), H, W).requires_grad_() for t in lows]
        preds = [y.view(B, D, P).permute(0, 2, 1) for y in imgs]
        if path == "fused":
            for p_, l_ in zip(preds, lows):
                resnet_dilated.attach_lowres(p_, l_, H, W)
        five = loss_composer.get_loss(pcl, mt, preds[0], preds[1], ma, mb, na, nb, ga, gb, xa, xb)
        five[0].backward()
        if path == "generic":      # push the full-resolution gradient through the upsample's adjoint
            g = [ops.upsample_bilinear_backward(y.grad, h, w).permute(0, 2, 3, 1).reshape(B, h * w, D) for y in imgs]
            assert lows[0].grad is None
        else:
            g = [t.grad for t in lows]
            assert imgs[0].grad is None                     # the full-resolution image was never differentiated
        res[path] = ([float(t) for t in five], pcl.debug_data["num_hard_negatives_device"].clone(), g)
    (f0, c0, g0), (f1, c1, g1) = res["generic"], res["fused"]
    assert torch.equal(c0, c1)
    for a, b in zip(f0, f1):
        assert abs(a - b) <= 2e-6 * max(1.0, abs(a)), (f0, f1)
    assert rel(g1[0], g0[0]) < 2e-5 and rel(g1[1], g0[1]) < 2e-5
    # a modified image must NOT use the stale low-resolution map
    y = ops.upsample_bilinear_forward(nchw(low[0]), H, W)
    resnet_dilated.attach_lowres(y, low[0], H, W)
    assert resnet_dilated.lowres_of(y) is not None
    y.mul_(2.0)
    assert resnet_dilated.lowres_of(y) is None
