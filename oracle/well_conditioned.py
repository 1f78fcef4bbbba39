"""Well-conditioned whole-network fixtures -- TEST INFRASTRUCTURE, NOT THE PRODUCT.

A randomly initialised Resnet34_8s has a ~1e-2 gradient noise floor even between PyTorch's own CPU and CUDA runs: ReLU /
max-pool decisions flip on 1-ulp differences and train-mode BatchNorm amplifies them.  These fixtures remove that floor by
making the ReLU decisions decisive (``decisive_relu_biases``), so that every parameter gradient of the network can be gated
tightly against the oracle in fp64.  ``reference`` also returns the fp32 CPU oracle's own distance from fp64, the conditioning
certificate: a fixture whose certificate is not < 1e-4 is a badly chosen input, not a kernel bug.

``CASES`` is the shape / descriptor-size / BatchNorm-group matrix the GPU suite runs (tests/test_gpu_network.py); the CPU suite
asserts the certificate of every one of them (tests/test_oracle_cpu.py).
"""
import torch

from oracle.resnet34_8s_oracle import seeded_oracle

SEEDS = (77, 78, 79, 80, 81, 82)

# (D, images per BatchNorm group, groups, H, W, BatchNorm mode, input seeds).  Sub-tiles of the implicit-GEMM convolutions are
# 4 x 16 pixels (two per CTA, four per CTA pair); the layer-1 halo kernels take 8 x 16 tiles and run when layer 1's map (H/4 x W/4)
# is made of whole tiles; the trunk (layer2..4, fc) runs at H/8 x W/8.
# The seeds are inputs on which the fp32 oracle itself flips no mask (certificate ~3e-6; D = 1: <= 2e-5).  Batches stay at or below
# ~8k pixels per step: the bf16x3 forward error (~1e-5) lands one non-decisive relu(bn2(.) + identity) element within rounding of
# zero in about every second input at 12k pixels (64x96 x 2), and in nearly every input at 16k+ (64x128 x 2: 6 of 6 seeds flipped).
CASES = [
    # layer 1 16x16 = 2 halo tiles per image: conv64_halo_kernel with BN statistics (forward) and BN-backward column sums (data
    # gradient), wgrad64_halo_kernel; eval: the same kernels without statistics (frozen BatchNorm, DDN_MODE_EVAL_SAVE)
    (3, 2, 1, 64, 64, "train", SEEDS),
    (3, 1, 2, 64, 64, "train", SEEDS),
    (3, 2, 1, 64, 64, "eval", SEEDS),
    (3, 1, 2, 64, 64, "eval", (77, 78, 79, 81, 82, 83)),
    # layer 1 10x12 = 3 sub-tiles per image: with one image per group the second CTA holds sub-tiles of both groups;
    # h*w = 30, so forward_pair's second half of the low-resolution map is not 16-byte aligned
    (3, 1, 2, 40, 48, "train", SEEDS),
    # trunk 9x5 = 3 sub-tiles per image: with one image per group a CTA (layer2) and a CTA pair (layer3/4) straddle the group
    # boundary; fc_wgrad_kernel with D < DM = 16; h*w = 45
    (12, 2, 1, 72, 40, "train", SEEDS),
    (12, 1, 2, 72, 40, "train", (78, 79, 80, 81, 82, 83)),
    # fc templates with DM = 32; one halo tile (the minimum size); one trunk sub-tile per image
    (32, 1, 1, 32, 64, "train", SEEDS),
    # the minimum shape and D = 1
    (1, 4, 1, 32, 32, "train", (77, 78, 82, 83, 85, 86)),
]


def case_id(case, with_mode=True):
    D, B, G, H, W, mode = case[:6]
    return "D%d-B%dx%d-%dx%d" % (D, B, G, H, W) + ("-" + mode if with_mode else "")


def decisive_relu_biases(net, amp=3.0, on_fraction=0.7, seed=5):
    """BatchNorm biases set to +-amp (70 % of the channels +amp, 30 % -amp): almost every ReLU input is then several standard
    deviations away from zero, so the ReLU masks -- both the passing and the blocking kind -- are the SAME in every arithmetic,
    and the gradient of the whole network becomes a well-conditioned function of its inputs (fp32 vs fp64 CPU oracle: ~3e-6 per
    tensor instead of ~1e-2 with the default biases, where a handful of mask flips at |pre-activation| ~ 1 ulp dominate)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, p in net.named_parameters():
            if ("bn" in k or "downsample.1" in k) and k.endswith(".bias"):
                sign = (torch.rand(p.shape, generator=g) < on_fraction).to(p.dtype) * 2 - 1
                p.copy_(amp * sign)
    return net


def build(mode, D, B, H, W, seed, groups=1):
    """-> (x [groups*B,3,H,W], cotangent [groups*B,D,H,W], fp32 oracle).  The batch is ``groups`` consecutive groups of B images
    (image-A batch, image-B batch for groups=2).  eval: frozen statistics that actually normalise -- one pass over the whole batch
    with momentum 1 copies its batch statistics into the running ones.  The oracle's state is what the network under test loads."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(groups * B, 3, H, W, generator=gen)
    cot = torch.randn(groups * B, D, H, W, generator=gen)
    oracle = decisive_relu_biases(seeded_oracle(D=D, seed=0))
    if mode == "eval":
        bns = [m for m in oracle.modules() if isinstance(m, torch.nn.BatchNorm2d)]
        for m in bns:
            m.momentum = 1.0
        oracle.train()
        with torch.no_grad():
            oracle(x)
        for m in bns:
            m.momentum = 0.1
    return x, cot, oracle


def reference(oracle, mode, x, cot, groups=1):
    """One call of the oracle per group, in order (what ``forward`` per image batch computes), in fp64 and in fp32, with the
    cotangent summed over the groups.  -> (y64, fp64 parameter gradients, names of the gradients that are not negligible,
    their scale, certificate = worst per-tensor distance of the fp32 oracle's gradients from fp64).  The fp32 ``oracle`` is left
    in the state the calls leave it in (running statistics updated group after group in train mode)."""
    ref64 = seeded_oracle(D=oracle.resnet34_8s.fc.out_channels, seed=0).double()
    ref64.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in oracle.state_dict().items()})
    for m in (oracle, ref64):
        m.train(mode == "train")
    y64 = torch.cat([ref64(xg.double()) for xg in x.chunk(groups)])
    (y64 * cot.double()).sum().backward()
    y32 = torch.cat([oracle(xg) for xg in x.chunk(groups)])
    (y32 * cot).sum().backward()
    g64 = {k: p.grad for k, p in ref64.named_parameters()}
    scale = max(float(v.norm()) for v in g64.values())
    big = [k for k in g64 if float(g64[k].norm()) >= 1e-6 * scale]
    cert = max(_rel(p.grad, g64[k]) for k, p in oracle.named_parameters() if k in big)
    return y64.detach(), g64, big, scale, cert


def _rel(a, b):
    a = a.double().cpu(); b = b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
