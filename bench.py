#!/usr/bin/env python
"""bench.py -- image-pairs/s of the dense-descriptor training hot path (fwd(A) + fwd(B) + loss + backward) at 640x480.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c5] [--two-calls]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One JSON line on stdout (rank 0).  Workload (default `--config c2`) = BASELINE.json configs[1] ("batch 8 pairs, Resnet34_8s
D=3, single B200, fused fwd+loss+bwd") per GPU; N GPUs = weak scaling, 8 pairs per GPU, the gradient all-reduce OVERLAPPED
with the backward (configs[3] at N=8).  `--config c5` (or DDN_BENCH_CONFIG=c5) = BASELINE.json configs[4]: 32 pairs over 8 GPUs
= 4 pairs per GPU, D=8, 1000 matches + 5000 masked + 5000 background non-matches per pair, hard-negative scaling.  Inputs are
synthetic (pdc_b200.synthetic, SURVEY.md 8d), weights are the reference's own random init.

  value            pairs/s with the step's inputs already resident in HBM (CUDA events, max over ranks)
  e2e              the same step through the reference-facing Python API starting from PINNED HOST buffers:
                   H2D copies of both image batches and all index tensors and the D2H read of the loss are inside
                   the timed region (what dense_correspondence/training/training.py:311-345 does per step)
  roofline         the convolution contraction kernels (forward, data-grad, weight-grad), timed individually with
                   CUDA events on the launching stream during the timed region; achieved = algorithmic conv FLOPs
                   (2*MACs, SURVEY.md 8d) / summed kernel time, against the measured dense bf16 peak
  train_step_with_adam   the same step + FusedAdam.step() (so the weight packs are re-made every step, as in real training)
  forward_b16      north_star's forward target: Resnet34_8s forward only, D=3, 640x480, batch 16 (train- and eval-mode BN)
  gpu_torch_baseline     configs[1] "vs reference GPU PyTorch": the oracle modules on the SAME GPU through PyTorch / cuDNN
  cpu_baseline     the CPU oracle port of the same step on this box's host cores (bounded sample)
  allreduce_check  (N > 1) the overlapped all-reduce left bit-identical gradients on every rank, equal to the mean of the
                   ranks' local gradients

``--impl reference`` times the reference's own algorithm on the host CPU (the oracle port, pinned bit-for-bit to the
executed reference source by tests/test_oracle_ref_cpu.py; the reference itself is Python 2 + needs its dataset stack, so it
cannot run as a whole here -- see DESIGN.md) for the same metric on the same 8-pair batches, without loading libddn_b200.so.
"""
import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

F_IMG = {3: 211.909e9, 8: 211.934e9, 16: 211.973e9}   # conv FLOPs per 640x480 image forward (SURVEY.md 8d)
CONV1_DGRAD = 1.445e9

CONFIGS = {
    # BASELINE.json configs[1] (and, at N = 8, configs[3]: 64 pairs over 8 GPUs)
    "c2": dict(name="configs[1]", pairs_per_gpu=8, D=3, matches=1000, masked=1000, background=1000, l2_pixel=False),
    # BASELINE.json configs[4]: batch 32 pairs over 8 GPUs, D=8, masked + background non-matches + hard-negative scaling
    "c5": dict(name="configs[4] per-GPU shard", pairs_per_gpu=4, D=8, matches=1000, masked=5000, background=5000, l2_pixel=False),
}


def flops_per_pair(D, H, W):
    f = F_IMG.get(D, 211.909e9 + (D - 3) * 2 * 512 * 4800) * (H * W) / (480.0 * 640.0)
    return 2 * f + 2 * (2 * f - CONV1_DGRAD * (H * W) / (480.0 * 640.0))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1400.0, "fallback"


def load_synthetic():
    """pdc_b200.synthetic loaded by path: pure torch, and importing it this way does NOT load libddn_b200.so (the reference
    arm must not map the product library)."""
    spec = importlib.util.spec_from_file_location(
        "_ddn_synthetic", os.path.join(ROOT, "pytorch-dense-correspondence_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class ClockSampler(object):
    """Samples SM clock / throttle reasons of one GPU every 50 ms while the timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self._stop = index, [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------------- CPU arm
_cpu_threads = [None]


def usable_cpu_threads():
    """Host threads the CPU arm can really use: affinity mask, cgroup quota, then a short calibration (a container can
    advertise 128 logical CPUs and still be throttled to a few -- 128 torch threads then run ~70x slower than 8)."""
    if _cpu_threads[0] is not None:
        return _cpu_threads[0]
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    from oracle.resnet34_8s_oracle import seeded_oracle
    net = seeded_oracle(D=3, seed=0).eval()
    x = torch.randn(1, 3, 240, 320)
    best, best_t = n, None
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n})
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            net(x)
            t0 = time.perf_counter(); net(x); dt = time.perf_counter() - t0
            if best_t is None or dt < best_t * 0.95:
                best, best_t = c, dt
    _cpu_threads[0] = best
    return best


def cpu_reference_rate(cfg, H, W, steps, warmup, budget_s, backward=True):
    """The oracle port (plain PyTorch fp32 on the host cores) on the SAME batches as the GPU arm: fwd(A), fwd(B) over all
    `pairs_per_gpu` pairs of a step, within-scene loss[, backward].  `steps`/`warmup` are cut down so that the whole call stays
    within ~budget_s seconds (the cut is reported).  -> (pairs/s, threads, timed steps, warm-up steps, wall seconds)"""
    from oracle import loss_oracle as LO
    from oracle.resnet34_8s_oracle import seeded_oracle, process_network_output
    synthetic = load_synthetic()
    torch.set_num_threads(usable_cpu_threads())
    D, B = cfg["D"], cfg["pairs_per_gpu"]
    net = seeded_oracle(D=D, seed=0).train()
    pcl = LO.TorchPixelwiseContrastiveLoss([H, W], dict(LO.DEFAULT_LOSS_CONFIG))
    data = synthetic.make_pair_batch(B, H, W, cfg["matches"], cfg["masked"], cfg["background"], 0, seed=1)
    times, t_start, done_warm = [], time.perf_counter(), 0
    it = 0
    while True:
        t0 = time.perf_counter()
        net.zero_grad(set_to_none=True)
        with torch.set_grad_enabled(backward):
            ya = net(data["img_a"]); yb = net(data["img_b"])
            five = LO.batched_within_scene_loss(pcl, process_network_output(ya, B, D, H, W),
                                                process_network_output(yb, B, D, H, W), data)
            if backward:
                five[0].backward()
        float(five[0].detach())
        dt = time.perf_counter() - t0
        it += 1
        if done_warm < warmup and (it == 1 or (time.perf_counter() - t_start) + 2 * dt < budget_s * 0.5):
            done_warm += 1              # warm-up steps as long as they fit in half the budget (always at least one)
            continue
        times.append(dt)
        if len(times) >= steps or (time.perf_counter() - t_start) + dt > budget_s:
            break
    times.sort()
    return B / times[len(times) // 2], torch.get_num_threads(), len(times), done_warm, time.perf_counter() - t_start


def workload_text(cfg, H, W, extra=""):
    return ("%s: batch %d pairs/GPU, Resnet34_8s D=%d, %dx%d, train-mode BN, %d matches + %d masked + %d background non-matches per "
            "pair, loss_composer.get_loss within-scene%s" % (cfg["name"], cfg["pairs_per_gpu"], cfg["D"], W, H, cfg["matches"],
                                                            cfg["masked"], cfg["background"], extra))


def _library_mapped():
    try:
        return "libddn_b200" in open("/proc/self/maps").read()
    except Exception:
        return None


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H, W = args.height, args.width
    rate, cores, steps, warm, wall = cpu_reference_rate(cfg, H, W, max(1, args.steps), max(1, args.warmup), budget_s=150.0)
    line = {
        "impl": "reference", "metric": "image-pairs/s (640x480, D=%d) fwd+loss+bwd" % cfg["D"], "value": rate, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1000.0 * cfg["pairs_per_gpu"] / rate,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(cfg, H, W, ", no optimizer step; the reference arm runs the same %d-pair batches on the host CPU"
                                             % cfg["pairs_per_gpu"]),
                   "requested_steps": args.steps, "requested_warmup": args.warmup},
        "cpu_baseline": {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": "%d timed steps of %d pairs each (fwd A, fwd B, loss, backward) after %d warm-up step(s), the oracle port on "
                                   "the host CPU, median; %.1f s wall (step counts are cut to a ~150 s budget)"
                                   % (steps, cfg["pairs_per_gpu"], warm, wall)},
        "e2e": {"value": rate, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "libddn_b200_mapped": _library_mapped(),      # must be false: this arm is the oracle alone
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------- GPU arm helpers
def _event_time(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def forward_b16_leg(N, pdc_b200, tf_peak, steps=6, warmup=3):
    """north_star: '>= 90 % of the tensor-pipe roofline for the Resnet34_8s forward at D=3, 640x480, batch 16'."""
    D, B, H, W = 3, 16, 480, 640
    net = pdc_b200.Resnet34_8s(num_classes=D).cuda()
    x = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(1)).cuda()
    rows = {}
    for mode in ("train", "eval"):
        net.train(mode == "train")
        with torch.no_grad():
            for _ in range(warmup):
                net(x)
            torch.cuda.synchronize()
            l0 = N.launch_count()
            ms = _event_time(lambda: net(x), steps)
            launches = (N.launch_count() - l0) // steps
            N.lib.ddn_profile_reset(); N.lib.ddn_profile_enable(1)
            for _ in range(steps):
                net(x)
            torch.cuda.synchronize()
            N.lib.ddn_profile_enable(0)
        conv = N.profile_read().get("conv_fwd_tc")
        useful_whole = B * F_IMG[3] / (ms * 1e-3) / 1e12
        row = {"ms_per_forward": ms, "imgs_per_s": B / (ms * 1e-3), "launches_per_forward": launches,
               "roofline": {"bound": "tensor", "achieved": useful_whole, "peak": tf_peak, "unit": "TFLOP/s", "frac": useful_whole / tf_peak,
                            "issued_frac": 3 * useful_whole / tf_peak, "traffic": None,
                            "note": "whole forward, algorithmic conv FLOPs / elapsed; bf16x3 issues 3 MMAs per useful MAC"}}
        if conv and conv["ms"] > 0:
            u = conv["flops"] / (conv["ms"] * 1e-3) / 1e12
            row["conv_kernels"] = {"ms": conv["ms"] / steps, "share_of_forward": conv["ms"] / steps / ms, "useful_TFLOPs": u,
                                   "issued_frac_of_peak": 3 * u / tf_peak}
        rows[mode + "_bn"] = row
    del net, x
    torch.cuda.empty_cache()
    out = {"workload": "Resnet34_8s forward only, D=3, 640x480, batch 16, bf16x3, inputs resident, %d timed forwards after %d warm-up" % (steps, warmup)}
    out.update(rows)
    return out


def gpu_torch_baseline_leg(cfg, H, W, dev):
    """configs[1] 'vs reference GPU PyTorch': the oracle modules (the reference's layers restated in plain PyTorch, bit-equal to
    the reference modules on CPU) on the same GPU through PyTorch / cuDNN: strict fp32 (the parity reference), TF32 convolutions
    (fails the 1e-3 gate) and bf16 autocast channels_last (context only).  Bounded: 2 warm-up + 3 timed steps each."""
    from oracle import loss_oracle as LO
    from oracle.resnet34_8s_oracle import seeded_oracle, process_network_output
    synthetic = load_synthetic()
    D, B = cfg["D"], cfg["pairs_per_gpu"]
    host = synthetic.make_pair_batch(B, H, W, cfg["matches"], cfg["masked"], cfg["background"], 0, seed=1)
    data = {k: v.to(dev) for k, v in host.items() if v is not None}
    pcl_o = LO.TorchPixelwiseContrastiveLoss([H, W], dict(LO.DEFAULT_LOSS_CONFIG))
    rows = []
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for label, tf32, autocast in (("fp32, TF32 off (the parity reference)", False, False),
                                      ("fp32 storage, TF32 convolutions", True, False),
                                      ("bf16 autocast, channels_last", True, True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            net = seeded_oracle(D=D, seed=0).to(dev).train()
            xa, xb = data["img_a"], data["img_b"]
            if autocast:
                net = net.to(memory_format=torch.channels_last)
                xa, xb = xa.contiguous(memory_format=torch.channels_last), xb.contiguous(memory_format=torch.channels_last)

            def step():
                net.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    ya, yb = net(xa), net(xb)
                ya, yb = ya.float().contiguous(), yb.float().contiguous()
                five = LO.batched_within_scene_loss(pcl_o, process_network_output(ya, B, D, H, W), process_network_output(yb, B, D, H, W), data)
                five[0].backward()
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            ms = _event_time(step, 3)
            rows.append({"impl": "oracle modules on PyTorch %s / cuDNN %s: %s" % (torch.__version__, torch.backends.cudnn.version(), label),
                         "ms_per_step": ms, "pairs_per_s": B / (ms * 1e-3)})
            del net
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return {"workload": "same step as `value` (inputs resident), 3 timed steps after 2 warm-up", "rows": rows}


DUMP_SAMPLE = 1 << 21      # elements kept of a larger array: three 8 MB samples + the loss values stay well under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy, float32 (float64 for the loss values).  An array of more than DUMP_SAMPLE
    elements is replaced by the flattened elements at DUMP_SAMPLE sorted flat indices drawn without replacement by
    numpy.random.default_rng(0) -- the same indices for the same shape -- so that two builds run with the same arguments
    can be compared element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def committed_traffic(kernel_class):
    """dram bytes per launch of the dominant kernel class from the committed `ncu --set full` capture, if there is one."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            if kernel_class in d:
                return d[kernel_class].get("dram_bytes_per_launch"), d[kernel_class].get("source")
        except Exception:
            pass
    return None, None


# ---------------------------------------------------------------------------------------------------- GPU arm
def run_ours(args, cfg):
    import torch.distributed as dist
    import pdc_b200
    from pdc_b200 import _native as N, synthetic, loss_composer, data_parallel as DP

    # stdout carries exactly ONE JSON line: anything a library prints while we run (NCCL's version banner ...) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    rank, world, local_rank = DP.init_from_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    H, W, D, Bp = args.height, args.width, cfg["D"], cfg["pairs_per_gpu"]
    prec_name = args.precision
    if prec_name == "auto":
        prec_name = "bf16x3"
    prec = {"fp32": N.PRECISION_FP32_SIMT, "bf16x3": N.PRECISION_BF16X3, "bf16": N.PRECISION_BF16}[prec_name]

    torch.manual_seed(0)
    dcn = pdc_b200.DenseCorrespondenceNetwork.from_config({"descriptor_dimension": D, "image_width": W, "image_height": H},
                                                          load_stored_params=False)
    dcn.fcn.precision = prec
    DP.broadcast_parameters(dcn)
    loss_cfg = dict(pdc_b200.DEFAULT_LOSS_CONFIG)
    if cfg["l2_pixel"]:
        loss_cfg["use_l2_pixel_loss_on_masked_non_matches"] = True
    pcl = pdc_b200.PixelwiseContrastiveLoss(image_shape=dcn.image_shape, config=loss_cfg)
    reducer = DP.GradientAllReducer(dcn.parameters(), module=dcn.fcn, overlap=not args.no_overlap)
    host = synthetic.make_pair_batch(Bp, H, W, cfg["matches"], cfg["masked"], cfg["background"], 0, seed=1 + rank)
    keys = [k for k, v in host.items() if v is not None]
    pinned = {k: host[k].pin_memory() for k in keys}
    resident = {k: host[k].to(dev) for k in keys}
    match_type = torch.zeros(Bp, dtype=torch.int64)          # SINGLE_OBJECT_WITHIN_SCENE, a CPU tensor like the DataLoader's
    blind = loss_composer.empty_tensor().to(dev)
    h2d_bytes = sum(pinned[k].numel() * pinned[k].element_size() for k in keys)

    side = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)] if args.two_streams else None
    last = {}                 # --dump-outputs: what the latest step handed back to its caller

    def forward_loss_backward(d):
        if args.two_streams:      # EXPERIMENT (timing only: shared BN buffers / pack cache / flat gradient are raced)
            cur = torch.cuda.current_stream()
            for s_ in side:
                s_.wait_stream(cur)
            with torch.cuda.stream(side[0]):
                ya = dcn.forward(d["img_a"])
            with torch.cuda.stream(side[1]):
                yb = dcn.forward(d["img_b"])
            for s_ in side:
                cur.wait_stream(s_)
        elif args.two_calls:
            ya, yb = dcn.forward(d["img_a"]), dcn.forward(d["img_b"])
        else:
            ya, yb = dcn.forward_pair(d["img_a"], d["img_b"])
        five = loss_composer.get_loss(pcl, match_type, dcn.process_network_output(ya, Bp), dcn.process_network_output(yb, Bp),
                                      d["matches_a"], d["matches_b"], d["masked_a"], d["masked_b"],
                                      d["background_a"], d["background_b"], blind, blind)
        five[0].backward()
        if args.dump_outputs:
            last.update(five=five, descriptors_a=ya, descriptors_b=yb)
        return five[0]

    def step(d):
        dcn.zero_grad(set_to_none=True)
        out = forward_loss_backward(d)
        reducer()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        step(resident)
    barrier()

    # ---- timed region 1: inputs resident in HBM.  Nothing but the step's own launches is on the stream: the per-kernel event
    # pairs of the roofline pass below would sit between dependent kernels (one event record after every convolution, ~220
    # per step) and defeat the programmatic dependent launch that overlaps one kernel's prologue with its predecessor's tail.
    def timed_steps(instrumented):
        N.lib.ddn_profile_reset()
        N.lib.ddn_profile_enable(1 if instrumented else 0)
        n0 = N.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_host = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            out = step(resident)
        e1.record()
        host_ms = (time.perf_counter() - t_host) * 1e3        # time the host needed to ENQUEUE the steps (the GPU runs behind it)
        barrier()
        N.lib.ddn_profile_enable(0)
        return max_over_ranks(e0.elapsed_time(e1)), N.launch_count() - n0, out, host_ms

    with ClockSampler(local_rank) as clk:
        ms_total, launches, loss, host_ms = timed_steps(False)
    if args.dump_outputs and rank == 0:
        # the last timed step: its five loss values, both descriptor batches and every parameter gradient (after the
        # all-reduce), concatenated in named_parameters() order
        dump_outputs(args.dump_outputs, {
            "loss": torch.tensor([float(t.detach()) for t in last["five"]], dtype=torch.float64),
            "descriptors_a": last["descriptors_a"], "descriptors_b": last["descriptors_b"],
            "param_grads": torch.cat([p.grad.reshape(-1) for _, p in dcn.named_parameters()])})
        last.clear()
    # ---- timed region 1b: the same K steps again with a CUDA-event pair around every convolution / loss kernel on the launching
    # stream (ddn_profile_*): the per-class kernel durations the roofline block is computed from
    if args.profile_run:      # under ncu: warm-up + the timed steps only, so the launch list is exactly `steps` steps
        if rank == 0:
            emit({"profile_run": True, "ms_per_step_under_profiler": ms_total / args.steps})
        return
    ms_instrumented, _, _, _ = timed_steps(True)
    prof = N.profile_read()

    # ---- timed region 2: end to end from pinned host memory, loss read back every step.  Every step's inputs are copied
    # host->device inside the timed region (through DevicePrefetcher: the copy of step i+1 overlaps the compute of step i,
    # like a pinned-memory DataLoader would) and every step's loss is read back with .item().
    def host_batches(n):
        for _ in range(n):
            yield pinned
    def e2e_loop(n):
        """The training loop a user writes around the public API: every step copies its batch host->device (DevicePrefetcher: the
        copy of batch i+1 is enqueued while step i computes) and reads its loss back with .item().  The host work that does not
        depend on that loss -- zero_grad, fetching the next batch -- is done BEFORE the blocking read, so the GPU waits for the host
        only between the read returning and the first launch of the next step."""
        it = iter(DP.DevicePrefetcher(host_batches(n), dev))
        d = next(it, None)
        val = None
        dcn.zero_grad(set_to_none=True)
        while d is not None:
            out = forward_loss_backward(d)
            reducer()                            # (an optimizer step would go here)
            dcn.zero_grad(set_to_none=True)
            d = next(it, None)
            val = float(out.item())
        return val

    e2e_loop(min(args.warmup, 2))
    barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    last_loss = e2e_loop(args.steps)
    ev3.record()
    barrier()
    ms_e2e = max_over_ranks(ev2.elapsed_time(ev3))

    # ---- the step + optimizer (real training re-packs the bf16 weights after every update; `value` above does not pay that)
    opt = pdc_b200.FusedAdam(dcn, lr=1e-6, weight_decay=1e-4)

    def train_step():
        out = step(resident)
        opt.step()
        return out
    for _ in range(2):
        train_step()
    barrier()
    ev4, ev5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev4.record()
    for _ in range(args.steps):
        train_step()
    ev5.record()
    barrier()
    ms_adam = max_over_ranks(ev4.elapsed_time(ev5))

    # ---- N > 1: the reduced gradient is bit-identical on every rank and equals the mean of the ranks' local gradients
    allreduce_check, allreduce_detail = None, None
    if world > 1:
        step(resident)
        g_over = dcn.fcn.flat_gradient.detach().clone()
        ref0 = g_over.clone()
        dist.broadcast(ref0, src=0)
        identical = torch.equal(ref0, g_over)
        overlapped_steps, bytes_last = reducer.overlapped_steps, reducer.bytes_last
        reducer.detach()                                   # local gradients, then the textbook mean
        dcn.zero_grad(set_to_none=True)
        forward_loss_backward(resident)
        g_mean = dcn.fcn.flat_gradient.detach().clone()
        dist.all_reduce(g_mean, op=dist.ReduceOp.SUM)
        g_mean /= world
        err = float((g_over.double() - g_mean.double()).norm() / (g_mean.double().norm() + 1e-30))
        flags = torch.tensor([1.0 if identical else 0.0, -err], device=dev, dtype=torch.float64)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        all_identical, worst_err = bool(flags[0].item() == 1.0), -float(flags[1].item())
        # the two runs differ by the summation order of the weight-gradient atomics (~1e-6 relative), never by more
        allreduce_check = bool(all_identical and worst_err < 1e-4)
        allreduce_detail = {"bit_identical_across_ranks": all_identical, "rel_err_vs_mean_of_local_gradients": worst_err,
                            "overlapped_steps": overlapped_steps, "bytes_per_step": bytes_last}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pairs = world * Bp * args.steps
    value = pairs / (ms_total / 1e3)
    e2e = pairs / (ms_e2e / 1e3)
    hbm_peak, tf_peak, peak_src = measured_peaks()
    conv_ms = sum(v["ms"] for k, v in prof.items() if k.startswith("conv"))
    conv_fl = sum(v["flops"] for k, v in prof.items() if k.startswith("conv"))
    dom = max((k for k in prof if k.startswith("conv")), key=lambda k: prof[k]["ms"], default=None)
    roof = None
    if dom:
        a = prof[dom]["flops"] / (prof[dom]["ms"] * 1e-3) / 1e12 if prof[dom]["ms"] > 0 else 0.0
        mma_per_mac = {"fp32": 0, "bf16x3": 3, "bf16": 1}[prec_name]
        traffic, traffic_src = committed_traffic(dom)
        roof = {"bound": "tensor", "kernel": dom, "achieved": a, "peak": tf_peak, "unit": "TFLOP/s", "frac": a / tf_peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "issued_tensor_TFLOPs": a * mma_per_mac, "issued_frac": a * mma_per_mac / tf_peak,
                "peak_source": peak_src + " bf16_tflops_sustained (kernel timed inside a long step)",
                "launches": prof[dom]["launches"], "avg_launch_ms": prof[dom]["ms"] / max(1, prof[dom]["launches"]),
                "all_conv_achieved": (conv_fl / (conv_ms * 1e-3) / 1e12) if conv_ms > 0 else 0.0,
                "conv_share_of_step": conv_ms / ms_instrumented if ms_instrumented > 0 else None,
                "timed": "a second pass of the same %d steps with a CUDA-event pair around every convolution / loss launch on the launching "
                         "stream; that pass took %.3f ms/step (the uninstrumented pass that `value` comes from: %.3f ms/step)"
                         % (args.steps, ms_instrumented / args.steps, ms_total / args.steps),
                "whole_step_achieved": value * flops_per_pair(D, H, W) / world / 1e12,
                "arithmetic": {"fp32": "fp32 FFMA (CUDA cores)", "bf16x3": "bf16x3 split: 3 tensor-core MMAs per useful MAC",
                               "bf16": "single bf16 MMA"}[prec_name],
                "classes": prof}
    fwd16 = gpu_base = cpu = None
    if world == 1 and not args.quick:
        del opt
        dcn.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
        if prec_name == "bf16x3":
            fwd16 = forward_b16_leg(N, pdc_b200, tf_peak)
        gpu_base = gpu_torch_baseline_leg(cfg, H, W, dev)
        t0 = time.perf_counter()
        rate, cores, n_t, n_w, wall = cpu_reference_rate(cfg, H, W, steps=2, warmup=1, budget_s=45.0, backward=True)
        cpu = {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
               "sample": "oracle port on the host CPU, the same %d-pair batches: %d timed fwd+loss+bwd step(s) (median) after %d warm-up; "
                         "%.1f s of CPU wall" % (Bp, n_t, n_w, time.perf_counter() - t0)}
    line = {
        "metric": "image-pairs/s (640x480, D=%d) fwd+loss+bwd" % D, "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "bf16x3": "f32 (bf16x3 split on tcgen05, fp32 accumulate)", "bf16": "bf16"}[prec_name],
        "data": "synthetic",
        "config": {"workload": workload_text(cfg, H, W, ", no optimizer step"),
                   "api": ("DenseCorrespondenceNetwork.forward(A), .forward(B)" if args.two_calls else
                           "DenseCorrespondenceNetwork.forward_pair(A, B): both reference forward calls as one launch sequence with per-image-batch "
                           "BatchNorm statistics (identical results; `--two-calls` times the two-call form)"),
                   "l2_pixel_loss_on_masked_non_matches": bool(cfg["l2_pixel"]), "global_batch_pairs": world * Bp,
                   "parallelism": "dp%d" % world, "precision": prec_name,
                   "allreduce": (None if world == 1 else ("overlapped with backward (4 buckets, issued as each residual layer's gradients "
                                                          "complete)" if not args.no_overlap else "after backward")),
                   "l2": "inputs+activations touched per step (~%.1f GB) are far larger than the 126 MB L2; no explicit flush" %
                         (N.lib.ddn_resnet34_8s_workspace_bytes(2 * Bp, H, W, D, 1, prec) / 1e9)},
        "clocks": clk.summary(),
        "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps, "last_loss": last_loss},
        "gpu_launches": launches,
        "launches_per_step": launches / float(args.steps),
        "host_enqueue_ms_per_step": host_ms / args.steps,
        "roofline": roof,
        "train_step_with_adam": {"value": pairs / (ms_adam / 1e3), "unit": "pairs/s", "ms_per_step": ms_adam / args.steps,
                                 "includes": "FusedAdam.step() over the flat arrays + the device-side fingerprint and re-pack of all bf16 weight "
                                             "packs that every parameter update triggers"},
        "forward_b16": fwd16,
        "gpu_torch_baseline": gpu_base,
        "cpu_baseline": cpu,
        "loss": float(loss.item()),
    }
    if world > 1:
        line["allreduce_check"] = allreduce_check
        line["allreduce_detail"] = allreduce_detail
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("DDN_BENCH_CONFIG", "c2"), choices=sorted(CONFIGS),
                    help="c2 = BASELINE.json configs[1] (default; configs[3] at --gpus 8), c5 = configs[4] per-GPU shard")
    ap.add_argument("--pairs-per-gpu", type=int, default=None)
    ap.add_argument("--D", type=int, default=None)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--matches", type=int, default=None)
    ap.add_argument("--non-matches", type=int, default=None)
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16x3", "bf16"])
    ap.add_argument("--quick", "--no-cpu-baseline", dest="quick", action="store_true",
                    help="skip the forward_b16 / gpu_torch_baseline / cpu_baseline legs")
    ap.add_argument("--two-calls", action="store_true",
                    help="forward(A), forward(B) as two calls (the reference API) instead of DenseCorrespondenceNetwork.forward_pair")
    ap.add_argument("--two-streams", action="store_true", help="experiment: the two forward calls (and their backwards) on two CUDA streams")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: all-reduce after backward instead of overlapped with it")
    ap.add_argument("--l2-pixel-loss", action="store_true",
                    help="configs[4] variant: use_l2_pixel_loss_on_masked_non_matches=True (M_pixel=50)")
    ap.add_argument("--profile-run", action="store_true",
                    help="short run for ncu: 1 warm-up + --steps timed steps, no e2e / cpu legs (numbers printed are NOT bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss values, descriptors, parameter "
                         "gradients; seeded samples of the large arrays) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.pairs_per_gpu is not None:
        cfg["pairs_per_gpu"] = args.pairs_per_gpu
    if args.D is not None:
        cfg["D"] = args.D
    if args.matches is not None:
        cfg["matches"] = args.matches
    if args.non_matches is not None:
        cfg["masked"] = cfg["background"] = args.non_matches
    if args.l2_pixel_loss:
        cfg["l2_pixel"] = True
    if cfg != CONFIGS[args.config]:
        cfg["name"] = "custom (from %s)" % cfg["name"]
    if args.impl == "reference":
        return run_reference_arm(args, cfg)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            sys.stderr.write("bench.py: --gpus %d needs a torchrun launch (WORLD_SIZE=%d); see the module docstring\n" % (args.gpus, world))
            sys.exit(2)
    if args.profile_run:
        args.warmup, args.quick = 1, True
    elif args.warmup < 3:
        args.warmup = 3
    run_ours(args, cfg)


if __name__ == "__main__":
    main()
