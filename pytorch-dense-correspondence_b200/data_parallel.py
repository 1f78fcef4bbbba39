"""Data parallelism for the dense-descriptor training step: one process per GPU, independent image pairs per
rank, and exactly one exchange per step -- an all-reduce (SUM, then 1/world) of the fp32 parameter gradients
over NCCL / NVLink (SURVEY.md 8e).  The reference itself is single-GPU (training.py:254-256); BatchNorm
statistics stay per rank, as N independent reference processes would have them.

Because every parameter (and therefore, after backward, every gradient) of ``Resnet34_8s`` aliases one flat
fp32 array, the exchange is a handful of large bucketed all-reduces over slices of that array instead of
110 small ones.  Works on CUDA (nccl) and, for the host-logic tests, on CPU tensors (gloo).
"""
import os

import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """torchrun-style rendezvous from RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT.
    Returns (rank, world_size, local_rank).  A single process (no env) returns (0, 1, 0) without initialising."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local_rank


def shard_range(global_count, rank, world):
    """Consecutive split of ``global_count`` units over ``world`` ranks: -> (start, count).  The first
    ``global_count % world`` ranks take one extra unit."""
    base, extra = divmod(global_count, world)
    count = base + (1 if rank < extra else 0)
    start = rank * base + min(rank, extra)
    return start, count


def broadcast_parameters(module, src=0, group=None):
    """Make every rank start from rank ``src``'s weights and BN buffers (one broadcast per flat array when the
    module exposes them, else per tensor)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    with torch.no_grad():
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t.data, src=src, group=group)
        for m in module.modules():         # writes through .data are invisible to autograd's version counters
            if hasattr(m, "mark_parameters_changed"):
                m.mark_parameters_changed()


def _flat_view_of(tensors):
    """If ``tensors`` tile one contiguous storage in order (gaps of < 16 bytes allowed), return
    (base_tensor_1d covering all of them); else None."""
    if not tensors:
        return None
    t0 = tensors[0]
    if any(t.dtype != t0.dtype or t.device != t0.device or not t.is_contiguous() for t in tensors):
        return None
    es = t0.element_size()
    storage_ptr = t0.untyped_storage().data_ptr()
    if any(t.untyped_storage().data_ptr() != storage_ptr for t in tensors):
        return None
    cursor = t0.data_ptr()
    for t in tensors:
        gap = t.data_ptr() - cursor
        if gap < 0 or gap >= 16:
            return None
        cursor = t.data_ptr() + t.numel() * es
    start = (t0.data_ptr() - storage_ptr) // es
    length = (cursor - t0.data_ptr()) // es
    return torch.empty(0, dtype=t0.dtype, device=t0.device).set_(t0.untyped_storage(), start, (length,), (1,))


class GradientAllReducer(object):
    """Averages ``p.grad`` of the given parameters across the process group.

        reducer = GradientAllReducer(dcn.parameters(), module=dcn.fcn)     # module: the Resnet34_8s that owns them
        loss.backward(); reducer(); optimizer.step()

    With ``module`` given (and ``overlap=True``) the exchange is OVERLAPPED with the backward: the library reports each
    gradient bucket the moment its last kernel is enqueued (ddn_resnet34_8s_backward's ``on_bucket``: layer4 + fc first --
    52 MB of the 85 MB -- then layer3, layer2, layer1 + stem) and the bucket's NCCL all-reduce is issued right there, so it
    runs on NCCL's stream while the remaining weight-gradient kernels still compute; the 1/world factor is folded into the
    cotangent, so no scaling pass exists.  ``reducer()`` after ``backward()`` then only has to confirm that nothing is left.
    Without ``module`` (or for gradients produced some other way) ``reducer()`` does the bucketed all-reduce itself.
    """

    def __init__(self, parameters, group=None, num_buckets=4, module=None, overlap=True):
        self.params = [p for p in parameters if p.requires_grad]
        self.group = group
        self.num_buckets = max(1, int(num_buckets))
        self.bytes_last = 0
        self.used_flat_path = False
        self.overlapped_steps = 0
        self._works = []
        self._covered = 0
        self._done_for = None
        self.module = module
        if module is not None and overlap and dist.is_initialized() and dist.get_world_size(group) > 1:
            module._bucket_hook = self
        elif module is not None:
            module._bucket_hook = None

    # ---- overlapped path: called by resnet_dilated._Backbone.backward
    def cotangent_scale(self):
        return 1.0 / dist.get_world_size(self.group)

    def __call_bucket__(self, flat_grads, bucket, offset, numel):
        if bucket == 0:
            self._works, self._covered = [], 0
        self._works.append(dist.all_reduce(flat_grads[offset:offset + numel], op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        self._covered += numel

    def finish(self, flat_grads):
        """All buckets of this backward are in flight: make the compute stream wait for them (only the tail of the last,
        smallest bucket is ever exposed)."""
        for w in self._works:
            w.wait()
        self._works = []
        self.bytes_last = self._covered * flat_grads.element_size()
        self.used_flat_path = True
        self.overlapped_steps += 1
        self._done_for = flat_grads.data_ptr()

    def detach(self):
        if self.module is not None and getattr(self.module, "_bucket_hook", None) is self:
            self.module._bucket_hook = None

    # ---- explicit path
    def __call__(self):
        if not dist.is_initialized():
            return
        world = dist.get_world_size(self.group)
        if world == 1:
            return
        if self.module is not None and getattr(self.module, "_bucket_hook", None) is self:
            return                        # every backward of this step already reduced its own gradients
        grads = [p.grad for p in self.params if p.grad is not None]
        if not grads:
            return
        flat = _flat_view_of(grads)
        self.used_flat_path = flat is not None
        if flat is None:   # gradients are scattered: pack, reduce, unpack
            flat = torch.cat([g.reshape(-1) for g in grads])
        n = flat.numel()
        self.bytes_last = n * flat.element_size()
        # reverse order: the tail of the flat array (layer4, fc) is what backward finishes first
        bounds = [n * i // self.num_buckets // 4 * 4 for i in range(self.num_buckets)] + [n]
        works = []
        for i in reversed(range(self.num_buckets)):
            if bounds[i + 1] > bounds[i]:
                works.append(dist.all_reduce(flat[bounds[i]:bounds[i + 1]], op=dist.ReduceOp.SUM, group=self.group,
                                             async_op=True))
        for w in works:
            w.wait()
        if flat.is_cuda:
            from . import ops
            ops.scale_inplace(flat, 1.0 / world)
        else:
            flat.mul_(1.0 / world)
        if not self.used_flat_path:
            off = 0
            for g in grads:
                g.copy_(flat[off:off + g.numel()].view_as(g))
                off += g.numel()


class DevicePrefetcher(object):
    """Double-buffered host->device staging of training batches (dicts of pinned CPU tensors): the copies of batch i+1 run on
    a side stream while batch i computes, which is what ``DataLoader(pin_memory=True)`` + ``.cuda(non_blocking=True)`` only
    achieves when somebody issues the next copy early.  The reference copies synchronously inside the step
    (dense_correspondence/training/training.py:311-323).  Two fixed sets of device buffers are reused (no allocation in
    steady state; batches must keep their shapes), so a batch is valid until the next-but-one ``next()``.

        for batch in DevicePrefetcher(iterable_of_dicts, device): ...     # tensors on `device`, ready on the current stream
    """

    def __init__(self, batches, device):
        self.it = iter(batches)
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self._sets = [None, None]
        self._i = 0
        self._next = None
        self._preload()

    def _preload(self):
        try:
            host = next(self.it)
        except StopIteration:
            self._next = None
            return
        slot = self._i & 1
        self._i += 1
        main = torch.cuda.current_stream(self.device)
        if self._sets[slot] is None or any(torch.is_tensor(v) and (k not in self._sets[slot] or self._sets[slot][k].shape != v.shape)
                                            for k, v in host.items()):
            self._sets[slot] = {k: torch.empty(v.shape, dtype=v.dtype, device=self.device) for k, v in host.items() if torch.is_tensor(v)}
        # the buffers of this slot were last read by the batch handed out two calls ago: everything enqueued so far covers it
        self.stream.wait_stream(main)
        with torch.cuda.stream(self.stream):
            out = {}
            for k, v in host.items():
                if torch.is_tensor(v):
                    self._sets[slot][k].copy_(v, non_blocking=True)
                    out[k] = self._sets[slot][k]
                else:
                    out[k] = v
        self._next = out

    def __iter__(self):
        return self

    def __next__(self):
        if self._next is None:
            raise StopIteration
        torch.cuda.current_stream(self.device).wait_stream(self.stream)
        batch = self._next
        self._preload()
        return batch
