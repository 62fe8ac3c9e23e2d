"""Data-parallel plumbing for the two hot paths (one process per GPU, torch.distributed).

Both paths shard over clips with no data-path collective (SURVEY.md section 8e): windows never
cross a clip and the reference loss never crosses a sample.  What remains is what the reference
does with ``DistributedSampler`` + DDP (``pixcontrast_18/main_pretrain_swinv5.py:54``,
``contrast/data/__init__.py:25``) and, for the segmentation scripts, with ``nn.DataParallel``
(``seg18/train_swin.py:131-135``): split the clips, all-reduce the gradients.

These helpers are backend-agnostic (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

import inspect
from typing import Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist


def shard_indices(n: int, rank: int, world: int) -> List[int]:
    """Indices of the samples rank ``rank`` owns: DistributedSampler(shuffle=False) semantics --
    the index list is padded by wrapping around to a multiple of ``world`` and dealt out
    round-robin (contrast/data/__init__.py:25)."""
    total = (n + world - 1) // world * world
    idx = list(range(n))
    pad = total - n
    if pad:
        idx += (idx * ((pad + n - 1) // n))[:pad]
    return idx[rank:total:world]


def scaled_lr(base_lr: float, batch_size: int, world: int) -> float:
    """lr = batch_size * world_size / 256 * base_lr  (main_pretrain_swinv5.py:38,45)."""
    return batch_size * world / 256.0 * base_lr


def average_gradients(params: Iterable[torch.nn.Parameter], *, bucket_bytes: int = 64 << 20,
                      comm_dtype: Optional[torch.dtype] = None, group=None) -> int:
    """All-reduce (mean) the ``.grad`` of every parameter in flat buckets of ``bucket_bytes``.
    ``comm_dtype=torch.bfloat16`` halves the bytes on the wire (the 96.6 M-parameter Swin head is
    386 MB in fp32).  Returns the number of collectives issued.  DDP does the same overlapped with
    backward; this explicit form is what the CPU tests exercise and what a DataParallel-free
    training loop can call."""
    world = dist.get_world_size(group)
    grads = [p.grad for p in params if p.grad is not None]
    if world == 1 or not grads:
        return 0
    calls, i = 0, 0
    while i < len(grads):
        bucket, size = [], 0
        while i < len(grads) and (not bucket or size + grads[i].numel() * grads[i].element_size() <= bucket_bytes):
            bucket.append(grads[i]); size += grads[i].numel() * grads[i].element_size(); i += 1
        flat = torch.cat([g.reshape(-1) for g in bucket])
        wire = flat.to(comm_dtype) if comm_dtype is not None and comm_dtype != flat.dtype else flat
        dist.all_reduce(wire, op=dist.ReduceOp.SUM, group=group)
        flat = wire.to(flat.dtype) if wire is not flat else flat
        flat.div_(world)
        off = 0
        for g in bucket:
            g.copy_(flat[off:off + g.numel()].view_as(g)); off += g.numel()
        calls += 1
    return calls


class FlatGradients:
    """One flat fp32 buffer holding the gradients of ``params`` (each view 16-byte aligned), for a single
    all-reduce per step instead of DDP's buckets -- the data-parallel exchange of ``bench.py --dp flat``:

        loss.backward()            # may be replayed from a CUDA graph together with ``gather()``
        flat.gather()              # copy every p.grad into the buffer (one multi-tensor copy)
        flat.all_reduce()          # ONE collective (mean over ranks)
        flat.bind()                # p.grad = view of the reduced buffer
        optimizer.step()

    Backend-agnostic (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        sizes = [(p.numel() + 3) // 4 * 4 for p in self.params]
        dev = self.params[0].device
        self.buffer = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        self.views, off = [], 0
        for p, n in zip(self.params, sizes):
            self.views.append(self.buffer[off:off + p.numel()].view_as(p))
            off += n

    def gather(self) -> None:
        grads = [p.grad for p in self.params]
        if any(g is None for g in grads):
            raise RuntimeError("FlatGradients.gather: a parameter has no gradient")
        torch._foreach_copy_(self.views, grads)

    def all_reduce(self, group=None) -> None:
        world = dist.get_world_size(group)
        if world == 1:
            return
        if dist.get_backend(group) == "nccl":
            dist.all_reduce(self.buffer, op=dist.ReduceOp.AVG, group=group)
        else:                                   # gloo has no AVG
            dist.all_reduce(self.buffer, op=dist.ReduceOp.SUM, group=group)
            self.buffer.div_(world)

    def bind(self) -> None:
        for p, v in zip(self.params, self.views):
            p.grad = v


def _takes_grads(opt) -> bool:
    """Whether ``opt.step`` accepts ``grads=``.  Read through the signature: ``torch.optim.Optimizer`` wraps ``step``
    in a ``(*args, **kwargs)`` profiling wrapper, whose own code object does not name the parameter."""
    try:
        return "grads" in inspect.signature(opt.step).parameters
    except (AttributeError, TypeError, ValueError):
        return False


class SegmentedStep:
    """Data-parallel training step whose gradient exchange overlaps the backward.

    ``model.stages(x)`` gives the forward as a chain of stages (``SwinTransformerLayerv5.stages``).  The autograd graph
    is cut at the stage boundaries, so the backward runs stage by stage, last stage first; as soon as a stage's
    backward is done its gradients are copied (and rounded to ``wire_dtype``) into that stage's flat bucket and the
    bucket is all-reduced (average) on a side stream while the earlier stages' backward still runs.  Only the first
    stage's bucket -- the smallest one for the Swin head -- is exposed.  The forward and every backward segment are
    captured as CUDA graphs sharing one memory pool and replayed in order (``use_graph``); the collectives and the
    optimizer step are issued between / after the replays.

    The optimizer step reads the reduced gradients straight from the buckets when the optimizer accepts
    ``step(grads=...)`` (``optim.FusedAdam``, ``optim.FusedSGD``, ``optim.LARS``: fp32 or bf16 gradients); otherwise they are copied back into
    ``p.grad`` first.  Backend-agnostic (NCCL on GPUs, gloo in the CPU tests; there ``use_graph=False``)."""

    def __init__(self, model, optimizer, loss_fn, *, segments: int = 4, wire_dtype: torch.dtype = torch.bfloat16,
                 use_graph: bool = True, group=None, example_input: Optional[torch.Tensor] = None):
        self.model, self.opt, self.loss_fn, self.group = model, optimizer, loss_fn, group
        self.wire_dtype = wire_dtype
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.nccl = self.world > 1 and dist.get_backend(group) == "nccl"
        self.segments = max(1, segments)
        self.use_graph = use_graph
        self.captured = False
        self._built = False
        self._static_x = None
        if example_input is not None:
            self._build(example_input)

    # ---- construction
    def _build(self, x):
        stages = self.model.stages(x)
        K = min(self.segments, len(stages))
        # merge neighbouring stages, keeping the LAST stages separate (their backward runs first, their buckets are the
        # large ones for the Swin head) -- e.g. 4 stages in 2 segments: [0,1,2] + [3]
        groups = [[] for _ in range(K)]
        n = len(stages)
        for i in range(n):
            groups[max(0, K - (n - i))].append(i)
        self._stage_fns = [[stages[i][0] for i in g] for g in groups]
        self._stage_params = [[p for i in g for p in stages[i][1] if p.requires_grad] for g in groups]
        dev = x.device
        self._buckets, self._views = [], []
        for ps in self._stage_params:
            sizes = [(p.numel() + 7) // 8 * 8 for p in ps]
            buf = torch.zeros(sum(sizes), dtype=self.wire_dtype, device=dev)
            views, off = [], 0
            for p, sz in zip(ps, sizes):
                views.append(buf[off:off + p.numel()].view_as(p))
                off += sz
            self._buckets.append(buf)
            self._views.append(views)
        self._view_of = {id(p): v for ps, vs in zip(self._stage_params, self._views) for p, v in zip(ps, vs)}
        self._direct = _takes_grads(self.opt)
        self._opt_grads = [self._view_of[id(p)] for g in self.opt.param_groups for p in g["params"] if p.requires_grad]
        self._cuda = dev.type == "cuda"
        if self._cuda:
            self._comm = torch.cuda.Stream(device=dev)
            self._events = [torch.cuda.Event() for _ in self._buckets]
        self._built = True

    def describe(self) -> str:
        sizes = ", ".join("%.0f MB" % (b.numel() * b.element_size() / 2 ** 20) for b in reversed(self._buckets))
        return ("backward in %d %s, one %s gradient bucket per segment (%s) all-reduced (average) on a side stream while the "
                "next segment's backward runs" % (len(self._buckets), "CUDA-graph segments" if self.captured else "eager segments",
                                                  str(self.wire_dtype).replace("torch.", ""), sizes))

    # ---- one step, segment by segment
    def _forward(self, x):
        self._ins, self._outs = [], []
        state = (x,)
        for k, fns in enumerate(self._stage_fns):
            ins = tuple(s if k == 0 else s.detach().requires_grad_(True) for s in state)
            state = ins
            for fn in fns:
                state = fn(*state)
            self._ins.append(ins)
            self._outs.append(state)
        self._loss = self.loss_fn(state)
        return self._loss

    def _backward_segment(self, k):
        if k == len(self._stage_fns) - 1:
            self._loss.backward()
        else:
            pairs = [(o, i.grad) for o, i in zip(self._outs[k], self._ins[k + 1]) if i.grad is not None]
            torch.autograd.backward([o for o, _ in pairs], [g for _, g in pairs])
        ps = self._stage_params[k]
        if ps:
            grads = [p.grad for p in ps]
            if self._cuda and all(g.dtype == torch.float32 and g.is_contiguous() for g in grads) and \
                    self.wire_dtype in (torch.float32, torch.bfloat16):
                from . import ops
                ops.gather_cast(self._views[k], grads)           # one multi-tensor launch per 48 tensors
            else:
                torch._foreach_copy_(self._views[k], grads)

    def _reduce(self, k):
        if self.world == 1 or self._buckets[k].numel() == 0:
            return
        buf = self._buckets[k]
        if self._cuda:
            self._events[k].record(torch.cuda.current_stream(buf.device))
            with torch.cuda.stream(self._comm):
                self._comm.wait_event(self._events[k])
                self._all_reduce(buf)
        else:
            self._all_reduce(buf)

    def _all_reduce(self, buf):
        if self.nccl:
            dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=self.group)
        else:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group)
            buf.div_(self.world)

    def _update(self):
        if self._cuda and self.world > 1:
            torch.cuda.current_stream().wait_stream(self._comm)
        if self._direct:
            self.opt.step(grads=self._opt_grads)
        else:
            ps = [p for st in self._stage_params for p in st]
            torch._foreach_copy_([p.grad for p in ps], [self._view_of[id(p)] for p in ps])
            self.opt.step()

    def eager(self, x):
        """The same step without graph replays (every kernel launched by the host: profiling, debugging)."""
        if not self._built:
            self._build(x)
        return self._eager(x)

    def _eager(self, x):
        self.opt.zero_grad(set_to_none=True)
        loss = self._forward(x)
        for k in reversed(range(len(self._stage_fns))):
            self._backward_segment(k)
            self._reduce(k)
        self._update()
        return loss

    def _capture(self, x):
        dev = x.device
        self._static_x = x.clone()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):                      # warm-up without side effects: no all-reduce, no optimizer step
                self.opt.zero_grad(set_to_none=True)
                self._forward(self._static_x)
                for k in reversed(range(len(self._stage_fns))):
                    self._backward_segment(k)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.opt.zero_grad(set_to_none=True)
        self._g_fwd = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._g_fwd):
            self._forward(self._static_x)
        pool = self._g_fwd.pool()
        self._g_bwd = {}
        for k in reversed(range(len(self._stage_fns))):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                self._backward_segment(k)
            self._g_bwd[k] = g
        self.captured = True

    def step(self, x):
        """One training step on ``x``; returns the (device) loss."""
        if not self._built:
            self._build(x)
        if not (self.use_graph and self._cuda):
            return self._eager(x)
        if not self.captured:
            try:
                self._capture(x)
            except Exception as e:                 # capture is an optimisation; every rank must agree (checked below)
                import sys
                print(f"SegmentedStep: CUDA graph capture failed ({type(e).__name__}: {e}); running eager segments", file=sys.stderr)
                self.use_graph = False
                torch.cuda.synchronize()
            if self.world > 1:
                ok = torch.tensor([1 if self.captured else 0], device=x.device)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
                if int(ok) == 0:
                    self.captured, self.use_graph = False, False
            if not self.captured:
                return self._eager(x)
        if x is not self._static_x:
            self._static_x.copy_(x, non_blocking=True)
        self._g_fwd.replay()
        for k in reversed(range(len(self._stage_fns))):
            self._g_bwd[k].replay()
            self._reduce(k)
        self._update()
        return self._loss


def broadcast_parameters(params: Iterable[torch.nn.Parameter], src: int = 0, group=None) -> None:
    """Replicas start from rank ``src``'s parameters (what DDP's constructor does)."""
    for p in params:
        dist.broadcast(p.data, src=src, group=group)


def gather_key_sets(tensors: Sequence[torch.Tensor], group=None) -> List[torch.Tensor]:
    """All-gather every tensor of ``tensors`` from all ranks; returns, per input tensor, the list of
    per-rank copies flattened into one list (own rank's copy first).  Building block of the
    'negatives span all ranks' extension (SURVEY D5 / C3): the gathered key sets are appended as
    extra sets of ``pixel_contrast_loss`` -- *not* reference behaviour (parity unpinned)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    out: List[torch.Tensor] = []
    for t in tensors:
        t = t.contiguous()
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        out.extend([parts[rank]] + [p for r, p in enumerate(parts) if r != rank])
    return out
