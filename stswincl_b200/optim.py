"""Drop-in replacements for the optimiser-side loops of the STswinCL training recipes (SURVEY.md section 8f, N2 / N4).

  * ``FusedAdam``                    -- ``torch.optim.Adam`` of ``seg18/train_swin.py``: multi-tensor, reads fp32 or bf16
    (all-reduce bucket) gradients, writes the bf16 shadow of the weights the Swin kernels read (``bf16_weight``).
  * ``FusedSGD``                     -- ``torch.optim.SGD`` of the fine-tune recipe
    ``train_CL_ft_mswin_sgd_minput.py:147-162`` (momentum, per-module groups, poly lr): the same contract as
    ``FusedAdam``, bit-identical with torch's single-tensor step, ``state_dict`` compatible with ``torch.optim.SGD``, and
    a device-tensor ``lr`` that a CUDA-graph-captured step reads on every replay.
  * ``LARS`` / ``add_weight_decay``  -- ``pixcontrast_18/contrast/lars.py`` (same names, constructor, wrapper
    semantics: ``LARS(torch.optim.SGD(add_weight_decay(model, wd), lr, momentum))``).  The reference calls
    ``p.norm()`` / ``p.grad.norm()`` per tensor and branches on the results in Python (:127-133), a host
    synchronisation for every weight tensor and step; here each parameter group is two multi-tensor
    launches (norms, update) per 48 tensors with every decision taken on the device
    (``stswin_lars_sgd_step``).  State stays in the wrapped optimiser (``momentum_buffer``), so
    ``state_dict`` / ``load_state_dict`` interoperate with the reference.  The same contract as ``FusedSGD``: the
    bf16 weight shadow, ``step(grads=...)`` over fp32 or bf16 bucket gradients, and a device-tensor ``lr``.
  * ``momentum_update``              -- the key-encoder EMA of ``PixPro._momentum_update_key_encoder``
    (``PixPro_swin_v5.py:258-289``): one multi-tensor stream instead of three eager ops per parameter, writing the
    bf16 shadow of the key weights; the momentum may be a device pair, so a captured update follows a schedule.

CUDA fp32 parameters only -- no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Iterable, Optional, Sequence

import torch
from torch.optim.optimizer import Optimizer

from . import _lib, ops
from ._lib import StswinError

__all__ = ["LARS", "FusedAdam", "FusedSGD", "add_weight_decay", "momentum_update", "bf16_weight"]


def add_weight_decay(model, weight_decay=1e-5, skip_list=()):
    """The two parameter groups of ``lars.py:7-32``: vectors (biases, norm scales) and anything named in ``skip_list``
    get no weight decay and are exempt from LARS scaling (``ignore``); every other trainable tensor decays."""
    groups = {True: [], False: []}
    for name, param in model.named_parameters():
        if param.requires_grad:
            groups[param.dim() == 1 or name in skip_list].append(param)
    return [dict(params=groups[True], weight_decay=0, ignore=True),
            dict(params=groups[False], weight_decay=weight_decay, ignore=False)]


def _check_f32(tensors: Iterable[torch.Tensor], what: str) -> None:
    for t in tensors:
        if not t.is_cuda:
            raise StswinError(f"{what}: tensors must be CUDA tensors (stswincl_b200 has no CPU path)")
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise StswinError(f"{what}: tensors must be contiguous fp32, got {t.dtype} (contiguous={t.is_contiguous()})")


def _ptrs(tensors: Sequence[Optional[torch.Tensor]]):
    return (ctypes.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def _numels(tensors: Sequence[torch.Tensor]):
    return (ctypes.c_int64 * len(tensors))(*[t.numel() for t in tensors])


def _group_grads(param_groups, grads, who: str):
    """List of (group, params, gradients) of every parameter group with parameters to update: those with ``p.grad``, or
    with ``grads`` every ``requires_grad`` parameter in group order with its entry of the list.  Parameters must be
    contiguous fp32 CUDA tensors; gradients dense contiguous CUDA tensors, all fp32 or all bf16, one per parameter and of
    its size.  Every group is checked before the list is returned, so a refused step updates no group."""
    if grads is not None:
        n_req = sum(p.requires_grad for group in param_groups for p in group["params"])
        if len(grads) != n_req:
            raise StswinError(f"{who}: {len(grads)} gradients for {n_req} parameters that require grad")
    out, gi = [], 0
    for group in param_groups:
        if grads is None:
            params = [p for p in group["params"] if p.grad is not None]
            gl = [p.grad for p in params]
        else:
            params = [p for p in group["params"] if p.requires_grad]
            gl = list(grads[gi:gi + len(params)])
            gi += len(params)
        if not params:
            continue
        _check_f32(params, who)
        gdt = gl[0].dtype
        if gdt not in (torch.float32, torch.bfloat16) or any(g.dtype != gdt or g.is_sparse or not g.is_cuda or
                                                             not g.is_contiguous() or g.numel() != p.numel()
                                                             for g, p in zip(gl, params)):
            raise StswinError(f"{who}: gradients must be dense contiguous CUDA tensors, all fp32 or all bf16, one per "
                              "parameter and of its size")
        out.append((group, params, gl))
    return out


def _momentum_buffers(state, params, who: str):
    """The momentum buffers of ``params`` and the host array of first-step flags.  A parameter without one gets an
    uninitialised buffer and the flag, on which the kernel writes buf = g to every element."""
    _check_f32([state[p]["momentum_buffer"] for p in params if state[p].get("momentum_buffer") is not None],
               f"{who} (momentum_buffer)")                  # before any new buffer exists
    bufs, first = [], (ctypes.c_uint8 * len(params))()
    for i, p in enumerate(params):
        st = state[p]
        if st.get("momentum_buffer") is None:
            st["momentum_buffer"] = torch.empty_like(p, memory_format=torch.contiguous_format)
            first[i] = 1
        bufs.append(st["momentum_buffer"])
    return bufs, first


@torch.no_grad()
def momentum_update(params_q: Iterable[torch.Tensor], params_k: Iterable[torch.Tensor], momentum, *,
                    shadow: bool = True) -> None:
    """``param_k = param_k * momentum + param_q * (1. - momentum)`` for every pair, in place
    (``PixPro_swin_v5.py:266-267``), bit-exact with the eager expression.

    ``momentum`` is a float, or a 2-element fp32 tensor ``[m, 1 - m]`` on the parameters' device, read by the kernel
    on the device (a CUDA-graph-captured update then follows a schedule written into the tensor between replays); for
    bit-exactness its entries are the fp32 roundings of the double ``m`` and ``1. - m``.  With ``shadow``, every key
    parameter of >= 2 dimensions keeps a bf16 shadow that the update rewrites (``bf16_weight``)."""
    pk = list(params_k)
    q = [p.data for p in params_q]
    k = [p.data for p in pk]
    if len(q) != len(k):
        raise ValueError(f"momentum_update: {len(q)} query tensors vs {len(k)} key tensors")
    if not q:
        return
    _check_f32(q, "momentum_update"); _check_f32(k, "momentum_update")
    for a, b in zip(q, k):
        if a.shape != b.shape or a.device != b.device:
            raise ValueError("momentum_update: query / key parameter mismatch")
    if torch.is_tensor(momentum):
        if momentum.dtype != torch.float32 or momentum.shape != (2,) or momentum.device != k[0].device or \
                not momentum.is_contiguous():
            raise StswinError(f"momentum_update: a tensor momentum must be the contiguous fp32 pair [m, 1 - m] on "
                              f"{k[0].device}, got {momentum.dtype} {tuple(momentum.shape)} on {momentum.device}")
        m, om, m_dev = 0.0, 0.0, momentum.data_ptr()
    else:
        m, om, m_dev = float(momentum), float(1. - momentum), None
    shadows = [_shadow(p, shadow) for p in pk]
    n_bytes = sum(t.numel() for t in k) * 12 + sum(t.numel() for t, s in zip(k, shadows) if s is not None) * 2
    with ops._launch("ema_update", float(n_bytes), k[0]):                   # read k, q; write k (+ shadow)
        st = _lib.load().stswin_ema_update(_ptrs(k), _ptrs(q), _ptrs(shadows), _numels(k), len(k), m, om, m_dev,
                                           ops._stream(k[0]))
    _lib.check(st, "stswin_ema_update")
    ops.count_extra_launches(ops.mt_launches(len(k)) - 1)


def _lr_arg(lr, dev, who: str):
    """(host lr, device lr pointer) of a group's ``lr``: a number, or a 0-dim fp32 tensor on ``dev`` that the kernel
    reads on the device."""
    if not torch.is_tensor(lr):
        return float(lr), None
    if lr.dim() != 0 or lr.dtype != torch.float32 or lr.device != dev:
        raise StswinError(f"{who}: a tensor lr must be a 0-dim fp32 tensor on {dev}, got {lr.dtype} "
                          f"{tuple(lr.shape)} on {lr.device}")
    return 0.0, lr.data_ptr()


class LARS(Optimizer):
    """'LARS (Layer-wise Adaptive Rate Scaling)' as a wrapper of ``torch.optim.SGD`` (``lars.py:34-152``).

    With ``shadow``, the update pass also writes the bf16 shadow of every >= 2-D parameter (``bf16_weight``).  A
    group's ``lr`` may be a 0-dim fp32 CUDA tensor (``torch.optim.SGD(..., lr=lr_t)``): the kernel reads it on the
    device, so a CUDA-graph-captured step follows a schedule that writes the tensor between replays.  The step is
    capturable once every momentum buffer exists (after one eager step).

    ``step(grads=...)`` takes the gradients from a list (fp32 or bf16, one per ``requires_grad`` parameter in group
    order) instead of ``p.grad`` -- the bucket views of a data-parallel all-reduce (``dist.SegmentedStep``).  On that
    path neither ``p.grad`` nor the list is written; on the ``p.grad`` path ``p.grad`` holds the decayed / scaled
    gradient afterwards, as in the reference."""

    def __init__(self, optimizer, eps=1e-8, trust_coef=0.001, *, shadow: bool = True):
        if eps < 0.0:
            raise ValueError('invalid epsilon value: , %f' % eps)
        if trust_coef < 0.0:
            raise ValueError("invalid trust coefficient: %f" % trust_coef)
        if not isinstance(optimizer, torch.optim.SGD):
            raise StswinError("LARS: the fused step wraps torch.optim.SGD (the optimiser main_pretrain_swinv5.py:43-47 builds)")
        self.optim = optimizer
        self.eps = eps
        self.trust_coef = trust_coef
        self.shadow = shadow

    def __getstate__(self):
        return (self.optim, {'eps': self.eps, 'trust_coef': self.trust_coef, 'shadow': self.shadow})

    def __setstate__(self, state):
        self.optim, lars_dict = state
        self.eps = lars_dict['eps']
        self.trust_coef = lars_dict['trust_coef']
        self.shadow = lars_dict.get('shadow', True)

    def __repr__(self):
        return '%s(%r)' % (self.__class__.__name__, self.optim)

    @property
    def param_groups(self):
        return self.optim.param_groups

    @property
    def state(self):
        return self.optim.state

    def state_dict(self):
        return self.optim.state_dict()

    def load_state_dict(self, state_dict):
        self.optim.load_state_dict(state_dict)

    def zero_grad(self, set_to_none: bool = True):
        self.optim.zero_grad(set_to_none=set_to_none)

    def add_param_group(self, param_group):
        self.optim.add_param_group(param_group)

    @torch.no_grad()
    def step(self, closure=None, grads=None):
        """Weight decay into the gradient, LARS scaling of the non-``ignore`` group, momentum SGD update
        (``lars.py:109-152``), from ``p.grad`` or from ``grads`` (see the class docstring)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for group, params, gl in _group_grads(self.optim.param_groups, grads, "LARS.step"):
            if group.get('maximize', False):
                raise StswinError("LARS: maximize=True is not supported")
            gdt = gl[0].dtype
            lr, lr_dev = _lr_arg(group['lr'], params[0].device, "LARS.step")
            momentum, dampening = float(group['momentum']), float(group['dampening'])
            ignore = group.get('ignore', None)
            lars = ignore is not None and not ignore          # lars.py:125
            bufs, first = _momentum_buffers(self.optim.state, params, "LARS.step") if momentum != 0 else (None, None)
            shadows = [_shadow(p, self.shadow) for p in params]
            dev = params[0].device
            norms = torch.empty(2 * len(params), dtype=torch.float64, device=dev) if lars else None
            write = grads is None                                               # the p.grad contract of the reference
            n_el, gsz = sum(p.numel() for p in params), gl[0].element_size()
            # norms: p, g; update: p in / out, g in (+ out), buf in / out, shadow out
            n_bytes = n_el * ((4 + gsz if lars else 0) + 8 + gsz + (4 if write else 0) + (8 if momentum != 0 else 0)) + \
                sum(p.numel() for p, s in zip(params, shadows) if s is not None) * 2
            with ops._launch("lars_sgd_step", float(n_bytes), params[0]):
                st = lib.stswin_lars_sgd_step(_ptrs(params), _ptrs(gl), _ptrs(bufs) if bufs else None,
                                              _ptrs(shadows), _numels(params), first,
                                              len(params), int(gdt == torch.bfloat16), int(write), lr, lr_dev, momentum,
                                              dampening, int(bool(group['nesterov'])), float(group['weight_decay']),
                                              int(lars), float(self.trust_coef), float(self.eps),
                                              norms.data_ptr() if norms is not None else None, ops._stream(params[0]))
            _lib.check(st, "stswin_lars_sgd_step")
            ops.count_extra_launches(ops.mt_launches(len(params), 2 if lars else 1) - 1)       # norms + update per launch
        return loss


# ---------------------------------------------------------------------------------------------------------------
# bf16 shadow of the weights
# ---------------------------------------------------------------------------------------------------------------
def bf16_weight(w: torch.Tensor) -> torch.Tensor:
    """The bf16 copy of a weight the GEMM kernels consume.  ``FusedAdam``, ``FusedSGD``, ``LARS`` and
    ``momentum_update`` (key weights) keep a shadow copy per parameter that their update kernel rewrites every step, so the forward needs no cast kernel; the shadow is valid as long as nobody else
    wrote the parameter (tracked by the tensor's version counter -- the kernel does not bump it).  Without a valid
    shadow this is ``w.to(bfloat16)``."""
    sh = getattr(w, "_stswin_shadow", None)
    if sh is not None:
        if sh[1] == w._version and sh[0].device == w.device:
            return sh[0]
        with torch.no_grad():                       # someone else updated the parameter: refresh
            sh[0].copy_(w)
        w._stswin_shadow = (sh[0], w._version)
        return sh[0]
    return w.to(torch.bfloat16)


class FusedAdam(Optimizer):
    """``torch.optim.Adam`` semantics (the optimiser of ``seg18/train_swin.py``; no amsgrad / maximize) as multi-tensor
    launches of ``stswin_adam_step``: 48 tensors per launch, step count on the device (CUDA-graph capturable), and the
    bf16 shadow of every >= 2-D weight written in the same pass (``bf16_weight``).  State keys ``exp_avg`` /
    ``exp_avg_sq`` as in torch; the step count is one device scalar per group (``group['step_t']``).

    ``step(grads=...)`` takes the gradients from a list (fp32 or bf16, one per ``requires_grad`` parameter in group
    order) instead of ``p.grad`` -- the bf16 bucket views of a data-parallel all-reduce (``dist.SegmentedStep``)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, shadow: bool = True):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("FusedAdam: invalid hyper-parameter")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self.shadow = shadow

    def _state(self, p):
        st = self.state[p]
        if not st:
            st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
            st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
        return st

    @torch.no_grad()
    def step(self, closure=None, grads=None, grad_scale: float = 1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for group, params, gl in _group_grads(self.param_groups, grads, "FusedAdam.step"):
            gdt = gl[0].dtype
            states = [self._state(p) for p in params]
            if "step_t" not in group:
                group["step_t"] = torch.zeros((), dtype=torch.float32, device=params[0].device)
            shadows = [_shadow(p, self.shadow) for p in params]
            n_bytes = sum(p.numel() for p in params) * (28 + gl[0].element_size() - 4 + 2)
            b1, b2 = group["betas"]
            with ops._launch("adam", float(n_bytes), params[0]):
                st = lib.stswin_adam_step(_ptrs(params), _ptrs(gl), _ptrs([s["exp_avg"] for s in states]),
                                          _ptrs([s["exp_avg_sq"] for s in states]), _ptrs(shadows), _numels(params), len(params),
                                          int(gdt == torch.bfloat16), float(group["lr"]), float(b1), float(b2), float(group["eps"]),
                                          float(group["weight_decay"]), float(grad_scale), group["step_t"].data_ptr(),
                                          ops._stream(params[0]))
            _lib.check(st, "stswin_adam_step")
            ops.count_extra_launches(ops.mt_launches(len(params)))                  # + the step-count tick
        return loss


def _shadow(p: torch.Tensor, enabled: bool) -> Optional[torch.Tensor]:
    """The bf16 shadow of ``p`` that an update kernel rewrites (created for >= 2-D weights when ``enabled``), or None."""
    sh = getattr(p, "_stswin_shadow", None)
    if sh is None or sh[0].device != p.device:
        if not enabled or p.dim() < 2:
            return None
        sh = p._stswin_shadow = (p.detach().to(torch.bfloat16), p._version)
    elif sh[1] != p._version:                      # stale shadow: the kernel rewrites it anyway
        sh = p._stswin_shadow = (sh[0], p._version)
    return sh[0]


class FusedSGD(Optimizer):
    """``torch.optim.SGD`` (momentum, dampening, nesterov, weight decay, maximize) as multi-tensor launches of
    ``stswin_sgd_step`` (48 tensors per launch), bit-identical with torch's single-tensor step, that also write the bf16
    shadow of every >= 2-D weight in the same pass (``bf16_weight``).  State is ``state[p]["momentum_buffer"]`` as in
    torch, so ``state_dict`` / ``load_state_dict`` interoperate with ``torch.optim.SGD`` both ways.  ``foreach`` /
    ``fused`` are accepted and ignored.

    ``lr`` may be a 0-dim fp32 CUDA tensor: the kernel reads it on the device, so a CUDA-graph-captured step follows a
    schedule that writes the tensor between replays.  The step is capturable once every parameter with momentum has a
    buffer (after one eager step), as for torch's SGD.

    ``step(grads=...)`` takes the gradients from a list (fp32 or bf16, one per ``requires_grad`` parameter in group
    order) instead of ``p.grad``, scaled by ``grad_scale`` -- the bf16 bucket views of a data-parallel all-reduce
    (``dist.SegmentedStep``).  ``p.grad`` is never written."""

    def __init__(self, params, lr=1e-3, momentum=0, dampening=0, weight_decay=0, nesterov=False, *, maximize=False,
                 foreach=None, differentiable=False, fused=None, shadow: bool = True):
        if isinstance(lr, torch.Tensor) and lr.numel() != 1:
            raise ValueError("Tensor lr must be 1-element")
        if lr < 0.0:
            raise ValueError(f"Invalid learning rate: {lr}")
        if momentum < 0.0:
            raise ValueError(f"Invalid momentum value: {momentum}")
        if weight_decay < 0.0:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        if nesterov and (momentum <= 0 or dampening != 0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")
        if differentiable:
            raise StswinError("FusedSGD: differentiable=True is not supported (the update runs in a CUDA kernel)")
        # foreach / fused are kept in the groups (unused here) so that a torch.optim.SGD loading this state takes them
        super().__init__(params, dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay,
                                      nesterov=nesterov, maximize=maximize, foreach=foreach, differentiable=False,
                                      fused=fused))
        self.shadow = shadow

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:
            group.setdefault("nesterov", False)
            group.setdefault("maximize", False)

    @torch.no_grad()
    def step(self, closure=None, grads=None, grad_scale: float = 1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for group, params, gl in _group_grads(self.param_groups, grads, "FusedSGD.step"):
            gdt = gl[0].dtype
            lr, lr_dev = _lr_arg(group["lr"], params[0].device, "FusedSGD.step")
            momentum = float(group["momentum"])
            bufs, first = _momentum_buffers(self.state, params, "FusedSGD.step") if momentum != 0 else (None, None)
            shadows = [_shadow(p, self.shadow) for p in params]
            n_el = sum(p.numel() for p in params)
            n_bytes = n_el * (8 + gl[0].element_size() + (8 if bufs else 0)) + \
                sum(p.numel() for p, s in zip(params, shadows) if s is not None) * 2
            with ops._launch("sgd_step", float(n_bytes), params[0]):
                st = lib.stswin_sgd_step(_ptrs(params), _ptrs(gl), _ptrs(bufs) if bufs else None,
                                         _ptrs(shadows), _numels(params), first, len(params),
                                         int(gdt == torch.bfloat16), lr, lr_dev, momentum, float(1 - group["dampening"]),
                                         int(bool(group["nesterov"])), int(bool(group["maximize"])),
                                         float(group["weight_decay"]), float(grad_scale), ops._stream(params[0]))
            _lib.check(st, "stswin_sgd_step")
            ops.count_extra_launches(ops.mt_launches(len(params)) - 1)
        return loss
