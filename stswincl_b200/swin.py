"""Drop-in replacements for the reference's spatio-temporal Swin head.

Same constructor signatures, same ``state_dict`` keys and shapes, same forward
contracts as ``seg18/net/Ours/swin_512.py`` (== ``segcata/net/Ours/swin_tem_cata.py``
== ``pixcontrast_*/contrast/models/Ours/swin_tem.py``):

  * ``WindowAttention``          swin_512.py:73-141
  * ``Mlp``                      swin_512.py:7-23
  * ``SwinTransformerBlock``     swin_512.py:143-237  (post-norm, mask fill -100)
  * ``PatchMerging``             swin_512.py:239-277
  * ``SwinTransformerLayerv5``   swin_512.py:280-327

so ``model.swin = stswincl_b200.swin.SwinTransformerLayerv5(...)`` followed by
``load_state_dict(reference_state, strict=True)`` is the whole integration.

All arithmetic runs in the sm_100a kernels behind ``include/stswin_b200.h`` through
``torch.autograd.Function`` wrappers: bf16 storage, fp32 accumulation / statistics.
Parameters stay fp32 (the reference's master copy under AMP) and are rounded to bf16
per call.  There is no CPU path and no PyTorch fallback: CPU tensors raise.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import ops, ops32
from ._lib import StswinError
from .ops import _wgrad_splits
from .optim import bf16_weight as _w16

_BF16 = torch.bfloat16
# bf16 mode: keep GELU'(fc1 output) for the backward as one byte per element (step 0.005 over [-0.14, 1.14]; the bf16 rounding
# of a value near 1 is 0.002-0.004) instead of bf16 -- the fc1 + GELU layer is HBM-write bound (DESIGN.md section 8).  False
# restores the bf16 form.
GELU_GRAD_Q8 = True


def to_2tuple(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x, x)


def _relative_position_index(ws_h: int, ws_w: int) -> torch.Tensor:
    """Closed form of swin_512.py:88-99."""
    n = torch.arange(ws_h * ws_w)
    h, w = n // ws_w, n % ws_w
    dh = h[:, None] - h[None, :] + ws_h - 1
    dw = w[:, None] - w[None, :] + ws_w - 1
    return dh * (2 * ws_w - 1) + dw


def _shift_attn_mask(H: int, W: int, ws: int, shift: int) -> torch.Tensor:
    """Closed form of swin_512.py:171-192 -- kept as a buffer for state_dict parity only; the
    kernels rebuild the mask from (H, W, ws, shift)."""
    def band(p, extent):
        return (p >= extent - ws).long() + (p >= extent - shift).long()
    ids = 3 * band(torch.arange(H), H)[:, None] + band(torch.arange(W), W)[None, :]
    per_win = ids.view(H // ws, ws, W // ws, ws).permute(0, 2, 1, 3).reshape(-1, ws * ws)
    differ = per_win[:, None, :] != per_win[:, :, None]
    return torch.where(differ, torch.tensor(-100.0), torch.tensor(0.0))


def _linear_wgrad(dy2d: torch.Tensor, x2d: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[N_out, K_in] = dy^T x, reduced over tokens on the tensor cores (fp32, split-K).
    ``out`` must be zero-filled (the split-K epilogue accumulates)."""
    ops.gemm(dy2d, x2d, a_mn_major=True, b_mn_major=True, mode=ops.EPI_F32_REDUCE, out=out,
             k_splits=_wgrad_splits(out.shape[0], out.shape[1], dy2d.shape[0]))
    return out


def _zeros_like_many(shapes, device):
    """One zero-filled fp32 allocation carved into the given shapes (one memset instead of many)."""
    sizes = [int(math.prod(s)) for s in shapes]
    offs, total = [], 0
    for n in sizes:
        offs.append(total)
        total += (n + 3) // 4 * 4            # keep every view 16-byte aligned (TMA reduce target)
    flat = torch.zeros(total, dtype=torch.float32, device=device)
    return [flat[o:o + n].view(s) for o, n, s in zip(offs, sizes, shapes)]


# ---------------------------------------------------------------------------------------------------------------
# The block's two halves on bf16 token rows x2 [rows, C], written once for the stand-alone Functions and the block.
# ``res`` / ``dres``: a residual (rows like the output) added in the epilogue of the half's last GEMM.  Gradient
# buffers are zero-filled fp32 (the kernels accumulate); the gradient of the half's last bias is the caller's.
# ---------------------------------------------------------------------------------------------------------------
def _attn_fwd(x2, shp, table, wq, b_qkv, wp, b_proj, geom, mask=None, res=None):
    """qkv GEMM -> window attention core -> proj GEMM (+ res); ``shp`` = (Bp, T, H*W) of the rows.
    Returns (qkv, attn, lse2, out)."""
    H, W, nH, ws, shift, qk_scale = geom[:6]
    C = x2.shape[1]
    qkv = ops.gemm(x2, wq, bias=b_qkv)
    attn, lse2 = ops.winattn_fwd(qkv.view(*shp, 3 * C), table, H, W, nH, ws, shift, qk_scale=qk_scale, mask=mask)
    out = ops.gemm(attn.view(-1, C), wp, bias=b_proj, aux=res, mode=ops.EPI_BIAS if res is None else ops.EPI_BIAS_RES)
    return qkv, attn, lse2, out


def _attn_bwd(dy, shp, x2, qkv, attn, lse2, table, wq, wp, geom, d_table, d_bqkv, d_wproj, d_wqkv, mask=None,
              need_dx=True, dres=None):
    """Backward of ``_attn_fwd`` from dy [rows, C]: proj dgrad -> proj wgrad -> attention core -> qkv dgrad (+ dres; only
    with ``need_dx``) -> qkv wgrad.  ``d_bqkv`` None: no qkv bias.  Returns dx [rows, C] or None."""
    H, W, nH, ws, shift, qk_scale = geom[:6]
    C = x2.shape[1]
    d_attn = ops.gemm(dy, wp, b_mn_major=True)
    _linear_wgrad(dy, attn.view(-1, C), d_wproj)
    d_qkv = ops.winattn_bwd(qkv.view(*shp, 3 * C), table, lse2, d_attn.view(*shp, C), H, W, nH, ws, shift,
                            d_table, d_bqkv, qk_scale=qk_scale, mask=mask)
    dq2 = d_qkv.view(-1, 3 * C)
    d_x = None
    if need_dx:
        d_x = ops.gemm(dq2, wq, b_mn_major=True, aux=dres, mode=ops.EPI_BIAS if dres is None else ops.EPI_BIAS_RES)
    _linear_wgrad(dq2, x2, d_wqkv)
    return d_x


def _mlp_fwd(x2, w1, b1, w2, b2, res=None, keep_dgelu=True):
    """fc1 + GELU -> fc2 (+ res).  With ``keep_dgelu`` the fc1 epilogue also writes GELU'(fc1 out) for the backward, one
    byte per element when GELU_GRAD_Q8 and the width allow (a bounded multiplier; fc1 + GELU is HBM-write bound), else
    bf16.  Returns (h, dgelu or None, y)."""
    dgelu = None
    if keep_dgelu:
        q8 = GELU_GRAD_Q8 and w1.shape[0] % 16 == 0
        dgelu = torch.empty((x2.shape[0], w1.shape[0]), dtype=torch.uint8 if q8 else _BF16, device=x2.device)
        h = ops.gemm(x2, w1, bias=b1, mode=ops.EPI_BIAS_GELU_Q8 if q8 else ops.EPI_BIAS_GELU, out2=dgelu)
    else:
        h = ops.gemm(x2, w1, bias=b1, mode=ops.EPI_BIAS_GELU_FWD)
    y = ops.gemm(h, w2, bias=b2, aux=res, mode=ops.EPI_BIAS if res is None else ops.EPI_BIAS_RES)
    return h, dgelu, y


def _mlp_bwd(dy, x2, h, dgelu, w1, w2, d_b1, d_w1, d_w2):
    """Backward of ``_mlp_fwd`` from dy [rows, C_out]: fc2 dgrad times GELU' (column sums into d_b1) -> fc2 wgrad ->
    fc1 dgrad -> fc1 wgrad.  Returns dx [rows, C_in]."""
    du = ops.gemm(dy, w2, b_mn_major=True, mode=ops.EPI_MUL_AUX_Q8 if dgelu.dtype == torch.uint8 else ops.EPI_MUL_AUX,
                  aux=dgelu, colsum=d_b1)
    _linear_wgrad(dy, h, d_w2)
    dx = ops.gemm(du, w1, b_mn_major=True)
    _linear_wgrad(du, x2, d_w1)
    return dx


class _AttentionFn(torch.autograd.Function):
    """qkv Linear -> window attention core -> proj Linear on tokens in natural order.

    x [Bp, T, H*W, C] bf16.  Gradients for x, table, qkv.{weight,bias}, proj.{weight,bias}."""

    @staticmethod
    def forward(ctx, x, table, w_qkv, b_qkv, w_proj, b_proj, geom, mask=None):
        x2 = x.reshape(-1, x.shape[-1])
        wq, wp = _w16(w_qkv), _w16(w_proj)
        qkv, attn, lse2, out = _attn_fwd(x2, x.shape[:3], table, wq, b_qkv, wp, b_proj, geom, mask)
        ctx.save_for_backward(x2, qkv, attn, lse2, table, wq, wp)
        ctx.geom, ctx.mask, ctx.has_qkv_bias = geom, mask, b_qkv is not None
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, d_out):
        x2, qkv, attn, lse2, table, wq, wp = ctx.saved_tensors
        C = x2.shape[1]
        d2 = d_out.contiguous().view(-1, C)
        d_table, d_bqkv, d_bproj, d_wproj, d_wqkv = _zeros_like_many([tuple(table.shape), (3 * C,), (C,), tuple(wp.shape), tuple(wq.shape)], d2.device)
        ops.colsum(d2, d_bproj)                           # proj bias gradient: one read of d_out
        if not ctx.has_qkv_bias:
            d_bqkv = None
        d_x = _attn_bwd(d2, d_out.shape[:3], x2, qkv, attn, lse2, table, wq, wp, ctx.geom, d_table, d_bqkv, d_wproj, d_wqkv,
                        ctx.mask)
        return d_x.view(d_out.shape), d_table, d_wqkv, d_bqkv, d_wproj, d_bproj, None, None


class _BlockFn(torch.autograd.Function):
    """One post-norm SwinTransformerBlock (swin_512.py:196-237) on bf16 tokens [Bp, T, H*W, C]:

        y   = x + proj(attn_core(qkv(x)))           residual fused into the proj GEMM epilogue
        z   = y + fc2(gelu(fc1(norm2(y))))          GELU / residual fused into the GEMM epilogues
        out = norm1(z)
    """

    @staticmethod
    def forward(ctx, x, table, w_qkv, b_qkv, w_proj, b_proj, g1, be1, g2, be2, w_fc1, b_fc1, w_fc2, b_fc2, geom):
        eps = geom[6]
        # inference (no_grad key encoders of the pre-training model, evaluation): no gelu' output, nothing kept for a backward
        infer = geom[7] or not any(ctx.needs_input_grad)
        x2 = x.reshape(-1, x.shape[-1])
        wq, wp, w1, w2 = _w16(w_qkv), _w16(w_proj), _w16(w_fc1), _w16(w_fc2)
        qkv, attn, lse2, y = _attn_fwd(x2, x.shape[:3], table, wq, b_qkv, wp, b_proj, geom, res=x2)
        yn, mean2, rstd2 = ops.layernorm_fwd(y, g2, be2, eps)
        h, dgelu, z = _mlp_fwd(yn, w1, b_fc1, w2, b_fc2, res=y, keep_dgelu=not infer)
        out, mean1, rstd1 = ops.layernorm_fwd(z, g1, be1, eps)
        if not infer:
            ctx.save_for_backward(x2, qkv, attn, lse2, y, yn, mean2, rstd2, dgelu, h, z, mean1, rstd1,
                                  table, wq, wp, w1, w2, g1, g2)
            ctx.geom, ctx.has_qkv_bias = geom[:7], b_qkv is not None
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, d_out):
        (x2, qkv, attn, lse2, y, yn, mean2, rstd2, dgelu, h, z, mean1, rstd1,
         table, wq, wp, w1, w2, g1, g2) = ctx.saved_tensors
        C = x2.shape[1]
        d2 = d_out.contiguous().view(-1, C)
        (d_g1, d_be1, d_bfc2, d_bfc1, d_g2, d_be2, d_bproj, d_table, d_bqkv, d_wfc2, d_wfc1, d_wproj, d_wqkv) = \
            _zeros_like_many([(C,), (C,), (C,), (w1.shape[0],), (C,), (C,), (C,), tuple(table.shape), (3 * C,),
                              tuple(w2.shape), tuple(w1.shape), tuple(wp.shape), tuple(wq.shape)], d2.device)
        if not ctx.has_qkv_bias:
            d_bqkv = None
        # out = norm1(z); z = y + mlp(yn), the fc2 bias gradient is the column sums of dz
        dz = ops.layernorm_bwd(d2, z, mean1, rstd1, g1, d_g1, d_be1, dx_colsum=d_bfc2)
        dyn = _mlp_bwd(dz, yn, h, dgelu, w1, w2, d_bfc1, d_wfc1, d_wfc2)
        # yn = norm2(y); y = x + attn(x), the proj bias gradient is the column sums of dy
        dy = ops.layernorm_bwd(dyn, y, mean2, rstd2, g2, d_g2, d_be2, dres=dz, dx_colsum=d_bproj)
        # the first block of a head fed with features that carry no gradient skips the qkv dgrad
        d_x = _attn_bwd(dy, d_out.shape[:3], x2, qkv, attn, lse2, table, wq, wp, ctx.geom, d_table, d_bqkv, d_wproj, d_wqkv,
                        need_dx=ctx.needs_input_grad[0], dres=dy)
        return (None if d_x is None else d_x.view(d_out.shape), d_table, d_wqkv, d_bqkv, d_wproj, d_bproj,
                d_g1, d_be1, d_g2, d_be2, d_wfc1, d_bfc1, d_wfc2, d_bfc2, None)


class _PatchMergeFn(torch.autograd.Function):
    """2x2 gather + LayerNorm(4C) in one pass, then the bias-free reduction GEMM (swin_512.py:255-277)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, w_red, geom):
        H, W, eps = geom
        B, T, L, C = x.shape
        xn, mean, rstd = ops.layernorm_fwd(x.reshape(B * T, L, C), gamma, beta, eps, patch_merge_hw=(H, W))
        wr = _w16(w_red)
        out = ops.gemm(xn, wr)
        ctx.save_for_backward(x, xn, mean, rstd, gamma, wr)
        ctx.geom = geom
        return out.view(B, T, L // 4, wr.shape[0])

    @staticmethod
    def backward(ctx, d_out):
        x, xn, mean, rstd, gamma, wr = ctx.saved_tensors
        H, W, eps = ctx.geom
        B, T, L, C = x.shape
        d2 = d_out.contiguous().view(-1, wr.shape[0])
        dxn = ops.gemm(d2, wr, b_mn_major=True)
        d_w = _linear_wgrad(d2, xn, torch.zeros(wr.shape, dtype=torch.float32, device=d2.device))
        d_gamma = torch.zeros(4 * C, dtype=torch.float32, device=x.device)
        d_beta = torch.zeros_like(d_gamma)
        dx = ops.layernorm_bwd(dxn, x.reshape(B * T, L, C), mean, rstd, gamma, d_gamma, d_beta, patch_merge_hw=(H, W))
        return dx.view(B, T, L, C), d_gamma, d_beta, d_w, None


class _TransposeFn(torch.autograd.Function):
    """[batch, R, Cc] -> [batch, Cc, R] with dtype change; the backward is the inverse move."""

    @staticmethod
    def forward(ctx, x, out_dtype):
        ctx.in_dtype = x.dtype
        return ops.transpose(x.contiguous(), out_dtype)

    @staticmethod
    def backward(ctx, g):
        return ops.transpose(g.contiguous(), ctx.in_dtype), None


class _FnCtx:
    """Minimal stand-in for an autograd context, used to run ``_BlockFn`` inside another Function."""

    def __init__(self, n_inputs: int):
        self.needs_input_grad = (True,) * n_inputs
        self.saved_tensors = ()

    def save_for_backward(self, *tensors):
        self.saved_tensors = tensors


def _mid_frames(x: torch.Tensor, blocks) -> torch.Tensor:
    """``cat([x[:, :1], blocks(x[:, 1:3]), x[:, 3:]])`` for x [B, 4, L, C] without a ``cat``: frames 1..2 are copied out
    and run through ``blocks``, and the output is assembled from the result and frames 0 / 3 of x."""
    B, _, L, C = x.shape
    xm = torch.empty((B, 2, L, C), dtype=x.dtype, device=x.device)
    ops.copy_frames(xm, x[:, 1:3])
    y = blocks(xm)
    out = torch.empty_like(x)
    ops.copy_frames(out[:, 0], x[:, 0])
    ops.copy_frames(out[:, 3], x[:, 3])
    ops.copy_frames(out[:, 1:3], y)
    return out


class _MidLayerFn(torch.autograd.Function):
    """The middle layer of a stage (swin_512.py:302-307): ``cat([x[:, :1], blk1(blk0(x[:, 1:3])), x[:, 3:]])`` as ONE
    autograd node; the forward is ``_mid_frames``.  Backward: the incoming gradient is only read; the gradient of
    x is a fresh buffer filled from three sources (frames 0 / 3 of d_out, the blocks' input gradient for frames 1..2),
    so there is no zero-fill and no gradient accumulation for the pass-through frames."""

    N_BLOCK_ARGS = 13

    @staticmethod
    def forward(ctx, x, geom0, geom1, *params):
        n = _MidLayerFn.N_BLOCK_ARGS
        c0, c1 = _FnCtx(n + 2), _FnCtx(n + 2)
        blk = ctx.blk = _BLOCK_FNS[x.dtype]
        out = _mid_frames(x, lambda xm: blk.forward(c1, blk.forward(c0, xm, *params[:n], geom0), *params[n:], geom1))
        ctx.blocks = (c0, c1)
        return out

    @staticmethod
    def backward(ctx, d_out):
        c0, c1 = ctx.blocks
        d_out = d_out.contiguous()
        B, _, L, C = d_out.shape
        d_y = torch.empty((B, 2, L, C), dtype=d_out.dtype, device=d_out.device)
        ops.copy_frames(d_y, d_out[:, 1:3])
        g1 = ctx.blk.backward(c1, d_y)
        g0 = ctx.blk.backward(c0, g1[0])
        d_x = torch.empty_like(d_out)
        ops.copy_frames(d_x[:, 0], d_out[:, 0])
        ops.copy_frames(d_x[:, 3], d_out[:, 3])
        ops.copy_frames(d_x[:, 1:3], g0[0].contiguous())
        return (d_x, None, None, *g0[1:-1], *g1[1:-1])


class _MlpFn(torch.autograd.Function):
    """Stand-alone Mlp.forward (swin_512.py:17-23) on bf16 rows [..., C_in]."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2):
        x2 = x.reshape(-1, x.shape[-1])
        w1b, w2b = _w16(w1), _w16(w2)
        h, dgelu, y = _mlp_fwd(x2, w1b, b1, w2b, b2)
        ctx.save_for_backward(x2, h, dgelu, w1b, w2b)
        return y.view(*x.shape[:-1], w2b.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, h, dgelu, w1b, w2b = ctx.saved_tensors
        d2 = dy.contiguous().view(-1, w2b.shape[0])
        d_b2, d_b1, d_w2, d_w1 = _zeros_like_many([(w2b.shape[0],), (w1b.shape[0],), tuple(w2b.shape), tuple(w1b.shape)], d2.device)
        ops.colsum(d2, d_b2)
        dx = _mlp_bwd(d2, x2, h, dgelu, w1b, w2b, d_b1, d_w1, d_w2)
        return dx.view(*dy.shape[:-1], w1b.shape[1]), d_w1, d_b1, d_w2, d_b2


# ---------------------------------------------------------------------------------------------------------------
# fp32-accurate mode (ops32): the reference's no-AMP run at <= 1e-3
# ---------------------------------------------------------------------------------------------------------------
_PRECISION = "bf16"


def set_precision(mode: str) -> str:
    """Arithmetic of the drop-in modules: ``"bf16"`` (default: bf16 storage, fp32 accumulation -- the counterpart of the
    reference under ``amp.autocast``), ``"fp32"`` (activations stay fp32, dense layers as split-bf16 tcgen05 GEMMs, the
    attention core as fp32 SIMT kernels: <= 1e-3 against the reference's fp32 run) or ``"auto"`` (fp32 for fp32 inputs
    outside autocast, bf16 otherwise).  A module's own ``precision`` attribute, when set, wins.  Returns the old mode."""
    global _PRECISION
    if mode not in ("bf16", "fp32", "auto"):
        raise ValueError("precision must be 'bf16', 'fp32' or 'auto'")
    old, _PRECISION = _PRECISION, mode
    return old


def _use_fp32(module, x: torch.Tensor) -> bool:
    mode = getattr(module, "precision", None) or _PRECISION
    if mode == "auto":
        return x.dtype == torch.float32 and not torch.is_autocast_enabled()
    return mode == "fp32"


def _zeros_f32(shape, dev):
    return torch.zeros(shape, dtype=torch.float32, device=dev)


# The two halves again over ops32 (fp32 rows), written once for the stand-alone Functions and the block.  They differ
# from the bf16 ones in what they fuse: the fc2 GEMM applies GELU to its split input (u is kept, not GELU'(u)) and the
# bias gradients are separate column sums.
def _attn_fwd32(x2, shp, table, w_qkv, b_qkv, w_proj, b_proj, geom, mask=None, res=None):
    """``_attn_fwd`` in fp32.  Returns (qkv, attn, lse, out)."""
    H, W, nH, ws, shift, qk_scale = geom[:6]
    C = x2.shape[1]
    qkv = ops32.linear(x2, w_qkv, b_qkv)
    attn, lse = ops32.winattn_fwd(qkv.view(*shp, 3 * C), table, H, W, nH, ws, shift, qk_scale, mask)
    return qkv, attn, lse, ops32.linear(attn.view(-1, C), w_proj, b_proj, res=res)


def _attn_bwd32(dy, shp, x2, qkv, attn, lse, table, w_qkv, w_proj, geom, has_qkv_bias, mask=None, dres=None):
    """``_attn_bwd`` in fp32, from dy [rows, C].  Returns (dx (+ dres), d_table, d_wqkv, d_bqkv or None, d_wproj, d_bproj)."""
    H, W, nH, ws, shift, qk_scale = geom[:6]
    C = x2.shape[1]
    dev = dy.device
    d_bproj = ops32.colsum(dy, _zeros_f32((C,), dev))
    d_attn = ops32.linear_dgrad(dy, w_proj)
    d_wproj = ops32.linear_wgrad(dy, attn.view(-1, C))
    d_table = _zeros_f32(tuple(table.shape), dev)
    d_qkv = ops32.winattn_bwd(qkv.view(*shp, 3 * C), table, attn, lse, d_attn.view(*shp, C), H, W, nH, ws, shift, d_table,
                              qk_scale, mask)
    dq2 = d_qkv.view(-1, 3 * C)
    d_bqkv = ops32.colsum(dq2, _zeros_f32((3 * C,), dev)) if has_qkv_bias else None
    d_x = ops32.linear_dgrad(dq2, w_qkv, res=dres)
    d_wqkv = ops32.linear_wgrad(dq2, x2)
    return d_x, d_table, d_wqkv, d_bqkv, d_wproj, d_bproj


def _mlp_fwd32(x2, w1, b1, w2, b2, res=None):
    """fc1 -> GELU -> fc2 (+ res) in fp32.  Returns (u = fc1 out, y)."""
    u = ops32.linear(x2, w1, b1)
    return u, ops32.linear(u, w2, b2, res=res, gelu_input=True)


def _mlp_bwd32(dy, x2, u, w1, w2):
    """Backward of ``_mlp_fwd32`` from dy [rows, C_out].  Returns (dx, d_w1, d_b1, d_w2, d_b2)."""
    dev = dy.device
    d_b2 = ops32.colsum(dy, _zeros_f32((w2.shape[0],), dev))
    dh = ops32.linear_dgrad(dy, w2)
    d_w2 = ops32.linear_wgrad(dy, u, gelu_input=True)
    du = ops32.mul_gelu_grad(dh, u)
    d_b1 = ops32.colsum(du, _zeros_f32((w1.shape[0],), dev))
    dx = ops32.linear_dgrad(du, w1)
    d_w1 = ops32.linear_wgrad(du, x2)
    return dx, d_w1, d_b1, d_w2, d_b2


class _AttentionFn32(torch.autograd.Function):
    """``_AttentionFn`` in the fp32-accurate mode: x [Bp, T, H*W, C] fp32."""

    @staticmethod
    def forward(ctx, x, table, w_qkv, b_qkv, w_proj, b_proj, geom, mask=None):
        x2 = x.reshape(-1, x.shape[-1])
        qkv, attn, lse, out = _attn_fwd32(x2, x.shape[:3], table, w_qkv, b_qkv, w_proj, b_proj, geom, mask)
        ctx.save_for_backward(x2, qkv, attn, lse, table, w_qkv, w_proj)
        ctx.geom, ctx.mask, ctx.has_qkv_bias = geom, mask, b_qkv is not None
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, d_out):
        d2 = d_out.contiguous().view(-1, d_out.shape[-1])
        d_x, *grads = _attn_bwd32(d2, d_out.shape[:3], *ctx.saved_tensors, ctx.geom, ctx.has_qkv_bias, ctx.mask)
        return (d_x.view(d_out.shape), *grads, None, None)


class _BlockFn32(torch.autograd.Function):
    """``_BlockFn`` (one post-norm SwinTransformerBlock, swin_512.py:196-237) in the fp32-accurate mode."""

    @staticmethod
    def forward(ctx, x, table, w_qkv, b_qkv, w_proj, b_proj, g1, be1, g2, be2, w_fc1, b_fc1, w_fc2, b_fc2, geom):
        eps, infer = geom[6], geom[7]
        x2 = x.reshape(-1, x.shape[-1])
        qkv, attn, lse, y = _attn_fwd32(x2, x.shape[:3], table, w_qkv, b_qkv, w_proj, b_proj, geom, res=x2)
        yn, mean2, rstd2 = ops32.layernorm_fwd(y, g2, be2, eps)
        u, z = _mlp_fwd32(yn, w_fc1, b_fc1, w_fc2, b_fc2, res=y)
        out, mean1, rstd1 = ops32.layernorm_fwd(z, g1, be1, eps)
        if not infer:
            ctx.save_for_backward(x2, qkv, attn, lse, y, yn, mean2, rstd2, u, z, mean1, rstd1, table, w_qkv, w_proj, w_fc1, w_fc2, g1, g2)
            ctx.geom, ctx.has_qkv_bias = geom[:7], b_qkv is not None
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, d_out):
        (x2, qkv, attn, lse, y, yn, mean2, rstd2, u, z, mean1, rstd1, table, w_qkv, w_proj, w_fc1, w_fc2, g1, g2) = ctx.saved_tensors
        C = x2.shape[1]
        d2 = d_out.contiguous().view(-1, C)
        d_g1, d_be1, d_g2, d_be2 = (_zeros_f32((C,), d2.device) for _ in range(4))
        dz = ops32.layernorm_bwd(d2, z, mean1, rstd1, g1, d_g1, d_be1)
        dyn, d_wfc1, d_bfc1, d_wfc2, d_bfc2 = _mlp_bwd32(dz, yn, u, w_fc1, w_fc2)
        dy = ops32.layernorm_bwd(dyn, y, mean2, rstd2, g2, d_g2, d_be2, dres=dz)
        d_x, d_table, d_wqkv, d_bqkv, d_wproj, d_bproj = _attn_bwd32(dy, d_out.shape[:3], x2, qkv, attn, lse, table, w_qkv,
                                                                     w_proj, ctx.geom, ctx.has_qkv_bias, dres=dy)
        return (d_x.view(d_out.shape), d_table, d_wqkv, d_bqkv, d_wproj, d_bproj, d_g1, d_be1, d_g2, d_be2,
                d_wfc1, d_bfc1, d_wfc2, d_bfc2, None)


class _PatchMergeFn32(torch.autograd.Function):
    """``_PatchMergeFn`` in the fp32-accurate mode."""

    @staticmethod
    def forward(ctx, x, gamma, beta, w_red, geom):
        H, W, eps = geom
        B, T, L, C = x.shape
        xn, mean, rstd = ops32.layernorm_fwd(x.reshape(B * T, L, C), gamma, beta, eps, patch_merge_hw=(H, W))
        out = ops32.linear(xn, w_red)
        ctx.save_for_backward(x, xn, mean, rstd, gamma, w_red)
        ctx.geom = geom
        return out.view(B, T, L // 4, w_red.shape[0])

    @staticmethod
    def backward(ctx, d_out):
        x, xn, mean, rstd, gamma, w_red = ctx.saved_tensors
        H, W, eps = ctx.geom
        B, T, L, C = x.shape
        d2 = d_out.contiguous().view(-1, w_red.shape[0])
        dxn = ops32.linear_dgrad(d2, w_red)
        d_w = ops32.linear_wgrad(d2, xn)
        d_gamma, d_beta = _zeros_f32((4 * C,), x.device), _zeros_f32((4 * C,), x.device)
        dx = ops32.layernorm_bwd(dxn, x.reshape(B * T, L, C), mean, rstd, gamma, d_gamma, d_beta, patch_merge_hw=(H, W))
        return dx.view(B, T, L, C), d_gamma, d_beta, d_w, None


class _MlpFn32(torch.autograd.Function):
    """``_MlpFn`` in the fp32-accurate mode."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2):
        x2 = x.reshape(-1, x.shape[-1])
        u, y = _mlp_fwd32(x2, w1, b1, w2, b2)
        ctx.save_for_backward(x2, u, w1, w2)
        return y.view(*x.shape[:-1], w2.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, u, w1, w2 = ctx.saved_tensors
        dx, *grads = _mlp_bwd32(dy.contiguous().view(-1, w2.shape[0]), x2, u, w1, w2)
        return (dx.view(*dy.shape[:-1], w1.shape[1]), *grads)


# The Function of each kind for the token dtype: fp32 tokens run the fp32-accurate mode.
_ATTENTION_FNS = {_BF16: _AttentionFn, torch.float32: _AttentionFn32}
_MLP_FNS = {_BF16: _MlpFn, torch.float32: _MlpFn32}
_BLOCK_FNS = {_BF16: _BlockFn, torch.float32: _BlockFn32}
_PATCH_MERGE_FNS = {_BF16: _PatchMergeFn, torch.float32: _PatchMergeFn32}


def _in_precision(module, x: torch.Tensor, fn) -> torch.Tensor:
    """``fn`` on x as contiguous tokens of the module's precision (fp32 in the fp32-accurate mode, else bf16), with the
    result cast back to x's dtype."""
    if not x.is_cuda:
        raise StswinError("stswincl_b200 modules need CUDA tensors (no CPU path)")
    dtype = torch.float32 if _use_fp32(module, x) else _BF16
    out = fn((x if x.dtype == dtype else x.to(dtype)).contiguous())
    return out if out.dtype == x.dtype else out.to(x.dtype)


class Mlp(nn.Module):
    """Parameter container with the reference's names (swin_512.py:7-23); the math runs fused
    inside the block (fc1 + GELU epilogue, fc2 + residual epilogue)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        if act_layer is not nn.GELU:
            raise NotImplementedError("only nn.GELU (erf) is implemented, as used by every reference config")
        if drop != 0.:
            raise NotImplementedError("dropout > 0 is not used by any reference config and is not implemented")
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        """fc1 -> GELU (erf) -> fc2 on the last dim (swin_512.py:17-23), stand-alone: two GEMMs with the bias / GELU
        epilogues fused.  Inside ``SwinTransformerBlock`` the same GEMMs run with the residual fused as well."""
        params = (self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias)
        return _in_precision(self, x, lambda t: _MLP_FNS[t.dtype].apply(t, *params))


class WindowAttention(nn.Module):
    """swin_512.py:73-141.  ``forward(x_v [B_, T, N, C], mask=None) -> [B_, T, N, C]``.

    Called stand-alone, every window is attended independently (it is treated as a ws x ws image
    with one un-shifted window); an explicit ``mask`` [nW, N, N] is added to the logits of window
    ``b_ % nW`` exactly as at :127-131.  ``SwinTransformerBlock`` does not go through this path: its
    kernels rebuild the shift mask from the geometry."""

    def __init__(self, dim, window_size, num_heads, qkv_bias=True, qk_scale=None, attn_drop=0., proj_drop=0.):
        super().__init__()
        self.dim = dim
        self.window_size = to_2tuple(window_size)
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5
        if attn_drop != 0. or proj_drop != 0.:
            raise NotImplementedError("dropout > 0 is not used by any reference config and is not implemented")
        if self.window_size[0] != self.window_size[1]:
            raise NotImplementedError("square windows only (the reference always passes to_2tuple(ws))")
        ws = self.window_size[0]
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * ws - 1) * (2 * ws - 1), num_heads))
        self.register_buffer("relative_position_index", _relative_position_index(ws, ws))
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)

    def _qk_scale_arg(self) -> float:
        default = (self.dim // self.num_heads) ** -0.5
        return 0.0 if abs(self.scale - default) < 1e-12 else float(self.scale)

    def forward(self, x_v, mask=None):
        B_, T, N, C = x_v.shape
        if mask is not None:
            assert mask.shape[1:] == (N, N) and B_ % mask.shape[0] == 0, "mask must be [nW, N, N] with B_ a multiple of nW"
            mask = mask.detach().to(device=x_v.device, dtype=torch.float32).contiguous()
        ws = self.window_size[0]
        assert N == ws * ws and C == self.dim, "input feature has wrong size"
        geom = (ws, ws, self.num_heads, ws, 0, self._qk_scale_arg())
        args = (self.relative_position_bias_table, self.qkv.weight, self.qkv.bias, self.proj.weight, self.proj.bias, geom, mask)
        return _in_precision(self, x_v, lambda t: _ATTENTION_FNS[t.dtype].apply(t, *args))


class SwinTransformerBlock(nn.Module):
    """swin_512.py:143-237.  ``forward(x_v [B, T, L, C]) -> [B, T, L, C]`` (same dtype as the input).

    The reference asserts T == 2; T == 1 is also accepted here (SURVEY D2) as long as
    T * window_size**2 is 16, 32, 64 or 128."""

    def __init__(self, dim, input_resolution, num_heads, window_size=8, shift_size=0, mlp_ratio=4., qkv_bias=True,
                 qk_scale=None, drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        self.dim = dim
        self.input_resolution = tuple(input_resolution)
        self.num_heads = num_heads
        self.window_size = window_size
        self.shift_size = shift_size
        self.mlp_ratio = mlp_ratio
        if min(self.input_resolution) <= self.window_size:
            self.shift_size = 0
            self.window_size = min(self.input_resolution)
        assert 0 <= self.shift_size < self.window_size, "shift_size must in 0-window_size"
        if norm_layer is not nn.LayerNorm:
            raise NotImplementedError("only nn.LayerNorm is implemented")
        if drop_path != 0.:
            raise NotImplementedError("drop_path > 0 is not used by any reference config and is not implemented")
        self.norm1 = norm_layer(dim)
        self.attn = WindowAttention(dim, window_size=to_2tuple(self.window_size), num_heads=num_heads,
                                    qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop, proj_drop=drop)
        self.drop_path = nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        if self.shift_size > 0:
            H, W = self.input_resolution
            attn_mask = _shift_attn_mask(H, W, self.window_size, self.shift_size)
        else:
            attn_mask = None
        self.register_buffer("attn_mask", attn_mask)

    def _geom(self):
        H, W = self.input_resolution
        return (H, W, self.num_heads, self.window_size, self.shift_size, self.attn._qk_scale_arg(), self.norm1.eps)

    def _block_params(self):
        a, m = self.attn, self.mlp
        return (a.relative_position_bias_table, a.qkv.weight, a.qkv.bias, a.proj.weight, a.proj.bias,
                self.norm1.weight, self.norm1.bias, self.norm2.weight, self.norm2.bias,
                m.fc1.weight, m.fc1.bias, m.fc2.weight, m.fc2.bias)

    def forward_tokens(self, x: torch.Tensor) -> torch.Tensor:
        """bf16 in, bf16 out; no dtype round trip (used by the layer container)."""
        # grad mode is decided here: inside autograd.Function.forward it always reads "disabled", and
        # ctx.needs_input_grad ignores torch.no_grad()
        infer = not torch.is_grad_enabled()
        return _BLOCK_FNS[x.dtype].apply(x, *self._block_params(), self._geom() + (infer,))

    def forward(self, x_v):
        H, W = self.input_resolution
        B, T, L, C = x_v.shape
        assert L == H * W, "input feature has wrong size"
        return _in_precision(self, x_v, self.forward_tokens)


class PatchMerging(nn.Module):
    """swin_512.py:239-277.  ``forward(x [B, T, L, C]) -> [B, T, L/4, 2C]``."""

    def __init__(self, input_resolution, dim, norm_layer=nn.LayerNorm):
        super().__init__()
        self.input_resolution = tuple(input_resolution)
        self.dim = dim
        self.reduction = nn.Linear(4 * dim, 2 * dim, bias=False)
        self.norm = norm_layer(4 * dim)

    def forward_tokens(self, x: torch.Tensor) -> torch.Tensor:
        H, W = self.input_resolution
        return _PATCH_MERGE_FNS[x.dtype].apply(x, self.norm.weight, self.norm.bias, self.reduction.weight, (H, W, self.norm.eps))

    def forward(self, x):
        H, W = self.input_resolution
        B, T, L, C = x.shape
        assert L == H * W, "input feature has wrong size"
        assert H % 2 == 0 and W % 2 == 0, f"x size ({H}*{W}) are not even."
        return _in_precision(self, x, self.forward_tokens)


class SwinTransformerLayerv5(nn.Module):
    """swin_512.py:280-327.  ``forward(x [B, 4, C, H, W]) -> (x3 [B,4,C,H,W], x6 [B,4,2C,H/2,W/2])``.

    Differences in mechanism, not in result: tokens stay bf16 and token-major between blocks;
    the two frame pairs of layers 0 / 2 (which are independent, :302-307) run as one batch of 2B;
    the NCHW <-> token-major moves are single transposing kernels."""

    def __init__(self, dim=512, input_resolution=(64, 80), num_heads=4):
        super().__init__()
        self.dim = dim
        self.input_resolution = tuple(input_resolution)
        self.num_heads = num_heads
        self.num_layers = 3
        self.pairs = [[slice(0, 2), slice(2, 4)], [slice(1, 3)], [slice(0, 2), slice(2, 4)]]  # t=4
        H, W = self.input_resolution
        self.layers = nn.ModuleList()
        for _ in range(self.num_layers):
            self.layers.append(nn.Sequential(
                SwinTransformerBlock(dim, (H, W), num_heads),
                SwinTransformerBlock(dim, (H, W), num_heads, shift_size=4)))
        for _ in range(self.num_layers):
            self.layers.append(nn.Sequential(
                SwinTransformerBlock(dim * 2, (H // 2, W // 2), num_heads, window_size=4),
                SwinTransformerBlock(dim * 2, (H // 2, W // 2), num_heads, window_size=4, shift_size=2)))
        self.downsample = PatchMerging((H, W), dim)

    def _run_layer(self, x: torch.Tensor, layer_idx: int, both_pairs: bool) -> torch.Tensor:
        """x [B, 4, L, C] bf16 -> same.  ``both_pairs``: frames (0,1) and (2,3); else frames (1,2),
        with frames 0 and 3 passing through (swin_512.py:302-307)."""
        B, T, L, C = x.shape
        blk0, blk1 = self.layers[layer_idx][0], self.layers[layer_idx][1]
        if both_pairs:
            y = blk1.forward_tokens(blk0.forward_tokens(x.view(B * 2, 2, L, C)))
            return y.view(B, 4, L, C)
        if not torch.is_grad_enabled():
            return _mid_frames(x, lambda xm: blk1.forward_tokens(blk0.forward_tokens(xm)))
        return _MidLayerFn.apply(x, blk0._geom() + (False,), blk1._geom() + (False,), *blk0._block_params(), *blk1._block_params())

    def _check_input(self, x_v):
        B, T, C, H, W = x_v.shape
        assert T == 4, "input feature has wrong size"
        assert (H, W) == self.input_resolution and C == self.dim, "input feature has wrong size"
        if not x_v.is_cuda:
            raise StswinError("stswincl_b200 modules need CUDA tensors (no CPU path)")
        # outputs keep the input dtype like the reference's (:326); under autocast its last op, LayerNorm, returns fp32
        keep = x_v.dtype if not torch.is_autocast_enabled() else torch.float32
        out_dtype = keep if keep in (torch.float32, _BF16) else torch.float32
        return keep, out_dtype

    def _to_tokens(self, x_v):
        B, T, C, H, W = x_v.shape
        x_in = x_v if x_v.dtype in (torch.float32, _BF16) else x_v.float()
        tok_dtype = torch.float32 if _use_fp32(self, x_v) else _BF16        # fp32 tokens select the fp32-accurate blocks
        return _TransposeFn.apply(x_in.reshape(B * T, C, H * W), tok_dtype).view(B, T, H * W, C)

    def _from_tokens(self, t, stage: int, out_dtype, keep):
        B, T = t.shape[:2]
        H, W = self.input_resolution
        C = self.dim
        if stage == 2:
            H, W, C = H // 2, W // 2, 2 * C
        out = _TransposeFn.apply(t.reshape(B * T, H * W, C), out_dtype).view(B, T, C, H, W)
        return out if keep == out_dtype else out.to(keep)       # fp16 / fp64 callers: cast at the boundary

    def stages(self, like: torch.Tensor):
        """The forward as a chain of four stages, each ``(fn, parameters)`` with ``fn`` mapping a tuple of tensors to
        the next tuple; composing them on ``(x,)`` gives ``forward(x)``.  ``dist.SegmentedStep`` cuts the autograd
        graph at the stage boundaries, so that the gradients of a stage are complete -- and can travel -- while the
        backward of the stages before it still runs.  ``like``: an input tensor (fixes the output dtype)."""
        keep, out_dtype = self._check_input(like)
        L = self.layers

        def s0(x):
            return (self._run_layer(self._to_tokens(x), 0, True),)

        def s1(t):
            return (self._run_layer(self._run_layer(t, 1, False), 2, True),)

        def s2(t):
            return (self._from_tokens(t, 1, out_dtype, keep), self._run_layer(self.downsample.forward_tokens(t.contiguous()), 3, True))

        def s3(out1, u):
            return (out1, self._from_tokens(self._run_layer(self._run_layer(u, 4, False), 5, True), 2, out_dtype, keep))

        return [(s0, list(L[0].parameters())), (s1, list(L[1].parameters()) + list(L[2].parameters())),
                (s2, list(self.downsample.parameters()) + list(L[3].parameters())),
                (s3, list(L[4].parameters()) + list(L[5].parameters()))]

    def forward(self, x_v):
        state = (x_v,)
        for fn, _ in self.stages(x_v):
            state = fn(*state)
        return state
