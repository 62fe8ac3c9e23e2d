"""fp32-accurate mode: torch-tensor wrappers over the ``stswin_f32_*`` / ``stswin_winattn_f32_*`` entry points and the
split-bf16 dense layer built on ``stswin_gemm_bf16`` (include/stswin_b200.h, "fp32-accurate mode").  No fallbacks."""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib, ops
from .ops import _al16, _launch, _ptr, _req, _stream

_F32 = torch.float32
SPLIT_A, SPLIT_B = 0, 1          # operand patterns (hi, hi, lo) / (hi, lo, hi)
COLS, ROWS = 0, 1                # reduction over columns ([R, 3C]) / over rows ([3R, C])


def split(x: torch.Tensor, layout: int, pattern: int, gelu: bool = False) -> torch.Tensor:
    """fp32 [R, C] -> the three bf16 terms of ``stswin_f32_split`` ([R, 3C] or [3R, C])."""
    x = _al16(x)
    _req(x, _F32, "x")
    assert x.dim() == 2
    R, C = x.shape
    out = torch.empty((R, 3 * C) if layout == COLS else (3 * R, C), dtype=torch.bfloat16, device=x.device)
    with _launch("f32_split", float(x.numel() * 10), x):
        st = _lib.load().stswin_f32_split(x.data_ptr(), out.data_ptr(), R, C, layout, pattern, int(gelu), _stream(x))
    _lib.check(st, "stswin_f32_split")
    return out


def rows_init(shape, device, bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[r, c] = bias[c] + res[r, c] -- what a ``D += acc`` GEMM starts from."""
    out = torch.empty(shape, dtype=_F32, device=device)
    bias = _al16(bias)
    if bias is None and res is None:
        return out.zero_()
    with _launch("f32_rowop", float(out.numel() * (8 if res is not None else 4)), out):
        st = _lib.load().stswin_f32_rowop(out.data_ptr(), _ptr(bias), _ptr(res), None, shape[0], shape[1], 0, _stream(out))
    _lib.check(st, "stswin_f32_rowop")
    return out


def mul_gelu_grad(a: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """a * gelu_erf'(u)."""
    _req(a, _F32, "a"); _req(u, _F32, "u")
    assert a.shape == u.shape and a.is_contiguous() and u.is_contiguous()
    out = torch.empty_like(a)
    with _launch("f32_rowop", float(a.numel() * 12), a):
        st = _lib.load().stswin_f32_rowop(out.data_ptr(), None, a.data_ptr(), u.data_ptr(), a.shape[0], a.shape[1], 1, _stream(a))
    _lib.check(st, "stswin_f32_rowop")
    return out


def colsum(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    _req(x, _F32, "x"); _req(out, _F32, "out")
    assert x.dim() == 2 and x.is_contiguous() and out.numel() == x.shape[1]
    with _launch("f32_colsum", float(x.numel() * 4), x):
        st = _lib.load().stswin_f32_colsum(x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], _stream(x))
    _lib.check(st, "stswin_f32_colsum")
    return out


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
           gelu_input: bool = False) -> torch.Tensor:
    """y = f(x) W^T + bias + res in fp32 accuracy: x [M, K], W [N, K] (``nn.Linear`` layout); f = GELU when
    ``gelu_input``.  One bf16 tcgen05 GEMM over K' = 3K."""
    M, N = x.shape[0], w.shape[0]
    y = rows_init((M, N), x.device, bias, res)
    ops.gemm(split(x, COLS, SPLIT_A, gelu=gelu_input), split(w, COLS, SPLIT_B), mode=ops.EPI_F32_REDUCE, out=y)
    return y


def linear_dgrad(dy: torch.Tensor, w: torch.Tensor, res: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dx = dy W (+ res): dy [M, N], W [N, K]."""
    dx = rows_init((dy.shape[0], w.shape[1]), dy.device, None, res)
    ops.gemm(split(dy, COLS, SPLIT_A), split(w, ROWS, SPLIT_B), b_mn_major=True, mode=ops.EPI_F32_REDUCE, out=dx)
    return dx


def linear_wgrad(dy: torch.Tensor, x: torch.Tensor, gelu_input: bool = False) -> torch.Tensor:
    """dW [N, K] = dy^T f(x), reduced over the rows (tokens) on the tensor cores, split-K."""
    N, K, tokens = dy.shape[1], x.shape[1], dy.shape[0]
    dw = torch.zeros((N, K), dtype=_F32, device=dy.device)
    ops.gemm(split(dy, ROWS, SPLIT_A), split(x, ROWS, SPLIT_B, gelu=gelu_input), a_mn_major=True, b_mn_major=True,
             mode=ops.EPI_F32_REDUCE, out=dw, k_splits=ops._wgrad_splits(N, K, 3 * tokens))   # the split rows are 3x
    return dw


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, patch_merge_hw=None):
    gamma, beta = gamma.contiguous(), beta.contiguous()
    _req(x, _F32, "x")
    assert x.is_contiguous()
    M, row_len, pm, H, W, C = ops._layernorm_rows(x, patch_merge_hw)
    y = torch.empty((M, row_len), dtype=_F32, device=x.device)
    mean = torch.empty(M, dtype=_F32, device=x.device)
    rstd = torch.empty(M, dtype=_F32, device=x.device)
    with _launch("f32_layernorm_fwd", 8.0 * M * row_len, x):
        st = _lib.load().stswin_f32_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                                  rstd.data_ptr(), M, row_len, eps, pm, H, W, C, _stream(x))
    _lib.check(st, "stswin_f32_layernorm_fwd")
    return y, mean, rstd


def layernorm_bwd(dy, x, mean, rstd, gamma, dgamma, dbeta, dres=None, patch_merge_hw=None):
    _req(dy, _F32, "dy"); _req(x, _F32, "x")
    assert dy.is_contiguous() and x.is_contiguous()
    M, row_len, pm, H, W, C = ops._layernorm_rows(x, patch_merge_hw)
    dx = torch.empty_like(x)
    with _launch("f32_layernorm_bwd", 20.0 * M * row_len, x):
        st = _lib.load().stswin_f32_layernorm_bwd(dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
                                                  _ptr(dres), dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), M, row_len,
                                                  pm, H, W, C, _stream(x))
    _lib.check(st, "stswin_f32_layernorm_bwd")
    ops.count_extra_launches(1)
    return dx


def winattn_fwd(qkv, table, H, W, nH, ws, shift, qk_scale=0.0, mask=None):
    """fp32 qkv [B, T, H*W, 3C] -> (out [B, T, H*W, C] fp32, lse)."""
    table = table.contiguous()
    _req(qkv, _F32, "qkv"); _req(table, _F32, "bias_table")
    B, T, L, C3 = qkv.shape
    C = C3 // 3
    assert L == H * W and qkv.is_contiguous()
    out = torch.empty((B, T, L, C), dtype=_F32, device=qkv.device)
    lse = torch.empty(B * T * L * nH, dtype=_F32, device=qkv.device)
    with _launch("winattn_f32_fwd", 16.0 * C * B * T * L, qkv):
        st = _lib.load().stswin_winattn_f32_fwd(qkv.data_ptr(), table.data_ptr(), out.data_ptr(), lse.data_ptr(), B, T, H, W, C, nH,
                                                ws, shift, float(qk_scale), _ptr(mask), ops._mask_windows(mask, ws), _stream(qkv))
    _lib.check(st, "stswin_winattn_f32_fwd")
    return out, lse


def winattn_bwd(qkv, table, out, lse, d_out, H, W, nH, ws, shift, d_table, qk_scale=0.0, mask=None):
    _req(qkv, _F32, "qkv"); _req(d_out, _F32, "d_out"); _req(out, _F32, "out")
    B, T, L, C3 = qkv.shape
    C = C3 // 3
    assert d_out.is_contiguous() and out.is_contiguous() and d_table.is_contiguous()
    d_qkv = torch.empty_like(qkv)
    delta = torch.empty_like(lse)
    with _launch("winattn_f32_bwd", 28.0 * C * B * T * L, qkv):
        st = _lib.load().stswin_winattn_f32_bwd(qkv.data_ptr(), table.data_ptr(), out.data_ptr(), lse.data_ptr(), d_out.data_ptr(),
                                                d_qkv.data_ptr(), d_table.data_ptr(), delta.data_ptr(), B, T, H, W, C, nH, ws, shift,
                                                float(qk_scale), _ptr(mask), ops._mask_windows(mask, ws), _stream(qkv))
    _lib.check(st, "stswin_winattn_f32_bwd")
    ops.count_extra_launches(1)
    return d_qkv
