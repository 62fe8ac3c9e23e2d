"""Thin torch-tensor wrappers over the C ABI (include/stswin_b200.h).

Each function checks shapes/dtypes, passes raw device pointers and the *current*
CUDA stream, and raises ``StswinError`` on a non-zero status.  No fallbacks.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import StswinError

EPI_BIAS, EPI_BIAS_RES, EPI_BIAS_GELU, EPI_MUL_AUX, EPI_F32_REDUCE, EPI_BIAS_GELU_FWD = 0, 1, 2, 3, 4, 5
EPI_BIAS_GELU_Q8, EPI_MUL_AUX_Q8 = 6, 7      # GELU' kept as one byte per element (include/stswin_b200.h)

# ---------------------------------------------------------------------------------------------
# launch accounting (bench.py): every C-ABI kernel launch is counted; with an EventProfiler
# installed each launch is also bracketed by CUDA events on the launching stream.  The counter and
# the profiler are shared by every thread that calls into the library (autograd workers,
# nn.DataParallel replica threads): both are only touched under ``_ACCT``.
import threading

_ACCT = threading.Lock()
_TLS = threading.local()          # per thread: devices whose context this thread has bound inside the library
LAUNCHES = 0


class EventProfiler:
    """Per-kernel-family device time from CUDA events recorded on the launching stream.
    ``work`` is the algorithmic FLOPs (tensor-bound kernels) or bytes (HBM-bound) of the launch."""

    def __init__(self):
        self.records = []          # (family, work, start_event, end_event)

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        with _ACCT:
            records = list(self.records)
        for fam, work, e0, e1 in records:
            d = out.setdefault(fam, {"launches": 0, "ms": 0.0, "work": 0.0})
            d["launches"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["work"] += work
        return out


_PROFILER: Optional["EventProfiler"] = None


def set_profiler(p: Optional["EventProfiler"]) -> None:
    global _PROFILER
    with _ACCT:
        _PROFILER = p


def count_extra_launches(n: int) -> None:
    """Kernels a C-ABI call launches beyond its first one (counted for bench.py's ``gpu_launches``)."""
    global LAUNCHES
    with _ACCT:
        LAUNCHES += n


class _launch:
    """Context of one C-ABI call: makes the tensor's device current for the duration of the call -- on the torch side
    (``torch.cuda.device``, restored on exit, so a call on a tensor of another GPU never changes the caller's current
    device) and inside the library (``stswin_set_device``: a fresh autograd-worker / DataParallel replica thread has no
    driver context bound yet, and tensor-map encoding is a driver call) -- counts the launch and, with a profiler
    installed, brackets it with CUDA events on the launching stream."""

    def __init__(self, family: str, work: float, ref: torch.Tensor):
        self.family, self.work, self.ref = family, work, ref

    def __enter__(self):
        global LAUNCHES
        dev = self.ref.device
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        # the common case -- the tensor lives on the thread's current device -- needs no guard
        self.guard = None
        if idx != torch.cuda.current_device():
            self.guard = torch.cuda.device(idx)
            self.guard.__enter__()
        try:
            bound = getattr(_TLS, "bound", None)
            if bound is None:
                bound = _TLS.bound = set()
            if idx not in bound or self.guard is not None:      # first call of this thread on this device, or a switch
                _lib.check(_lib.load().stswin_set_device(idx), "stswin_set_device")
                bound.add(idx)
            with _ACCT:
                LAUNCHES += 1
                self.prof = _PROFILER
            if self.prof is not None:
                self.e0 = torch.cuda.Event(enable_timing=True)
                self.e0.record(torch.cuda.current_stream(dev))
        except BaseException:
            if self.guard is not None:
                self.guard.__exit__(None, None, None)
            raise
        return self

    def __exit__(self, *exc):
        try:
            if self.prof is not None and exc[0] is None:
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record(torch.cuda.current_stream(self.ref.device))
                with _ACCT:
                    self.prof.records.append((self.family, self.work, self.e0, e1))
        finally:
            if self.guard is not None:
                self.guard.__exit__(*exc)      # restores the caller's device (torch issues the cudaSetDevice)
        return False


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor):
    """Current stream of the tensor's device (call inside a ``_launch`` block)."""
    return torch.cuda.current_stream(t.device).cuda_stream


def _al16(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """A 16-byte aligned, contiguous version of a small parameter tensor (bias, LayerNorm scale, bias table).  Replica
    parameters of nn.DataParallel are views into one coalesced broadcast buffer and can start at any 4-byte offset; the
    kernels read these vectors with 16-byte loads."""
    if t is None:
        return None
    if t.data_ptr() % 16 != 0 or not t.is_contiguous():
        t = t.contiguous()
        if t.data_ptr() % 16 != 0:
            t = t.clone()
    return t


def _req(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise StswinError(f"{name} must be a CUDA tensor (stswincl_b200 has no CPU path)")
    if t.dtype != dtype:
        raise StswinError(f"{name} must be {dtype}, got {t.dtype}")


def gemm(a: torch.Tensor, b: torch.Tensor, *, a_mn_major: bool = False, b_mn_major: bool = False,
         mode: int = EPI_BIAS, bias: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None, out2: Optional[torch.Tensor] = None,
         colsum: Optional[torch.Tensor] = None, k_splits: int = 1) -> torch.Tensor:
    """D[M,N] = sum_k A[m,k] B[n,k] with a fused epilogue (stswin_gemm_bf16).

    a: [M,K] (K-major) or [K,M] (``a_mn_major``); b: [N,K] or [K,N] (``b_mn_major``).
    Rows may be strided (last dim contiguous)."""
    _req(a, torch.bfloat16, "a"); _req(b, torch.bfloat16, "b")
    assert a.dim() == 2 and b.dim() == 2 and a.stride(1) == 1 and b.stride(1) == 1
    (K, M) = a.shape if a_mn_major else a.shape[::-1]
    (Kb, N) = b.shape if b_mn_major else b.shape[::-1]
    assert K == Kb, f"reduction dims differ: {K} vs {Kb}"
    if mode == EPI_F32_REDUCE:
        assert out is not None and out.dtype == torch.float32, "fp32 reduce epilogue accumulates into `out`"
    elif out is None:
        out = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
    assert out.shape == (M, N) and out.stride(1) == 1
    if mode in (EPI_BIAS_GELU, EPI_BIAS_GELU_Q8) and out2 is None:
        out2 = torch.empty((M, N), dtype=torch.uint8 if mode == EPI_BIAS_GELU_Q8 else torch.bfloat16, device=a.device)
    if out2 is not None:
        _req(out2, torch.uint8 if mode == EPI_BIAS_GELU_Q8 else torch.bfloat16, "out2")
        assert out2.shape == (M, N) and out2.stride() == out.stride()
    if aux is not None:
        _req(aux, torch.uint8 if mode == EPI_MUL_AUX_Q8 else torch.bfloat16, "aux"); assert aux.shape == (M, N) and aux.stride(1) == 1
    if bias is not None:
        bias = _al16(bias)
        _req(bias, torch.float32, "bias"); assert bias.numel() == N
    if colsum is not None:
        _req(colsum, torch.float32, "colsum"); assert colsum.numel() == N and colsum.is_contiguous()
    lib = _lib.load()
    fam = "gemm_wgrad" if mode == EPI_F32_REDUCE else "gemm"
    with _launch(fam, 2.0 * M * N * K, a):
        st = lib.stswin_gemm_bf16(a.data_ptr(), int(a_mn_major), a.stride(0), b.data_ptr(), int(b_mn_major), b.stride(0),
                                  out.data_ptr(), out.stride(0), _ptr(out2), _ptr(aux), aux.stride(0) if aux is not None else 0,
                                  _ptr(bias), _ptr(colsum), M, N, K, mode, k_splits, _stream(a))
    _lib.check(st, "stswin_gemm_bf16")
    return out


def _wgrad_splits(n_out: int, k_in: int, tokens: int) -> int:
    """Split-K factor of a weight-gradient GEMM dW [n_out, k_in] reduced over ``tokens`` rows: about two work items per
    CTA pair of the 148 SMs, and at least 64 rows per split."""
    tiles = ((n_out + 127) // 128) * ((k_in + 255) // 256)
    return max(1, min((tokens + 63) // 64, round(2 * 148 / tiles)))


def _mask_windows(mask: Optional[torch.Tensor], ws: int) -> int:
    if mask is None:
        return 0
    _req(mask, torch.float32, "mask")
    assert mask.dim() == 3 and mask.shape[1] == ws * ws and mask.shape[2] == ws * ws and mask.is_contiguous()
    return mask.shape[0]


def winattn_lse_elems(B, T, H, W, C, nH, ws) -> int:
    n = _lib.load().stswin_winattn_lse_elems(B, T, H, W, C, nH, ws)
    if n < 0:
        _lib.check(-2, "stswin_winattn_lse_elems")
    return n


def winattn_fwd(qkv: torch.Tensor, bias_table: torch.Tensor, H: int, W: int, num_heads: int, ws: int, shift: int,
                out: Optional[torch.Tensor] = None, qk_scale: float = 0.0, mask: Optional[torch.Tensor] = None):
    """qkv [B, T, H*W, 3C] bf16 (natural token order) -> (out [B, T, H*W, C] bf16, lse2 fp32).
    stswin_winattn_fwd: gather (roll+partition) / QK^T / bias+mask / softmax / PV / scatter."""
    bias_table = _al16(bias_table)
    _req(qkv, torch.bfloat16, "qkv"); _req(bias_table, torch.float32, "bias_table")
    B, T, L, C3 = qkv.shape
    assert L == H * W and C3 % 3 == 0 and qkv.is_contiguous()
    C = C3 // 3
    assert bias_table.shape == ((2 * ws - 1) ** 2, num_heads)
    if out is None:
        out = torch.empty((B, T, L, C), dtype=torch.bfloat16, device=qkv.device)
    lse2 = torch.empty(winattn_lse_elems(B, T, H, W, C, num_heads, ws), dtype=torch.float32, device=qkv.device)
    with _launch("winattn_fwd", 8.0 * C * B * T * L, qkv):     # bytes: q,k,v in + o out, bf16 = 8*C per token (SURVEY 8d)
        st = _lib.load().stswin_winattn_fwd(qkv.data_ptr(), bias_table.data_ptr(), out.data_ptr(), lse2.data_ptr(),
                                            B, T, H, W, C, num_heads, ws, shift, float(qk_scale),
                                            _ptr(mask), _mask_windows(mask, ws), _stream(qkv))
    _lib.check(st, "stswin_winattn_fwd")
    return out, lse2


def winattn_bwd(qkv: torch.Tensor, bias_table: torch.Tensor, lse2: torch.Tensor, d_out: torch.Tensor,
                H: int, W: int, num_heads: int, ws: int, shift: int, d_table: torch.Tensor,
                d_qkv_colsum: Optional[torch.Tensor] = None, d_qkv: Optional[torch.Tensor] = None,
                qk_scale: float = 0.0, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Gradient of winattn_fwd: returns d_qkv [B,T,H*W,3C] bf16; accumulates into d_table (fp32
    [(2ws-1)^2, nH]) and, if given, into d_qkv_colsum (fp32 [3C])."""
    bias_table = _al16(bias_table)
    _req(qkv, torch.bfloat16, "qkv"); _req(d_out, torch.bfloat16, "d_out")
    _req(d_table, torch.float32, "d_table"); _req(lse2, torch.float32, "lse2")
    B, T, L, C3 = qkv.shape
    C = C3 // 3
    assert d_out.shape == (B, T, L, C) and d_out.is_contiguous() and qkv.is_contiguous()
    assert d_table.shape == bias_table.shape and d_table.is_contiguous()
    if d_qkv is None:
        d_qkv = torch.empty_like(qkv)
    if d_qkv_colsum is not None:
        _req(d_qkv_colsum, torch.float32, "d_qkv_colsum"); assert d_qkv_colsum.numel() == C3
    with _launch("winattn_bwd", 14.0 * C * B * T * L, qkv):    # bytes: q,k,v,dO in + dq,dk,dv out, bf16 = 14*C per token
        st = _lib.load().stswin_winattn_bwd(qkv.data_ptr(), bias_table.data_ptr(), lse2.data_ptr(), d_out.data_ptr(),
                                            d_qkv.data_ptr(), d_table.data_ptr(), _ptr(d_qkv_colsum),
                                            B, T, H, W, C, num_heads, ws, shift, float(qk_scale),
                                            _ptr(mask), _mask_windows(mask, ws), _stream(qkv))
    _lib.check(st, "stswin_winattn_bwd")
    return d_qkv


def _layernorm_rows(x: torch.Tensor, patch_merge_hw):
    """Row geometry of a LayerNorm over x: ``(M, row_len, pm, H, W, C)`` as the C ABI takes it.  Rows are the last dim of
    x, or with ``patch_merge_hw=(H, W)`` the 2x2-gathered 4C vectors of PatchMerging (x [BT, H*W, C])."""
    if patch_merge_hw is None:
        return x.numel() // x.shape[-1], x.shape[-1], 0, 0, 0, 0
    H, W = patch_merge_hw
    C = x.shape[-1]
    return x.numel() // C // 4, 4 * C, 1, H, W, C


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, *,
                  patch_merge_hw=None):
    """LayerNorm over the last dim of x [M, C] (bf16) -> (y bf16, mean fp32 [M], rstd fp32 [M]).
    With ``patch_merge_hw=(H, W)``: x is [BT, H*W, C]; rows are the 2x2-gathered 4C vectors of
    PatchMerging (swin_512.py:266-274) and y is [BT*H*W/4, 4C]."""
    gamma, beta = _al16(gamma), _al16(beta)
    _req(x, torch.bfloat16, "x"); _req(gamma, torch.float32, "gamma"); _req(beta, torch.float32, "beta")
    assert x.is_contiguous()
    M, row_len, pm, H, W, C = _layernorm_rows(x, patch_merge_hw)
    assert gamma.numel() == row_len and beta.numel() == row_len
    y = torch.empty((M, row_len), dtype=torch.bfloat16, device=x.device)
    mean = torch.empty(M, dtype=torch.float32, device=x.device)
    rstd = torch.empty(M, dtype=torch.float32, device=x.device)
    with _launch("layernorm_fwd", 4.0 * M * row_len, x):            # read x, write y (bf16)
        st = _lib.load().stswin_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                              rstd.data_ptr(), M, row_len, eps, pm, H, W, C, _stream(x))
    _lib.check(st, "stswin_layernorm_fwd")
    return y, mean, rstd


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, gamma: torch.Tensor,
                  dgamma: torch.Tensor, dbeta: torch.Tensor, *, dres: Optional[torch.Tensor] = None,
                  dx_colsum: Optional[torch.Tensor] = None, patch_merge_hw=None) -> torch.Tensor:
    """Returns dx (layout of x); accumulates dgamma / dbeta (fp32) and optionally the column sums of dx."""
    gamma = _al16(gamma)
    _req(dy, torch.bfloat16, "dy"); _req(x, torch.bfloat16, "x")
    assert dy.is_contiguous() and x.is_contiguous()
    M, row_len, pm, H, W, C = _layernorm_rows(x, patch_merge_hw)
    assert dy.numel() == M * row_len
    dx = torch.empty_like(x)
    if dres is not None:
        _req(dres, torch.bfloat16, "dres"); assert dres.is_contiguous() and dres.numel() == dy.numel()
    with _launch("layernorm_bwd", (6.0 + (2.0 if dres is not None else 0.0)) * M * row_len, x):
        st = _lib.load().stswin_layernorm_bwd(dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
                                              _ptr(dres), dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _ptr(dx_colsum),
                                              M, row_len, pm, H, W, C, _stream(x))
    _lib.check(st, "stswin_layernorm_bwd")
    return dx


def transpose(x: torch.Tensor, out_dtype: torch.dtype) -> torch.Tensor:
    """[batch, R, Cc] -> [batch, Cc, R] with fp32/bf16 conversion (stswin_transpose)."""
    assert x.dim() == 3 and x.is_contiguous() and x.is_cuda
    assert x.dtype in (torch.float32, torch.bfloat16) and out_dtype in (torch.float32, torch.bfloat16)
    b, R, Cc = x.shape
    out = torch.empty((b, Cc, R), dtype=out_dtype, device=x.device)
    with _launch("transpose", float(x.numel() * x.element_size() + out.numel() * out.element_size()), x):
        st = _lib.load().stswin_transpose(x.data_ptr(), int(x.dtype == torch.float32), out.data_ptr(),
                                          int(out_dtype == torch.float32), b, R, Cc, _stream(x))
    _lib.check(st, "stswin_transpose")
    return out


def copy_frames(dst: torch.Tensor, src: torch.Tensor) -> None:
    """dst[b] = src[b] for two [batch, ...] views whose trailing dims are dense (only the batch stride
    may differ): the frame slices of the middle Swin layer (stswin_copy_strided)."""
    assert dst.shape == src.shape and dst.dtype == src.dtype and dst.is_cuda and src.is_cuda
    b = dst.shape[0]
    inner = dst[0].numel() * dst.element_size()
    assert dst[0].is_contiguous() and src[0].is_contiguous()
    ds = dst.stride(0) * dst.element_size() if b > 1 else inner
    ss = src.stride(0) * src.element_size() if b > 1 else inner
    with _launch("copy", float(2 * b * inner), dst):
        st = _lib.load().stswin_copy_strided(dst.data_ptr(), ds, src.data_ptr(), ss, inner, b, _stream(dst))
    _lib.check(st, "stswin_copy_strided")



def colsum(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[c] += sum_r x[r, c] for bf16 x [R, C] (bias gradient of a Linear whose output gradient is x);
    ``out`` fp32 [C], accumulated into (stswin_colsum)."""
    _req(x, torch.bfloat16, "x"); _req(out, torch.float32, "out")
    assert x.dim() == 2 and x.is_contiguous() and out.numel() == x.shape[1] and out.is_contiguous()
    with _launch("colsum", float(x.numel() * 2), x):
        st = _lib.load().stswin_colsum(x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], _stream(x))
    _lib.check(st, "stswin_colsum")
    return out


def gather_cast(dst, src) -> None:
    """dst[i].copy_(src[i]) for lists of contiguous CUDA tensors, src fp32, dst fp32 or bf16 (all the same), as
    multi-tensor launches (stswin_gather_cast): the gradient gather of ``dist.SegmentedStep``."""
    import ctypes
    assert len(dst) == len(src) and len(dst) > 0
    to_bf16 = dst[0].dtype == torch.bfloat16
    for d, s in zip(dst, src):
        _req(s, torch.float32, "src"); _req(d, torch.bfloat16 if to_bf16 else torch.float32, "dst")
        assert d.numel() == s.numel() and d.is_contiguous() and s.is_contiguous()
    n = len(dst)
    with _launch("gather_cast", float(sum(s.numel() for s in src) * (4 + dst[0].element_size())), dst[0]):
        st = _lib.load().stswin_gather_cast((ctypes.c_void_p * n)(*[d.data_ptr() for d in dst]),
                                            (ctypes.c_void_p * n)(*[s.data_ptr() for s in src]),
                                            (ctypes.c_int64 * n)(*[s.numel() for s in src]), n, int(to_bf16), _stream(dst[0]))
    _lib.check(st, "stswin_gather_cast")
    count_extra_launches((n + 47) // 48 - 1)
