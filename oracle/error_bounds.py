"""Per-element error bounds for the bf16 / fp32 kernels.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  For each operation the functions below return the exact result
``ref`` (fp64) on the kernel's own inputs together with a magnitude ``mag`` of the same shape, and
``check_bound(got, ref, mag, kappa, u, floor)`` reports the worst ``|got - ref| / (kappa * u * mag + floor)``.  A
kernel that is right up to its documented rounding points stays at or below 1 on every element; an error confined to
one tile, one window or one row shows up there even when it is far below a max-relative bar.

Numerics the bounds rest on (u = 2^-8 for a bf16 result, gamma(n) = n * 2^-24 for a chain of n fp32 additions):

* GEMM.  Products of bf16 operands are exact in fp32; a dot product of length K is a chain of K additions, the bias
  and the residual one more each, and the bf16 store rounds once: ``u |ref| + gamma(K + 2) (|A| |B|^T + |bias| + |aux|)``.
  The x-aux modes multiply the fp32 ``acc + bias`` by aux (the kernel adds ``bias`` before the product; aux is
  dequantised from the kernel's own bytes in the one-byte mode).  GELU: the epilogue evaluates
  Phi(u) ~ 0.5 + 0.5 tanh(u (c0 + c1 u^2)) with tanh.approx: the fit is good to 2.7e-4 on GELU and 8.7e-4 on GELU',
  tanh.approx adds 2.4e-4 (DESIGN.md section 8), so h gets ``2.7e-4 + 2.4e-4`` absolute and GELU' 1.5e-3; the
  accumulation error moves h by at most max|GELU'| = 1.13 times itself and GELU' by max|GELU''| = 0.8 times itself.
  The byte form of GELU' adds half a quantisation step (0.64 / 255).  The split-K fp32 reduce is a chain of
  ceil(K / splits) MMA additions, then ``splits`` reduce-adds onto the base; column sums of D are a chain of the
  kernel's sequential depth over the bf16 values it stored.
* Window attention (bf16).  S and the softmax are fp32; the unnormalised P is rounded to bf16 before P V, the output
  once more: per element ``kappa u M_i`` with M_i = sum_j P_ij |v_j| and kappa = 2 (an fp64 simulation of those
  rounding points peaks at 1.03-1.39 u M).  Backward: P and dS enter their MMAs as bf16 and the outputs are stored as
  bf16, so with A_ij = P_ij (|dP_ij| + sum_j' P_ij' |dP_ij'|) (a bound on |dS_ij|) kappa = 4 on
  dV_j: sum_i P_ij |dO_i|, dQ_i: scale sum_j A_ij |k_j|, dK_j: scale sum_i A_ij |q_i|, d_table[r, h]: the A_ij of the
  pairs at relative index r, and the qkv column sums: the sums of the d_qkv magnitudes.  The last two are fp32 sums over
  many windows / tokens; their chain (gamma of the number of terms times the sum of magnitudes) is added as an
  absolute floor, because a kappa u bound does not grow with the number of terms.
* fp32 attention (SIMT kernels): the same magnitudes with u = 2^-24 and kappa = 4 (L + head_dim).
* LayerNorm.  Mean and variance are fp32 sums over the row (chain C each).  The error of the mean is at most
  gamma(C) mean|x|, which moves x_hat by rstd times that even where x_hat is 0, so the bounds use
  xa = |x_hat| + rstd mean_j |x_j| wherever |x_hat| enters: forward ``u |y| + gamma(2C) (xa |gamma| + |beta|)``;
  backward ``u |dx| + gamma(2C) (rstd (|gamma dy| + mean|gamma dy| + xa mean|gamma dy| xa) + |dres|)``; the column
  reductions (dgamma, dbeta, dx column sums) are chains of the kernel's depth (rows per warp + 8 warps + one atomic per
  CTA) over their absolute terms.  Statistics: a lane sums C/32 values in sequence and five shuffle steps fold the
  warp, so the mean is good to gamma(C/32 + 5) mean|x| and rstd (half the relative error of the variance, plus two
  ulp of rsqrt) to gamma(C/32 + 5) / 2 + 2^-22 relative.
"""
from __future__ import annotations

import math
from typing import Callable, NamedTuple, Optional

import torch

from . import index_oracle as ix

U_BF16 = 2.0 ** -8
U_F32 = 2.0 ** -24
GELU_ABS = 2.7e-4 + 2.4e-4        # tanh-form fit + tanh.approx, on GELU
GELU_GRAD_ABS = 1.5e-3             # on GELU' (fit 8.7e-4 + tanh.approx)
Q8_STEP = 1.28 / 255.0             # one-byte GELU' (include/stswin_b200.h)
Q8_OFF = 0.14
KAPPA_ATTN_FWD = 2.0
KAPPA_ATTN_BWD = 4.0

EPI_BIAS, EPI_BIAS_RES, EPI_BIAS_GELU, EPI_MUL_AUX, EPI_F32_REDUCE, EPI_BIAS_GELU_FWD = 0, 1, 2, 3, 4, 5
EPI_BIAS_GELU_Q8, EPI_MUL_AUX_Q8 = 6, 7


def gamma(n) -> float:
    """Error factor of a chain of n fp32 additions."""
    return float(n) * U_F32


class Bound(NamedTuple):
    ratio: float          # worst |got - ref| / (kappa u mag + floor); inf for a non-finite element
    n_over: int           # elements above 1
    worst: str            # the worst element, in the kernel's terms

    def message(self, what: str = "") -> str:
        return f"{what}: worst ratio {self.ratio:.3g} at {self.worst}; {self.n_over} element(s) above the bound"


def check_bound(got, ref, mag, kappa: float = 1.0, u: float = 1.0, floor=0.0,
                locate: Optional[Callable[[tuple], str]] = None) -> Bound:
    """Worst ratio |got - ref| / (kappa u mag + floor) and the number of elements above 1 (fp64, on ref's device).
    ``locate`` turns the index of the worst element into words (``gemm_locator`` / ``attn_locator`` / ``ln_locator``)."""
    ref = torch.as_tensor(ref).double()
    got = torch.as_tensor(got).to(ref.device).double().reshape(ref.shape)
    mag = torch.as_tensor(mag).to(ref.device).double()
    bound = kappa * u * mag + (floor.to(ref.device).double() if torch.is_tensor(floor) else floor)
    err = (got - ref).abs()
    ratio = torch.where(torch.isfinite(got), err / bound.clamp_min(1e-300), torch.full_like(err, math.inf))
    ratio = torch.where((err == 0) & torch.isfinite(got), torch.zeros_like(ratio), ratio)
    flat = int(torch.argmax(ratio.reshape(-1)))
    idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), ref.shape)) if ref.dim() else ()
    worst = float(ratio.reshape(-1)[flat])
    where = locate(idx) if locate is not None else f"index {idx}"
    where += f" (got {float(got.reshape(-1)[flat]):.6g}, ref {float(ref.reshape(-1)[flat]):.6g}, bound {float(bound.reshape(-1)[flat]):.3g})"
    return Bound(worst, int((ratio > 1).sum()), where)


def gemm_locator(row_offset: int = 0) -> Callable[[tuple], str]:
    def loc(idx):
        if len(idx) == 1:
            return f"column {idx[0]} (256-column tile {idx[0] // 256})"
        r, c = idx[0] + row_offset, idx[1]
        return f"row {r}, column {c}, 256x256 tile ({r // 256}, {c // 256})"
    return loc


def attn_locator(H: int, W: int, ws: int, shift: int, C: int, nH: int) -> Callable[[tuple], str]:
    """Index of a [B, T, H*W, C or 3C] tensor -> token, window (roll + partition order) and head."""
    hd = C // nH

    def loc(idx):
        if len(idx) == 1:                        # a [3C] column sum
            c = idx[0]
            return f"column {c} ({'qkv'[c // C]}, head {(c % C) // hd})"
        if len(idx) == 2:                        # a [(2ws-1)^2, nH] bias-table gradient
            return f"bias-table entry {idx[0]}, head {idx[1]}"
        b, t, l, c = idx
        h, w = l // W, l % W
        win = (((h - shift) % H) // ws) * (W // ws) + ((w - shift) % W) // ws
        return f"batch {b}, frame {t}, token {l} (h {h}, w {w}), window {win}, head {(c % C) // hd}, channel {c}"
    return loc


def ln_locator(idx) -> str:
    return f"row {idx[0]}, channel {idx[1]}" if len(idx) == 2 else f"channel {idx[0]}"


# ---------------------------------------------------------------------------------------------------------------
# GEMM (stswin_gemm_bf16)
# ---------------------------------------------------------------------------------------------------------------

def q8_dequant(q: torch.Tensor) -> torch.Tensor:
    return q.double() * Q8_STEP - Q8_OFF


def gemm(a: torch.Tensor, b: torch.Tensor, mode: int, bias=None, aux=None, base=None, k_splits: int = 1):
    """a [M, K], b [N, K] (logical K-major views, any dtype) -> dict of fp64 references and magnitudes on a's device.

    Keys: ``d`` / ``d_mag`` (bounds with kappa u = 1; for F32_REDUCE ``base + A B^T``), and for the GELU modes
    ``g`` / ``g_mag`` (GELU' in bf16, or dequantised bytes)."""
    A, B = a.double(), b.double()
    K = A.shape[1]
    acc = A @ B.t()
    macc = A.abs() @ B.abs().t()
    bias64 = bias.double().reshape(1, -1) if bias is not None else torch.zeros(1, B.shape[0], dtype=torch.float64, device=A.device)
    g = gamma(K + 2)
    out = {}
    if mode == EPI_F32_REDUCE:
        base64 = base.double()
        ref = base64 + acc
        chain = -(-((K + 63) // 64) // k_splits) * 64 + k_splits + 1
        out["d"], out["d_mag"] = ref, gamma(chain) * (macc + base64.abs()) + U_F32 * ref.abs()
        return out
    if mode in (EPI_BIAS, EPI_BIAS_RES):
        ref = acc + bias64
        m = macc + bias64.abs()
        if mode == EPI_BIAS_RES:
            ref = ref + aux.double()
            m = m + aux.double().abs()
        out["d"], out["d_mag"] = ref, U_BF16 * ref.abs() + g * m
    elif mode in (EPI_MUL_AUX, EPI_MUL_AUX_Q8):
        mul = q8_dequant(aux) if mode == EPI_MUL_AUX_Q8 else aux.double()
        ref = (acc + bias64) * mul
        out["d"], out["d_mag"] = ref, U_BF16 * ref.abs() + g * (macc + bias64.abs()) * mul.abs()
    else:                                        # the GELU modes
        uu = acc + bias64
        cdf = 0.5 * (1.0 + torch.erf(uu / math.sqrt(2.0)))
        h = uu * cdf
        gd = cdf + uu * torch.exp(-0.5 * uu * uu) / math.sqrt(2.0 * math.pi)
        du = g * (macc + bias64.abs())
        out["d"], out["d_mag"] = h, U_BF16 * h.abs() + GELU_ABS + 1.13 * du
        if mode == EPI_BIAS_GELU:
            out["g"], out["g_mag"] = gd, U_BF16 * gd.abs() + GELU_GRAD_ABS + 0.8 * du
        elif mode == EPI_BIAS_GELU_Q8:
            out["g"], out["g_mag"] = gd, 0.5 * Q8_STEP + GELU_GRAD_ABS + 0.8 * du
    return out


def colsum(d: torch.Tensor, base: Optional[torch.Tensor] = None, chain: Optional[int] = None):
    """Column sums of the kernel's own bf16 D (+ base) and the bound (kappa u = 1).  ``chain`` defaults to the GEMM
    epilogue's depth: 8 rows per lane + 2 shuffle steps per 32-row group, one atomic per group."""
    D = d.double()
    M = D.shape[0]
    if chain is None:
        chain = -(-M // 32) + 32
    ref = D.sum(0)
    mag = D.abs().sum(0)
    if base is not None:
        ref = ref + base.double()
        mag = mag + base.double().abs()
    return ref, gamma(chain + 1) * mag


# ---------------------------------------------------------------------------------------------------------------
# window attention (stswin_winattn_*, stswin_winattn_f32_*)
# ---------------------------------------------------------------------------------------------------------------

def _attn_setup(qkv, table, H, W, ws, shift, nH, qk_scale, mask):
    dev = qkv.device
    B, T, Ltok, C3 = qkv.shape
    C, N = C3 // 3, ws * ws
    hd, L, nW = C // nH, T * N, (H // ws) * (W // ws)
    scale = qk_scale if (qk_scale is not None and qk_scale > 0) else hd ** -0.5
    gidx = torch.from_numpy(ix.window_gather_index(H, W, ws, shift)).reshape(-1).to(dev)
    qw = qkv.double()[:, :, gidx].reshape(B, T, nW, N, 3, nH, hd).permute(0, 2, 4, 5, 1, 3, 6).reshape(B, nW, 3, nH, L, hd)
    rel = torch.from_numpy(ix.relative_position_index(ws)).to(dev).repeat(T, T)             # [L, L]
    s_add = table.double().to(dev)[rel.reshape(-1)].reshape(L, L, nH).permute(2, 0, 1)[None, None]   # [1, 1, nH, L, L]
    sm = ix.shift_attn_mask(H, W, ws, shift)
    if sm is not None:
        s_add = s_add + torch.from_numpy(sm).to(dev).double().repeat(1, T, T)[None, :, None]
    if mask is not None:
        mw = mask.shape[0]
        dm = mask.double().to(dev)[torch.arange(nW, device=dev) % mw].repeat(1, T, T)
        s_add = s_add + dm[None, :, None]
    return dict(B=B, T=T, Ltok=Ltok, C=C, N=N, hd=hd, L=L, nW=nW, nH=nH, scale=scale, gidx=gidx, rel=rel,
                q=qw[:, :, 0], k=qw[:, :, 1], v=qw[:, :, 2], s_add=s_add)


def _to_tokens(g, x):
    """[B, nW, X, nH, L, hd] windowed (X = 1 or 3 blocks of C) -> [B, T, H*W, X*C] natural order."""
    B, T, nW, N, nH, hd = g["B"], g["T"], g["nW"], g["N"], g["nH"], g["hd"]
    X = x.shape[2]
    y = x.reshape(B, nW, X, nH, T, N, hd).permute(0, 4, 1, 5, 2, 3, 6).reshape(B, T, nW * N, X * nH * hd)
    out = torch.empty_like(y)
    out[:, :, g["gidx"]] = y
    return out


def attention(qkv, table, H, W, ws, shift, nH, d_out=None, qk_scale=None, mask=None, simulate_bf16: bool = False):
    """Exact (fp64) window attention on the kernel's inputs and the magnitudes of the module docstring.

    qkv [B, T, H*W, 3C] (natural token order), table [(2ws-1)^2, nH], optional dense additive mask [mw, N, N] applied
    on top of the shift mask (window w uses mask[w % mw]).  Returns a dict: out / out_mag, and with ``d_out``
    d_qkv / d_qkv_mag, d_table / d_table_mag / d_table_terms (pairs per entry), colsum / colsum_mag.
    ``simulate_bf16`` instead rounds at the kernels' documented points (unnormalised P before P V, P and dS before
    their MMAs, every bf16 output): the results are then a simulation of the kernels, not the reference."""
    g = _attn_setup(qkv, table, H, W, ws, shift, nH, qk_scale, mask)
    bf = (lambda t: t.to(torch.bfloat16).double()) if simulate_bf16 else (lambda t: t)
    q, k, v, scale = g["q"], g["k"], g["v"], g["scale"]
    s = scale * (q @ k.transpose(-1, -2)) + g["s_add"]
    e = torch.exp(s - s.amax(-1, keepdim=True))
    Z = e.sum(-1, keepdim=True)
    P = e / Z
    o = bf((bf(e) @ v) / Z)
    res = {"out": _to_tokens(g, o[:, :, None]), "out_mag": _to_tokens(g, (P @ v.abs())[:, :, None])}
    if d_out is None:
        return res
    B, T, nW, N, C, nHh, hd = g["B"], g["T"], g["nW"], g["N"], g["C"], g["nH"], g["hd"]
    dw = d_out.double()[:, :, g["gidx"]].reshape(B, T, nW, N, nHh, hd).permute(0, 2, 4, 1, 3, 5).reshape(B, nW, nHh, g["L"], hd)
    dP = dw @ v.transpose(-1, -2)
    dv = bf(bf(P).transpose(-1, -2) @ dw)
    dS = P * (dP - (P * dP).sum(-1, keepdim=True))
    dq = bf(scale * (bf(dS) @ k))
    dk = bf(scale * (bf(dS).transpose(-1, -2) @ q))
    A = P * (dP.abs() + (P * dP.abs()).sum(-1, keepdim=True))
    dv_m = P.transpose(-1, -2) @ dw.abs()
    dq_m = scale * (A @ k.abs())
    dk_m = scale * (A.transpose(-1, -2) @ q.abs())
    res["d_qkv"] = _to_tokens(g, torch.stack([dq, dk, dv], 2))
    res["d_qkv_mag"] = _to_tokens(g, torch.stack([dq_m, dk_m, dv_m], 2))
    R = (2 * ws - 1) ** 2
    rel = g["rel"].reshape(-1)
    L2 = g["L"] * g["L"]
    res["d_table"] = torch.zeros(R, nHh, dtype=torch.float64, device=qkv.device).index_add_(
        0, rel, dS.sum((0, 1)).reshape(nHh, L2).t())
    res["d_table_mag"] = torch.zeros(R, nHh, dtype=torch.float64, device=qkv.device).index_add_(
        0, rel, A.sum((0, 1)).reshape(nHh, L2).t())
    res["d_table_terms"] = torch.bincount(rel, minlength=R).double() * (B * nW)
    res["colsum"] = res["d_qkv"].sum((0, 1, 2))
    res["colsum_mag"] = res["d_qkv_mag"].sum((0, 1, 2))
    res["tokens"] = B * T * g["Ltok"]
    return res


# ---------------------------------------------------------------------------------------------------------------
# LayerNorm (stswin_layernorm_*)
# ---------------------------------------------------------------------------------------------------------------

def pm_gather(x: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """PatchMerging 2x2 gather: x [BT, H*W, C] -> rows [BT*H*W/4, 4C] (swin_512.py:266-274)."""
    BT, C = x.shape[0], x.shape[-1]
    return x.reshape(BT, H // 2, 2, W // 2, 2, C).permute(0, 1, 3, 4, 2, 5).reshape(BT * H * W // 4, 4 * C)


def pm_scatter(rows: torch.Tensor, BT: int, H: int, W: int) -> torch.Tensor:
    """Inverse of ``pm_gather``: rows [BT*H*W/4, 4C] -> [BT, H*W, C]."""
    C = rows.shape[-1] // 4
    return rows.reshape(BT, H // 2, W // 2, 2, 2, C).permute(0, 1, 4, 2, 3, 5).reshape(BT, H * W, C)


def ln_chain(M: int, sms: int = 148) -> int:
    """Sequential depth of the backward's column reductions: rows per warp (8 warps per CTA, at most 2 CTAs per SM),
    the CTA's 8 warps, one atomic per CTA, and the start value."""
    want = -(-M // 8)
    lo, hi = min(want, sms), min(want, 2 * sms)
    return -(-M // (8 * lo)) + 8 + hi + 1


def layernorm(x, gam, bet, eps: float = 1e-5, dy=None, dres=None, sms: int = 148):
    """x [M, C] rows (already gathered for PatchMerging) -> dict: y / y_mag, mean / rstd (fp64), and with dy:
    dx / dx_mag (rows), dgamma / dbeta with their bounds, and the absolute terms of every column reduction
    (``dgamma_terms``, ``dbeta_terms``) for controls that drop one row.  All bounds with kappa u = 1."""
    X = x.double()
    M, C = X.shape
    g64, b64 = gam.double().to(X.device), bet.double().to(X.device)
    mu = X.mean(-1, keepdim=True)
    var = ((X - mu) ** 2).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    xh = (X - mu) * rstd
    xa = xh.abs() + rstd * X.abs().mean(-1, keepdim=True)
    y = xh * g64 + b64
    gc = gamma(2 * C)
    stat = gamma(-(-C // 32) + 5)
    res = {"mean": mu[:, 0], "rstd": rstd[:, 0], "mean_tol": stat * X.abs().mean(-1), "rstd_rel_tol": stat / 2 + 2.0 ** -22, "y": y,
           "y_mag": U_BF16 * y.abs() + gc * (xa * g64.abs() + b64.abs())}
    if dy is None:
        return res
    DY = dy.double()
    gdy = DY * g64
    m1 = gdy.mean(-1, keepdim=True)
    m2 = (gdy * xh).mean(-1, keepdim=True)
    dx = rstd * (gdy - m1 - xh * m2)
    mag = rstd * (gdy.abs() + gdy.abs().mean(-1, keepdim=True) + xa * (gdy.abs() * xa).mean(-1, keepdim=True))
    if dres is not None:
        dx = dx + dres.double()
        mag = mag + dres.double().abs()
    res["dx"], res["dx_mag"] = dx, U_BF16 * dx.abs() + gc * mag
    ch = gamma(ln_chain(M, sms))
    res["dgamma_terms"], res["dbeta_terms"] = DY * xh, DY
    res["dgamma"], res["dgamma_mag"] = (DY * xh).sum(0), ch * (DY.abs() * xa).sum(0)
    res["dbeta"], res["dbeta_mag"] = DY.sum(0), ch * DY.abs().sum(0)
    return res
