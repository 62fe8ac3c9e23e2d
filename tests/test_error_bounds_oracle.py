"""CPU: the per-element error bounds of ``oracle/error_bounds.py``.

Each reference equals the existing oracle; an fp64 simulation of the kernels' documented rounding points stays inside
its bound; and small defects of the kind a kernel bug produces (a wrong scale, one wrong value row or bias entry, a
misplaced 32-row group or bias group, a dropped row of a column reduction) exceed it -- most of them while today's
max-relative bars of the GPU tests still accept them."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from oracle import error_bounds as eb
from oracle import swin_oracle as so
from test_gpu_winattn import make_case

D = torch.float64
# a handful of the GPU cases: ws 8 shifted, 7x7 padded slots, 2x2 windows with head_dim 32, stage-2-like, 3x3 windows
SIM_CASES = [(2, 2, 16, 24, 256, 2, 8, 4), (3, 1, 14, 21, 128, 2, 7, 3), (2, 1, 8, 12, 128, 4, 2, 0),
             (1, 2, 8, 12, 256, 2, 4, 2), (2, 2, 9, 12, 64, 1, 3, 1)]
CTRL_CASES = [(2, 2, 16, 24, 256, 2, 8, 4), (1, 2, 64, 80, 512, 4, 8, 4), (3, 1, 14, 21, 128, 2, 7, 3)]
TOL_ATTN_TODAY = 2e-2        # the max-relative bar of tests/test_gpu_winattn.py
TOL_GEMM_TODAY = 1e-2        # ... of tests/test_gpu_gemm.py and tests/test_gpu_lnorm.py


def _bf(t):
    return t.to(torch.bfloat16).to(D)


def _dout(case, seed=5):
    B, T, H, W, C = case[:5]
    return torch.randn(B, T, H * W, C, generator=torch.Generator().manual_seed(seed)).to(torch.bfloat16)


@pytest.mark.parametrize("case", SIM_CASES[:3], ids=str)
def test_attention_reference_equals_oracle(case):
    B, T, H, W, C, nH, ws, shift = case
    qkv, table = make_case(*case)
    d_out = _dout(case)
    q64 = qkv.to(D).requires_grad_(True)
    t64 = table.to(D).requires_grad_(True)
    ref = so.attention_core_unrolled(q64, t64, (H, W), ws, shift, nH)
    (ref * d_out.to(D)).sum().backward()
    r = eb.attention(qkv, table, H, W, ws, shift, nH, d_out=d_out)
    assert (r["out"] - ref.detach()).abs().max() < 1e-12
    assert (r["d_qkv"] - q64.grad).abs().max() < 1e-12
    assert (r["d_table"] - t64.grad).abs().max() < 1e-12
    assert (r["colsum"] - q64.grad.sum((0, 1, 2))).abs().max() < 1e-11
    assert (r["out_mag"] >= r["out"].abs() * (1 - 1e-12)).all()


def test_attention_reference_qk_scale_and_mask():
    """qk_scale and a dense mask on top of the shift mask, against attention_core on explicitly gathered windows."""
    B, T, H, W, C, nH, ws, shift = 2, 2, 16, 24, 128, 2, 8, 4
    qkv, table = make_case(B, T, H, W, C, nH, ws, shift, seed=3)
    nW, N = (H // ws) * (W // ws), ws * ws
    mask = torch.where(torch.rand(3, N, N, generator=torch.Generator().manual_seed(1)) < 0.2, -100.0, 0.0)
    r = eb.attention(qkv, table, H, W, ws, shift, nH, qk_scale=0.11, mask=mask)
    from oracle import index_oracle as ix
    gidx = torch.from_numpy(ix.window_gather_index(H, W, ws, shift)).reshape(-1)
    full = torch.from_numpy(ix.shift_attn_mask(H, W, ws, shift)).to(D) + mask.to(D)[torch.arange(nW) % 3]
    qw = qkv.to(D)[:, :, gidx].reshape(B, T, nW, N, 3 * C).permute(0, 2, 1, 3, 4).reshape(B * nW, T * N, 3 * C)
    ow = so.attention_core(qw, table.to(D), ws, nH, full, T, qk_scale=0.11)
    ow = ow.reshape(B, nW, T, N, C).permute(0, 2, 1, 3, 4).reshape(B, T, nW * N, C)
    ref = torch.empty_like(ow)
    ref[:, :, gidx] = ow
    assert (r["out"] - ref).abs().max() < 1e-12


def test_layernorm_reference_equals_oracle():
    g = torch.Generator().manual_seed(4)
    for pm in (False, True):
        BT, Hh, Ww, C0 = 3, 8, 12, 64
        x = (torch.randn(BT, Hh * Ww, C0, generator=g) * 2 + 0.5).to(torch.bfloat16)
        C = 4 * C0 if pm else C0
        rows = eb.pm_gather(x, Hh, Ww) if pm else x.reshape(-1, C0)
        dy = torch.randn(rows.shape, generator=g).to(torch.bfloat16)
        dres = None if pm else torch.randn(rows.shape, generator=g).to(torch.bfloat16)
        gam, bet = 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
        x64 = x.to(D).requires_grad_(True)
        g64, b64 = gam.to(D).requires_grad_(True), bet.to(D).requires_grad_(True)
        xin = eb.pm_gather(x64, Hh, Ww) if pm else x64.reshape(-1, C0)
        y = so.layer_norm(xin, g64, b64)
        (y * dy.to(D)).sum().backward()
        r = eb.layernorm(rows, gam, bet, dy=dy, dres=dres)
        assert (r["y"] - y.detach()).abs().max() < 1e-12
        dx = eb.pm_scatter(r["dx"], BT, Hh, Ww) if pm else r["dx"].reshape(x.shape)
        want = x64.grad + (0 if dres is None else dres.to(D).reshape(x.shape))
        assert (dx - want).abs().max() < 1e-12
        assert (r["dgamma"] - g64.grad).abs().max() < 1e-11
        assert (r["dbeta"] - b64.grad).abs().max() < 1e-11
        assert torch.equal(eb.pm_scatter(eb.pm_gather(x, Hh, Ww), BT, Hh, Ww), x)


@pytest.mark.parametrize("mode", [eb.EPI_BIAS, eb.EPI_BIAS_RES, eb.EPI_BIAS_GELU, eb.EPI_MUL_AUX, eb.EPI_MUL_AUX_Q8,
                                  eb.EPI_F32_REDUCE])
def test_gemm_reference_equals_linear(mode):
    g = torch.Generator().manual_seed(7)
    M, N, K = 70, 48, 40
    a = torch.randn(M, K, generator=g).to(torch.bfloat16)
    b = torch.randn(N, K, generator=g).to(torch.bfloat16)
    bias = torch.randn(N, generator=g)
    aux = torch.randint(0, 256, (M, N), generator=g, dtype=torch.uint8) if mode == eb.EPI_MUL_AUX_Q8 else \
        torch.randn(M, N, generator=g).to(torch.bfloat16)
    base = torch.randn(M, N, generator=g)
    r = eb.gemm(a, b, mode, bias=bias, aux=aux, base=base, k_splits=3)
    lin = F.linear(a.to(D), b.to(D), bias.to(D))
    if mode == eb.EPI_BIAS:
        want = lin
    elif mode == eb.EPI_BIAS_RES:
        want = lin + aux.to(D)
    elif mode == eb.EPI_MUL_AUX:
        want = lin * aux.to(D)
    elif mode == eb.EPI_MUL_AUX_Q8:
        want = lin * (aux.to(D) * (1.28 / 255) - 0.14)
    elif mode == eb.EPI_F32_REDUCE:
        want = base.to(D) + F.linear(a.to(D), b.to(D))
    else:
        u = lin.clone().requires_grad_(True)
        h = F.gelu(u)
        h.sum().backward()
        assert (r["g"] - u.grad).abs().max() < 1e-12
        want = h.detach()
    assert (r["d"] - want).abs().max() < 1e-11
    assert (r["d_mag"] > 0).all()


@pytest.mark.parametrize("case", SIM_CASES, ids=str)
def test_simulated_kernel_numerics_inside_bound(case):
    """The kernels' documented rounding points, simulated in fp64, stay inside kappa u M (forward kappa 2, backward
    kappa 4) on every element; the forward sits near 1.0-1.4 u M, i.e. <= 0.7 of its bound."""
    B, T, H, W, C, nH, ws, shift = case
    qkv, table = make_case(*case)
    d_out = _dout(case)
    ref = eb.attention(qkv, table, H, W, ws, shift, nH, d_out=d_out)
    sim = eb.attention(qkv, table, H, W, ws, shift, nH, d_out=d_out, simulate_bf16=True)
    loc = eb.attn_locator(H, W, ws, shift, C, nH)
    fwd = eb.check_bound(sim["out"], ref["out"], ref["out_mag"], eb.KAPPA_ATTN_FWD, eb.U_BF16, locate=loc)
    assert fwd.n_over == 0 and fwd.ratio <= 0.75, fwd.message("out")
    bwd = eb.check_bound(sim["d_qkv"], ref["d_qkv"], ref["d_qkv_mag"], eb.KAPPA_ATTN_BWD, eb.U_BF16, locate=loc)
    assert bwd.n_over == 0, bwd.message("d_qkv")
    cs = eb.check_bound(sim["colsum"], ref["colsum"], ref["colsum_mag"], eb.KAPPA_ATTN_BWD, eb.U_BF16, locate=loc)
    assert cs.n_over == 0, cs.message("colsum")


def _attn_ratio(got, ref, case):
    B, T, H, W, C, nH, ws, shift = case
    return eb.check_bound(got, ref["out"], ref["out_mag"], eb.KAPPA_ATTN_FWD, eb.U_BF16,
                          locate=eb.attn_locator(H, W, ws, shift, C, nH))


@pytest.mark.parametrize("case", CTRL_CASES, ids=str)
def test_negative_controls_attention(case):
    """qk scale x 1.01, one value row x 0.97, one bias-table entry + 0.05: each exceeds the bound on at least one
    element while the max-relative bar of the GPU tests (2e-2) still accepts it."""
    B, T, H, W, C, nH, ws, shift = case
    qkv, table = make_case(*case)
    ref = eb.attention(qkv, table, H, W, ws, shift, nH)
    hd = C // nH
    scaled = eb.attention(qkv, table, H, W, ws, shift, nH, qk_scale=1.01 * hd ** -0.5)["out"]
    q2 = qkv.to(D).clone()
    q2[0, 0, 5, 2 * C:2 * C + hd] *= 0.97
    vrow = eb.attention(q2, table, H, W, ws, shift, nH)["out"]
    t2 = table.clone()
    t2[table.shape[0] // 3, 0] += 0.05
    bias = eb.attention(qkv, t2, H, W, ws, shift, nH)["out"]
    report = {}
    for name, got in (("qk_scale x1.01", scaled), ("v row x0.97", vrow), ("bias entry +0.05", bias)):
        got = _bf(got)
        r = _attn_ratio(got, ref, case)
        report[name] = (r.ratio, rel_err(got, ref["out"]))
        assert r.ratio > 1, f"{name}: invisible to the bound ({r.message()})"
        assert report[name][1] < TOL_ATTN_TODAY, f"{name}: today's bar already sees it"
    print(case, {k: "ratio %.2f rel_err %.1e" % v for k, v in report.items()})


def test_negative_controls_gemm():
    """A 32-row group of a 256x256 tile taken from the neighbouring tile, and the bias applied to the wrong 8-column
    group: both exceed the bound, localised to the tile / columns they hit."""
    g = torch.Generator().manual_seed(11)
    M, N, K = 512, 520, 200
    a = (torch.randn(M, K, generator=g) * K ** -0.5).to(torch.bfloat16)
    b = torch.randn(N, K, generator=g).to(torch.bfloat16)
    bias = torch.randn(N, generator=g)
    r = eb.gemm(a, b, eb.EPI_BIAS, bias=bias)
    good = _bf(r["d"])
    ok = eb.check_bound(good, r["d"], r["d_mag"])
    assert ok.n_over == 0, ok.message("bf16-rounded reference")
    swapped = good.clone()
    swapped[256 + 64:256 + 96, 256:512] = good[256 + 64:256 + 96, 0:256]
    bad = eb.check_bound(swapped, r["d"], r["d_mag"], locate=eb.gemm_locator())
    assert bad.ratio > 1 and "tile (1, 1)" in bad.worst, bad.message("32-row group from the neighbouring tile")
    shifted_bias = bias.clone()
    shifted_bias[264:272] = bias[272:280]
    wrong = _bf(eb.gemm(a, b, eb.EPI_BIAS, bias=shifted_bias)["d"])
    bad2 = eb.check_bound(wrong, r["d"], r["d_mag"], locate=eb.gemm_locator())
    assert bad2.ratio > 1 and 264 <= int(bad2.worst.split("column ")[1].split(",")[0]) < 272, bad2.message("bias group")
    print("gemm controls: tile group ratio %.1f rel_err %.1e | bias group ratio %.1f rel_err %.1e"
          % (bad.ratio, rel_err(swapped, r["d"]), bad2.ratio, rel_err(wrong, r["d"])))


def test_negative_controls_layernorm_dropped_row():
    """At M = 163840 rows the column reductions (dgamma, dbeta, column sums of dx) are long fp32 chains; dropping the
    row with the largest term in the checked column still exceeds their bound, and today's 1e-2 bar accepts it."""
    M, C = 163840, 64
    g = torch.Generator().manual_seed(2)
    x = (torch.randn(M, C, generator=g) * 2 + 0.5).to(torch.bfloat16)
    dy = torch.randn(M, C, generator=g).to(torch.bfloat16)
    gam, bet = 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    r = eb.layernorm(x, gam, bet, dy=dy)
    col = 5
    dx_bf = _bf(r["dx"])
    cs_ref, cs_mag = eb.colsum(dx_bf, chain=eb.ln_chain(M))
    terms = {"dgamma": (r["dgamma"], r["dgamma_mag"], r["dgamma_terms"][:, col]),
             "dbeta": (r["dbeta"], r["dbeta_mag"], r["dbeta_terms"][:, col]),
             "dx_colsum": (cs_ref, cs_mag, dx_bf[:, col])}
    for name, (ref, mag, t) in terms.items():
        row = int(t.abs().argmax())
        got = ref.clone()
        got[col] -= t[row]
        b = eb.check_bound(got, ref, mag, locate=eb.ln_locator)
        assert b.ratio > 1 and b.worst.startswith(f"channel {col} "), b.message(f"{name} without row {row}")
        assert rel_err(got, ref) < TOL_GEMM_TODAY, name
        print(f"{name}: row {row} dropped -> ratio {b.ratio:.2f}, rel_err {rel_err(got, ref):.1e}")


def test_check_bound_reports_nonfinite_and_location():
    ref = torch.zeros(300, 300, dtype=D)
    mag = torch.ones(300, 300, dtype=D)
    got = ref.clone()
    got[260, 17] = float("nan")
    b = eb.check_bound(got, ref, mag, locate=eb.gemm_locator())
    assert b.ratio == float("inf") and b.n_over == 1 and "row 260, column 17, 256x256 tile (1, 0)" in b.worst
