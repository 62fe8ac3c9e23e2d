"""GPU: the GEMM, window-attention (bf16 and fp32) and LayerNorm kernels held to per-element error bounds
(``oracle/error_bounds.py``), with every output element written and nothing outside it.

Harness: each output is a view into a larger allocation with 1 KB guard bands before and after it (and, for GEMM
outputs, a padded row pitch ldd = N + 64).  The bands hold a seeded byte pattern and must be bitwise unchanged after
the call.  Overwritten outputs are produced twice, once over 0x00 bytes and once over 0xFF bytes; both results must
be bitwise identical (an unwritten element differs; so does a non-deterministic one).  Accumulated outputs (split-K
fp32 GEMM, bias-table gradient, column sums, dgamma / dbeta) start from a random base and get the bands only.
Run with ``-s`` to see the worst ratio of every quantity ("BOUND" lines)."""
import math

import pytest
import torch

from oracle import error_bounds as eb
from test_gpu_winattn import CASES, make_case

pytestmark = pytest.mark.gpu

PAD = 1024
F64 = torch.float64


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


class Guarded:
    """An output view of ``shape`` (row pitch ``pitch`` elements, byte offset ``offset`` into the allocation) between
    two PAD-byte guard bands."""

    def __init__(self, shape, dtype, pitch=None, offset=0):
        esz = torch.tensor([], dtype=dtype).element_size()
        shape = tuple(shape)
        rows, cols = int(math.prod(shape[:-1])), shape[-1]
        pitch = pitch or cols
        assert (pitch - cols) * esz <= PAD
        start, size = PAD + offset, rows * pitch * esz
        self.buf = torch.empty(start + size + PAD, dtype=torch.uint8, device="cuda")
        base = self.buf[start:start + size].view(dtype)
        strides = [pitch]
        for d in reversed(shape[1:-1]):
            strides.insert(0, strides[0] * d)
        self.view = base.as_strided(shape, tuple(strides) + (1,)) if len(shape) > 1 else base
        inside = torch.zeros(self.buf.numel(), dtype=torch.bool, device="cuda")
        inside[start:start + size].view(rows, pitch * esz)[:, :cols * esz] = True
        self.outside = ~inside
        g = torch.Generator(device="cuda").manual_seed(1234)
        self.pattern = torch.randint(0, 256, (self.buf.numel(),), generator=g, dtype=torch.uint8, device="cuda")[self.outside]

    def fill(self, byte=None, base=None):
        """Bands <- pattern; the output <- ``byte`` everywhere, or the values of ``base``."""
        if byte is not None:
            self.buf.fill_(byte)
        if base is not None:
            self.view.copy_(base)
        self.buf[self.outside] = self.pattern

    def check_bands(self, what):
        torch.cuda.synchronize()
        bad = (self.buf[self.outside] != self.pattern).nonzero()
        assert bad.numel() == 0, f"{what}: {bad.numel()} guard-band byte(s) written (first at band offset {int(bad[0])})"


def run_twice(fn, outs, accs=(), what=""):
    """Runs ``fn`` over 0x00- and 0xFF-filled outputs (``outs``: Guarded) and returns the first run's results, after
    checking that both agree bitwise and that no band moved.  ``accs``: (Guarded, base) pairs reset before each run."""
    got = []
    for byte in (0x00, 0xFF):
        for o in outs:
            o.fill(byte)
        for a, base in accs:
            a.fill(base=base)
        fn()
        for o in list(outs) + [a for a, _ in accs]:
            o.check_bands(what)
        got.append([o.view.clone() for o in outs])
    for i, (x, y) in enumerate(zip(*got)):
        eq = x.view(torch.uint8) == y.view(torch.uint8) if x.element_size() == 1 else \
            x.contiguous().view(torch.int16 if x.element_size() == 2 else torch.int32) == \
            y.contiguous().view(torch.int16 if y.element_size() == 2 else torch.int32)
        assert eq.all(), f"{what}: output {i} differs between the 0x00 and 0xFF runs at {(~eq).nonzero()[:4].tolist()} " \
                         f"(unwritten or non-deterministic elements)"
    return got[0]


def assert_bound(what, got, ref, mag, kappa=1.0, u=1.0, floor=0.0, locate=None):
    b = eb.check_bound(got, ref, mag, kappa, u, floor, locate)
    print(f"BOUND {what} ratio {b.ratio:.3f}")
    assert b.n_over == 0, b.message(what)
    return b


def _bf16(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).cuda()


# ---------------------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------------------
MAJORS = [(0, 0), (0, 1), (1, 1)]
MODES = [eb.EPI_BIAS, eb.EPI_BIAS_RES, eb.EPI_BIAS_GELU, eb.EPI_MUL_AUX, eb.EPI_F32_REDUCE, eb.EPI_BIAS_GELU_FWD,
         eb.EPI_BIAS_GELU_Q8, eb.EPI_MUL_AUX_Q8]
BYTE_MODES = (eb.EPI_BIAS_GELU_Q8, eb.EPI_MUL_AUX_Q8)
MS, NS, NS8, KS = [1, 100, 129, 384, 1000], [8, 24, 136, 520], [16, 144, 528], [8, 40, 200, 512]


def _ragged_cases():
    """A pairwise-style walk over (majors, mode) x M x N x K x bias x strided operands x colsum placement: every
    instantiation gets two shapes, every value of each factor appears with every mode."""
    out = []
    i = 0
    for mi, majors in enumerate(MAJORS):
        for mode in MODES:
            for rep in range(2):
                M = MS[i % 5]
                N = (NS8 if mode in BYTE_MODES else NS)[(i + mi) % (3 if mode in BYTE_MODES else 4)]
                K = KS[(i // 2 + rep) % 4]
                out.append(dict(majors=majors, mode=mode, M=M, N=N, K=K, bias=(i % 2 == 0), strided=(i % 3 != 0),
                                colsum=(mode != eb.EPI_F32_REDUCE and rep == 0), cs_offset=4 if (mi == 1 and rep == 0) else 0,
                                splits=1 + (i % 3) if mode == eb.EPI_F32_REDUCE else 1))
                i += 1
    return out


def _production_cases():
    """Every GEMM call of swin.py's block at 20480 tokens, both stages (C = 512 / 1024, MLP hidden 4C)."""
    from stswincl_b200.swin import _wgrad_splits
    T = 20480
    out = []
    for C in (512, 1024):
        Hd = 4 * C
        fwd = [("qkv", eb.EPI_BIAS, 3 * C, C), ("proj+res", eb.EPI_BIAS_RES, C, C), ("fc1+gelu", eb.EPI_BIAS_GELU, Hd, C),
               ("fc1+gelu_q8", eb.EPI_BIAS_GELU_Q8, Hd, C), ("fc2+res", eb.EPI_BIAS_RES, C, Hd),
               ("fc1+gelu_fwd", eb.EPI_BIAS_GELU_FWD, Hd, C)]
        for name, mode, N, K in fwd:
            out.append(dict(name=f"C{C}_{name}", majors=(0, 0), mode=mode, M=T, N=N, K=K, bias=True, strided=False,
                            colsum=False, cs_offset=0, splits=1))
        dgrad = [("fc2_dgrad_q8+colsum", eb.EPI_MUL_AUX_Q8, Hd, C), ("fc2_dgrad+colsum", eb.EPI_MUL_AUX, Hd, C),
                 ("fc1_dgrad", eb.EPI_BIAS, C, Hd), ("proj_dgrad", eb.EPI_BIAS, C, C), ("qkv_dgrad+res", eb.EPI_BIAS_RES, C, 3 * C)]
        for name, mode, N, K in dgrad:
            out.append(dict(name=f"C{C}_{name}", majors=(0, 1), mode=mode, M=T, N=N, K=K, bias=False, strided=False,
                            colsum=name.endswith("colsum"), cs_offset=0, splits=1))
        for name, n_out, k_in in (("qkv", 3 * C, C), ("proj", C, C), ("fc1", Hd, C), ("fc2", C, Hd)):
            out.append(dict(name=f"C{C}_{name}_wgrad", majors=(1, 1), mode=eb.EPI_F32_REDUCE, M=n_out, N=k_in, K=T, bias=False,
                            strided=False, colsum=False, cs_offset=0, splits=_wgrad_splits(n_out, k_in, T)))
    # a split-K reduce with more than two items per CTA pair (the block's own wgrad splits aim at about two)
    out.append(dict(name="wgrad_many_items", majors=(1, 1), mode=eb.EPI_F32_REDUCE, M=2048, N=2048, K=1024, bias=False,
                    strided=False, colsum=False, cs_offset=0, splits=4))
    return out


RAGGED, PRODUCTION = _ragged_cases(), _production_cases()


def _items_per_pair(c, sms):
    num_m, num_n = -(-c["M"] // 128), -(-c["N"] // 256)
    kb = -(-c["K"] // 64)
    s = min(c["splits"], kb)
    while s > 1 and (s - 1) * (-(-kb // s)) >= kb:
        s -= 1
    items = ((num_m + 1) // 2) * num_n * s
    return -(-items // min(items, sms // 2))


def _operand(rows, cols, seed, scale, strided):
    """[rows, cols] bf16 with a leading dimension that is a multiple of 8 (+ 8 more when ``strided``)."""
    ld = -(-cols // 8) * 8 + (8 if strided else 0)
    full = torch.zeros(rows, ld, dtype=torch.bfloat16, device="cuda")
    full[:, :cols] = _bf16((rows, cols), seed, scale)
    return full[:, :cols]


def _run_gemm(c):
    from stswincl_b200 import ops
    (am, bm), mode, M, N, K = c["majors"], c["mode"], c["M"], c["N"], c["K"]
    a_in = _operand(M, K, 1, K ** -0.5, c["strided"]) if not am else _operand(K, M, 1, K ** -0.5, c["strided"])
    a_log = a_in if not am else a_in.t()
    b_in = _operand(N, K, 2, 1.0, c["strided"]) if not bm else _operand(K, N, 2, 1.0, c["strided"])
    b_log = b_in if not bm else b_in.t()
    bias = torch.randn(N, generator=torch.Generator().manual_seed(3)).cuda() if c["bias"] else None
    aux = None
    if mode in (eb.EPI_BIAS_RES, eb.EPI_MUL_AUX):
        aux = _operand(M, N, 4, 1.0, c["strided"])
    elif mode == eb.EPI_MUL_AUX_Q8:
        full = torch.randint(0, 256, (M, N + (16 if c["strided"] else 0)), generator=torch.Generator().manual_seed(4),
                             dtype=torch.uint8).cuda()
        aux = full[:, :N]
    ldd = N + 64
    tag = f"{c.get('name', '')} majors {c['majors']} mode {mode} M {M} N {N} K {K}"
    if mode == eb.EPI_F32_REDUCE:
        D = Guarded((M, N), torch.float32, pitch=ldd)
        base = torch.randn(M, N, generator=torch.Generator().manual_seed(5)).cuda()
        D.fill(base=base)
        ops.gemm(a_in, b_in, a_mn_major=bool(am), b_mn_major=bool(bm), mode=mode, bias=bias, out=D.view, k_splits=c["splits"])
        D.check_bands(tag)
        r = eb.gemm(a_log, b_log, mode, base=base, k_splits=c["splits"])
        assert_bound(f"gemm mode {mode} D ({tag})", D.view, r["d"], r["d_mag"], locate=eb.gemm_locator())
        return
    D = Guarded((M, N), torch.bfloat16, pitch=ldd)
    outs = [D]
    D2 = None
    if mode in (eb.EPI_BIAS_GELU, eb.EPI_BIAS_GELU_Q8):
        D2 = Guarded((M, N), torch.uint8 if mode == eb.EPI_BIAS_GELU_Q8 else torch.bfloat16, pitch=ldd)
        outs.append(D2)
    accs = []
    cs = cs_base = None
    if c["colsum"]:
        cs = Guarded((N,), torch.float32, offset=c["cs_offset"])
        cs_base = torch.randn(N, generator=torch.Generator().manual_seed(6)).cuda()
        accs.append((cs, cs_base))

    def call():
        ops.gemm(a_in, b_in, a_mn_major=bool(am), b_mn_major=bool(bm), mode=mode, bias=bias, aux=aux, out=D.view,
                 out2=D2.view if D2 is not None else None, colsum=cs.view if cs is not None else None)
    got = run_twice(call, outs, accs, tag)
    r = eb.gemm(a_log, b_log, mode, bias=bias, aux=aux)
    loc = eb.gemm_locator()
    assert_bound(f"gemm mode {mode} D ({tag})", got[0], r["d"], r["d_mag"], locate=loc)
    if D2 is not None:
        g2 = eb.q8_dequant(got[1]) if mode == eb.EPI_BIAS_GELU_Q8 else got[1]
        assert_bound(f"gemm mode {mode} D2 ({tag})", g2, r["g"], r["g_mag"], locate=loc)
    if cs is not None:
        ref, mag = eb.colsum(got[0], cs_base)
        assert_bound(f"gemm mode {mode} colsum ({tag})", cs.view, ref, mag, locate=loc)


@pytest.mark.parametrize("c", RAGGED, ids=lambda c: "mj%d%d_m%d_M%d_N%d_K%d" % (*c["majors"], c["mode"], c["M"], c["N"], c["K"]))
def test_gemm_ragged(c):
    _run_gemm(c)


@pytest.mark.parametrize("c", PRODUCTION, ids=lambda c: c["name"])
def test_gemm_production_shapes(c):
    _run_gemm(c)


def test_gemm_mn_k_pair_raises():
    from stswincl_b200 import ops
    from stswincl_b200._lib import StswinError
    for mode in MODES:
        out = torch.zeros(128, 256, dtype=torch.float32 if mode == eb.EPI_F32_REDUCE else torch.bfloat16, device="cuda")
        with pytest.raises(StswinError, match="not instantiated"):
            ops.gemm(_bf16((64, 128), 1), _bf16((256, 64), 2), a_mn_major=True, b_mn_major=False, mode=mode, out=out,
                     aux=torch.zeros(128, 256, dtype=torch.uint8 if mode == eb.EPI_MUL_AUX_Q8 else torch.bfloat16, device="cuda"),
                     out2=torch.zeros(128, 256, dtype=torch.uint8 if mode == eb.EPI_BIAS_GELU_Q8 else torch.bfloat16, device="cuda")
                     if mode in (eb.EPI_BIAS_GELU, eb.EPI_BIAS_GELU_Q8) else None)


def test_gemm_every_mode_runs_past_two_items_per_cta_pair():
    """The persistent loop's second use of each TMEM accumulator, the staging ping-pong across items and the next item's
    aux prefetch only run from the third item of a CTA pair on."""
    sms = _sms()
    for mode in MODES:
        best = max(_items_per_pair(c, sms) for c in RAGGED + PRODUCTION if c["mode"] == mode)
        assert best > 2, f"mode {mode}: at most {best} items per CTA pair"


def test_gemm_mul_aux_adds_bias_before_the_product():
    """STSWIN_EPI_MUL_AUX(_Q8) with a bias computes (acc + bias) * aux (include/stswin_b200.h)."""
    from stswincl_b200 import ops
    M, N, K = 256, 256, 64
    A, B = _bf16((M, K), 1, 0.0), _bf16((N, K), 2)
    bias = torch.full((N,), 2.0, device="cuda")
    aux = torch.full((M, N), 3.0, dtype=torch.bfloat16, device="cuda")
    assert torch.all(ops.gemm(A, B, mode=ops.EPI_MUL_AUX, bias=bias, aux=aux).float() == 6.0)
    q = torch.full((M, N), 255, dtype=torch.uint8, device="cuda")          # dequantises to 1.28 - 0.14 = 1.14
    d = ops.gemm(A, B, mode=ops.EPI_MUL_AUX_Q8, bias=bias, aux=q).float()
    assert torch.allclose(d, torch.full_like(d, 2.28), rtol=2 ** -8)


# ---------------------------------------------------------------------------------------------------------------
# window attention
# ---------------------------------------------------------------------------------------------------------------
EXTRA = [((2, 2, 16, 24, 256, 2, 8, 4), 0.07, False), ((3, 1, 14, 21, 128, 2, 7, 3), 0.3, False),
         ((2, 2, 16, 24, 128, 2, 8, 0), 0.0, True), ((2, 1, 8, 12, 128, 2, 4, 2), 0.2, True),
         # the look-up-table kernels for 64- and 32-token windows (a dense mask rules out the compile-time maps)
         ((2, 1, 16, 24, 128, 2, 8, 0), 0.0, True), ((1, 2, 8, 12, 256, 4, 4, 2), 0.0, True)]
ATTN = [(c, 0.0, False) for c in CASES] + EXTRA


def _attn_id(p):
    c, s, m = p
    return "B%d_T%d_%dx%d_C%d_h%d_ws%d_s%d" % c + (f"_scale{s}" if s else "") + ("_mask" if m else "")


def _dense_mask(case):
    B, T, H, W, C, nH, ws, shift = case
    nW, N = (H // ws) * (W // ws), ws * ws
    m = torch.where(torch.rand(nW, N, N, generator=torch.Generator().manual_seed(8)) < 0.25, -100.0, 0.0)
    m[:, torch.arange(N), torch.arange(N)] = 0.0
    return m.cuda()


def _attn_inputs(p, f32=False):
    case, scale, masked = p
    B, T, H, W, C, nH, ws, shift = case
    qkv, table = make_case(*case)
    if f32:
        qkv = torch.randn(qkv.shape, generator=torch.Generator().manual_seed(1)) * 1.2
    d_out = torch.randn(B, T, H * W, C, generator=torch.Generator().manual_seed(5))
    d_out = d_out if f32 else d_out.to(torch.bfloat16)
    return qkv.cuda(), table.cuda(), d_out.cuda(), scale, (_dense_mask(case) if masked else None)


def _attn_check(tag, case, res, out, d_qkv, d_table, colsum, d_table_base, colsum_base, kappa_f, kappa_b, u):
    B, T, H, W, C, nH, ws, shift = case
    loc = eb.attn_locator(H, W, ws, shift, C, nH)
    tag = f"{tag} {case}"
    assert_bound(f"attn{tag} out", out, res["out"], res["out_mag"], kappa_f, u, locate=loc)
    assert_bound(f"attn{tag} d_qkv", d_qkv, res["d_qkv"], res["d_qkv_mag"], kappa_b, u, locate=loc)
    for part, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        b = eb.check_bound(d_qkv[..., sl], res["d_qkv"][..., sl], res["d_qkv_mag"][..., sl], kappa_b, u)
        print(f"BOUND attn{tag} {part} ratio {b.ratio:.3f}")
    # fp32 sums over many windows / tokens: their chain is an absolute floor (error_bounds docstring)
    fl = eb.gamma(res["d_table_terms"].max() + 1) * res["d_table_mag"] + eb.U_F32 * d_table_base.double().abs()
    assert_bound(f"attn{tag} d_table", d_table, d_table_base.double() + res["d_table"], res["d_table_mag"], kappa_b, u,
                 floor=fl, locate=loc)
    if colsum is not None:
        fl = eb.gamma(res["tokens"] + 1) * res["colsum_mag"] + eb.U_F32 * colsum_base.double().abs()
        assert_bound(f"attn{tag} colsum", colsum, colsum_base.double() + res["colsum"], res["colsum_mag"], kappa_b, u,
                     floor=fl, locate=loc)


@pytest.mark.parametrize("p", ATTN, ids=_attn_id)
def test_winattn_bf16_bounds(p):
    from stswincl_b200 import ops
    case = p[0]
    B, T, H, W, C, nH, ws, shift = case
    qkv, table, d_out, scale, mask = _attn_inputs(p)
    res = eb.attention(qkv, table, H, W, ws, shift, nH, d_out=d_out, qk_scale=scale or None, mask=mask)
    out = Guarded((B, T, H * W, C), torch.bfloat16)
    lse = {}

    def fwd():
        lse["v"] = ops.winattn_fwd(qkv, table, H, W, nH, ws, shift, out=out.view, qk_scale=scale, mask=mask)[1]
    o = run_twice(fwd, [out], what=f"winattn_fwd {case}")[0]
    dq = Guarded((B, T, H * W, 3 * C), torch.bfloat16)
    dt = Guarded(tuple(table.shape), torch.float32)
    cs = Guarded((3 * C,), torch.float32)
    dt_base = torch.randn(table.shape, generator=torch.Generator().manual_seed(9)).cuda()
    cs_base = torch.randn(3 * C, generator=torch.Generator().manual_seed(10)).cuda()

    def bwd():
        ops.winattn_bwd(qkv, table, lse["v"], d_out, H, W, nH, ws, shift, dt.view, cs.view, d_qkv=dq.view, qk_scale=scale,
                        mask=mask)
    g = run_twice(bwd, [dq], [(dt, dt_base), (cs, cs_base)], what=f"winattn_bwd {case}")[0]
    _attn_check("", case, res, o, g, dt.view, cs.view, dt_base, cs_base, eb.KAPPA_ATTN_FWD, eb.KAPPA_ATTN_BWD, eb.U_BF16)


def test_winattn_bf16_negative_controls():
    """On real kernel output: qk_scale x 1.01, and separately one bias-table entry + 0.05, against the unperturbed
    reference must exceed the forward bound (an input change, not a kernel edit)."""
    from stswincl_b200 import ops
    case = (1, 2, 64, 80, 512, 4, 8, 4)
    B, T, H, W, C, nH, ws, shift = case
    qkv, table, _, _, _ = _attn_inputs((case, 0.0, False))
    res = eb.attention(qkv, table, H, W, ws, shift, nH)
    loc = eb.attn_locator(H, W, ws, shift, C, nH)
    o = ops.winattn_fwd(qkv, table, H, W, nH, ws, shift, qk_scale=1.01 * (C // nH) ** -0.5)[0]
    b1 = eb.check_bound(o, res["out"], res["out_mag"], eb.KAPPA_ATTN_FWD, eb.U_BF16, locate=loc)
    t2 = table.clone()
    t2[table.shape[0] // 3, 0] += 0.05
    o2 = ops.winattn_fwd(qkv, t2, H, W, nH, ws, shift)[0]
    b2 = eb.check_bound(o2, res["out"], res["out_mag"], eb.KAPPA_ATTN_FWD, eb.U_BF16, locate=loc)
    print(f"CONTROL qk_scale x1.01 ratio {b1.ratio:.2f}; bias entry +0.05 ratio {b2.ratio:.2f}")
    assert b1.ratio > 1 and b2.ratio > 1


def _f32_call(name, *args):
    from stswincl_b200 import _lib, ops
    with ops._launch(name, 0.0, args[0]):
        st = getattr(_lib.load(), "stswin_" + name)(*[a.data_ptr() if torch.is_tensor(a) else a for a in args[1:]])
    _lib.check(st, name)


@pytest.mark.parametrize("p", ATTN, ids=_attn_id)
def test_winattn_fp32_bounds(p):
    from stswincl_b200 import ops
    case = p[0]
    B, T, H, W, C, nH, ws, shift = case
    qkv, table, d_out, scale, mask = _attn_inputs(p, f32=True)
    L, hd = T * ws * ws, C // nH
    res = eb.attention(qkv, table, H, W, ws, shift, nH, d_out=d_out, qk_scale=scale or None, mask=mask)
    out = Guarded((B, T, H * W, C), torch.float32)
    lse = torch.empty(B * T * H * W * nH, device="cuda")
    mw = ops._mask_windows(mask, ws)
    s = torch.cuda.current_stream().cuda_stream
    o = run_twice(lambda: _f32_call("winattn_f32_fwd", qkv, qkv, table, out.view, lse, B, T, H, W, C, nH, ws, shift,
                                    float(scale), mask if mask is not None else None, mw, s), [out], what=f"f32 fwd {case}")[0]
    dq = Guarded((B, T, H * W, 3 * C), torch.float32)
    dt = Guarded(tuple(table.shape), torch.float32)
    dt_base = torch.randn(table.shape, generator=torch.Generator().manual_seed(9)).cuda()
    delta = torch.empty_like(lse)
    g = run_twice(lambda: _f32_call("winattn_f32_bwd", qkv, qkv, table, o.contiguous(), lse, d_out, dq.view, dt.view, delta,
                                    B, T, H, W, C, nH, ws, shift, float(scale), mask, mw, s),
                  [dq], [(dt, dt_base)], what=f"f32 bwd {case}")[0]
    kappa = 4.0 * (L + hd)
    _attn_check("_f32", case, res, o, g, dt.view, None, dt_base, None, kappa, kappa, eb.U_F32)


def test_winattn_fp32_unsupported_raises():
    from stswincl_b200 import ops32
    from stswincl_b200._lib import StswinError
    for (C, nH, ws, msg) in ((512, 4, 16, "> 128"), (24, 2, 4, "multiple of 8")):
        qkv = torch.zeros(1, 2, 64 * 80, 3 * C, device="cuda")
        with pytest.raises(StswinError, match=msg):
            ops32.winattn_fwd(qkv, torch.zeros((2 * ws - 1) ** 2, nH, device="cuda"), 64, 80, nH, ws, 0)


# ---------------------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------------------
LN_CS = [64, 256, 384, 512, 1024, 2048]
LN_MS = [1, 9, 33, 163840]
LN_VARIANTS = [(False, False), (True, False), (False, True), (True, True)]      # (dx_colsum, dres)
LN_CASES = [(C, LN_MS[(ci + vi) % 4], cs, res) for ci, C in enumerate(LN_CS) for vi, (cs, res) in enumerate(LN_VARIANTS)]


def _ln_x(M, C, seed):
    """2 randn + 0.5, with adversarial rows among the first 33: mean 100 (bf16 spacing 0.5), constant, one outlier."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, C, generator=g) * 2 + 0.5
    for r in range(min(M, 33)):
        if r % 4 == 1:
            x[r] = 100 + torch.randn(C, generator=g)
        elif r % 4 == 2:
            x[r] = 1.25
        elif r % 4 == 3:
            x[r, (7 * r) % C] = 60.0
    return x.to(torch.bfloat16).cuda()


def _ln_run(tag, x_in, rows, C, pm_geom, with_cs, with_res):
    """x_in: the kernel's x (plain [M, C] or [BT, H*W, C0]); rows: the gathered [M, C] view of it."""
    from stswincl_b200 import _lib, ops
    M = rows.shape[0]
    g = torch.Generator().manual_seed(4)
    gam = (1.0 + 0.2 * torch.randn(C, generator=g)).cuda()
    bet = (0.2 * torch.randn(C, generator=g)).cuda()
    pm, H, W, C0 = (1, *pm_geom, C // 4) if pm_geom else (0, 0, 0, 0)
    dy = _bf16((M, C), 2)
    dres = _bf16((M, C), 3) if with_res else None
    r = eb.layernorm(rows, gam, bet, dy=dy, dres=dres, sms=_sms())
    lib = _lib.load()
    y, mean, rstd = (Guarded((M, C), torch.bfloat16), Guarded((M,), torch.float32), Guarded((M,), torch.float32))
    s = torch.cuda.current_stream().cuda_stream

    def fwd():
        with ops._launch("layernorm_fwd", 0.0, x_in):
            _lib.check(lib.stswin_layernorm_fwd(x_in.data_ptr(), gam.data_ptr(), bet.data_ptr(), y.view.data_ptr(),
                                                mean.view.data_ptr(), rstd.view.data_ptr(), M, C, 1e-5, pm, H, W, C0, s), "ln fwd")
    yo, mo, ro = run_twice(fwd, [y, mean, rstd], what=f"layernorm_fwd {tag}")
    loc = eb.ln_locator
    assert_bound(f"ln y ({tag})", yo, r["y"], r["y_mag"], locate=loc)
    assert_bound(f"ln mean ({tag})", mo, r["mean"], r["mean_tol"])
    assert_bound(f"ln rstd ({tag})", ro, r["rstd"], r["rstd"] * r["rstd_rel_tol"])
    # the backward takes the exact statistics (rounded to fp32), so that dx is checked against the exact gradient
    mean32, rstd32 = r["mean"].float(), r["rstd"].float()
    dx = Guarded(tuple(x_in.shape), torch.bfloat16)
    dg, db, cs = Guarded((C,), torch.float32), Guarded((C,), torch.float32), Guarded((C,), torch.float32)
    bases = [torch.randn(C, generator=torch.Generator().manual_seed(20 + i)).cuda() for i in range(3)]
    accs = [(dg, bases[0]), (db, bases[1])] + ([(cs, bases[2])] if with_cs else [])

    def bwd():
        with ops._launch("layernorm_bwd", 0.0, x_in):
            _lib.check(lib.stswin_layernorm_bwd(dy.data_ptr(), x_in.data_ptr(), mean32.data_ptr(), rstd32.data_ptr(),
                                                gam.data_ptr(), dres.data_ptr() if dres is not None else None, dx.view.data_ptr(),
                                                dg.view.data_ptr(), db.view.data_ptr(), cs.view.data_ptr() if with_cs else None,
                                                M, C, pm, H, W, C0, s), "ln bwd")
    dxo = run_twice(bwd, [dx], accs, what=f"layernorm_bwd {tag}")[0]
    dx_rows = eb.pm_gather(dxo, H, W) if pm else dxo
    assert_bound(f"ln dx ({tag})", dx_rows, r["dx"], r["dx_mag"], locate=loc)
    fl = eb.U_F32 * 2
    assert_bound(f"ln dgamma ({tag})", dg.view, bases[0].double() + r["dgamma"], r["dgamma_mag"] + fl * bases[0].double().abs(), locate=loc)
    assert_bound(f"ln dbeta ({tag})", db.view, bases[1].double() + r["dbeta"], r["dbeta_mag"] + fl * bases[1].double().abs(), locate=loc)
    if with_cs:
        ref, mag = eb.colsum(dx_rows, bases[2], chain=eb.ln_chain(M, _sms()))
        assert_bound(f"ln dx_colsum ({tag})", cs.view, ref, mag, locate=loc)


@pytest.mark.parametrize("C,M,with_cs,with_res", LN_CASES, ids=lambda v: str(v))
def test_layernorm_bounds(C, M, with_cs, with_res):
    x = _ln_x(M, C, 1)
    _ln_run(f"M {M} C {C} colsum {with_cs} dres {with_res}", x, x, C, None, with_cs, with_res)


@pytest.mark.parametrize("BT,H,W,C0", [(4, 16, 24, 128), (3, 8, 12, 64), (2, 16, 20, 512)])
@pytest.mark.parametrize("with_cs", [False, True])
def test_layernorm_patch_merging_bounds(BT, H, W, C0, with_cs):
    x = _ln_x(BT * H * W, C0, 7).reshape(BT, H * W, C0)
    _ln_run(f"PM BT {BT} {H}x{W} C {C0} colsum {with_cs}", x, eb.pm_gather(x, H, W), 4 * C0, (H, W), with_cs, False)
