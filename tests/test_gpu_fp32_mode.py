"""GPU: the fp32-accurate mode (BASELINE.json north_star: <= 1e-3 relative error against the reference's fp32 run,
exact arg-max labels) -- split-bf16 tcgen05 GEMMs, fp32 SIMT window attention, fp32 LayerNorm -- against the
reference's goldens and the CPU oracle.  Tolerance 1e-3 (stated bar); inputs are NOT rounded to bf16 here."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _g(name):
    return np.load(os.path.join(GOLDEN, name))


def _load(module, params):
    module.load_state_dict(params, strict=True)
    module = module.cuda()
    module.precision = "fp32"
    return module


def test_split_gemm_is_fp32_accurate():
    from stswincl_b200 import ops32
    gen = torch.Generator().manual_seed(1)
    x, w, b = torch.randn(300, 520, generator=gen), torch.randn(136, 520, generator=gen), torch.randn(136, generator=gen)
    ref = x.double() @ w.double().t() + b.double()
    y = ops32.linear(x.cuda(), w.cuda(), b.cuda())
    assert rel_err(y.cpu(), ref) < 5e-5
    dy = torch.randn(300, 136, generator=gen)
    assert rel_err(ops32.linear_dgrad(dy.cuda(), w.cuda()).cpu(), dy.double() @ w.double()) < 5e-5
    assert rel_err(ops32.linear_wgrad(dy.cuda(), x.cuda()).cpu(), dy.double().t() @ x.double()) < 5e-5
    u = torch.randn(300, 136, generator=gen)
    ref = torch.nn.functional.gelu(u.double()) @ torch.randn(64, 136, generator=torch.Generator().manual_seed(2)).double().t()
    w2 = torch.randn(64, 136, generator=torch.Generator().manual_seed(2))
    assert rel_err(ops32.linear(u.cuda(), w2.cuda(), gelu_input=True).cpu(), ref) < 5e-5


BLOCK_CASES = [("b0", 128, (16, 24), 2, 8, 0, 2, 1), ("b1", 128, (16, 24), 2, 8, 4, 2, 1),
               ("b2", 256, (8, 12), 4, 4, 2, 2, 2), ("b3", 128, (16, 24), 2, 8, 4, 1, 1)]
BLOCK_GRADS = ["attn.relative_position_bias_table", "attn.qkv.bias", "attn.proj.bias", "norm1.weight", "norm1.bias",
               "norm2.weight", "norm2.bias", "mlp.fc1.bias", "mlp.fc2.bias"]


@pytest.mark.parametrize("case", BLOCK_CASES, ids=lambda c: c[0])
def test_block_vs_reference_golden_fp32(case):
    """SwinTransformerBlock forward + backward against the goldens written from the reference's fp32 run."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, (H, W), heads, ws, shift, T, B = case
    g = _g("swin_block.npz")
    params = so.make_block_params(dim, (H, W), heads, ws, shift, seed=31)
    m = _load(swin.SwinTransformerBlock(dim, (H, W), heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(41, B, T, H * W, dim).cuda().requires_grad_(True)
    w = (so.make_features(42, B, T, H * W, dim) - 0.4).cuda()
    y = m(x)
    assert y.dtype == torch.float32
    (y * w).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), g[f"{tag}_y"]) < TOL
    assert rel_err(x.grad.cpu(), g[f"{tag}_dx"]) < TOL
    sd = dict(m.named_parameters())
    for n in BLOCK_GRADS:
        assert rel_err(sd[n].grad.cpu(), g[f"{tag}_d_{n}"]) < TOL, n
    for n in ["attn.qkv.weight", "attn.proj.weight", "mlp.fc1.weight", "mlp.fc2.weight"]:
        assert rel_err(sd[n].grad.cpu()[::23], g[f"{tag}_d_{n}_rows"]) < TOL, n


def test_layer_vs_reference_golden_fp32():
    from oracle import make_goldens as mg, swin_oracle as so
    from stswincl_b200 import swin
    c = mg.LAYER_CASE
    g = _g("swin_layer.npz")
    H, W = c["res"]
    params = so.make_layer_params(c["dim"], c["res"], c["heads"], c["seed"])
    m = _load(swin.SwinTransformerLayerv5(dim=c["dim"], input_resolution=c["res"], num_heads=c["heads"]), params)
    x = so.make_features(61, c["B"], 4, c["dim"], H, W).cuda().requires_grad_(True)
    w1 = (so.make_features(62, c["B"], 4, c["dim"], H, W) - 0.4).cuda()
    w2 = (so.make_features(63, c["B"], 4, 2 * c["dim"], H // 2, W // 2) - 0.4).cuda()
    y1, y2 = m(x)
    ((y1 * w1).sum() + (y2 * w2).sum()).backward()
    torch.cuda.synchronize()
    assert rel_err(y1.cpu(), g["y1"]) < TOL and rel_err(y2.cpu(), g["y2"]) < TOL
    assert rel_err(x.grad.cpu(), g["dx"]) < TOL
    sd = dict(m.named_parameters())
    for n in ["layers.0.0.attn.relative_position_bias_table", "layers.1.1.attn.relative_position_bias_table",
              "layers.4.1.attn.relative_position_bias_table", "layers.2.1.norm1.weight", "layers.5.0.mlp.fc2.bias",
              "downsample.norm.weight", "downsample.norm.bias"]:
        assert rel_err(sd[n].grad.cpu(), g[f"d_{n}"]) < TOL, n
    assert rel_err(sd["downsample.reduction.weight"].grad.cpu()[::29], g["d_downsample.reduction.weight_rows"]) < TOL
    assert rel_err(sd["layers.1.0.attn.qkv.weight"].grad.cpu()[::29], g["d_layers.1.0.attn.qkv.weight_rows"]) < TOL


@pytest.mark.parametrize("case", [("S1_shifted", 512, (64, 80), 4, 8, 4), ("S2_shifted", 1024, (32, 40), 4, 4, 2),
                                  ("w7_general", 256, (28, 42), 4, 7, 3)], ids=lambda c: c[0])
def test_real_geometry_block_fp32_vs_oracle(case):
    """The shipped geometries (and a 7x7 / shift 3 window) at 1e-3: output, input gradient, all 13 parameter gradients."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, res, heads, ws, shift = case
    L = res[0] * res[1]
    params = so.make_block_params(dim, res, heads, ws, shift, seed=91)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(92, 1, 2, L, dim)
    w = so.make_features(93, 1, 2, L, dim) - 0.4
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and k != "attn_mask" else v) for k, v in params.items()}
    xr = x.clone().requires_grad_(True)
    ref = so.swin_block(xr, leaf, res, heads, ws, shift)
    (ref * w).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    (y * w.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL
    assert rel_err(xg.grad.cpu(), xr.grad) < TOL
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), leaf[n].grad) < TOL, n


def test_standalone_window_attention_with_dense_mask_fp32():
    """WindowAttention.forward(x, mask) (swin_512.py:109-141) on its own, dense [nW, N, N] mask, fp32 mode."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, ws, heads, nW = 128, 4, 4, 3
    params = so.make_attention_params(dim, ws, heads, seed=5)
    m = _load(swin.WindowAttention(dim, (ws, ws), heads), params)
    gen = torch.Generator().manual_seed(6)
    x = torch.randn(2 * nW, 2, ws * ws, dim, generator=gen)
    mask = torch.where(torch.rand(nW, ws * ws, ws * ws, generator=gen) < 0.2, torch.tensor(-100.0), torch.tensor(0.0))
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in params.items()}
    xr = x.clone().requires_grad_(True)
    ref = so.window_attention(xr, leaf, ws, heads, mask=mask)
    wgt = torch.randn(x.shape, generator=gen)
    (ref * wgt).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg, mask.cuda())
    (y * wgt.cuda()).sum().backward()
    assert rel_err(y.cpu(), ref) < TOL and rel_err(xg.grad.cpu(), xr.grad) < TOL
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), leaf[n].grad) < TOL, n


def test_standalone_mlp_fp32_vs_oracle():
    """Mlp.forward (swin_512.py:17-23) on its own in the fp32-accurate mode, forward + backward, against the CPU oracle."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    gen = torch.Generator().manual_seed(3)
    params = {"fc1.weight": torch.randn(512, 128, generator=gen) * 128 ** -0.5, "fc1.bias": 0.5 * torch.randn(512, generator=gen),
              "fc2.weight": torch.randn(128, 512, generator=gen) * 512 ** -0.5, "fc2.bias": 0.5 * torch.randn(128, generator=gen)}
    m = _load(swin.Mlp(128, 512), params)
    x = torch.randn(2, 50, 128, generator=gen)
    wgt = torch.randn(2, 50, 128, generator=gen)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    xr = x.clone().requires_grad_(True)
    ref = so.mlp(xr, leaf)
    (ref * wgt).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    assert y.dtype == torch.float32 and y.shape == ref.shape
    (y * wgt.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL and rel_err(xg.grad.cpu(), xr.grad) < TOL
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), leaf[n].grad) < TOL, n


def test_precision_auto_follows_the_input_dtype():
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads, ws, shift = 128, (16, 24), 2, 8, 4
    params = so.make_block_params(dim, res, heads, ws, shift, seed=3)
    m = swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift)
    m.load_state_dict(params, strict=True)
    m = m.cuda()
    x = so.make_features(4, 1, 2, res[0] * res[1], dim)
    ref = so.swin_block(x, params, res, heads, ws, shift)
    old = swin.set_precision("auto")
    try:
        with torch.no_grad():
            y32 = m(x.cuda())
            y16 = m(x.cuda().to(torch.bfloat16))
            with torch.autocast("cuda", dtype=torch.float16):
                yac = m(x.cuda())
    finally:
        swin.set_precision(old)
    assert rel_err(y32.cpu(), ref) < TOL                      # fp32 input outside autocast: the accurate path
    assert 1e-3 < rel_err(y16.float().cpu(), ref) < 2e-2      # bf16 input: the bf16 path
    assert 1e-3 < rel_err(yac.float().cpu(), ref) < 2e-2      # under autocast: the bf16 path


def test_full_model_fp32_mode_exact_argmax():
    """TswinPlus with the head swapped, head in fp32 mode: logits within 1e-3 of the reference's fp32 run and the
    arg-max label map EXACTLY equal (north_star: exact match of arg-max segmentation labels on fp32 runs)."""
    import json
    from oracle import tswin_oracle as to
    from stswincl_b200 import swin
    g = _g("tswinplus.npz")
    head = swin.SwinTransformerLayerv5()
    head.precision = "fp32"
    model = to.TswinPlus(12, head)
    model.load_state_dict(to.synth_state_dict(model.state_dict(), 5), strict=True)
    model = model.cuda().eval()
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        torch.backends.cuda.matmul.allow_tf32 = False
        logits = model(to.make_clip(6).cuda())
    scale = float(g["logit_absmax"])
    err = float(np.abs(logits[0, :, ::8, ::8].float().cpu().numpy() - g["logits_sub"]).max()) / scale
    assert err < TOL, err
    am = logits.argmax(1)[0].cpu().numpy()
    assert np.array_equal(am, g["argmax"]), int((am != g["argmax"]).sum())


@pytest.mark.parametrize("idx", range(5))
def test_regression_loss_fp32_vs_reference_golden(idx):
    """regression_loss (PixPro_swin_v5.py:71-129) with precision='fp32' against the goldens written from the reference's
    fp32 run: loss value and dq at 1e-3 (incl. the absent-class and single-class key-set cases)."""
    from oracle import make_goldens as mg
    from stswincl_b200 import contrast
    case = mg.LOSS_CASES[idx]
    tag, N, C, H, W, K, special = case
    g = _g("loss_cases.npz")
    labels, emb = mg.loss_case_inputs(*case)
    q = emb[0].cuda().requires_grad_(True)
    loss = contrast.regression_loss(q, *[e.cuda() for e in emb[1:]], *[l.cuda() for l in labels], K, precision="fp32")
    loss.backward()
    torch.cuda.synchronize()
    ref = float(g[f"{tag}_loss"])
    assert abs(float(loss) - ref) < TOL * abs(ref)
    assert rel_err(q.grad.cpu(), g[f"{tag}_dq"]) < TOL


@pytest.mark.parametrize("N,C,H,W,K,coarse", [(2, 256, 32, 56, 12, (4, 7)), (1, 64, 28, 28, 26, (28, 28))])
def test_symmetric_tail_fp32_fused_normalize_vs_oracle(N, C, H, W, K, coarse):
    """The fused symmetric step (ConsistencyLoss tail with F.normalize inside) in fp32 mode against the un-rounded fp32
    oracle: loss and both query gradients at 1e-3."""
    from oracle import loss_oracle as lo
    from stswincl_b200 import contrast
    full = lo.make_label_maps(121, 6, N, 8 * H, 8 * W, K, coarse=coarse)
    ds = [torch.nn.functional.interpolate(m, size=[H, W], mode="nearest") for m in full]
    gen = torch.Generator().manual_seed(122)
    raw = [e * (0.5 + 2.0 * torch.rand(N, 1, H, W, generator=gen)) for e in lo.make_embeddings(123, ds + ds[:2], C, K)]
    pred = [raw[6].clone().requires_grad_(True), raw[7].clone().requires_grad_(True)]
    nrm = lo.l2_normalize
    ref = lo.consistency_tail(nrm(pred[0]), nrm(pred[1]), nrm(raw[0]), nrm(raw[1]), [nrm(r) for r in raw[2:6]], full[0], full[1], full[2:], K)
    ref.backward()
    c = lambda t: t.cuda()
    p1, p2 = c(raw[6]).requires_grad_(True), c(raw[7]).requires_grad_(True)
    loss = contrast.consistency_loss_tail(p1, p2, *[c(r) for r in raw[:6]], *[c(m) for m in full], K, normalize=True, precision="fp32")
    loss.backward()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref)) < TOL * abs(float(ref))
    assert rel_err(p1.grad.cpu(), pred[0].grad) < TOL
    assert rel_err(p2.grad.cpu(), pred[1].grad) < TOL
