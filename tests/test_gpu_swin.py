"""GPU: the drop-in Swin modules against (a) the reference's own outputs stored in tests/golden
(produced by oracle/make_goldens.py from the unmodified reference) and (b) the CPU oracle.
Tolerance: 2e-2 relative error for the bf16 path (BASELINE north_star)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err, rel_l2

pytestmark = pytest.mark.gpu
TOL = 2e-2


def _g(name):
    return np.load(os.path.join(GOLDEN, name))


def _load(module, params):
    missing, unexpected = module.load_state_dict(params, strict=True)
    assert not missing and not unexpected
    return module.cuda()


@pytest.mark.parametrize("case", [("a0", 128, 4, 2, 2, (8, 12), 2, 2), ("a1", 128, 4, 2, 1, (8, 12), 0, 2),
                                  ("a2", 256, 8, 2, 2, (16, 24), 4, 1)], ids=lambda c: c[0])
def test_attention_module_vs_reference_golden(case):
    """WindowAttention.forward semantics (windows in, windows out) reproduced by moving the
    golden's window-ordered tokens to natural order, running the fused path with the block's
    geometry, and moving the result back."""
    from oracle import index_oracle as ix, swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, ws, heads, T, (H, W), shift, B = case
    g = _g("swin_attention.npz")
    nW, N = (H // ws) * (W // ws), ws * ws
    params = so.make_attention_params(dim, ws, heads, seed=11)
    m = _load(swin.WindowAttention(dim, (ws, ws), heads), params)
    x_win = so.make_features(21, B * nW, T, N, dim) - 0.4
    w_win = so.make_features(22, B * nW, T, N, dim) - 0.4
    gidx = torch.from_numpy(ix.window_gather_index(H, W, ws, shift)).reshape(-1)

    def to_natural(t):     # [B*nW, T, N, C] -> [B, T, H*W, C]
        t = t.reshape(B, nW, T, N, dim).permute(0, 2, 1, 3, 4).reshape(B, T, nW * N, dim)
        out = torch.empty_like(t)
        out[:, :, gidx] = t
        return out

    def to_windows(t):     # inverse
        return t[:, :, gidx].reshape(B, T, nW, N, dim).permute(0, 2, 1, 3, 4).reshape(B * nW, T, N, dim)

    x = to_natural(x_win).to(torch.bfloat16).cuda().requires_grad_(True)
    geom = (H, W, heads, ws, shift, 0.0)
    y = swin._AttentionFn.apply(x, m.relative_position_bias_table, m.qkv.weight, m.qkv.bias, m.proj.weight, m.proj.bias, geom)
    (y.float() * to_natural(w_win).cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(to_windows(y.float().cpu()), g[f"{tag}_y"]) < TOL
    assert rel_err(to_windows(x.grad.float().cpu()), g[f"{tag}_dx"]) < TOL
    assert rel_err(m.relative_position_bias_table.grad.cpu(), g[f"{tag}_d_relative_position_bias_table"]) < TOL
    assert rel_err(m.qkv.bias.grad.cpu(), g[f"{tag}_d_qkv.bias"]) < TOL
    assert rel_err(m.proj.bias.grad.cpu(), g[f"{tag}_d_proj.bias"]) < TOL
    assert rel_err(m.qkv.weight.grad.cpu()[::17], g[f"{tag}_d_qkv.weight_rows"]) < TOL
    assert rel_err(m.proj.weight.grad.cpu()[::17], g[f"{tag}_d_proj.weight_rows"]) < TOL


def test_attention_module_standalone_unmasked():
    """Stand-alone WindowAttention(x_windows, mask=None) == oracle.window_attention."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, ws, heads, T, Bw = 128, 4, 2, 2, 12
    params = so.make_attention_params(dim, ws, heads, seed=11)
    m = _load(swin.WindowAttention(dim, (ws, ws), heads), params)
    x = so.make_features(21, Bw, T, ws * ws, dim) - 0.4
    ref = so.window_attention(x.to(torch.bfloat16).float(), params, ws, heads, None)
    y = m(x.cuda())
    assert y.dtype == torch.float32
    assert rel_err(y.cpu(), ref) < TOL


@pytest.mark.parametrize("case", [("a0", 128, 4, 2, 2, (8, 12), 2, 2), ("a2", 256, 8, 2, 2, (16, 24), 4, 1)], ids=lambda c: c[0])
def test_attention_module_with_dense_mask_vs_reference_golden(case):
    """WindowAttention.forward(x_windows, mask=attn_mask) called exactly like the reference's block calls it
    (swin_512.py:221): windows in, windows out, the dense {0,-100} mask tensor as an argument."""
    from oracle import index_oracle as ix, swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, ws, heads, T, (H, W), shift, B = case
    g = _g("swin_attention.npz")
    nW, N = (H // ws) * (W // ws), ws * ws
    m = _load(swin.WindowAttention(dim, (ws, ws), heads), so.make_attention_params(dim, ws, heads, seed=11))
    x = (so.make_features(21, B * nW, T, N, dim) - 0.4).cuda().requires_grad_(True)
    w = (so.make_features(22, B * nW, T, N, dim) - 0.4).cuda()
    mask = torch.from_numpy(ix.shift_attn_mask(H, W, ws, shift)).cuda()
    y = m(x, mask=mask)
    (y * w).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), g[f"{tag}_y"]) < TOL
    assert rel_err(x.grad.cpu(), g[f"{tag}_dx"]) < TOL
    assert rel_err(m.relative_position_bias_table.grad.cpu(), g[f"{tag}_d_relative_position_bias_table"]) < TOL
    assert rel_err(m.qkv.bias.grad.cpu(), g[f"{tag}_d_qkv.bias"]) < TOL


BLOCK_CASES = [("b0", 128, (16, 24), 2, 8, 0, 2, 1), ("b1", 128, (16, 24), 2, 8, 4, 2, 1),
               ("b2", 256, (8, 12), 4, 4, 2, 2, 2), ("b3", 128, (16, 24), 2, 8, 4, 1, 1)]


@pytest.mark.parametrize("case", BLOCK_CASES, ids=lambda c: c[0])
def test_block_vs_reference_golden(case):
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, (H, W), heads, ws, shift, T, B = case
    g = _g("swin_block.npz")
    params = so.make_block_params(dim, (H, W), heads, ws, shift, seed=31)
    m = _load(swin.SwinTransformerBlock(dim, (H, W), heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(41, B, T, H * W, dim).cuda().requires_grad_(True)
    w = (so.make_features(42, B, T, H * W, dim) - 0.4).cuda()
    y = m(x)
    assert y.dtype == torch.float32 and y.shape == x.shape
    (y * w).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), g[f"{tag}_y"]) < TOL
    assert rel_err(x.grad.cpu(), g[f"{tag}_dx"]) < TOL
    sd = dict(m.named_parameters())
    for n in ["attn.relative_position_bias_table", "attn.qkv.bias", "attn.proj.bias", "norm1.weight", "norm1.bias",
              "norm2.weight", "norm2.bias", "mlp.fc1.bias", "mlp.fc2.bias"]:
        assert rel_err(sd[n].grad.cpu(), g[f"{tag}_d_{n}"]) < TOL, n
    for n in ["attn.qkv.weight", "attn.proj.weight", "mlp.fc1.weight", "mlp.fc2.weight"]:
        assert rel_err(sd[n].grad.cpu()[::23], g[f"{tag}_d_{n}_rows"]) < TOL, n


def test_layer_vs_reference_golden():
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
    assert y1.shape == (c["B"], 4, c["dim"], H, W) and y2.shape == (c["B"], 4, 2 * c["dim"], H // 2, W // 2)
    ((y1 * w1).sum() + (y2 * w2).sum()).backward()
    torch.cuda.synchronize()
    assert rel_err(y1.cpu(), g["y1"]) < TOL
    assert rel_err(y2.cpu(), g["y2"]) < TOL
    assert rel_err(x.grad.cpu(), g["dx"]) < 2 * TOL          # 12 blocks deep in bf16
    sd = dict(m.named_parameters())
    for n in ["layers.0.0.attn.relative_position_bias_table", "layers.1.1.attn.relative_position_bias_table",
              "layers.2.1.norm1.weight", "layers.5.0.mlp.fc2.bias", "downsample.norm.weight", "downsample.norm.bias"]:
        assert rel_err(sd[n].grad.cpu(), g[f"d_{n}"]) < 2 * TOL, n
    # layers.4.1 sees ONE pair of 8x12-token frames (6 windows): its bias-table gradient is a heavily
    # cancelling sum over very few windows and is ~5x more sensitive than every other quantity -- the
    # fp32 oracle itself moves by 3.8e-2 when only the block boundaries are rounded to bf16
    # (tools/conditioning_check.py).  The kernel that produces it is held to 2e-2 on this exact
    # geometry in tests/test_gpu_winattn.py.
    n = "layers.4.1.attn.relative_position_bias_table"
    assert rel_err(sd[n].grad.cpu(), g[f"d_{n}"]) < 1e-1, n
    assert rel_err(sd["downsample.reduction.weight"].grad.cpu()[::29], g["d_downsample.reduction.weight_rows"]) < 2 * TOL
    assert rel_err(sd["layers.1.0.attn.qkv.weight"].grad.cpu()[::29], g["d_layers.1.0.attn.qkv.weight_rows"]) < 2 * TOL


def test_full_size_block_vs_oracle():
    """The real stage-1 geometry (C=512, 64x80, ws 8, shift 4, 4 heads), one clip pair."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads, ws, shift = 512, (64, 80), 4, 8, 4
    params = so.make_block_params(dim, res, heads, ws, shift, seed=77)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(78, 1, 2, res[0] * res[1], dim)
    ref = so.swin_block(x.to(torch.bfloat16).float(), params, res, heads, ws, shift)
    y = m(x.cuda())
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL


def test_block_inference_path_matches_training_path():
    """Under no_grad (the six key-encoder passes of the pre-training model, SURVEY N2) the block takes the
    forward-only GELU epilogue and keeps nothing for a backward: same output as the training forward."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads, ws, shift = 512, (32, 40), 4, 8, 4
    params = so.make_block_params(dim, res, heads, ws, shift, seed=83)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(84, 2, 2, res[0] * res[1], dim).cuda()
    y_train = m(x)
    with torch.no_grad():
        y_eval = m(x)
    assert y_train.requires_grad and not y_eval.requires_grad
    assert rel_err(y_eval.float().cpu(), y_train.detach().float().cpu()) < 5e-3
    ref = so.swin_block(x.cpu().to(torch.bfloat16).float(), params, res, heads, ws, shift)
    assert rel_err(y_eval.float().cpu(), ref) < TOL


def test_cadis_shaped_block_vs_oracle():
    """Config 5: CaDIS-shaped crop 512x960 -> 64x120 tokens (SURVEY D7), shifted block, 8 heads."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads, ws, shift = 512, (64, 120), 8, 8, 4
    params = so.make_block_params(dim, res, heads, ws, shift, seed=79)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(80, 1, 2, res[0] * res[1], dim)
    ref = so.swin_block(x.to(torch.bfloat16).float(), params, res, heads, ws, shift)
    y = m(x.cuda())
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL


def test_window7_block_fwd_bwd_vs_oracle():
    """Config 5 corner: 7x7 windows, shift 3, on a 56x84-token crop (98-token windows, unequal rectangles)."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads, ws, shift = 256, (28, 42), 4, 7, 3
    params = so.make_block_params(dim, res, heads, ws, shift, seed=81)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(82, 1, 2, res[0] * res[1], dim)
    w = so.make_features(83, 1, 2, res[0] * res[1], dim) - 0.4
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and k != "attn_mask" else v) for k, v in params.items()}
    xr = x.to(torch.bfloat16).float().requires_grad_(True)
    ref = so.swin_block(xr, leaf, res, heads, ws, shift)
    (ref * w).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    (y * w.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL
    assert rel_err(xg.grad.cpu(), xr.grad) < TOL
    assert rel_err(m.attn.relative_position_bias_table.grad.cpu(), leaf["attn.relative_position_bias_table"].grad) < TOL
    assert rel_err(m.attn.qkv.bias.grad.cpu(), leaf["attn.qkv.bias"].grad) < TOL


def test_cpu_tensor_raises():
    from stswincl_b200 import swin
    from stswincl_b200._lib import StswinError
    m = swin.SwinTransformerBlock(128, (16, 24), 2)
    with pytest.raises(StswinError):
        m(torch.zeros(1, 2, 384, 128))


def test_standalone_mlp_forward_backward():
    """Mlp.forward (swin_512.py:17-23) called on its own, against fp32 torch."""
    from stswincl_b200 import swin
    torch.manual_seed(3)
    m = swin.Mlp(128, 512).cuda()
    x = torch.randn(2, 50, 128).cuda()
    xr = x.clone().requires_grad_(True)
    ref = torch.nn.functional.linear(torch.nn.functional.gelu(torch.nn.functional.linear(xr.to(torch.bfloat16).float(), m.fc1.weight, m.fc1.bias)),
                                     m.fc2.weight, m.fc2.bias)
    w = torch.randn_like(ref)
    (ref * w).sum().backward()
    ref_grads = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    xg = x.clone().requires_grad_(True)
    y = m(xg)
    assert y.dtype == torch.float32 and y.shape == ref.shape
    (y * w).sum().backward()
    assert rel_err(y, ref) < 2e-2 and rel_err(xg.grad, xr.grad) < 2e-2
    for p, g in zip(m.parameters(), ref_grads):
        assert rel_err(p.grad, g) < 2e-2


@pytest.mark.parametrize("precision,tol", [("bf16", TOL), ("fp32", 1e-3)])
def test_standalone_patch_merging_vs_oracle(precision, tol):
    """PatchMerging.forward (swin_512.py:255-277) called on its own, forward + backward, against the CPU oracle in both
    precisions (the bf16 mode's input is rounded to bf16 for the oracle too)."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, (H, W) = 128, (16, 24)
    gen = torch.Generator().manual_seed(7)
    params = {"reduction.weight": torch.randn(2 * dim, 4 * dim, generator=gen) * (4 * dim) ** -0.5,
              "norm.weight": 1.0 + 0.2 * torch.randn(4 * dim, generator=gen), "norm.bias": 0.2 * torch.randn(4 * dim, generator=gen)}
    m = _load(swin.PatchMerging((H, W), dim), params)
    m.precision = precision
    x = so.make_features(8, 2, 2, H * W, dim)
    if precision == "bf16":
        x = x.to(torch.bfloat16).float()
    wgt = torch.randn(2, 2, H * W // 4, 2 * dim, generator=gen)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    xr = x.clone().requires_grad_(True)
    ref = so.patch_merging(xr, leaf, (H, W))
    (ref * wgt).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    assert y.dtype == torch.float32 and y.shape == ref.shape
    (y * wgt.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < tol and rel_err(xg.grad.cpu(), xr.grad) < tol
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), leaf[n].grad) < tol, n


def test_layer_dtype_contract_fp16_and_autocast():
    """The reference's layer returns its input dtype (:326); under amp.autocast its last op (LayerNorm) returns fp32."""
    from stswincl_b200 import swin
    torch.manual_seed(4)
    layer = swin.SwinTransformerLayerv5(dim=128, input_resolution=(16, 24), num_heads=2).cuda()
    x = torch.relu(torch.randn(1, 4, 128, 16, 24)).cuda()
    with torch.no_grad():
        a1, a2 = layer(x)
        h1, h2 = layer(x.half())
        with torch.autocast("cuda", dtype=torch.float16):
            c1, c2 = layer(x.half())
    assert a1.dtype == torch.float32 and h1.dtype == torch.float16 and h2.dtype == torch.float16 and c1.dtype == torch.float32
    assert rel_err(h1.float(), a1) < 2e-2 and rel_err(c2, a2) < 2e-2


REAL_GEOMETRIES = [("S1_unshifted", 512, (64, 80), 4, 8, 0), ("S1_shifted", 512, (64, 80), 4, 8, 4),
                   ("S2_unshifted", 1024, (32, 40), 4, 4, 0), ("S2_shifted", 1024, (32, 40), 4, 4, 2)]
BLOCK_GRADS = ["attn.relative_position_bias_table", "attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias",
               "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias",
               "mlp.fc2.weight", "mlp.fc2.bias"]


@pytest.mark.parametrize("case", REAL_GEOMETRIES, ids=lambda c: c[0])
def test_real_geometry_block_forward_backward_vs_oracle(case):
    """SwinTransformerBlock forward AND backward at the shipped geometries (stage 1: C 512, 64x80 tokens, ws 8,
    shift 0 / 4; stage 2: C 1024, 32x40, ws 4, shift 0 / 2; 4 heads, B = 2 frame pairs) against the CPU oracle
    (swin_512.py:196-237): output, input gradient and all 13 parameter gradients at the bf16 bar, 2e-2."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    tag, dim, res, heads, ws, shift = case
    L = res[0] * res[1]
    params = so.make_block_params(dim, res, heads, ws, shift, seed=91)
    m = _load(swin.SwinTransformerBlock(dim, res, heads, window_size=ws, shift_size=shift), params)
    x = so.make_features(92, 2, 2, L, dim)
    # the upstream gradient is made bf16-representable: half of relu(N) - 0.4 is the single value -0.4, whose bf16
    # rounding error (+1e-3 relative, the same sign for every element) would otherwise add up over the 20480 rows into
    # a 1.6e-2 bias of the norm1 gradients that no kernel could avoid
    w = (so.make_features(93, 2, 2, L, dim) - 0.4).to(torch.bfloat16).float()
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and k != "attn_mask" else v) for k, v in params.items()}
    xr = x.to(torch.bfloat16).float().requires_grad_(True)
    ref = so.swin_block(xr, leaf, res, heads, ws, shift)
    (ref * w).sum().backward()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    (y * w.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_err(y.cpu(), ref) < TOL and rel_l2(y.cpu(), ref) < TOL
    assert rel_err(xg.grad.cpu(), xr.grad) < TOL and rel_l2(xg.grad.cpu(), xr.grad) < TOL
    sd = dict(m.named_parameters())
    for n in BLOCK_GRADS:
        assert rel_err(sd[n].grad.cpu(), leaf[n].grad) < TOL, n
        assert rel_l2(sd[n].grad.cpu(), leaf[n].grad) < TOL, n         # norm-wise too: many small outliers would show here


def test_full_size_layer_forward_backward_vs_oracle():
    """The whole SwinTransformerLayerv5 at the bench geometry (dim 512, 64x80 tokens, 4 heads, 12 blocks + PatchMerging;
    swin_512.py:280-327), one clip, forward and backward against the CPU oracle.  Outputs at 2e-2; the gradients have
    passed 12 blocks of bf16 storage: 4e-2 (input gradient, first / last blocks' parameters)."""
    from oracle import swin_oracle as so
    from stswincl_b200 import swin
    dim, res, heads = 512, (64, 80), 4
    params = so.make_layer_params(dim, res, heads, seed=95)
    m = _load(swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads), params)
    x = so.make_features(96, 1, 4, dim, res[0], res[1])
    w1 = (so.make_features(97, 1, 4, dim, res[0], res[1]) - 0.4).to(torch.bfloat16).float()       # bf16-representable upstream gradients
    w2 = (so.make_features(98, 1, 4, 2 * dim, res[0] // 2, res[1] // 2) - 0.4).to(torch.bfloat16).float()
    names = ["layers.0.0.attn.relative_position_bias_table", "layers.0.0.attn.qkv.weight", "layers.0.1.mlp.fc1.bias",
             "layers.2.1.norm1.weight", "layers.3.0.attn.qkv.bias", "layers.5.1.mlp.fc2.weight", "layers.5.1.norm1.bias",
             "downsample.norm.weight", "downsample.reduction.weight"]
    leaf = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in params.items()}
    xr = x.to(torch.bfloat16).float().requires_grad_(True)
    r1, r2 = so.swin_layer_v5(xr, leaf, dim, res, heads)
    ((r1 * w1).sum() + (r2 * w2).sum()).backward()
    xg = x.cuda().requires_grad_(True)
    y1, y2 = m(xg)
    ((y1 * w1.cuda()).sum() + (y2 * w2.cuda()).sum()).backward()
    torch.cuda.synchronize()
    assert rel_err(y1.cpu(), r1) < TOL and rel_err(y2.cpu(), r2) < TOL
    assert rel_err(xg.grad.cpu(), xr.grad) < 2 * TOL
    sd = dict(m.named_parameters())
    for n in names:
        assert rel_err(sd[n].grad.cpu(), leaf[n].grad) < 2 * TOL, n


def _swapped_model():
    """The reference's full segmentation model with ``model.swin`` replaced by the product (INTEGRATION.md): the caller
    side (ResNet-18 OS8, ASPP, projections, classifier -- plain torch on the GPU) is the restatement pinned against the
    reference by tests/test_oracle_golden.py; weights are the synthetic state_dict of the golden."""
    import json
    from oracle import tswin_oracle as to
    from stswincl_b200 import swin
    g = np.load(os.path.join(GOLDEN, "tswinplus.npz"))
    model = to.TswinPlus(12, swin.SwinTransformerLayerv5())
    assert {k: list(v.shape) for k, v in model.state_dict().items()} == json.loads(str(g["keys"]))
    model.load_state_dict(to.synth_state_dict(model.state_dict(), 5), strict=True)
    return model.cuda(), g, to


def test_full_model_with_swapped_head_logits_and_argmax():
    """TswinPlus (seg18/net/Ours/base18.py:52-108, head call at :94) with the head swapped, eval mode, one 4-frame
    512x640 clip: logits within 2e-2 of the reference's fp32 run, arg-max labels equal wherever the reference's top-2
    margin exceeds the bf16 noise floor."""
    model, g, to = _swapped_model()
    model.eval()
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        torch.backends.cuda.matmul.allow_tf32 = False
        logits = model(to.make_clip(6).cuda())
    scale = float(g["logit_absmax"])
    err = float(np.abs(logits[0, :, ::8, ::8].float().cpu().numpy() - g["logits_sub"]).max()) / scale
    assert err < TOL, err
    am = logits.argmax(1)[0].cpu().numpy()
    margin = g["margin"].astype(np.float32)
    decided = margin > 2 * TOL * scale
    assert np.array_equal(am[decided], g["argmax"][decided])
    assert (am == g["argmax"]).mean() > 0.97


def test_full_model_three_step_loss_trajectory():
    """Three SGD steps (lr 2e-4, momentum 0.9, cross-entropy, train mode with the image-pool BatchNorm in eval, SURVEY D8)
    of the swapped model follow the reference's loss trajectory within 2e-2 (see oracle/make_goldens_tswin.py for why
    not Adam 1e-4: that trajectory is chaotic on this synthetic model)."""
    model, g, to = _swapped_model()
    model.train()
    model.aspp.bn_conv_1x1_2.eval()
    clip = to.make_clip(6).cuda()
    target = to.make_targets(7, 1, 512, 640, 12).cuda()
    opt = torch.optim.SGD(model.parameters(), lr=2e-4, momentum=0.9)
    losses = []
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        for _ in range(3):
            opt.zero_grad()
            loss = torch.nn.functional.cross_entropy(model(clip), target)
            loss.backward()
            opt.step()
            losses.append(float(loss))
    ref = g["losses"]
    assert all(abs(a - b) < TOL * abs(b) for a, b in zip(losses, ref)), (losses, list(ref))
