"""GPU: the training-step kernels (OHEM cross-entropy, LARS-scaled SGD, key-encoder EMA) through the C ABI against the
reference's goldens and the CPU oracle.  fp32 element work: tolerance 2e-5 relative (summation order); the EMA is bit-exact;
bf16 logits: 2e-2 (the bf16 bar of BASELINE.json)."""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err

pytestmark = pytest.mark.gpu
TOL = 2e-5


def _g():
    return np.load(os.path.join(GOLDEN, "trainaux_cases.npz"))


def _cases():
    from oracle import trainaux_oracle as ta
    return ta.OHEM_CASES


@pytest.mark.parametrize("idx", range(9))
def test_ohem_vs_reference_golden(idx):
    from oracle import trainaux_oracle as ta
    from stswincl_b200.losses import OhemCELoss2D
    tag, B, K, H, W, _, margin, ign = ta.OHEM_CASES[idx]
    g = _g()
    n_min = int(g[f"ohem_{tag}_nmin"])
    logits, labels = ta.make_ohem_case(ta.ohem_seed(idx), B, K, H, W, margin, ign)
    x = logits.cuda().requires_grad_(True)
    loss = OhemCELoss2D(n_min)(x, labels.cuda())
    (loss * 1.0).backward()
    torch.cuda.synchronize()
    ref = float(g[f"ohem_{tag}_loss"])
    assert abs(float(loss) - ref) < TOL * abs(ref), (float(loss), ref)
    assert rel_err(x.grad.cpu(), g[f"ohem_{tag}_dlogits"]) < TOL


@pytest.mark.parametrize("margin,n_div", [(0.0, 16), (12.0, 16), (4.0, 16), (12.0, 3)])
def test_ohem_full_size_vs_oracle(margin, n_div):
    """EndoVis18 shape of train_swin.py:123 (batch 2, 12 classes, 512x640, n_min = H*W/16) against the oracle, with an
    upstream gradient different from 1; (12, 3): n_min beyond the labelled hard pixels."""
    from oracle import trainaux_oracle as ta
    from stswincl_b200.losses import OhemCELoss2D
    B, K, H, W = 2, 12, 512, 640
    n_min = H * W // n_div
    logits, labels = ta.make_ohem_case(5, B, K, H, W, margin, 0.05)
    xr = logits.clone().requires_grad_(True)
    ref = ta.ohem_ce(xr, labels, n_min)
    (ref * 0.37).backward()
    x = logits.cuda().requires_grad_(True)
    loss = OhemCELoss2D(n_min)(x, labels.cuda())
    (loss * 0.37).backward()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref)) < TOL * abs(float(ref))
    # pixels whose loss is within rounding of the selection cut may fall on either side of it (the reference's own
    # choice among them depends on its sort): compare the gradient away from the cut, and bound the rest in norm
    px = torch.nn.functional.cross_entropy(logits, labels, ignore_index=-1, reduction="none")
    t = -math.log(ta.OHEM_THRESH)
    kth = float(torch.topk(px.view(-1), n_min + 1).values[n_min])
    cut = t if kth > t else float(torch.topk(px.view(-1), n_min).values[-1])
    away = ((px - cut).abs() > 1e-5 * (1 + cut)).unsqueeze(1)
    got = x.grad.cpu()
    assert float(away.float().mean()) > 0.98
    assert rel_err(got * away, xr.grad * away) < 1e-4
    assert float((got - xr.grad).norm() / xr.grad.norm()) < 2e-2


def test_ohem_bf16_logits_and_ties():
    from oracle import trainaux_oracle as ta
    from stswincl_b200.losses import OhemCELoss2D
    logits, labels = ta.make_ohem_case(9, 2, 12, 32, 40, 12.0, 0.1)
    xb = logits.to(torch.bfloat16)
    xr = xb.float().requires_grad_(True)
    ref = ta.ohem_ce(xr, labels, 200)
    ref.backward()
    x = xb.cuda().requires_grad_(True)
    loss = OhemCELoss2D(200)(x, labels.cuda())
    loss.backward()
    assert x.grad.dtype == torch.bfloat16
    assert abs(float(loss) - float(ref)) < 1e-4 * abs(float(ref))
    assert rel_err(x.grad.float().cpu(), xr.grad) < 2e-2
    # identical logits everywhere: every loss equals the n_min-th value; the value is exact and the gradient weight
    # is shared by the ties (sum of weights = 1)
    K = 4
    flat = torch.zeros(1, K, 8, 8, device="cuda", requires_grad=True)
    lab = torch.zeros(1, 8, 8, dtype=torch.long, device="cuda")
    loss = OhemCELoss2D(16, thresh=0.1)(flat, lab)          # ln 4 = 1.386 < -ln 0.1 = 2.30 -> top-n_min branch
    loss.backward()
    assert abs(float(loss) - math.log(K)) < 1e-6
    assert abs(float(flat.grad[:, 0].sum()) - (1.0 / K - 1.0)) < 1e-5


def test_ohem_errors():
    from stswincl_b200._lib import StswinError
    from stswincl_b200.losses import OhemCELoss2D
    x = torch.zeros(1, 3, 4, 4, device="cuda")
    with pytest.raises(IndexError):
        OhemCELoss2D(16)(x, torch.zeros(1, 4, 4, dtype=torch.long, device="cuda"))
    with pytest.raises(ValueError):
        OhemCELoss2D(4)(x, torch.zeros(1, 4, 5, dtype=torch.long, device="cuda"))
    with pytest.raises(StswinError):
        OhemCELoss2D(4)(x.cpu(), torch.zeros(1, 4, 4, dtype=torch.long))


@pytest.mark.parametrize("run", [("wd", 1e-5, 0.9), ("wd0", 0.0, 0.9), ("nomom", 1e-4, 0.0)])
def test_lars_vs_reference_golden(run):
    from oracle import trainaux_oracle as ta
    from stswincl_b200.optim import LARS, add_weight_decay
    tag, wd, mom = run
    g = _g()
    params = ta.make_param_set(7)

    class Holder(torch.nn.Module):
        def __init__(self):
            super().__init__()
            for k, v in params.items():
                self.register_parameter(k.replace(".", "_"), torch.nn.Parameter(v.clone()))

    model = Holder().cuda()
    opt = LARS(torch.optim.SGD(add_weight_decay(model, wd), lr=0.5, momentum=mom))
    named = dict(model.named_parameters())
    for step in range(3):
        grads = ta.make_grads(20 + step, params)
        for k in params:
            named[k.replace(".", "_")].grad = grads[k].cuda()
        opt.step()
        torch.cuda.synchronize()
        for k in params:
            p = named[k.replace(".", "_")]
            assert rel_err(p.detach().cpu(), g[f"lars_{tag}_s{step}_p_{k}"]) < TOL, (k, step)
            gref = g[f"lars_{tag}_s{step}_g_{k}"]
            assert float((p.grad.cpu().double() - torch.as_tensor(gref).double()).abs().max()) <= TOL * max(1e-30, float(np.abs(gref).max())), (k, step)
            if mom != 0:
                bref = g[f"lars_{tag}_s{step}_b_{k}"]
                b = opt.state[p]["momentum_buffer"].cpu()
                assert float((b.double() - torch.as_tensor(bref).double()).abs().max()) <= TOL * max(1e-30, float(np.abs(bref).max())), (k, step)
    sd = opt.state_dict()                       # same layout as the wrapped torch.optim.SGD
    assert len(sd["param_groups"]) == 2 and sd["param_groups"][0]["ignore"] is True


def test_lars_many_tensors_vs_oracle():
    """More tensors than one launch holds (48), sizes around the 4096-element block size, nesterov momentum."""
    from oracle import trainaux_oracle as ta
    from stswincl_b200.optim import LARS
    g = torch.Generator().manual_seed(3)
    sizes = [1, 3, 4095, 4096, 4097, 8193, 50000] + [17 + 5 * i for i in range(60)]
    ps = [torch.randn(n, 2, generator=g) for n in sizes]
    gs = [torch.randn(n, 2, generator=g) * 0.1 for n in sizes]
    cu = [torch.nn.Parameter(p.cuda()) for p in ps]
    opt = LARS(torch.optim.SGD([{"params": cu, "weight_decay": 1e-3, "ignore": False}], lr=0.1, momentum=0.9, nesterov=True))
    bufs = [None] * len(ps)
    for step in range(2):
        for c, gr in zip(cu, gs):
            c.grad = (gr * (step + 1)).cuda()
        opt.step()
        for i in range(len(ps)):
            ps[i], _, bufs[i] = ta.lars_sgd_step(ps[i], gs[i] * (step + 1), bufs[i], lr=0.1, momentum=0.9, weight_decay=1e-3,
                                                 lars=True, nesterov=True)
    torch.cuda.synchronize()
    for c, p in zip(cu, ps):
        assert rel_err(c.detach().cpu(), p) < TOL


def test_ema_bit_exact_vs_reference_golden():
    from oracle import trainaux_oracle as ta
    from stswincl_b200.optim import momentum_update
    g = _g()
    q, k = ta.make_param_set(31), ta.make_param_set(32)
    qc = [torch.nn.Parameter(v.cuda()) for v in q.values()]
    kc = [torch.nn.Parameter(v.cuda()) for v in k.values()]
    for step in (3, 4):
        momentum_update(qc, kc, ta.cosine_momentum(0.99, step, 40))
    torch.cuda.synchronize()
    for n, t in zip(k.keys(), kc):
        assert np.array_equal(t.detach().cpu().numpy(), g[f"ema_{n.replace('.', '_')}"]), n


def test_ema_large_and_unaligned_bit_exact():
    from stswincl_b200.optim import momentum_update
    g = torch.Generator().manual_seed(11)
    sizes = [(2048, 512), (1536, 512), (513,), (7,), (1, 1), (4097, 3)] + [(33 + i,) for i in range(70)]
    q = [torch.randn(*s, generator=g).cuda() for s in sizes]
    k = [torch.randn(*s, generator=g).cuda() for s in sizes]
    base = torch.randn(1001, generator=g).cuda()
    q.append(base[1:]); k.append(torch.randn(1001, generator=g).cuda()[1:])      # 4-byte aligned views
    m = 0.9937
    want = [kk * m + qq * (1. - m) for kk, qq in zip(k, q)]                       # the reference's eager expression
    momentum_update(q, k, m)
    torch.cuda.synchronize()
    for a, b in zip(k, want):
        assert torch.equal(a, b)


def test_fused_adam_matches_torch_adam_and_keeps_the_bf16_shadow():
    """stswin_adam_step against torch.optim.Adam (the optimiser of seg18/train_swin.py) run on the CPU in fp32: three
    steps, weight decay, odd sizes (unaligned tails), fp32 and bf16 gradients; the bf16 shadow equals bf16(param)."""
    from stswincl_b200 import optim as so
    gen = torch.Generator().manual_seed(5)
    shapes = [(33, 17), (128,), (7,), (64, 96), (1, 5, 3)]
    for wd, gdtype in ((0.0, torch.float32), (1e-2, torch.float32), (0.0, torch.bfloat16)):
        ref = [torch.nn.Parameter(torch.randn(s, generator=gen)) for s in shapes]
        ours = [torch.nn.Parameter(p.detach().clone().cuda()) for p in ref]
        o_ref = torch.optim.Adam(ref, lr=1e-2, betas=(0.9, 0.99), eps=1e-8, weight_decay=wd)
        o_our = so.FusedAdam(ours, lr=1e-2, betas=(0.9, 0.99), eps=1e-8, weight_decay=wd)
        for step in range(3):
            grads = [torch.randn(s, generator=gen) * (0.1 + step) for s in shapes]
            if gdtype == torch.bfloat16:
                grads = [g.to(torch.bfloat16).float() for g in grads]
            for p, g in zip(ref, grads):
                p.grad = g.clone()
            o_ref.step()
            if gdtype == torch.bfloat16:
                o_our.step(grads=[g.to(torch.bfloat16).cuda() for g in grads])
            else:
                for p, g in zip(ours, grads):
                    p.grad = g.cuda()
                o_our.step()
        torch.cuda.synchronize()
        for p, q in zip(ref, ours):
            assert rel_err(q.detach().cpu(), p.detach()) < 1e-5
            assert rel_err(o_our.state[q]["exp_avg_sq"].cpu(), o_ref.state[p]["exp_avg_sq"]) < 1e-5
            if q.dim() >= 2:
                assert torch.equal(so.bf16_weight(q), q.detach().to(torch.bfloat16))       # written by the update kernel
                assert so.bf16_weight(q).data_ptr() == q._stswin_shadow[0].data_ptr()
        with torch.no_grad():                                # someone else writes the parameter: the shadow is refreshed
            ours[0].mul_(2.0)
        assert torch.equal(so.bf16_weight(ours[0]), ours[0].detach().to(torch.bfloat16))


def test_fused_adam_many_tensors_matches_torch_adam():
    """80 tensors in two groups of 60 and 20 (the first takes two launches: 48, then 12), fp32 and bf16 gradients, sizes
    around the 4096-element block size, and a 4-byte-offset view (the scalar path) in each launch of the first group."""
    from stswincl_b200 import optim as so
    gen = torch.Generator().manual_seed(7)
    shapes = [(1,), (3,), (4095,), (4096,), (4097,), (100, 1000)] + [(5 + 11 * i,) for i in range(74)]
    for gdtype in (torch.float32, torch.bfloat16):
        ref = [torch.nn.Parameter(torch.randn(s, generator=gen)) for s in shapes]
        ours = [torch.nn.Parameter(p.detach().clone().cuda()) for p in ref]
        for i in (4, 52):                                                  # misaligned data pointers
            host = torch.empty(ref[i].numel() + 1, device="cuda")
            ours[i] = torch.nn.Parameter(host[1:].copy_(ref[i].detach()))
        split = 60
        o_ref = torch.optim.Adam([dict(params=ref[:split]), dict(params=ref[split:], lr=3e-3)], lr=1e-2, weight_decay=1e-2)
        o_our = so.FusedAdam([dict(params=ours[:split]), dict(params=ours[split:], lr=3e-3)], lr=1e-2, weight_decay=1e-2)
        for step in range(2):
            grads = [(torch.randn(s, generator=gen) * (0.1 + step)).to(gdtype) for s in shapes]
            for p, g in zip(ref, grads):
                p.grad = g.float()
            o_ref.step()
            o_our.step(grads=[g.cuda() for g in grads])
        torch.cuda.synchronize()
        for p, q in zip(ref, ours):
            assert rel_err(q.detach().cpu(), p.detach()) < 1e-5
            assert rel_err(o_our.state[q]["exp_avg"].cpu(), o_ref.state[p]["exp_avg"]) < 1e-5


def test_fused_adam_errors():
    import ctypes
    from stswincl_b200 import _lib, optim
    ps = [torch.zeros(3, device="cuda", requires_grad=True), torch.zeros(5, device="cuda", requires_grad=True)]
    o = optim.FusedAdam([dict(params=ps[:1]), dict(params=ps[1:])], lr=0.1)
    # grads= lists that are short, long, or hold a gradient of another size (in the second group): refused before any
    # group is updated
    for gl in ([torch.ones(3, device="cuda")], [torch.ones(3, device="cuda"), torch.ones(5, device="cuda")] * 2,
               [torch.ones(3, device="cuda"), torch.ones(4, device="cuda")]):
        with pytest.raises(_lib.StswinError, match="gradients"):
            o.step(grads=gl)
    assert all(not torch.any(q) for q in ps) and not o.state
    # a null tensor in the table: refused before the step count advances
    lib = _lib.load()
    p, step = torch.zeros(3, device="cuda"), torch.zeros((), device="cuda")
    ptr, null = (ctypes.c_void_p * 1)(p.data_ptr()), (ctypes.c_void_p * 1)(None)
    n = (ctypes.c_int64 * 1)(3)
    stream = torch.cuda.current_stream().cuda_stream
    assert lib.stswin_adam_step(ptr, null, ptr, ptr, None, n, 1, 0, 0.1, 0.9, 0.99, 1e-8, 0.0, 1.0, step.data_ptr(), stream) != 0
    assert float(step) == 0.0 and not torch.any(p)


def test_launch_counts_match_the_profiler():
    """ops.LAUNCHES (bench.py's gpu_launches) counts every kernel of the multi-tensor calls, over 49 tensors: one more
    than a launch takes."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    from stswincl_b200 import ops, optim
    n = 49

    def params():
        return [torch.nn.Parameter(torch.randn(100 + 7 * i, 3, device="cuda")) for i in range(n)]

    def with_grads(ps):
        for p in ps:
            p.grad = torch.randn_like(p)
        return ps
    adam = optim.FusedAdam(with_grads(params()))
    sgd = optim.FusedSGD(with_grads(params()), lr=0.1, momentum=0.9)
    lars = optim.LARS(torch.optim.SGD(optim.add_weight_decay(torch.nn.ParameterList(with_grads(params() + [
        torch.nn.Parameter(torch.randn(50 + i, device="cuda")) for i in range(n)])), 1e-4), lr=0.1, momentum=0.9))
    assert [len(g["params"]) for g in lars.param_groups] == [n, n]           # an `ignore` group and a LARS group
    q, k = params(), params()
    src = [torch.randn(1000 + i, device="cuda") for i in range(n)]
    dst = [torch.empty(s.numel(), dtype=torch.bfloat16, device="cuda") for s in src]
    calls = {"adam": adam.step, "sgd": sgd.step, "lars": lars.step, "ema": lambda: optim.momentum_update(q, k, 0.99),
             "gather_cast": lambda: ops.gather_cast(dst, src)}
    for name, fn in calls.items():
        fn()                                     # optimizer state and shadows exist before the counted call
        torch.cuda.synchronize()
        n0 = ops.LAUNCHES
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and not e.is_user_annotation and
                   not e.name.startswith(("Memset", "Memcpy"))]
        assert ops.LAUNCHES - n0 == len(kernels), (name, ops.LAUNCHES - n0, kernels)


def test_colsum_and_gather_cast():
    from stswincl_b200 import ops
    gen = torch.Generator().manual_seed(9)
    for R, C in ((1000, 512), (37, 64), (5000, 1024), (3, 2048)):
        x = torch.randn(R, C, generator=gen).to(torch.bfloat16)
        out = torch.full((C,), 0.5, dtype=torch.float32).cuda()
        ops.colsum(x.cuda(), out)
        assert rel_err(out.cpu(), x.double().sum(0) + 0.5) < 1e-5
    src = [torch.randn(n, generator=gen).cuda() for n in (5, 4096, 100003, 8)] * 15     # 60 tensors: two launches
    for dt in (torch.bfloat16, torch.float32):
        dst = [torch.empty(s.numel(), dtype=dt, device="cuda") for s in src]
        ops.gather_cast(dst, src)
        assert all(torch.equal(d, s.to(dt)) for d, s in zip(dst, src))
