"""optim.FusedSGD (stswin_sgd_step) against torch.optim.SGD, the optimiser of the fine-tune recipe
train_CL_ft_mswin_sgd_minput.py:147-162: bit-identical parameters and momentum buffers with torch's single-tensor step on
the same GPU over the hyper-parameter grid, bf16 bucket gradients, the bf16 weight shadow, state_dict interchange, a
CUDA-graph-captured step with a device lr, and the data-parallel step (dist.SegmentedStep) on one and two GPUs."""
import copy
import ctypes
import itertools
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import rel_err

pytestmark = pytest.mark.gpu

# odd sizes (unaligned tails), sizes above one block's chunk, a >= 2-D weight of each kind, and in total more tensors than
# one launch takes (48)
SHAPES = [(1,), (3,), (7, 5), (1031,), (64, 129), (70001,), (3, 17, 19), (128, 512)] + [(5 + 7 * i,) for i in range(44)]


def _params(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(s, generator=g, device="cuda") for s in SHAPES]


def _pair(seed, **kw):
    """The same parameters for FusedSGD and torch.optim.SGD(foreach=False), in two groups with a 10x lr ratio (the
    classifier group of the recipe).  One FusedSGD parameter is a 4-byte-offset view (the kernel's scalar path)."""
    from stswincl_b200 import optim
    base = _params(seed)
    ours = [p.clone().requires_grad_() for p in base]
    host = torch.empty(base[3].numel() + 1, device="cuda")
    ours[3] = host[1:].copy_(base[3]).requires_grad_()          # misaligned data pointer
    ref = [p.clone().requires_grad_() for p in base]
    split = len(SHAPES) // 2
    groups = lambda ps, lr: [dict(params=ps[:split]), dict(params=ps[split:], lr=10 * lr)]
    lr = kw.pop("lr", 0.01)
    o = optim.FusedSGD(groups(ours, lr), lr=lr, **kw)
    r = torch.optim.SGD(groups(ref, lr), lr=lr, foreach=False, **kw)
    return ours, o, ref, r


def _assert_same(ours, o, ref, r):
    for i, (p, q) in enumerate(zip(ours, ref)):
        assert torch.equal(p, q), (i, float((p - q).abs().max()))
        b1, b2 = o.state[p].get("momentum_buffer"), r.state[q].get("momentum_buffer")
        assert (b1 is None) == (b2 is None), i
        if b1 is not None:
            assert torch.equal(b1, b2), (i, float((b1 - b2).abs().max()))


def _assert_shadows(ours):
    from stswincl_b200 import optim
    for p in ours:
        if p.dim() >= 2:
            w = optim.bf16_weight(p)
            assert w.data_ptr() == p._stswin_shadow[0].data_ptr()          # no cast: the shadow itself
            assert torch.equal(w, p.to(torch.bfloat16))


GRID = [dict(momentum=m, dampening=d, weight_decay=wd, maximize=mx)
        for (m, d), wd, mx in itertools.product([(0.0, 0.0), (0.0, 0.1), (0.9, 0.0), (0.9, 0.1)], [0.0, 1e-4], [False, True])]
GRID += [dict(momentum=0.9, dampening=0.0, nesterov=True, weight_decay=wd, maximize=mx)
         for wd, mx in itertools.product([0.0, 1e-4], [False, True])]


@pytest.mark.parametrize("hp", GRID, ids=lambda hp: "-".join(f"{k}={v}" for k, v in hp.items()))
def test_fused_sgd_bit_identical_with_torch_sgd(hp):
    """Five steps with new gradients each step and a new lr from step 3 on; one parameter has no gradient on step 2 and
    must keep its value and momentum buffer."""
    ours, o, ref, r = _pair(1, **hp)
    g = torch.Generator(device="cuda").manual_seed(2)
    for step in range(5):
        if step == 3:
            for opt in (o, r):
                for k, group in enumerate(opt.param_groups):
                    group["lr"] = (0.003, 0.03)[k]
        for i, (p, q) in enumerate(zip(ours, ref)):
            gr = torch.randn(p.shape, generator=g, device="cuda")
            p.grad, q.grad = (None, None) if (step == 2 and i == 4) else (gr.clone(), gr.clone())
        keep = (ours[4].clone(), o.state[ours[4]].get("momentum_buffer"))
        keep = (keep[0], None if keep[1] is None else keep[1].clone())
        o.step()
        r.step()
        _assert_same(ours, o, ref, r)
        _assert_shadows(ours)
        for p, q in zip(ours, ref):                             # p.grad is left as the caller set it (torch's too)
            assert (p.grad is None and q.grad is None) or torch.equal(p.grad, q.grad)
        if step == 2:
            assert torch.equal(ours[4], keep[0])
            if keep[1] is not None:
                assert torch.equal(o.state[ours[4]]["momentum_buffer"], keep[1])


@pytest.mark.parametrize("nesterov", [False, True])
def test_fused_sgd_bf16_bucket_gradients(nesterov):
    """step(grads=[bf16 ...], grad_scale=s) equals torch SGD fed g.float() * s."""
    hp = dict(momentum=0.9, dampening=0.0, weight_decay=1e-4, nesterov=nesterov)
    ours, o, ref, r = _pair(3, **hp)
    g = torch.Generator(device="cuda").manual_seed(4)
    s = 0.37
    for step in range(5):
        gb = [torch.randn(p.shape, generator=g, device="cuda").to(torch.bfloat16) for p in ours]
        for q, gr in zip(ref, gb):
            q.grad = gr.float() * s
        o.step(grads=gb, grad_scale=s)
        r.step()
        _assert_same(ours, o, ref, r)
        _assert_shadows(ours)
    assert all(p.grad is None for p in ours)


def test_fused_sgd_shadow_refreshed_after_an_outside_write():
    from stswincl_b200 import optim
    ours, o, _, _ = _pair(5, momentum=0.9)
    for p in ours:
        p.grad = torch.ones_like(p)
    o.step()
    _assert_shadows(ours)
    w = ours[4]
    with torch.no_grad():
        w.mul_(1.5)
    assert torch.equal(optim.bf16_weight(w), w.to(torch.bfloat16))
    o.step()
    _assert_shadows(ours)


@pytest.mark.parametrize("torch_first", [True, False])
def test_fused_sgd_state_dict_interchange_with_torch_sgd(torch_first):
    """Two steps in one optimiser, its state_dict loaded into the other, three more steps: equals the first optimiser
    continued for three steps."""
    from stswincl_b200 import optim
    hp = dict(lr=0.02, momentum=0.9, dampening=0.1, weight_decay=1e-4, foreach=False)     # the groups carry foreach
    base = _params(6)
    a_ps = [p.clone() for p in base]
    cls_a, cls_b = (lambda ps: torch.optim.SGD(ps, **hp)), (lambda ps: optim.FusedSGD(ps, **hp))
    if not torch_first:
        cls_a, cls_b = cls_b, cls_a
    a = cls_a(a_ps)
    g = torch.Generator(device="cuda").manual_seed(7)
    grads = [[torch.randn(s, generator=g, device="cuda") for s in SHAPES] for _ in range(5)]
    for k in range(2):
        for p, gr in zip(a_ps, grads[k]):
            p.grad = gr.clone()
        a.step()
    b_ps = [p.clone() for p in a_ps]
    b = cls_b(b_ps)
    b.load_state_dict(copy.deepcopy(a.state_dict()))        # a checkpoint: load_state_dict keeps same-device tensors
    for k in range(2, 5):
        for ps, opt in ((a_ps, a), (b_ps, b)):
            for p, gr in zip(ps, grads[k]):
                p.grad = gr.clone()
            opt.step()
    for p, q in zip(a_ps, b_ps):
        assert torch.equal(p, q)
        assert torch.equal(a.state[p]["momentum_buffer"], b.state[q]["momentum_buffer"])


def test_fused_sgd_graph_capture_with_device_lr():
    """One eager step, then step() captured with lr a device tensor; four replays with new gradients and a new lr
    written before each: equals the same five steps of torch SGD run eagerly."""
    from stswincl_b200 import optim
    hp = dict(momentum=0.9, dampening=0.0, weight_decay=1e-4)
    lrs = [0.05, 0.04, 0.03, 0.025, 0.01]
    base = _params(8)
    ours, ref = [p.clone() for p in base], [p.clone() for p in base]
    lr_t = torch.tensor(lrs[0], device="cuda")
    o = optim.FusedSGD(ours, lr=lr_t, **hp)
    r = torch.optim.SGD(ref, lr=lrs[0], foreach=False, **hp)
    g = torch.Generator(device="cuda").manual_seed(9)
    grads = [[torch.randn(s, generator=g, device="cuda") for s in SHAPES] for _ in range(5)]
    for p, gr in zip(ours, grads[0]):
        p.grad = gr.clone()
    o.step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph):
            o.step()
    torch.cuda.current_stream().wait_stream(side)
    for k in range(1, 5):
        for p, gr in zip(ours, grads[k]):
            p.grad.copy_(gr)
        lr_t.fill_(lrs[k])
        graph.replay()
    for k in range(5):
        for q, gr in zip(ref, grads[k]):
            q.grad = gr.clone()
        for group in r.param_groups:
            group["lr"] = float(torch.tensor(lrs[k]))            # the fp32 value the device scalar holds
        r.step()
    torch.cuda.synchronize()
    _assert_same(ours, o, ref, r)
    _assert_shadows(ours)


def _layer_setup(seed):
    from oracle import swin_oracle as so
    dim, res, heads = 128, (16, 24), 2
    params = so.make_layer_params(dim, res, heads, seed=seed)
    x = so.make_features(seed + 1, 2, 4, dim, res[0], res[1]).cuda().to(torch.bfloat16)
    w1 = (so.make_features(seed + 2, 2, 4, dim, res[0], res[1]) - 0.4).cuda().to(torch.bfloat16)
    w2 = (so.make_features(seed + 3, 2, 4, 2 * dim, res[0] // 2, res[1] // 2) - 0.4).cuda().to(torch.bfloat16)
    loss_fn = lambda y: torch.sum(y[0] * w1, dtype=torch.float32) + torch.sum(y[1] * w2, dtype=torch.float32)
    return dim, res, heads, params, x, loss_fn


@pytest.mark.parametrize("use_graph", [False, True])
def test_segmented_step_single_gpu_fused_sgd_direct_path(use_graph):
    """dist.SegmentedStep on one GPU with bf16 buckets.  FusedSGD takes the reduced gradients straight from the buckets
    (stepper._direct); every step equals torch.optim.SGD fed the same buckets the way the copy-back path feeds it
    (p.grad = fp32 copy of the bucket view), bit for bit.  A second stepper with torch.optim.SGD (copy-back path) takes
    the same first update within the bf16 bound: its own backward may reorder the fp32 atomic sums of the LayerNorm /
    bias gradients, which can move a bf16 rounding of a gradient by one step."""
    from stswincl_b200 import dist as sdist, optim, swin
    dim, res, heads, params, x, loss_fn = _layer_setup(27)
    hp = dict(lr=0.01, momentum=0.9, weight_decay=1e-4)

    def fresh():
        m = swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads)
        m.load_state_dict(params, strict=True)
        return m.cuda()

    mine = fresh()
    opt = optim.FusedSGD(mine.parameters(), **hp)
    stepper = sdist.SegmentedStep(mine, opt, loss_fn, segments=4, wire_dtype=torch.bfloat16, use_graph=use_graph)
    ref_ps = [p.detach().clone() for p in mine.parameters()]
    ref_opt = torch.optim.SGD(ref_ps, foreach=False, **hp)
    other = fresh()
    other_opt = torch.optim.SGD(other.parameters(), foreach=False, **hp)
    other_stepper = sdist.SegmentedStep(other, other_opt, loss_fn, segments=4, wire_dtype=torch.bfloat16, use_graph=use_graph)
    for step in range(3):
        stepper.step(x)
        other_stepper.step(x)
        if step == 0:           # from the same weights; later steps start from weights that differ and drift apart
            for (n, p), q in zip(mine.named_parameters(), other.parameters()):
                assert rel_err(p - params[n].cuda(), q - params[n].cuda()) < 2e-2, n
        for q, p in zip(ref_ps, mine.parameters()):
            q.grad = stepper._view_of[id(p)].float()
        ref_opt.step()
        torch.cuda.synchronize()
        for q, p in zip(ref_ps, mine.parameters()):
            assert torch.equal(p, q)
            assert torch.equal(opt.state[p]["momentum_buffer"], ref_opt.state[q]["momentum_buffer"])
            if p.dim() >= 2:
                assert torch.equal(optim.bf16_weight(p), p.detach().to(torch.bfloat16))
    assert stepper._direct and not other_stepper._direct
    assert stepper.captured == use_graph and other_stepper.captured == use_graph


def _dp_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from oracle import swin_oracle as so
        from stswincl_b200 import dist as sdist, optim, swin
        dim, res, heads = 128, (16, 24), 2
        params = so.make_layer_params(dim, res, heads, seed=7)
        x = so.make_features(8, world, 4, dim, res[0], res[1]).to(dev)
        w1 = (so.make_features(9, world, 4, dim, res[0], res[1]) - 0.4).to(dev)
        w2 = (so.make_features(10, world, 4, 2 * dim, res[0] // 2, res[1] // 2) - 0.4).to(dev)
        lr, ok, worst = 0.5, True, 0.0
        for use_graph, wire in ((False, torch.float32), (True, torch.float32), (True, torch.bfloat16)):
            full = swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads)
            full.load_state_dict(params, strict=True)
            full = full.to(dev)
            y1, y2 = full(x)
            (((y1 * w1).sum() + (y2 * w2).sum()) / world).backward()            # the whole batch on one rank
            want = {n: p.grad.clone() for n, p in full.named_parameters()}
            mine = swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads)
            mine.load_state_dict(params, strict=True)
            mine = mine.to(dev)
            p0 = {n: p.detach().clone() for n, p in mine.named_parameters()}
            opt = optim.FusedSGD(mine.parameters(), lr=lr, momentum=0.9)
            r = slice(rank, rank + 1)
            stepper = sdist.SegmentedStep(mine, opt, lambda y: (y[0] * w1[r]).sum() + (y[1] * w2[r]).sum(), segments=4,
                                          wire_dtype=wire, use_graph=use_graph)
            stepper.step(x[r].contiguous())
            torch.cuda.synchronize()
            tol = 2e-2 if wire == torch.bfloat16 else 5e-3
            for n, p in mine.named_parameters():
                e = max(rel_err(opt.state[p]["momentum_buffer"], want[n]),          # first step: buf = reduced gradient
                        rel_err(p.detach() - p0[n], -lr * want[n]))
                worst = max(worst, e)
                ok = ok and e < tol
            ok = ok and stepper._direct and (stepper.captured == use_graph) and len(stepper._buckets) == 4
        ret[rank] = (bool(ok), worst)
    finally:
        dist.destroy_process_group()


def test_two_rank_segmented_step_with_fused_sgd_equals_one_rank_step():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dp_worker, args=(2, 29500 + os.getpid() % 200, ret), nprocs=2, join=True)
    assert all(v[0] for v in dict(ret).values()) and len(ret) == 2, dict(ret)


def test_fused_sgd_errors():
    from stswincl_b200 import _lib, optim
    with pytest.raises(ValueError):
        optim.FusedSGD([torch.zeros(3, device="cuda")], nesterov=True)                   # nesterov without momentum
    with pytest.raises(ValueError):
        optim.FusedSGD([torch.zeros(3, device="cuda")], momentum=0.9, dampening=0.1, nesterov=True)
    with pytest.raises(ValueError):
        optim.FusedSGD([torch.zeros(3, device="cuda")], lr=-1.0)
    with pytest.raises(_lib.StswinError):
        optim.FusedSGD([torch.zeros(3, device="cuda")], differentiable=True)
    for p in (torch.zeros(3), torch.zeros(3, device="cuda", dtype=torch.float16)):        # CPU, fp16 parameters
        o = optim.FusedSGD([p], lr=0.1, momentum=0.9)
        p.grad = torch.ones_like(p)
        with pytest.raises(_lib.StswinError):
            o.step()
    p = torch.zeros(3, device="cuda")
    p.grad = torch.ones(6, device="cuda")[::2]                                            # non-contiguous gradient
    with pytest.raises(_lib.StswinError):
        optim.FusedSGD([p], lr=0.1).step()
    with pytest.raises(_lib.StswinError):                                                 # lr tensor on the host
        p.grad = torch.ones(3, device="cuda")
        optim.FusedSGD([p], lr=torch.tensor(0.1)).step()
    # grads= lists that are short, long, or hold a gradient of another size (in the second group): refused before any
    # group is updated
    ps = [torch.zeros(3, device="cuda", requires_grad=True), torch.zeros(5, device="cuda", requires_grad=True)]
    o = optim.FusedSGD([dict(params=ps[:1]), dict(params=ps[1:])], lr=0.1, momentum=0.9)
    for gl in ([torch.ones(3, device="cuda")], [torch.ones(3, device="cuda"), torch.ones(5, device="cuda")] * 2,
               [torch.ones(3, device="cuda"), torch.ones(4, device="cuda")]):
        with pytest.raises(_lib.StswinError, match="gradients"):
            o.step(grads=gl)
    assert all(not torch.any(q) for q in ps) and not o.state
    # the C ABI refuses what the constructor refuses, and momentum without buffers
    lib = _lib.load()
    ptr = (ctypes.c_void_p * 1)(p.data_ptr())
    n = (ctypes.c_int64 * 1)(3)
    stream = torch.cuda.current_stream().cuda_stream
    assert lib.stswin_sgd_step(ptr, ptr, ptr, None, n, None, 1, 0, 0.1, None, 0.0, 1.0, 1, 0, 0.0, 1.0, stream) != 0
    assert lib.stswin_sgd_step(ptr, ptr, ptr, None, n, None, 1, 0, 0.1, None, 0.9, 0.9, 1, 0, 0.0, 1.0, stream) != 0
    assert lib.stswin_sgd_step(ptr, ptr, None, None, n, None, 1, 0, 0.1, None, 0.9, 1.0, 0, 0, 0.0, 1.0, stream) != 0
    assert lib.stswin_sgd_step(None, ptr, None, None, n, None, 1, 0, 0.1, None, 0.0, 1.0, 0, 0, 0.0, 1.0, stream) != 0
    assert torch.equal(p, torch.zeros(3, device="cuda"))
