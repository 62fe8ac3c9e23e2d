"""The pre-training recipe's optimizer side (main_pretrain_swinv5.py): optim.LARS and optim.momentum_update with the bf16
weight shadow, bf16 bucket gradients (step(grads=...), dist.SegmentedStep's direct path), a device-tensor lr and a device
momentum pair that CUDA-graph-captured steps read on every replay, and PixPro's momentum schedule kept on the device.
Every comparison is bit for bit unless a tolerance is stated."""
import copy
import math
import types

import numpy as np
import pytest
import torch

from conftest import rel_err

# two add_weight_decay groups (vectors / everything else), 52 tensors: odd sizes (scalar tails), sizes above one block's
# chunk, >= 2-D weights, more tensors than one launch takes (48)
SHAPES = [(1,), (3,), (7, 5), (1031,), (64, 129), (70001,), (3, 17, 19), (128, 512)] + \
    [(5 + 7 * i,) if i % 2 else (3 + i, 11) for i in range(44)]


class _Params(torch.nn.Module):
    def __init__(self, tensors):
        super().__init__()
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(t) for t in tensors])


def _model(seed):
    """The SHAPES parameters; the (7, 5) weight is a 4-byte-offset view (the kernels' scalar path)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ts = [torch.randn(s, generator=g, device="cuda") for s in SHAPES]
    host = torch.empty(ts[2].numel() + 1, device="cuda")
    ts[2] = host[1:].view(SHAPES[2]).copy_(ts[2])
    return _Params(ts)


def _clone(m):
    c = _model(0)
    with torch.no_grad():
        for p, q in zip(c.parameters(), m.parameters()):
            p.copy_(q)
    return c


def _lars(model, shadow=True, lr=0.1, **kw):
    from stswincl_b200 import optim
    hp = dict(momentum=0.9, nesterov=True)
    hp.update(kw)
    return optim.LARS(torch.optim.SGD(optim.add_weight_decay(model, 1e-4), lr=lr, **hp), shadow=shadow)


def _grads(seed, n_steps, dtype=torch.float32):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [[torch.randn(s, generator=g, device="cuda").to(dtype) for s in SHAPES] for _ in range(n_steps)]


def _req_order(opt):
    """Parameters in the order step(grads=...) takes them: group order, requires_grad only."""
    return [p for g in opt.param_groups for p in g["params"] if p.requires_grad]


def _assert_same(m1, o1, m2, o2, grads_too=True):
    for i, (p, q) in enumerate(zip(m1.parameters(), m2.parameters())):
        assert torch.equal(p, q), (i, float((p - q).abs().max()))
        if grads_too:
            assert torch.equal(p.grad, q.grad), i
        assert torch.equal(o1.state[p]["momentum_buffer"], o2.state[q]["momentum_buffer"]), i


def _assert_shadows(model):
    from stswincl_b200 import optim
    n = 0
    for p in model.parameters():
        if p.dim() >= 2:
            w = optim.bf16_weight(p)
            assert w.data_ptr() == p._stswin_shadow[0].data_ptr()          # no cast: the shadow itself
            assert torch.equal(w, p.detach().to(torch.bfloat16))
            n += 1
    assert n > 0


@pytest.mark.gpu
def test_lars_shadow_changes_nothing_else():
    """LARS with the shadow vs shadow=False, 3 nesterov steps over two groups: parameters, p.grad (the decayed / scaled
    gradient the reference leaves there) and momentum buffers identical; every shadow equals bf16(p)."""
    a = _model(1)
    b = _clone(a)
    oa, ob = _lars(a, shadow=True), _lars(b, shadow=False)
    assert len(oa.param_groups) == 2 and len(list(a.parameters())) >= 49
    for gs in _grads(2, 3):
        for m in (a, b):
            for p, g in zip(m.parameters(), gs):
                p.grad = g.clone()
        oa.step()
        ob.step()
    torch.cuda.synchronize()
    _assert_same(a, oa, b, ob)
    _assert_shadows(a)
    assert all(getattr(p, "_stswin_shadow", None) is None for p in b.parameters())


@pytest.mark.gpu
def test_lars_bf16_bucket_grads_equal_p_grad_path():
    """step(grads=bf16 list) vs step() with p.grad = the same buckets widened: identical parameters and buffers; the
    buckets and p.grad stay untouched on the grads= path."""
    a = _model(3)
    b = _clone(a)
    oa, ob = _lars(a), _lars(b)
    sentinel = [torch.full_like(p, 7.0) for p in a.parameters()]
    for p, s in zip(a.parameters(), sentinel):
        p.grad = s.clone()
    order = {id(p): i for i, p in enumerate(a.parameters())}
    for gs in _grads(4, 3, torch.bfloat16):
        buckets = [gs[order[id(p)]] for p in _req_order(oa)]
        kept = [t.clone() for t in buckets]
        oa.step(grads=buckets)
        for q, g in zip(b.parameters(), gs):
            q.grad = g.float()
        ob.step()
        torch.cuda.synchronize()
        assert all(torch.equal(t, k) for t, k in zip(buckets, kept))
        assert all(torch.equal(p.grad, s) for p, s in zip(a.parameters(), sentinel))
    _assert_same(a, oa, b, ob, grads_too=False)
    _assert_shadows(a)


@pytest.mark.gpu
def test_lars_captured_step_follows_device_lr():
    """One eager step, then LARS.step captured with lr a device tensor; five replays with new gradients and lr_t
    rewritten before each equal an eager twin stepped with the same (fp32) lrs as floats."""
    lrs = [float(torch.tensor(v)) for v in (0.3, 0.25, 0.2, 0.1, 0.05, 0.01)]
    a = _model(5)
    b = _clone(a)
    lr_t = torch.tensor(lrs[0], device="cuda")
    oa, ob = _lars(a, lr=lr_t, nesterov=False), _lars(b, lr=lrs[0], nesterov=False)
    grads = _grads(6, 6)
    for p, g in zip(a.parameters(), grads[0]):
        p.grad = g.clone()
    oa.step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph):
            oa.step()
    torch.cuda.current_stream().wait_stream(side)
    for k in range(1, 6):
        for p, g in zip(a.parameters(), grads[k]):
            p.grad.copy_(g)
        lr_t.fill_(lrs[k])
        graph.replay()
    for k in range(6):
        for q, g in zip(b.parameters(), grads[k]):
            q.grad = g.clone()
        for group in ob.param_groups:
            group["lr"] = lrs[k]
        ob.step()
    torch.cuda.synchronize()
    _assert_same(a, oa, b, ob)
    _assert_shadows(a)


def _ema_lists(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = [torch.nn.Parameter(torch.randn(s, generator=g, device="cuda")) for s in SHAPES]
    k = [torch.nn.Parameter(torch.randn(s, generator=g, device="cuda"), requires_grad=False) for s in SHAPES]
    return q, k


@pytest.mark.gpu
def test_momentum_update_device_pair_captured():
    """momentum_update with a device pair [m, 1-m], captured and replayed with a new pair (and new query weights) before
    each replay: equals the eager float calls and the reference expression k * m + q * (1. - m); the key shadows equal
    bf16(k) and are what bf16_weight returns."""
    from stswincl_b200 import optim
    ms = [0.99, 0.9913, 0.995, 0.99712, 0.999, 1.0]
    q, k = _ema_lists(7)
    k_eager = [torch.nn.Parameter(t.detach().clone(), requires_grad=False) for t in k]
    k_ref = [t.detach().clone() for t in k]
    pair = torch.tensor([ms[0], 1. - ms[0]], dtype=torch.float32, device="cuda")
    optim.momentum_update(q, k, pair)                      # eager first call: creates the shadows
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph):
            optim.momentum_update(q, k, pair)
    torch.cuda.current_stream().wait_stream(side)
    for i, m in enumerate(ms):
        if i > 0:
            pair.copy_(torch.tensor([m, 1. - m], dtype=torch.float32))
            graph.replay()
        optim.momentum_update(q, k_eager, m)
        with torch.no_grad():
            for r, qq in zip(k_ref, q):
                r.copy_(r * m + qq * (1. - m))
            for qq in q:                                       # the query encoder moves between updates
                qq.mul_(1.001)
    torch.cuda.synchronize()
    for i, (a, b, r) in enumerate(zip(k, k_eager, k_ref)):
        assert torch.equal(a, b), i
        assert torch.equal(a, r), i
    _assert_shadows(types.SimpleNamespace(parameters=lambda: iter(k)))
    _assert_shadows(types.SimpleNamespace(parameters=lambda: iter(k_eager)))


def test_pixpro_momentum_table_is_the_host_formula():
    """CPU: every row k < K of the device schedule is the double expression of PixPro_swin_v5.py:262 rounded to fp32
    once; row K, served for every k >= K, is (1, 0)."""
    from stswincl_b200 import pixpro
    for base, K in ((0.99, 1), (0.99, 7), (0.9, 1000), (0.996, 1313)):
        t = pixpro.momentum_table(base, K)
        assert t.dtype == torch.float32 and t.shape == (K + 1, 2)
        want = np.empty((K + 1, 2), dtype=np.float32)
        for k in range(K):
            m = 1. - (1. - base) * (math.cos(math.pi * k / K) + 1) / 2.
            want[k] = (np.float32(m), np.float32(1. - m))
        want[K] = (1.0, 0.0)
        assert np.array_equal(t.numpy(), want)


class _Seg(torch.nn.Module):
    def __init__(self):
        super().__init__()
        from stswincl_b200 import swin
        self.resnet = torch.nn.Conv2d(3, 8, 1)
        self.swin = swin.SwinTransformerLayerv5(128, (16, 24), 2)
        self.aspp = torch.nn.Conv2d(256, 8, 1)
        self.project1, self.project2, self.project3 = (torch.nn.Conv2d(8, 4, 1), torch.nn.Conv2d(128, 4, 1),
                                                        torch.nn.Conv2d(256, 4, 1))


def _pixpro(K=20):
    from stswincl_b200 import pixpro
    torch.manual_seed(11)
    args = types.SimpleNamespace(pixpro_momentum=0.99, num_instances=2 * K, batch_size=2, epochs=1, start_epoch=1)
    pp = pixpro.PixPro(args, lambda: _Seg().cuda(), lambda: torch.nn.Conv2d(16, 8, 1).cuda()).cuda()
    with torch.no_grad():                                      # the query encoder differs from the key encoder
        for p in pp.encoder_2.parameters():
            p.add_(0.01 * torch.randn_like(p))
    assert pp.K == K and pp.k == 0
    return pp


def _key_params(pp):
    return [pk for _, pk in pp._pairs()]


@pytest.mark.gpu
def test_pixpro_captured_schedule_follows_k():
    """A captured _momentum_update_key_encoder replayed N times from k0 leaves the key encoder equal to N eager calls
    (and to the reference expression with the host-double momenta), and k == k0 + N."""
    pp = _pixpro()
    twin = copy.deepcopy(pp)
    k0, N = 5, 8
    ref = [p.detach().clone() for p in _key_params(pp)]
    qs = [pq.detach().clone() for pq, _ in pp._pairs()]
    pp.k = k0
    twin.k = k0
    pp._momentum_update_key_encoder()                          # eager first call: shadows; then the graph replays
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph):
            pp._momentum_update_key_encoder()
    torch.cuda.current_stream().wait_stream(side)
    assert pp.k == k0 + 1                                      # capture does not run the update
    for _ in range(N - 1):
        graph.replay()
    for _ in range(N):
        twin._momentum_update_key_encoder()
    with torch.no_grad():
        for k in range(k0, k0 + N):
            m = 1. - (1. - 0.99) * (math.cos(math.pi * k / pp.K) + 1) / 2.
            for r, q in zip(ref, qs):
                r.copy_(r * m + q * (1. - m))
    torch.cuda.synchronize()
    assert pp.k == k0 + N and twin.k == k0 + N
    for i, (a, b, r) in enumerate(zip(_key_params(pp), _key_params(twin), ref)):
        assert torch.equal(a, b), i
        assert torch.equal(a, r), i
    from stswincl_b200 import optim
    w = pp.encoder_k_2.layers[0][0].attn.qkv.weight
    assert optim.bf16_weight(w).data_ptr() == w._stswin_shadow[0].data_ptr()
    assert torch.equal(optim.bf16_weight(w), w.detach().to(torch.bfloat16))


@pytest.mark.gpu
def test_pixpro_schedule_end_holds_key_encoder():
    """At k = K - 1 the update takes the last momentum of the cosine; from k = K on (m = 1, 1 - m = 0) the key encoder
    stays where it is, while k keeps counting."""
    pp = _pixpro()
    pp.k = pp.K - 1
    pp._momentum_update_key_encoder()
    after_last = [p.detach().clone() for p in _key_params(pp)]
    for _ in range(3):
        pp._momentum_update_key_encoder()
    torch.cuda.synchronize()
    assert pp.k == pp.K + 3
    assert all(torch.equal(a, b) for a, b in zip(_key_params(pp), after_last))
    with pytest.raises(ValueError):
        pp.k = -1


def _layer_setup(seed):
    from oracle import swin_oracle as so
    dim, res, heads = 128, (16, 24), 2
    params = so.make_layer_params(dim, res, heads, seed=seed)
    x = so.make_features(seed + 1, 2, 4, dim, res[0], res[1]).cuda().to(torch.bfloat16)
    w1 = (so.make_features(seed + 2, 2, 4, dim, res[0], res[1]) - 0.4).cuda().to(torch.bfloat16)
    w2 = (so.make_features(seed + 3, 2, 4, 2 * dim, res[0] // 2, res[1] // 2) - 0.4).cuda().to(torch.bfloat16)
    loss_fn = lambda y: torch.sum(y[0] * w1, dtype=torch.float32) + torch.sum(y[1] * w2, dtype=torch.float32)
    return dim, res, heads, params, x, loss_fn


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True])
def test_segmented_step_single_gpu_lars_direct_path(use_graph):
    """dist.SegmentedStep(LARS) on one GPU with bf16 buckets takes the direct path (stepper._direct): LARS reads the
    reduced gradients straight from the buckets, and every step equals a LARS stepped through p.grad = the same
    buckets widened, bit for bit."""
    from stswincl_b200 import dist as sdist, optim, swin
    dim, res, heads, params, x, loss_fn = _layer_setup(31)

    def fresh():
        m = swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads)
        m.load_state_dict(params, strict=True)
        return m.cuda()

    mine, ref = fresh(), fresh()
    mk = lambda m: optim.LARS(torch.optim.SGD(optim.add_weight_decay(m, 1e-5), lr=0.05, momentum=0.9))
    opt, ref_opt = mk(mine), mk(ref)
    stepper = sdist.SegmentedStep(mine, opt, loss_fn, segments=4, wire_dtype=torch.bfloat16, use_graph=use_graph)
    for _ in range(3):
        stepper.step(x)
        for q, p in zip(ref.parameters(), mine.parameters()):
            q.grad = stepper._view_of[id(p)].float()
        ref_opt.step()
        torch.cuda.synchronize()
        for q, p in zip(ref.parameters(), mine.parameters()):
            assert torch.equal(p, q)
            assert torch.equal(opt.state[p]["momentum_buffer"], ref_opt.state[q]["momentum_buffer"])
    assert stepper._direct and stepper.captured == use_graph
    _assert_shadows(mine)


@pytest.mark.gpu
def test_head_outputs_with_shadows_equal_casts():
    """The Swin head after the same LARS steps with shadows and with shadow=False, and a key encoder updated by
    momentum_update with and without shadows: no-grad forwards bit-identical (the same bf16 values, from the shadow
    instead of a cast).  A training forward + backward agrees up to the fp32-atomic reordering two runs already show."""
    from stswincl_b200 import optim, swin
    dim, res, heads, params, x, loss_fn = _layer_setup(41)

    def fresh():
        m = swin.SwinTransformerLayerv5(dim=dim, input_resolution=res, num_heads=heads)
        m.load_state_dict(params, strict=True)
        return m.cuda()

    qa, qb, ka, kb = fresh(), fresh(), fresh(), fresh()
    for k in (ka, kb):
        for p in k.parameters():
            p.requires_grad_(False)
    oa = optim.LARS(torch.optim.SGD(optim.add_weight_decay(qa, 1e-5), lr=0.05, momentum=0.9), shadow=True)
    ob = optim.LARS(torch.optim.SGD(optim.add_weight_decay(qb, 1e-5), lr=0.05, momentum=0.9), shadow=False)
    g = torch.Generator(device="cuda").manual_seed(42)
    for _ in range(3):
        gs = [torch.randn(p.shape, generator=g, device="cuda") * 1e-2 for p in qa.parameters()]
        for m in (qa, qb):
            for p, gr in zip(m.parameters(), gs):
                p.grad = gr.clone()
        oa.step()
        ob.step()
        optim.momentum_update(qa.parameters(), ka.parameters(), 0.99, shadow=True)
        optim.momentum_update(qb.parameters(), kb.parameters(), 0.99, shadow=False)
    torch.cuda.synchronize()
    _assert_shadows(qa)
    _assert_shadows(ka)
    assert all(getattr(p, "_stswin_shadow", None) is None for m in (qb, kb) for p in m.parameters())
    with torch.no_grad():
        for a, b in ((qa, qb), (ka, kb)):
            for pa, pb in zip(a.parameters(), b.parameters()):
                assert torch.equal(pa, pb)
            ya, yb = a(x), b(x)
            assert all(torch.equal(u, v) for u, v in zip(ya, yb))
    for m in (qa, qb):
        m.zero_grad(set_to_none=True)
        loss_fn(m(x)).backward()
    for (n, pa), pb in zip(qa.named_parameters(), qb.parameters()):
        assert rel_err(pa.grad, pb.grad) <= 1e-6, n


@pytest.mark.gpu
def test_errors():
    from stswincl_b200 import optim
    from stswincl_b200._lib import StswinError
    m = _model(9)
    for g, p in zip(_grads(10, 1)[0], m.parameters()):
        p.grad = g
    for lr in (torch.tensor(0.1, dtype=torch.float64, device="cuda"), torch.tensor(0.1),
               torch.tensor([0.1], device="cuda")):
        with pytest.raises(StswinError, match="tensor lr"):
            _lars(m, lr=lr).step()
    o = _lars(m)
    n = len(_req_order(o))
    with pytest.raises(StswinError, match="gradients"):
        o.step(grads=[p.grad for p in _req_order(o)][:n - 1])
    mixed = [p.grad if i % 2 else p.grad.to(torch.bfloat16) for i, p in enumerate(_req_order(o))]
    with pytest.raises(StswinError, match="all fp32 or all bf16"):
        o.step(grads=mixed)
    q, k = _ema_lists(12)
    for bad in (torch.tensor([0.9, 0.1, 0.0], device="cuda"), torch.tensor([0.9, 0.1], dtype=torch.float64, device="cuda"),
                torch.tensor([0.9, 0.1])):
        with pytest.raises(StswinError, match="tensor momentum"):
            optim.momentum_update(q, k, bad)
