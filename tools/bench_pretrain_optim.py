"""The pre-training recipe's optimizer side (main_pretrain_swinv5.py: LARS around SGD momentum 0.9, add_weight_decay groups;
the key-encoder EMA of PixPro) with and without the bf16 weight shadows that LARS and momentum_update now write.

  kernel  the 159 tensors / 96.6 M parameters of the Swin head (512 ch, 4 heads) in the two add_weight_decay groups:
          LARS with fp32 p.grad or bf16 step(grads=...) and the shadow off / on, and momentum_update with the shadow off /
          on.  CUDA-graph replays (386 MB of fp32 weights: larger than L2); ms and GB/s of the bytes each pass needs,
          against the copy peak.
  step    the pre-training step of bench.py --config pretrain on one GPU (6 sequences x 4 clips x 4 frames, 512 ch, 32x56:
          2 query passes fwd + bwd, EMA, 6 no-grad key passes, the fused contrastive loss, LARS), captured whole:
            bench      the query passes batched into one head call and the key passes into another (as bench.py does);
            reference  2 query head calls and 6 separate key head calls (PixPro.forward, PixPro_swin_v5.py:291-366);
          shadows off (LARS(shadow=False), momentum_update(shadow=False)) and on, alternated --runs times.

    python tools/bench_pretrain_optim.py [--runs 3] [--steps 30] [--out profiles/bench_pretrain_optim.json]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import ClockSampler  # noqa: E402
from bench_sgd import COPY_PEAK_GBS, gpu_info, graphed, time_ms  # noqa: E402
from stswincl_b200 import contrast, optim, swin  # noqa: E402

DIM, HEADS, T = 512, 4, 4
HEAD_RES = (64, 80)             # parameter count of the head does not depend on the resolution except the masks
STEP_RES, CLIPS, K_CLASSES = (32, 56), 4, 12


def lars(model, shadow, lr=0.1):
    return optim.LARS(torch.optim.SGD(optim.add_weight_decay(model, 1e-5), lr=lr, momentum=0.9), shadow=shadow)


_HELD = []                      # shadows a captured graph writes: alive as long as the graphs


def strip_shadows(model):
    for p in model.parameters():
        if hasattr(p, "_stswin_shadow"):
            _HELD.append(p._stswin_shadow)
            del p._stswin_shadow


# ---------------------------------------------------------------------------------------------------------------
def bench_kernels(runs):
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=HEAD_RES, num_heads=HEADS).to(dev)
    key = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=HEAD_RES, num_heads=HEADS).to(dev)
    ps, pk = list(model.parameters()), list(key.parameters())
    n = sum(p.numel() for p in ps)
    n2 = sum(p.numel() for p in ps if p.dim() >= 2)
    g = torch.Generator(device=dev).manual_seed(1)
    g32 = [torch.randn(p.shape, generator=g, device=dev) * 1e-3 for p in ps]
    g16 = [t.to(torch.bfloat16) for t in g32]
    opts = {}

    def lars_step(shadow, bf16):
        key_ = (shadow, bf16)
        if key_ not in opts:
            opts[key_] = lars(model, shadow)
        o = opts[key_]
        idx = {id(p): i for i, p in enumerate(ps)}
        gl = [g16[idx[id(p)]] for grp in o.param_groups for p in grp["params"]]       # step(grads=) takes group order

        def fn():
            if bf16:
                o.step(grads=gl)
            else:
                for p, t in zip(ps, g32):
                    p.grad = t
                o.step()
        return fn

    # bytes per pass (fp32 = 4, bf16 = 2 per element): norms read p, g; update reads p, g, buf and writes p, buf
    # (+ g on the p.grad path), + the bf16 shadow of the >= 2-D weights; EMA reads k, q and writes k (+ shadow)
    variants = {}
    for bf16 in (False, True):
        gsz = 2 if bf16 else 4
        for shadow in (False, True):
            name = "lars_%s_grads_shadow_%s" % ("bf16" if bf16 else "fp32", "on" if shadow else "off")
            nbytes = n * ((4 + gsz) + 8 + gsz + (0 if bf16 else 4) + 8) + (n2 * 2 if shadow else 0)
            variants[name] = (lars_step(shadow, bf16), nbytes)
    for shadow in (False, True):
        variants["ema_shadow_%s" % ("on" if shadow else "off")] = (
            (lambda s=shadow: optim.momentum_update(ps, pk, 0.99, shadow=s)), n * 12 + (n2 * 2 if shadow else 0))
    replays = {}
    for k, (fn, _) in variants.items():      # capture each with only its own shadows present
        strip_shadows(model); strip_shadows(key)
        replays[k] = graphed(fn)
    times = {k: [] for k in variants}
    for _ in range(runs):                    # alternated
        for k, rep in replays.items():
            times[k].append(time_ms(rep, 50))
    out = {"tensors": len(ps), "parameters": n, "parameters_2d": n2, "copy_peak_GBps": COPY_PEAK_GBS,
           "bytes_note": "bytes each pass needs (LARS: norms p, g; update p, g, buf in, p, buf out, g out on the p.grad "
                         "path; EMA k, q in, k out; + bf16 shadow of the >= 2-D weights when on)"}
    for k, (_, nbytes) in variants.items():
        ms = min(times[k])
        out[k] = {"ms_runs": [round(t, 4) for t in times[k]], "ms_best": round(ms, 4), "MB": round(nbytes / 1e6, 1),
                  "GBps": round(nbytes / (ms * 1e-3) / 1e9, 1), "frac_copy_peak": round(nbytes / (ms * 1e-3) / 1e9 / COPY_PEAK_GBS, 3)}
    return out


# ---------------------------------------------------------------------------------------------------------------
def make_step(shape, shadow, dev):
    """One captured pre-training step (bench.py --config pretrain, one GPU) with the shadows on or off."""
    torch.manual_seed(0)
    model = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=STEP_RES, num_heads=HEADS).to(dev)
    key_model = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=STEP_RES, num_heads=HEADS).to(dev)
    key_model.load_state_dict(model.state_dict())
    for p in key_model.parameters():
        p.requires_grad_(False)
    opt = lars(model, shadow, lr=CLIPS / 256)
    B = CLIPS
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.relu(torch.randn(6 * B, T, DIM, STEP_RES[0], STEP_RES[1], generator=g, device=dev)).to(torch.bfloat16)
    masks = [torch.randint(0, K_CLASSES, (B, 1, 8, 14), generator=g, device=dev).float()
             .repeat_interleave(STEP_RES[0], 2).repeat_interleave(8 * STEP_RES[1] // 14, 3).contiguous() for _ in range(6)]

    def embed(y1, y2):
        up = torch.nn.functional.interpolate(y2[:, -1, :256], size=y1.shape[-2:], mode="nearest")
        return y1[:, -1, :256] + up

    def step():
        opt.zero_grad(set_to_none=True)
        if shape == "bench":
            y1, y2 = model(x[:2 * B])
            preds = [embed(y1[:B], y2[:B]), embed(y1[B:], y2[B:])]
        else:
            preds = [embed(*model(x[i * B:(i + 1) * B])) for i in range(2)]
        with torch.no_grad():
            optim.momentum_update(list(model.parameters()), list(key_model.parameters()), 0.99, shadow=shadow)
            if shape == "bench":
                k1, k2 = key_model(x)
                keys = [embed(k1[i * B:(i + 1) * B], k2[i * B:(i + 1) * B]) for i in range(6)]
            else:
                keys = [embed(*key_model(x[i * B:(i + 1) * B])) for i in range(6)]
        loss = contrast.consistency_loss_tail(*preds, *keys, *masks, K_CLASSES, normalize=True)
        loss.backward()
        opt.step()

    step()                                   # eager: momentum buffers and shadows exist before the capture
    replay = graphed(step, warm=2)

    def run():
        return replay() if step is not None else None      # holds the step's tensors as long as the graph
    return run


def bench_steps(runs, steps):
    dev = torch.device("cuda", 0)
    out = {}
    for shape in ("bench", "reference"):
        fns = {"shadow_off": make_step(shape, False, dev), "shadow_on": make_step(shape, True, dev)}
        res = {k: [] for k in fns}
        with ClockSampler(0) as clk:
            for fn in fns.values():
                for _ in range(10):
                    fn()
            torch.cuda.synchronize()
            for _ in range(runs):
                for k, fn in fns.items():
                    for _ in range(3):
                        fn()
                    res[k].append(time_ms(fn, steps))
        out[shape] = {k: {"ms_per_step": [round(t, 3) for t in v]} for k, v in res.items()}
        out[shape]["delta_ms_on_minus_off"] = [round(a - b, 3) for a, b in zip(res["shadow_on"], res["shadow_off"])]
        out[shape]["clock"] = clk.summary()
        del fns
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_pretrain_optim.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pretrain_optim.py: needs a CUDA device")
    report = {"gpu": gpu_info(0), "kernels": bench_kernels(args.runs)}
    torch.cuda.empty_cache()
    report["step_1gpu"] = {"workload": "bench.py --config pretrain on one GPU: %d sequences x %d clips x %d frames, %d ch, "
                                       "%dx%d tokens, LARS + key-encoder EMA, captured whole; bench = batched head calls, "
                                       "reference = 2 query + 6 key head calls" % (6, CLIPS, T, DIM, *STEP_RES),
                           "result": bench_steps(args.runs, args.steps)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
