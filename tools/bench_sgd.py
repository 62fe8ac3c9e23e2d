"""optim.FusedSGD against torch.optim.SGD(foreach=True) for the fine-tune recipe (train_CL_ft_mswin_sgd_minput.py:147-162:
SGD momentum 0.9, weight decay 1e-4, per-module groups, poly lr every iteration; bench.py --config finetune_sgd).

  optimizer  the 159 tensors / 96.6 M parameters of the Swin head (512 ch, 64x80, 4 heads): FusedSGD with fp32 gradients,
             FusedSGD with bf16 gradients (step(grads=...), the all-reduce buckets), and torch.optim.SGD(foreach=True)
             plus the per-call bf16 casts of the >= 2-D weights the forward then needs.  CUDA-graph replays (386 MB of
             fp32 weights: larger than L2); ms and GB/s of the bytes the fused pass needs, against the copy peak.
  step       the finetune_sgd step of bench.py (4 clips x 4 frames, 512 ch, 64x80, the same synthetic two-output loss),
             forward + backward + optimizer captured whole on one GPU; torch SGD and FusedSGD (lr a device tensor
             rewritten with the poly schedule before every replay) alternated --runs times; frames/s and the SM clock.
  dp         with two or more GPUs: the same A/B through dist.SegmentedStep (4 segments, bf16 buckets) on two ranks --
             torch SGD reads the buckets back into fp32 p.grad, FusedSGD reads them directly.

    python tools/bench_sgd.py [--runs 3] [--steps 40] > bench_sgd.json      (the JSON report goes to stdout)
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ClockSampler  # noqa: E402
from stswincl_b200 import dist as sdist, optim, swin  # noqa: E402

COPY_PEAK_GBS = 6542.0         # device-to-device copy rate measured on a B200 (1000 W power limit)
DIM, RES, HEADS, T, CLIPS = 512, (64, 80), 4, 4, 4
HP = dict(momentum=0.9, weight_decay=1e-4)
BASE_LR, ITERS, POWER = 1e-3, 10000, 0.9


def poly(i):
    return BASE_LR * (1 - i / ITERS) ** POWER


def gpu_info(index=0):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(index), "nvidia_smi": q}


def graphed(fn, warm=3):
    """fn captured as a CUDA graph after `warm` eager calls on a side stream; returns the replay."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def time_ms(fn, n, between=None):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        if between is not None:
            between(i)
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def head(dev):
    torch.manual_seed(0)
    return swin.SwinTransformerLayerv5(dim=DIM, input_resolution=RES, num_heads=HEADS).to(dev)


# ---------------------------------------------------------------------------------------------------------------
def bench_optimizer(runs):
    dev = torch.device("cuda", 0)
    model = head(dev)
    ps = list(model.parameters())
    n = sum(p.numel() for p in ps)
    n2 = sum(p.numel() for p in ps if p.dim() >= 2)
    g = torch.Generator(device=dev).manual_seed(1)
    g32 = [torch.randn(p.shape, generator=g, device=dev) * 1e-3 for p in ps]
    g16 = [t.to(torch.bfloat16) for t in g32]
    for p, t in zip(ps, g32):
        p.grad = t
    fused = optim.FusedSGD(ps, lr=BASE_LR, **HP)
    ref = torch.optim.SGD(ps, lr=BASE_LR, foreach=True, **HP)

    def torch_step():
        ref.step()
        for p in ps:
            if p.dim() >= 2:
                p.to(torch.bfloat16)                 # what bf16_weight does per call without a shadow

    variants = {
        "fused_sgd_fp32_grads": (lambda: fused.step(), n * 20 + n2 * 2),
        "fused_sgd_bf16_grads": (lambda: fused.step(grads=g16), n * 18 + n2 * 2),
        "torch_sgd_foreach_plus_bf16_casts": (torch_step, n * 20 + n2 * 2),
    }
    replays = {k: graphed(fn) for k, (fn, _) in variants.items()}
    times = {k: [] for k in variants}
    for _ in range(runs):                            # alternated
        for k, rep in replays.items():
            times[k].append(time_ms(rep, 50))
    out = {"tensors": len(ps), "parameters": n, "parameters_2d": n2, "copy_peak_GBps": COPY_PEAK_GBS,
           "bytes_note": "bytes the fused pass needs: p, buf, g read; p, buf written; bf16 shadow of the >= 2-D weights "
                         "written (the same count is used for torch's rate)"}
    for k, (_, nbytes) in variants.items():
        ms = min(times[k])
        out[k] = {"ms_runs": [round(t, 4) for t in times[k]], "ms_best": round(ms, 4), "MB": round(nbytes / 1e6, 1),
                  "GBps": round(nbytes / (ms * 1e-3) / 1e9, 1), "frac_copy_peak": round(nbytes / (ms * 1e-3) / 1e9 / COPY_PEAK_GBS, 3)}
    return out


# ---------------------------------------------------------------------------------------------------------------
def make_step(kind, dev, rank=0, world=1):
    """(run one step, lr setter or None) of the finetune_sgd step with torch SGD or FusedSGD."""
    model = head(dev)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.relu(torch.randn(CLIPS, T, DIM, RES[0], RES[1], generator=g, device=dev)).to(torch.bfloat16)
    g1 = (torch.randn(CLIPS, T, DIM, RES[0], RES[1], generator=g, device=dev) * 0.1).to(torch.bfloat16)
    g2 = (torch.randn(CLIPS, T, 2 * DIM, RES[0] // 2, RES[1] // 2, generator=g, device=dev) * 0.1).to(torch.bfloat16)
    loss_fn = lambda y: torch.sum(y[0] * g1, dtype=torch.float32) + torch.sum(y[1] * g2, dtype=torch.float32)
    lr_t = None
    if kind == "torch":
        opt = torch.optim.SGD(model.parameters(), lr=BASE_LR, foreach=True, **HP)
    else:
        lr_t = torch.tensor(BASE_LR, device=dev)
        opt = optim.FusedSGD(model.parameters(), lr=lr_t, **HP)
    set_lr = (lambda i: lr_t.fill_(poly(i))) if lr_t is not None else None
    if world > 1:
        stepper = sdist.SegmentedStep(model, opt, loss_fn, segments=4, wire_dtype=torch.bfloat16, use_graph=True)
        for _ in range(3):
            stepper.step(x)
        torch.cuda.synchronize()
        assert stepper.captured and stepper._direct == (kind == "fused")
        return (lambda: stepper.step(x)), set_lr

    def step():
        opt.zero_grad(set_to_none=True)
        loss_fn(model(x)).backward()
        opt.step()

    step()                                           # eager: momentum buffers and shadows exist before the capture
    replay = graphed(step, warm=2)

    def run():
        # holds `step` -- model, optimizer, inputs -- as long as the graph that reads and writes their memory (the next
        # capture empties the allocator's cache, so freed blocks would be unmapped)
        return replay() if step is not None else None

    return run, set_lr


def ab(dev, runs, steps, rank=0, world=1):
    fns = {k: make_step(k, dev, rank, world) for k in ("torch", "fused")}
    res = {k: [] for k in fns}
    with ClockSampler(dev.index if rank == 0 else None) as clk:
        for fn, _ in fns.values():                   # untimed: nvidia-smi's start-up stalls kernel launches for ~0.2 s
            for _ in range(20):
                fn()
        torch.cuda.synchronize()
        for _ in range(runs):
            for k, (fn, set_lr) in fns.items():
                for _ in range(3):
                    fn()
                if world > 1:
                    torch.distributed.barrier()
                ms = time_ms(fn, steps, set_lr)
                if world > 1:
                    t = torch.tensor([ms], device=dev)
                    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
                    ms = float(t)
                res[k].append(ms)
    frames = CLIPS * T * world
    out = {}
    for k, v in res.items():
        out[k] = {"ms_per_step": [round(t, 3) for t in v], "frames_per_s": [round(frames / (t * 1e-3), 1) for t in v]}
    return out, clk.summary()


def _dp_worker(rank, world, port, runs, steps, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        out, clock = ab(dev, runs, steps, rank, world)
        if rank == 0:
            ret["dp"] = {"world": world, "result": out, "clock": clock}
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--skip-dp", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sgd.py: needs a CUDA device")
    report = {"gpu": gpu_info(0), "optimizer_alone": bench_optimizer(args.runs)}
    torch.cuda.empty_cache()
    step, clock = ab(torch.device("cuda", 0), args.runs, args.steps)
    report["step_1gpu"] = {"workload": "finetune_sgd step: %d clips x %d frames, %d ch, %dx%d, fwd + bwd + optimizer, one CUDA "
                                       "graph; torch: SGD(foreach=True, momentum 0.9, wd 1e-4, constant lr); fused: FusedSGD "
                                       "(same), lr a device tensor rewritten with the poly schedule before every replay"
                                       % (CLIPS, T, DIM, RES[0], RES[1]), "result": step, "clock": clock}
    torch.cuda.empty_cache()
    if torch.cuda.device_count() >= 2 and not args.skip_dp:
        import torch.multiprocessing as mp
        ret = mp.Manager().dict()
        mp.spawn(_dp_worker, args=(2, 29300 + os.getpid() % 200, args.runs, args.steps, ret), nprocs=2, join=True)
        report["step_2gpu_segmented"] = dict(ret).get("dp")
    else:
        report["step_2gpu_segmented"] = "not measured: %d GPU(s) visible" % torch.cuda.device_count()
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
