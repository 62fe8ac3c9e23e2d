#!/usr/bin/env python
"""Headline benchmark: one training step of the STswinCL Swin head (the window-attention hot
path, BASELINE.json north_star) on synthetic EndoVis18-shaped clips, plus the pixel contrastive
loss step (the second hot path) timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--config seg|cadis|finetune_sgd|pretrain] [--dump-outputs DIR]

Default (``--config seg`` = configs[1] of BASELINE.json: batch 8, bf16, 1 B200): a step = forward +
backward + optimizer step of ``SwinTransformerLayerv5`` (dim 512, 64x80 tokens, 4 heads, 12 blocks +
PatchMerging -- seg18/net/Ours/swin_512.py:280-327) over one batch of ``--clips`` clips x 4 frames of
OS-8 features [clips, 4, 512, 64, 80].  frames/s counts input frames (clips x 4 per step).
The other configs are the remaining BASELINE.json configs at the same boundary:

  cadis         configs[4]: the same head on CaDIS-shaped features (64x120 tokens), 4 clips per GPU
  finetune_sgd  configs[2]: the fine-tune recipe of seg18/train_CL_ft_mswin_sgd_minput.py:147-165 (SGD momentum 0.9,
                weight decay 1e-4, batch 4 per GPU) on the head
  pretrain      configs[3]: the pre-training step of pixcontrast_18/main_pretrain_swinv5.py:150-185 on the head:
                2 query passes (forward + backward) + key-encoder EMA + 6 no-grad key passes at 32x56 tokens, the fused
                symmetric pixel contrastive loss (keys all-gathered across ranks when N > 1), LARS-SGD step

Prints ONE JSON line (rank 0).  ``value`` has the inputs resident in HBM; ``e2e`` feeds the same
module from pinned HOST buffers (H2D copy every step, loss read back every step).  ``roofline``
is measured with CUDA events around every launch of the dominant kernel family during extra,
separately timed steps; ``pixloss`` is the symmetric two-call loss step of ConsistencyLoss.forward
(PixPro_swin_v5.py:584-597) at the reference batch, replayed from CUDA graphs; ``cpu_baseline`` is the CPU
oracle (a port of the reference path, see oracle/) timed on this box's host cores on a bounded sample (N=1,
rank 0 only).

``--impl reference`` times the reference's CPU path with all host threads and prints the same line with
"impl": "reference": the UNMODIFIED reference module when a copy of the reference tree is present
(``baseline/_ref`` or $STSWIN_REFERENCE_ROOT; kind "reference"), otherwise the oracle port (kind "port":
the reference is pure Python/PyTorch with no build or install step, and /root/reference does not exist
on the GPU box).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "STswin-T train frames/s at 1/2/4/8 B200; window-attn TFLOP/s vs tensor peak"
DIM, HEADS, T = 512, 4, 4
CONFIGS = {
    # name: (token grid, default clips per GPU, optimizer, description)
    "seg": ((64, 80), 8, "adam",
            "configs[1]: Swin head train step (SwinTransformerLayerv5 dim 512, 64x80 tokens, 4 heads; fwd+bwd+Adam) on "
            "EndoVis18-shaped OS-8 features, bf16"),
    "cadis": ((64, 120), 4, "adam",
              "configs[4]: Swin head train step (SwinTransformerLayerv5 dim 512, 64x120 tokens, 4 heads; fwd+bwd+Adam) on "
              "CaDIS-shaped (512x960 crop) OS-8 features, bf16"),
    "finetune_sgd": ((64, 80), 4, "sgd",
                     "configs[2]: multi-frame fine-tune recipe (train_CL_ft_mswin_sgd_minput.py:147-165: SGD momentum 0.9, "
                     "weight decay 1e-4, batch 4 per GPU) on the Swin head, 64x80 tokens, bf16"),
    "pretrain": ((32, 56), 4, "lars",
                 "configs[3]: contrastive pre-training step on the Swin head at 32x56 tokens (main_pretrain_swinv5.py:150-185): "
                 "2 query passes fwd+bwd, key-encoder EMA, 6 no-grad key passes, fused symmetric pixel contrastive loss "
                 "(256 ch, 12 classes; shared key sets all-gathered across ranks when N > 1), LARS-SGD step; bf16"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="seg", choices=sorted(CONFIGS))
    ap.add_argument("--clips", type=int, default=0, help="clips per GPU per step (default: the config's recipe)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pixloss", action="store_true", help="skip the pixel contrastive loss object")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step in a CUDA graph")
    ap.add_argument("--gelu-grad", default="q8", choices=["q8", "bf16"],
                    help="storage of the MLP's saved GELU derivative: one byte per element (default) or bf16")
    ap.add_argument("--dp", default="flat", choices=["flat", "ddp"],
                    help="N > 1: 'flat' = forward + backward replayed from CUDA graph segments whose gradient buckets are "
                         "all-reduced (NCCL, average) on a side stream while the next segment runs, then the optimizer "
                         "step; 'ddp' = torch DistributedDataParallel, eager steps")
    ap.add_argument("--wire", default="bf16", choices=["fp32", "bf16"], help="--dp flat: dtype of the gradients on the wire")
    ap.add_argument("--segments", type=int, default=4, help="--dp flat: graph segments of the backward (1 = one all-reduce)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (float32): the loss, "
                         "the head's two outputs, every parameter and its gradient (a fixed seeded sample of the large ones, "
                         "64 MB at most), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.clips <= 0:
        args.clips = CONFIGS[args.config][1]
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def __enter__(self):
        if self.index is None:
            return self
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.path or not os.path.exists(self.path):
            return out
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_BYTES = 64 << 20          # --dump-outputs: the whole dump
DUMP_OUTPUT_CAP = 1 << 22      # elements kept of the loss / head outputs
DUMP_PARAM_CAP = 1 << 14       # elements kept of each parameter, gradient and key-encoder parameter


def dump_outputs(out_dir, arrays):
    """Write each (name, tensor, cap) as ``out_dir/<name>.npy`` in float32: the whole tensor when it has at most ``cap``
    elements, else ``cap`` of them at positions drawn from a generator seeded by the name (the same positions on every
    run and every build, for a tensor of the same size)."""
    import zlib
    import numpy as np
    import torch
    nbytes = sum(4 * min(t.numel(), cap) for _, t, cap in arrays)
    if nbytes > DUMP_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {nbytes} bytes, more than {DUMP_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, t, cap in arrays:
        t = t.detach()
        if t.numel() > cap:
            gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(0, t.numel(), (cap,), generator=gen).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    print(f"bench.py: wrote {len(arrays)} arrays ({nbytes / 2 ** 20:.1f} MB) to {out_dir}", file=sys.stderr)


def reset_training_state(params, initial, opt):
    """Put ``params`` back to ``initial`` and ``opt`` back to its state before its first step, in place (a captured step
    graph reads these very tensors).  Every state tensor of FusedAdam, SGD and LARS -- moments, momentum buffers, Adam's
    device step count -- is zero before the first step.  The bf16 weight shadows are rewritten from the weights."""
    import torch
    from stswincl_b200 import optim as soptim
    with torch.no_grad():
        for p, v in zip(params, initial):
            p.copy_(v)
        for t in [v for st in opt.state.values() for v in st.values()] + [v for g in opt.param_groups for v in g.values()]:
            if torch.is_tensor(t):
                t.zero_()
    for p in params:
        if getattr(p, "_stswin_shadow", None) is not None:
            soptim.bf16_weight(p)


def workload_config(name, clips, graph=None, extra=None):
    res = CONFIGS[name][0]
    opt = {"adam": "multi-tensor Adam (stswin kernel; writes the bf16 shadow of the weights) on the 96.6M Swin-head parameters",
           "sgd": "torch.optim.SGD(momentum 0.9, weight_decay 1e-4), foreach",
           "lars": "stswincl_b200.optim.LARS(torch.optim.SGD(add_weight_decay(...), momentum 0.9)) -- fused LARS-SGD kernels"}
    cfg = {"cuda_graph": graph, "workload": CONFIGS[name][3], "clips_per_gpu": clips, "frames_per_clip": T,
           "feature_shape": [clips, T, DIM, res[0], res[1]], "optimizer": opt[CONFIGS[name][2]],
           "l2": "inputs larger than L2 (%d MB of features per step, GBs of activations touched)"
                 % (clips * T * DIM * res[0] * res[1] * 2 * (6 if name == "pretrain" else 1) // 2 ** 20)}
    if extra:
        cfg.update(extra)
    return cfg


# ----------------------------------------------------------------------------------------------
# CPU path -- cpu_baseline leg and --impl reference
# ----------------------------------------------------------------------------------------------
def _reference_root():
    for cand in (os.environ.get("STSWIN_REFERENCE_ROOT"), os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "seg18", "net", "Ours", "swin_512.py")):
            return cand
    return None


def cpu_step_factory(res):
    """One clip (4 frames) of the config's workload, fp32, forward + backward on the host cores.
    Returns (step, threads, kind, sample text)."""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    from oracle import swin_oracle as so          # checker / CPU baseline only (never on the product path)
    x = so.make_features(1, 1, T, DIM, res[0], res[1])
    g1 = so.make_features(2, 1, T, DIM, res[0], res[1]) - 0.4
    g2 = so.make_features(3, 1, T, 2 * DIM, res[0] // 2, res[1] // 2) - 0.4
    ref_root = _reference_root()
    shape = "[1,4,%d,%d,%d]" % (DIM, res[0], res[1])
    if ref_root is not None:
        os.environ["STSWIN_REFERENCE_ROOT"] = ref_root
        from oracle import ref_shims                  # arranges sys.path so the reference's own file imports unmodified
        torch.manual_seed(0)
        model = ref_shims.import_swin().SwinTransformerLayerv5(dim=DIM, input_resolution=res, num_heads=HEADS)

        def step():
            model.zero_grad(set_to_none=True)
            y1, y2 = model(x)
            loss = (y1 * g1).sum() + (y2 * g2).sum()
            loss.backward()
            return float(loss)

        return step, torch.get_num_threads(), "reference", ("1 clip (4 frames) of the same workload %s, fp32, forward+backward, "
                                                             "the unmodified reference module (%s)" % (shape, ref_root))
    params = so.make_layer_params(DIM, res, HEADS, seed=0)
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and not k.endswith("attn_mask") else v)
            for k, v in params.items()}

    def step():
        for v in leaf.values():
            if v.is_floating_point() and v.requires_grad:
                v.grad = None
        y1, y2 = so.swin_layer_v5(x, leaf, DIM, res, HEADS)
        loss = (y1 * g1).sum() + (y2 * g2).sum()
        loss.backward()
        return float(loss)

    return step, torch.get_num_threads(), "port", ("1 clip (4 frames) of the same workload %s, fp32, forward+backward, oracle "
                                                   "port of the reference (no copy of the reference tree on this box)" % shape)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    res = CONFIGS[args.config][0]
    step, threads, kind, sample = cpu_step_factory(res)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    fps = T / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # this arm steps ONE clip per step on the host cores (a bounded sample of the workload), normalised to frames/s
            "config": workload_config(args.config, 1, extra={"optimizer": "none (forward + backward only)",
                                                             "arm": "CPU, %s, %d threads" % (kind, threads)}),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# pixel contrastive loss (HP-2): the symmetric two-call step of ConsistencyLoss.forward
# ----------------------------------------------------------------------------------------------
def bench_pixloss(dev, pk, timed, n=4, sets_in_rotation=3):
    """N = 4 per GPU (main_pretrain_swinv5.py recipe), C 256, 32x56 = 1792 pixels, 5 key sets per call, 12 classes,
    six full-resolution 256x448 label maps, fp32 projector outputs with F.normalize fused in: forward + backward of both
    symmetric calls as one step, replayed from CUDA graphs.  `sets_in_rotation` independent input sets (each its own
    captured graph) are replayed round-robin so the inputs of a step are not L2-resident from the previous one."""
    import torch
    from stswincl_b200 import contrast, ops
    K, C, H, W = 12, 256, 32, 56
    graphs = []
    gen = torch.Generator(device=dev).manual_seed(7)
    for _ in range(sets_in_rotation):
        # SURVEY 8d config 4: label maps built by nearest-upsampling a random [n, 1, 8, 14] integer map (coherent blobs)
        labels = [torch.randint(0, K, (n, 1, 8, 14), generator=gen, device=dev).float()
                  .repeat_interleave(32, 2).repeat_interleave(32, 3).contiguous() for _ in range(6)]
        emb = [torch.randn(n, C, H, W, generator=gen, device=dev) for _ in range(8)]
        q1, q2 = emb[6].requires_grad_(True), emb[7].requires_grad_(True)

        def step(q1=q1, q2=q2, emb=emb, labels=labels):
            q1.grad = None; q2.grad = None
            loss = contrast.consistency_loss_tail(q1, q2, *emb[:6], *labels, K, normalize=True)
            loss.backward()
            return loss

        for _ in range(2):
            step()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        graphs.append((g, step))
    for g, _ in graphs:
        g.replay()
    ms = timed(lambda i: graphs[i % len(graphs)][0].replay(), 30)
    l0 = ops.LAUNCHES
    graphs[0][1]()
    launches = ops.LAUNCHES - l0
    prof = ops.EventProfiler()
    for g, step in graphs[:2]:
        g.replay()
        ops.set_profiler(prof)
        step()
        ops.set_profiler(None)
    fam = prof.summary()
    dense = 2.0 * 2 * 5 * 2 * (H * W) ** 2 * C * n            # fwd + bwd, 2 queries x 5 key sets
    in_bytes = 8 * n * C * H * W * 4
    out = {"workload": "ConsistencyLoss.forward tail (PixPro_swin_v5.py:584-597): 2 symmetric regression_loss calls x 5 key sets, "
                       "N=%d per GPU, C=256, 32x56 pixels, 12 classes, 6 label maps 256x448 (random 8x14 blobs, SURVEY 8d), fp32 inputs with F.normalize fused, "
                       "forward + backward, CUDA-graph replay" % n,
           "ms_per_step": ms, "dense_gflop": dense / 1e9, "tflops": dense / ms / 1e9, "peak_tflops": pk["tflops_burst"],
           "frac_of_peak": dense / ms / 1e9 / pk["tflops_burst"], "bound": "tensor (dense form)",
           "launches_per_step": launches, "host_syncs_per_step": 0, "graph": True,
           "l2": "%d input sets in rotation (%d MB of inputs, > L2)" % (sets_in_rotation, sets_in_rotation * in_bytes // 2 ** 20),
           "kernels": {}}
    for k, v in fam.items():
        d = {"ms": v["ms"] / v["launches"]}
        if k in ("pixloss_fwd", "pixloss_bwd"):
            d.update(tflops=v["work"] / v["ms"] / 1e9, frac_of_peak=v["work"] / v["ms"] / 1e9 / pk["tflops_burst"],
                     note="includes the finalize / dq-finish kernel launched by the same C-ABI call")
        else:
            d.update(gbs=v["work"] / v["ms"] / 1e6, frac_of_hbm=v["work"] / v["ms"] / 1e6 / pk["hbm_gbs"])
        out["kernels"][k] = d
    return out


# ----------------------------------------------------------------------------------------------
# GPU path
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from stswincl_b200 import contrast, ops, optim as soptim, swin
    swin.GELU_GRAD_Q8 = args.gelu_grad == "q8"

    RES, _, opt_kind, _ = CONFIGS[args.config]
    pretrain = args.config == "pretrain"
    torch.manual_seed(0)
    model = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=RES, num_heads=HEADS).to(dev)
    for blk in model.modules():
        if isinstance(blk, swin.WindowAttention):       # sigma 0.02 init is nearly a no-op bias; use a visible one
            torch.nn.init.normal_(blk.relative_position_bias_table, std=0.5)
    key_model = None
    if pretrain:
        key_model = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=RES, num_heads=HEADS).to(dev)
        key_model.load_state_dict(model.state_dict())
        for p in key_model.parameters():
            p.requires_grad_(False)
    net = model
    side = torch.cuda.Stream(device=dev)
    flat_dp = world > 1 and args.dp == "flat"
    params = list(model.parameters())
    if world > 1 and not flat_dp:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True,
                                                        bucket_cap_mb=64, broadcast_buffers=False)
    from stswincl_b200 import dist as sdist
    if world > 1:
        sdist.broadcast_parameters(params)                 # replicas start identical (DDP's constructor does the same)
    state_params = params + (list(key_model.parameters()) if key_model is not None else [])
    initial = [p.detach().clone() for p in state_params] if args.dump_outputs else None
    if opt_kind == "adam":
        opt = soptim.FusedAdam(model.parameters(), lr=3e-5)
    elif opt_kind == "sgd":
        opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, foreach=True)
    else:
        opt = soptim.LARS(torch.optim.SGD(soptim.add_weight_decay(model, 1e-5), lr=sdist.scaled_lr(1.0, args.clips, world),
                                          momentum=0.9))
    B = args.clips
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    n_seq = 6 if pretrain else 1
    x_dev = torch.relu(torch.randn(n_seq * B, T, DIM, RES[0], RES[1], generator=g, device=dev)).to(torch.bfloat16)
    if pretrain:
        K = 12
        masks = [torch.randint(0, K, (B, 1, 8, 14), generator=g, device=dev).float()
                 .repeat_interleave(8 * RES[0] // 8, 2).repeat_interleave(8 * RES[1] // 14, 3).contiguous() for _ in range(6)]
    else:
        g1 = (torch.randn(B, T, DIM, RES[0], RES[1], generator=g, device=dev) * 0.1).to(torch.bfloat16)
        g2 = (torch.randn(B, T, 2 * DIM, RES[0] // 2, RES[1] // 2, generator=g, device=dev) * 0.1).to(torch.bfloat16)

    def embed(y1, y2):
        # stand-in for the projection head (ResNet / ASPP / projector are the caller's side of the boundary, PixPro_swin_v5.py:
        # 311-330): 256 channels of the last frame's stage-1 output plus the nearest-upsampled stage-2 output are the pixel
        # embedding, un-normalised (F.normalize is fused in the loss)
        up = torch.nn.functional.interpolate(y2[:, -1, :256], size=y1.shape[-2:], mode="nearest")
        return y1[:, -1, :256] + up

    kept = {}

    def keep(loss, y1, y2):
        # --dump-outputs: hold the step's loss and head outputs (a captured graph rewrites these tensors on every replay).
        # Detached: a reference to the autograd graph would keep its AccumulateGrad nodes alive into the next step, whose
        # stream mismatch breaks the graph capture.
        if args.dump_outputs:
            kept.update(loss=loss.detach(), y1=y1.detach(), y2=y2.detach())
        return loss

    def forward_loss(x):
        if not pretrain:
            y1, y2 = net(x)
            return keep(torch.sum(y1 * g1, dtype=torch.float32) + torch.sum(y2 * g2, dtype=torch.float32), y1, y2)
        # PixPro.forward (PixPro_swin_v5.py:291-561) on the Swin head: two query passes, EMA, six no-grad key passes
        y1, y2 = net(x[:2 * B])
        pred_1, pred_2 = embed(y1[:B], y2[:B]), embed(y1[B:], y2[B:])
        with torch.no_grad():
            soptim.momentum_update(list(model.parameters()), list(key_model.parameters()), 0.99)
            k1, k2 = key_model(x)
            keys = [embed(k1[i * B:(i + 1) * B], k2[i * B:(i + 1) * B]) for i in range(6)]
        return keep(contrast.consistency_loss_tail(pred_1, pred_2, *keys, *masks, K, normalize=True, cross_rank_negatives=world > 1),
                    y1, y2)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / n

    # ------------------------------------------------------------------------------------------
    # the step.  1 GPU: forward + backward + optimizer, captured whole.  N GPUs (--dp flat): the backward is cut into
    # `--segments` autograd segments, each captured as its own CUDA graph; after a segment's replay its gradient bucket
    # (bf16 on the wire by default) is all-reduced on a side stream while the next segment runs, so only the last
    # bucket's collective is exposed (sdist.SegmentedStep).
    # ------------------------------------------------------------------------------------------
    use_graph = not args.no_graph and not (pretrain and world > 1)      # NCCL all-gather inside the loss: eager
    stepper = None
    if flat_dp and not pretrain:
        stepper = sdist.SegmentedStep(model, opt, lambda y: keep(torch.sum(y[0] * g1, dtype=torch.float32) + torch.sum(y[1] * g2, dtype=torch.float32), *y),
                                      segments=max(1, args.segments), wire_dtype=torch.bfloat16 if args.wire == "bf16" else torch.float32,
                                      use_graph=use_graph)
    flat = sdist.FlatGradients(params) if (flat_dp and stepper is None) else None

    def fwd_bwd(x):
        opt.zero_grad(set_to_none=True)
        loss = forward_loss(x)
        loss.backward()
        if flat is not None:
            flat.gather()
        return loss

    def reduce_and_update():
        if flat is not None:
            flat.all_reduce()
            flat.bind()
        opt.step()

    def step(x):
        if stepper is not None:
            return stepper.step(x)
        loss = fwd_bwd(x)
        reduce_and_update()
        return loss

    for _ in range(args.warmup):
        step(x_dev)
    launches0 = ops.LAUNCHES
    step(x_dev)
    launches_per_step = ops.LAUNCHES - launches0

    graph, static_x, static_loss = None, None, None
    if stepper is not None:
        graph = stepper if stepper.captured else None
        static_x = x_dev
    elif use_graph and (world == 1 or flat is not None):
        captured = fwd_bwd if flat is not None else step
        try:
            static_x = x_dev.clone()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    step(static_x)
            torch.cuda.current_stream().wait_stream(side)
            opt.zero_grad(set_to_none=True)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss = captured(static_x)
            graph.replay()
            if flat is not None:
                reduce_and_update()
            torch.cuda.synchronize()
        except Exception as e:                      # capture is an optimisation of the harness, not of the product
            print(f"bench.py: CUDA graph capture failed ({type(e).__name__}: {e}); timing eager steps", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
        if flat is not None:          # every rank replays, or none does
            ok = torch.tensor([1 if graph is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok) == 0:
                graph = None

    def run_step(x):
        if stepper is not None:
            return stepper.step(x)
        if graph is None:
            return step(x)
        if x is not static_x:
            static_x.copy_(x, non_blocking=True)
        graph.replay()
        if flat is not None:
            reduce_and_update()
        return static_loss

    def cur_x():
        return static_x if (graph is not None and stepper is None) else x_dev

    for _ in range(2):
        run_step(x_dev)
    # nvidia-smi is started by rank 0 only and well before the timed steps: its start-up (NVML initialisation over
    # all GPUs of the box) stalls kernel launches of every process for ~0.1-0.2 s
    with ClockSampler(local if rank == 0 else None) as clk:
        for _ in range(12):
            run_step(cur_x())
        if args.dump_outputs:
            # the last timed step starts from the seeded initial weights and a fresh optimizer, so that its inputs are the
            # same on every run: the steps before it repeat one batch, and Adam turns the reordered fp32 sums of a step into
            # weight differences that grow from step to step.  The reset itself is not timed.
            ms_step = timed(lambda i: run_step(cur_x()), args.steps - 1) * (args.steps - 1) if args.steps > 1 else 0.0
            reset_training_state(state_params, initial, opt)
            ms_step = (ms_step + timed(lambda i: run_step(cur_x()), 1)) / args.steps
        else:
            ms_step = timed(lambda i: run_step(cur_x()), args.steps)
    launches = launches_per_step * args.steps
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        # with --dp flat the optimizer reads the all-reduced gradients from the stepper's buckets, not from p.grad
        grad_of = (lambda p: stepper._view_of[id(p)]) if stepper is not None else (lambda p: p.grad)
        arrays = [(k, kept[k], DUMP_OUTPUT_CAP) for k in ("loss", "y1", "y2")]
        for n, p in model.named_parameters():
            arrays += [("param." + n, p, DUMP_PARAM_CAP), ("grad." + n, grad_of(p), DUMP_PARAM_CAP)]
        if key_model is not None:
            arrays += [("key_param." + n, p, DUMP_PARAM_CAP) for n, p in key_model.named_parameters()]
        dump_outputs(args.dump_outputs, arrays)

    # ---- end to end: pinned host features -> H2D (copy stream, double buffered) -> step -> loss.item()
    x_host = x_dev.cpu().pin_memory()
    bufs = [torch.empty_like(x_dev), torch.empty_like(x_dev)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    d2h_bytes = 4

    def prefetch(i):
        b = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            bufs[b].copy_(x_host, non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_step(i):
        b = i & 1
        if i == 0:
            prefetch(0)
        prefetch(i + 1)                      # next step's features travel while this step computes
        torch.cuda.current_stream().wait_event(ready[b])
        loss = run_step(bufs[b])
        consumed[b].record(torch.cuda.current_stream())
        return loss.item()                   # D2H read of the step's result

    for b in range(2):
        consumed[b].record(torch.cuda.current_stream())
    for i in range(max(2, args.warmup)):
        e2e_step(i)
    ms_e2e = timed(e2e_step, args.steps)

    # ---- roofline of the dominant kernel family: CUDA events around every launch (separate, eager steps).  A replay of
    # the captured step is queued in front of each, so the host stays ahead of the GPU and every event pair brackets its
    # kernel back to back with its neighbours on a GPU as warm as in the timed region.
    pk = peaks()
    prof = ops.EventProfiler()
    for _ in range(2):
        run_step(cur_x())
        ops.set_profiler(prof)
        (stepper.eager if stepper is not None else step)(x_dev)
        ops.set_profiler(None)
    fam = prof.summary()
    total_ms = sum(v["ms"] for v in fam.values()) or 1.0
    shares = {k: round(v["ms"] / total_ms, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    gsum = {"ms": fam["gemm"]["ms"] + fam["gemm_wgrad"]["ms"], "work": fam["gemm"]["work"] + fam["gemm_wgrad"]["work"],
            "launches": fam["gemm"]["launches"] + fam["gemm_wgrad"]["launches"]}
    achieved = gsum["work"] / (gsum["ms"] * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("gemm_dram_bytes_per_launch")
    roofline = {"kernel": "stswin::gemm_kernel (tcgen05 dense layers, fwd + dgrad + wgrad)", "bound": "tensor",
                "achieved": achieved, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["tflops_sustained"], "traffic": traffic, "peak_source": pk["source"] + ", sustained",
                "launches_timed": gsum["launches"], "avg_launch_ms": gsum["ms"] / gsum["launches"],
                "share_of_step": round(gsum["ms"] / total_ms, 4), "family_time_shares": shares}
    # secondary, HBM-bound: the window-attention core kernels and the row-wise / layout kernels
    for k in ("winattn_fwd", "winattn_bwd", "layernorm_fwd", "layernorm_bwd", "transpose", "copy", "adam", "ema_update", "lars_sgd_step"):
        if k in fam:
            gbs = fam[k]["work"] / (fam[k]["ms"] * 1e-3) / 1e9
            roofline[k] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                           "avg_launch_ms": fam[k]["ms"] / fam[k]["launches"]}

    # ---- "window-attn TFLOP/s vs tensor peak" (second half of the metric): the WindowAttention module (qkv Linear +
    # shifted-window core + proj Linear, SURVEY 8d: 8C^2 + 4LC FLOPs per token forward, 2x that backward) at this
    # workload's batch, stage-1 (C 512, ws 8, shift 4) and stage-2 (C 1024, ws 4, shift 2) geometry,
    # replayed from a CUDA graph and timed alone -> against the measured burst bf16 peak
    window_attn = None
    if rank == 0 and world == 1 and not pretrain:
        window_attn = {}
        for name, dim, res, ws in (("stage1", DIM, RES, 8), ("stage2", 2 * DIM, (RES[0] // 2, RES[1] // 2), 4)):
            attn = swin.WindowAttention(dim, (ws, ws), HEADS).to(dev)
            torch.nn.init.normal_(attn.relative_position_bias_table, std=0.5)
            xa = torch.relu(torch.randn(2 * B, 2, res[0] * res[1], dim, device=dev)).to(torch.bfloat16).requires_grad_(True)
            ga = (torch.randn_like(xa) * 0.1)
            geom = (res[0], res[1], HEADS, ws, ws // 2, 0.0)

            def attn_fwd_bwd():
                xa.grad = None
                attn.zero_grad(set_to_none=True)
                y = swin._AttentionFn.apply(xa, attn.relative_position_bias_table, attn.qkv.weight, attn.qkv.bias,
                                            attn.proj.weight, attn.proj.bias, geom)
                y.backward(ga)

            def attn_fwd():
                with torch.no_grad():
                    swin._AttentionFn.apply(xa, attn.relative_position_bias_table, attn.qkv.weight, attn.qkv.bias,
                                            attn.proj.weight, attn.proj.bias, geom)

            res_ms = {}
            for tag, fn in (("fwd", attn_fwd), ("fwd_bwd", attn_fwd_bwd)):
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                side2 = torch.cuda.Stream(device=dev)
                side2.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side2):
                    fn()
                torch.cuda.current_stream().wait_stream(side2)
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    fn()
                for _ in range(3):
                    gr.replay()
                res_ms[tag] = timed(lambda i: gr.replay(), 10)
            tok = 2 * B * 2 * res[0] * res[1]
            f_fwd = (8.0 * dim * dim + 4.0 * (2 * ws * ws) * dim) * tok
            window_attn[name] = {
                "tokens": tok, "gflop_fwd": f_fwd / 1e9, "fwd_ms": res_ms["fwd"], "fwd_bwd_ms": res_ms["fwd_bwd"],
                "fwd_tflops": f_fwd / res_ms["fwd"] / 1e9, "fwd_bwd_tflops": 3 * f_fwd / res_ms["fwd_bwd"] / 1e9,
                "peak_tflops": pk["tflops_burst"], "fwd_frac_of_peak": f_fwd / res_ms["fwd"] / 1e9 / pk["tflops_burst"],
                "fwd_bwd_frac_of_peak": 3 * f_fwd / res_ms["fwd_bwd"] / 1e9 / pk["tflops_burst"]}
            del attn, xa, ga

    pixloss = None
    if rank == 0 and world == 1 and not args.no_pixloss:
        pixloss = bench_pixloss(dev, pk, timed)

    # ---- the fp32-accurate mode (north_star: <= 1e-3 against the reference's fp32 run): the same head step, fp32 features,
    # 2 clips, forward + backward, eager (stated throughput of the accuracy mode, not a headline)
    fp32_mode = None
    if rank == 0 and world == 1 and not pretrain and not args.no_pixloss:
        m32 = swin.SwinTransformerLayerv5(dim=DIM, input_resolution=RES, num_heads=HEADS).to(dev)
        m32.precision = "fp32"
        x32 = torch.relu(torch.randn(2, T, DIM, RES[0], RES[1], device=dev))
        w32a, w32b = torch.randn_like(x32) * 0.1, torch.randn(2, T, 2 * DIM, RES[0] // 2, RES[1] // 2, device=dev) * 0.1

        def step32(i):
            m32.zero_grad(set_to_none=True)
            a, b = m32(x32)
            ((a * w32a).sum() + (b * w32b).sum()).backward()

        step32(0)
        ms32 = timed(step32, 3)
        fp32_mode = {"workload": "SwinTransformerLayerv5 forward + backward, 2 clips x 4 frames, fp32 features, precision='fp32' "
                                 "(split-bf16 tcgen05 GEMMs over K' = 3K, fp32 SIMT window attention, fp32 LayerNorm), eager",
                     "ms_per_step": ms32, "frames_per_s": 2 * T / (ms32 * 1e-3), "parity_bar": "1e-3 (tests/test_gpu_fp32_mode.py)"}
        del m32, x32, w32a, w32b

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cstep, threads, kind, sample = cpu_step_factory(RES)
        cstep()                                           # warm-up (page-in, thread pool)
        t0 = time.perf_counter(); cstep(); dt = time.perf_counter() - t0
        cpu = {"value": T / dt, "unit": "frames/s", "cores": threads, "kind": kind, "sample": sample, "seconds": dt}

    if rank == 0:
        frames = n_seq * B * T * world
        if world == 1:
            par = "single GPU"
        elif stepper is not None:
            par = "dp%d: %s" % (world, stepper.describe())
        elif flat is not None:
            par = "dp%d: one flat fp32 gradient all-reduce (NCCL, average) per step" % world
        else:
            par = "dp%d: torch DDP, bucketed all-reduce overlapped with backward" % world
        line = {"metric": METRIC, "value": frames / (ms_step * 1e-3), "unit": "frames/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": dict(workload_config(args.config, B, graph is not None), parallelism=par,
                               saved_activations="bf16" + ("; the MLP's GELU derivative (a multiplier in [-0.13, 1.13] that only the backward's "
                                                           "epilogue reads) as a one-byte code with step 0.005, parity tests at the unchanged "
                                                           "2e-2 bar (--gelu-grad bf16 keeps it in bf16)" if args.gelu_grad == "q8" else "")),
                "clocks": clocks,
                "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": x_host.numel() * x_host.element_size(), "d2h_bytes_per_step": d2h_bytes},
                "gpu_launches": launches, "roofline": roofline, "window_attn": window_attn, "pixloss": pixloss, "fp32_mode": fp32_mode,
                "cpu_baseline": cpu, "clips_per_s": n_seq * B * world / (ms_step * 1e-3)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: self-launch one rank per GPU (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
