"""BASELINE config 3: VmambaIR SRx4 training step (fwd + L1 + bwd + gradient all-reduce + Adam), 4 images / GPU.
Reference recipe: SRGAN/options/MambaSISR15_x4.yml:26-32,60-61,78-82 (Adam 2e-4, betas .9/.99, L1, GT 256 = 4 x LQ 64, EMA 0.999),
step = MambaSISRModel.optimize_parameters (SRGAN/VmambaIR/models/MambaSISR_model.py:120-147).

The step here: forward + backward of every OSS block on this library's kernels (vmambair_b200.fused_train; bf16 activations under
autocast, fp32 parameters), captured in ONE CUDA graph; then the single collective of the path -- one flat fp32 all-reduce of the
gradients over NCCL -- and one fused Adam + EMA kernel over the flat parameter buffers (vmambair_b200.optim.FlatAdam)."""
from __future__ import annotations

import os
import time

import torch
import torch.nn.functional as F

B_PER_GPU = 4
H = W = 64


def run_train(args, build_net, ClockSampler, env_rank, dist_max, barrier, peaks, sample_clocks=True, outputs=None):
    """-> the JSON record (dict) of the training workload on this rank's GPU; the process group is the caller's.
    outputs (a dict) receives the loss of the last timed step and the parameters after it."""
    from . import archs, ops
    from .optim import FlatAdam
    rank, local, world = env_rank()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.manual_seed(0)  # same init on every rank (+ broadcast, as DDP does at construction)
    net = build_net("full").to(dev).train()
    if world > 1:
        for p in net.parameters():
            torch.distributed.broadcast(p.data, 0)
    opt = FlatAdam(net.parameters(), lr=2e-4, betas=(0.9, 0.99), eps=1e-8, weight_decay=0.0, ema_decay=0.999)
    g = torch.Generator().manual_seed(100 + rank)
    B = B_PER_GPU
    lq_host = torch.rand(B, 3, H, W, generator=g).pin_memory()
    gt_host = torch.rand(B, 3, 4 * H, 4 * W, generator=g).pin_memory()
    lq, gt = lq_host.to(dev), gt_host.to(dev)
    loss_host = torch.zeros(1).pin_memory()
    path = archs._TRAIN_PATH

    def fwd_bwd(lq_t, gt_t):
        # gradients accumulate straight into opt.flat_grad (zeroed by the optimizer kernel of the previous step)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = net(lq_t)
        loss = F.l1_loss(out.float(), gt_t)
        loss.backward()
        return loss

    # forward + loss + backward of the static-shape step captured in ONE CUDA graph; the all-reduce and the optimizer kernel follow it
    graph, static_loss = None, None
    lq_s, gt_s = lq.clone(), gt.clone()
    if os.environ.get("VMB_TRAIN_GRAPH", "1") == "1":
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    opt.flat_grad.zero_()
                    fwd_bwd(lq_s, gt_s)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            opt.check_views()
            opt.flat_grad.zero_()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss = fwd_bwd(lq_s, gt_s)
            # the replayed step must reproduce the eager one (loss and gradients) before it is trusted
            opt.flat_grad.zero_()
            graph.replay()
            torch.cuda.synchronize(dev)
            l_g, g_g = float(static_loss), opt.flat_grad.clone()
            opt.flat_grad.zero_()
            l_e = float(fwd_bwd(lq_s, gt_s))
            torch.cuda.synchronize(dev)
            rel = float((opt.flat_grad - g_g).norm() / opt.flat_grad.norm().clamp_min(1e-12))
            opt.flat_grad.zero_()
            if abs(l_g - l_e) > 1e-3 * abs(l_e) + 1e-6 or rel > 2e-2:
                raise RuntimeError(f"graph replay differs from eager: loss {l_g} vs {l_e}, grad rel diff {rel}")
        except Exception as e:  # report and fall back to the eager step (never silently)
            print(f"[train_bench] CUDA-graph capture of fwd+bwd failed, running eagerly: {type(e).__name__}: {e}", flush=True)
            graph = None
            torch.cuda.synchronize(dev)
            opt.check_views()
            opt.flat_grad.zero_()

    def step(lq_t, gt_t):
        if graph is not None:
            lq_s.copy_(lq_t, non_blocking=True)
            gt_s.copy_(gt_t, non_blocking=True)
            graph.replay()
            loss = static_loss
        else:
            loss = fwd_bwd(lq_t, gt_t)
        if world > 1:
            torch.distributed.all_reduce(opt.flat_grad)  # the single collective of the step: flat fp32 gradient sum
        opt.step(grad_scale=1.0 / world, zero_grad=True)  # Adam + EMA + gradient reset, one kernel
        return loss

    K, Wm = args.steps, max(args.warmup, 3)
    for _ in range(Wm):
        step(lq, gt)
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local) if sample_clocks else None
    if rank == 0 and sampler:
        sampler.start()
    # kernels of this library inside one step (counted on an eager pass; the gradients it leaves are cleared again)
    c0 = ops.launch_count()
    fwd_bwd(lq, gt)
    per_step_launches = ops.launch_count() - c0 + 3  # + sqsum-free Adam: update kernel, step counter (+1 memset-free)
    torch.cuda.synchronize(dev)
    opt.flat_grad.zero_()
    barrier(world)
    torch.cuda.synchronize(dev)
    s, e = torch.cuda.Event(True), torch.cuda.Event(True)
    s.record()
    for _ in range(K):
        loss = step(lq, gt)
    e.record()
    torch.cuda.synchronize(dev)
    barrier(world)
    if outputs is not None:  # before the end-to-end steps below update the parameters again
        outputs["train_loss"] = loss.detach().float().view(1).cpu()
        outputs["train_params"] = opt.flat_param.cpu()
    total_ms = dist_max(s.elapsed_time(e), world, dev)
    # collective share: the all-reduce alone, timed on the device
    ar_ms = 0.0
    if world > 1:
        a, b_ = torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        for _ in range(5):
            torch.distributed.all_reduce(opt.flat_grad)
        b_.record()
        torch.cuda.synchronize(dev)
        ar_ms = a.elapsed_time(b_) / 5
        opt.flat_grad.zero_()
    # end to end: pinned host batch -> device every step, loss read back every step
    barrier(world)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(K):
        l = step(lq_host.to(dev, non_blocking=True), gt_host.to(dev, non_blocking=True))
        loss_host.copy_(l.detach().view(1), non_blocking=True)
        torch.cuda.synchronize(dev)
    e2e_s = dist_max(time.perf_counter() - t0, world, dev)
    clocks = sampler.stop() if (rank == 0 and sampler) else None
    final_loss = float(loss_host[0])
    if not (final_loss == final_loss and abs(final_loss) < 1e6):
        raise SystemExit(f"train_bench: loss is not finite ({final_loss})")
    # roofline: scan kernels of one profiled (eager) forward + backward
    rec = []
    ops.set_timing(rec)
    fwd_bwd(lq, gt)
    torch.cuda.synchronize(dev)
    ops.set_timing(None)
    opt.flat_grad.zero_()
    peak, peak_src = peaks()
    by = {}
    for tag, nb, a, b_ in rec:
        t = by.setdefault(tag, [0, 0.0, 0])
        t[0] += nb
        t[1] += a.elapsed_time(b_)
        t[2] += 1
    fw = by.get("scan_fwd", [0, 1e-9, 0])
    bw = by.get("scan_bwd", [0, 1e-9, 0])
    value = world * B * K / (total_ms * 1e-3)
    ms_step = total_ms / K
    out = {
        "metric": "SRx4 training-step images/sec (64x64 LQ, bf16 autocast)", "value": round(value, 2), "unit": "images/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "VmambaIR full (MambaSISR6 [15,1,1,1]+15, 12.0M params) SRx4 training step: fwd + L1 + bwd + "
                               "flat gradient all-reduce + fused Adam/EMA; 4 x 3x64x64 LQ / 3x256x256 GT per GPU",
                   "global_batch": world * B, "parallelism": f"dp{world}: batch-sharded replicas, one NCCL all-reduce of {opt.n * 4 / 1e6:.1f} MB fp32 grads per step",
                   "l2": "activations of one step (>1 GB) exceed L2; no explicit flush",
                   "path": ("fused_train: forward + backward of the OSS blocks on this library's kernels" if path == "fused" else
                            "compose: torch ops + this repo's scan fwd/bwd kernels") + "; fwd+bwd " +
                           ("replayed from one CUDA graph" if graph is not None else "eager") + "; EMA (0.999) inside the optimizer kernel"},
        "e2e": {"value": round(world * B * K / e2e_s, 2), "unit": "images/s",
                "h2d_bytes_per_step": int(lq_host.numel() * 4 + gt_host.numel() * 4), "d2h_bytes_per_step": 4},
        "gpu_launches": int(per_step_launches * K),
        "collective": {"op": "all_reduce(sum) of the flat fp32 gradient buffer", "bytes": int(opt.n * 4),
                       "ms": round(ar_ms, 3), "share_of_step": round(ar_ms / ms_step, 4)},
        "loss_last": round(final_loss, 5),
        "roofline": {"kernel": "scan_bwd_kernel + scan_fwd kernels (all launches of one step)", "bound": "hbm",
                     "achieved": round((fw[0] + bw[0]) / ((fw[1] + bw[1]) * 1e-3) / 1e9, 1), "peak": peak, "peak_source": peak_src,
                     "unit": "GB/s", "frac": round((fw[0] + bw[0]) / ((fw[1] + bw[1]) * 1e-3) / 1e9 / peak, 4), "traffic": None,
                     "scan_fwd": {"launches": fw[2], "ms": round(fw[1], 3)}, "scan_bwd": {"launches": bw[2], "ms": round(bw[1], 3)},
                     "share_of_step": round((fw[1] + bw[1]) / ms_step, 3)},
        "clocks": clocks,
    }
    return out
