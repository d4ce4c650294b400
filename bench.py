#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native OSS operator stack.

Metric (BASELINE.json): SRx4 images/sec on synthetic B x 3 x 64 x 64 LQ tiles, bf16.
Default workload (N=1): BASELINE configs[1] -- "VmambaIR-light SRx4 inference, B=8 3x64x64 LQ, bf16, 1xB200"
(VmambaIR-light = the class-default MambaSISR6 [6,2,2,1]+6, SURVEY.md 8d); `--workload train` runs configs[2]
(full SR net training step, 4 img/GPU, gradient all-reduce over NCCL).  Images shard on the batch axis: every
rank processes its own batch (weak scaling), inference has no collective.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload infer|train] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

One JSON line on rank 0.  `--impl reference` times the CPU oracle port of the reference path (oracle/),
rank 0 only, one image per step.

--dump-outputs DIR: rank 0 writes what the timed path computed in its last timed step as DIR/<name>.npy (float32), so that
two builds run with the same arguments (same seeded inputs and weights) can be compared output for output:
  sr            the SR output batch (N x 3 x 4H x 4W) of the inference engine (--impl reference: of image 0 through the oracle)
  train_loss    the L1 loss of the training step (--workload train, and the training sub-record of the default run)
  train_params  the flat fp32 parameter buffer after that step's optimizer update
Two runs of one build already differ slightly (fp32 atomics in the out_norm statistics and the backward, then bf16 storage
over 27 blocks: max |diff| of sr 0.032 between two runs on one B200 at its 1000 W limit), so compare with a tolerance.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

B_PER_GPU_INFER = 8
B_PER_GPU_TRAIN = 4
H = W = 64
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, out_dir):
    """outputs: name -> tensor; written as out_dir/<name>.npy in float32"""
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: outputs to dump ({total} bytes) exceed {DUMP_LIMIT_BYTES} bytes")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = sorted(int(float(r[1])) for r in rows if len(r) >= 8)
        reasons = set()
        for r in rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(float(rows[0][2])) if rows else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_net(kind):
    from vmambair_b200 import archs
    torch.manual_seed(0)
    if kind == "light":
        return archs.MambaSISR6()  # class default [6,2,2,1] + 6 refinement, 10.5 M params
    if kind == "derain":  # BASELINE configs[3]: Deraining/Options/Deraining_mamber33.yml:53-63
        return archs.Mamber32(num_blocks=[3, 5, 7, 9], num_refinement_blocks=2)
    if kind == "realsr":  # BASELINE configs[4]: RealSR/options/mambaSR11_x4.yml:82-92 (class default [6,2,2,1] + 6)
        return archs.MambaRealSR11()
    return archs.MambaSISR6(num_blocks=[15, 1, 1, 1], num_refinement_blocks=15)  # options/MambaSISR15_x4.yml


# --config N (1-based index into BASELINE.json configs): net, images per GPU, LQ size, oracle kind, metric, workload
CONFIGS = {
    2: dict(net=None, B=8, hw=64, kind="sisr", metric=None, workload=None),
    4: dict(net="derain", B=4, hw=256, kind="mamber32", metric="deraining images/sec (256x256, bf16)",
            workload="Deraining Mamber32 [3,5,7,9]+2 (28.7M params) inference, B=4 x 3x256x256 per GPU (level-1 scans: L = 65 536)"),
    5: dict(net="realsr", B=2, hw=128, kind="realsr", metric="RealSR x4 images/sec (128x128 LQ, bf16)",
            workload="MambaRealSR11 [6,2,2,1]+6 (10.5M params) SRx4 inference, B=2 x 3x128x128 LQ per GPU (16 images over 8 GPUs)"),
}


METRIC = "SRx4 images/sec (64x64 LQ, bf16)"  # BASELINE.json's metric; both arms print this exact string


def workload_name(net):
    return ("VmambaIR-light (MambaSISR6 [6,2,2,1]+6, 10.5M params)" if net == "light" else
            "VmambaIR full (MambaSISR6 [15,1,1,1]+15, 12.0M params)") + " SRx4 inference, B=8 x 3x64x64 LQ per GPU"


def host_threads():
    """CPU threads for the CPU arm: physical cores inside the affinity mask, capped by the cgroup quota (oracle/cscan.py)"""
    from oracle import cscan
    return cscan.host_threads()


def bench_input(rank=0):
    """the synthetic LQ batch of the bench (B_PER_GPU_INFER x 3 x 64 x 64 in [0,1]); image 0 of rank 0 is the CPU sample"""
    g = torch.Generator().manual_seed(1234 + rank)
    return torch.rand(B_PER_GPU_INFER, 3, H, W, generator=g)


def cpu_oracle_images_per_s(steps, warmup, threads=None, x=None, kind="light"):
    """The reference path on the host CPU: oracle port (oracle/oss_ref.py + C scan), one image per step.
    -> (images/s, mean seconds, output of the last forward)"""
    from oracle import oss_ref, cscan
    cscan.build()
    threads = threads or host_threads()  # torchrun would otherwise pin OMP_NUM_THREADS=1
    torch.set_num_threads(threads)
    cscan.set_threads(threads)
    net = build_net(kind)
    sd = {k: v.detach().float() for k, v in net.state_dict().items()}
    if x is None:
        x = bench_input(0)[:1]
    ts = []
    y = None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            y = oss_ref.net_forward(sd, x.float(), "sisr")
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    mean = sum(ts) / len(ts)
    return 1.0 / mean, mean, y


def run_reference(args, outputs=None):
    rank, _, world = env_rank()
    if rank != 0:
        return
    cores = os.cpu_count()
    ips, mean, y = cpu_oracle_images_per_s(args.steps, args.warmup, kind=args.net)
    if outputs is not None:
        outputs["sr"] = y
    out = {
        "impl": "reference", "metric": METRIC, "value": round(ips, 4), "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(mean * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.net),
                   "sample": "bounded sample: 1 image of the batch per step through the CPU oracle port of the reference path"},
        "cpu_baseline": {"value": round(ips, 4), "unit": "images/s", "cores": torch.get_num_threads(), "host_cores": cores,
                         "affinity_cores": host_threads(),
                         "kind": "port", "sample": "full VmambaIR-light forward of one 3x64x64 image per step (fp32 arithmetic: the reference has no bf16 CPU path; oracle/oss_ref.py + OpenMP C scan)"},
        "e2e": {"value": round(ips, 4), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def dist_max(x, world, device):
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        torch.distributed.barrier()


def run_infer(args, outputs=None):
    from vmambair_b200 import ops
    from vmambair_b200.engine import InferenceEngine
    rank, local, world = env_rank()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    cfg = CONFIGS[args.config]
    B, H, W = cfg["B"], cfg["hw"], cfg["hw"]
    net_kind = cfg["net"] or args.net
    chains = int(os.environ.get("VMB_CHAINS", "1"))
    lowres = int(os.environ.get("VMB_LOWRES_CHAINS", "1"))
    eng = InferenceEngine(build_net(net_kind), B, H, W, dtype=torch.bfloat16, device=dev, chains=chains, lowres_chains=lowres)
    if args.config == 2:
        x_host = bench_input(rank).to(torch.bfloat16).pin_memory()
    else:
        x_host = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(1234 + rank)).to(torch.bfloat16).pin_memory()
    eng.x_dev.copy_(x_host)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    K, Wm = args.steps, max(args.warmup, 3)
    for _ in range(Wm):
        eng.step_device()
    torch.cuda.synchronize(dev)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- device-resident timing: K steps, L2 flushed between steps, CUDA events on the launching stream ----
    evs = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(K)]
    barrier(world)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(eng.stream):
        for s, e in evs:
            flush.zero_()
            s.record(eng.stream)
            eng.step_device()
            e.record(eng.stream)
    torch.cuda.synchronize(dev)
    barrier(world)
    if outputs is not None:
        outputs["sr"] = eng.y_dev.float().cpu()  # the last timed step's result, before the end-to-end runs below
    step_ms = [s.elapsed_time(e) for s, e in evs]
    total_ms = dist_max(sum(step_ms), world, dev)
    # ---- end-to-end through the public API: pinned host -> device -> net -> host, every step ----
    for _ in range(2):
        eng.run(x_host)
    barrier(world)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(K):
        y = eng.run(x_host)
    torch.cuda.synchronize(dev)
    e2e_s = dist_max(time.perf_counter() - t0, world, dev)
    clocks = sampler.stop() if rank == 0 else None
    # ---- roofline of the dominant kernel (selective scan fwd): per-launch CUDA events over eager steps ----
    rec = []
    y_bench = eng.run(x_host).float().clone()  # result of the benchmarked engine: sanity / parity check below
    if not bool(torch.isfinite(y_bench).all()):
        raise SystemExit("bench.py: the benchmarked forward produced non-finite values")
    eager = InferenceEngine(build_net(net_kind), B, H, W, dtype=torch.bfloat16, device=dev, use_graph=False)
    eager.x_dev.copy_(x_host)
    eager.step_device()
    torch.cuda.synchronize(dev)
    ops.set_timing(rec)
    for _ in range(3):
        flush.zero_()
        eager.step_device()
    torch.cuda.synchronize(dev)
    ops.set_timing(None)
    tot_b = sum(r[1] for r in rec if r[0] == "scan_fwd")
    tot_ms = sum(r[2].elapsed_time(r[3]) for r in rec if r[0] == "scan_fwd")
    big = [(r[1], r[2].elapsed_time(r[3])) for r in rec if r[0] == "scan_fwd"]
    top_b = max(b for b, _ in big)
    top = [(b, t) for b, t in big if b == top_b]
    peak, peak_src = peaks()
    ach = sum(b for b, _ in top) / (sum(t for _, t in top) * 1e-3) / 1e9
    ms_per_step = total_ms / K
    value = world * B * K / (total_ms * 1e-3)
    out = {
        "metric": cfg["metric"] or METRIC, "value": round(value, 2), "unit": "images/s", "n_gpus": world,
        "steps": K, "warmup": Wm, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "lq_mpix_per_s": round(value * H * W / 1e6, 3),
        "config": {"workload": cfg["workload"] or workload_name(args.net),
                   "global_batch": world * B, "parallelism": f"batch-sharded x{world}, no collective",
                   "l2": "256 MiB memset between timed steps", "graph": f"CUDA graph replay, {chains} whole-net sub-batch chains, levels below full resolution on {lowres} parallel sub-batch branches",
                   "path": f"fused OSS kernels ({eng.launches_per_step} launches of this library per step)" if eng.launches_per_step else "compose"},
        "e2e": {"value": round(world * B * K / e2e_s, 2), "unit": "images/s",
                "h2d_bytes_per_step": int(x_host.numel() * x_host.element_size()),
                "d2h_bytes_per_step": int(y.numel() * y.element_size())},
        "gpu_launches": int(eng.launches_per_step * K),
        "roofline": {"kernel": f"scan_fwd_tma_kernel (largest scan of the step, {top_b / 1e6:.1f} MB of operands; config 2: u (8,384,4096) bf16)", "bound": "hbm",
                     "achieved": round(ach, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": round(ach / peak, 4),
                     # dram__bytes_* of this launch are not measurable outside ncu: null here, the committed capture is cited
                     "traffic": None, "traffic_cited": "profiles/ncu_scan_fwd_r2.txt (ncu --set full of this kernel inside this command)",
                     "algorithmic_bytes_per_launch": int(top_b),
                     "all_scans_per_step": {"launches": len(big) // 3, "GB": round(tot_b / 3 / 1e9, 4),
                                            "ms": round(tot_ms / 3, 4), "share_of_step": round(tot_ms / 3 / ms_per_step, 3)},
                     "note": "not HBM-bound at bf16 I/O: the MUFU (ex2), LDS and SHFL instructions of a warp queue on one path (tools/microbench.cu, profiles/scan_fwd_r2.md)"},
        "clocks": clocks,
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and args.config == 2:
            ips, mean, y_ref = cpu_oracle_images_per_s(steps=2, warmup=1, x=x_host[:1], kind=args.net)
            out["cpu_baseline"] = {"value": round(ips, 4), "unit": "images/s", "cores": torch.get_num_threads(),
                                   "host_cores": os.cpu_count(), "kind": "port",
                                   "sample": f"2 timed forwards of image 0 of the bench batch (3x64x64), fp32 CPU oracle port ({mean:.2f} s each)"}
            # the benchmarked bf16 result against the fp32 oracle on the same image (bound of tests/test_bench_parity_gpu.py)
            err = (y_bench[:1].cpu() - y_ref).abs()
            out["parity"] = {"vs": "oracle/oss_ref.net_forward (fp32) on image 0", "max_abs_err": round(float(err.max()), 5),
                             "mean_abs_err": round(float(err.mean()), 6), "bound": {"max": 0.5, "mean": 0.05},
                             "note": "the oracle itself evaluated with bf16 storage is 0.028 mean / 0.18 max off its fp32 result on this net (tests/test_bench_parity_gpu.py)"}
            if float(err.max()) > 0.5 or float(err.mean()) > 0.05:
                raise SystemExit(f"bench.py: benchmarked output off the oracle: {out['parity']}")
    del eng, eager
    torch.cuda.empty_cache()
    return out


def train_record(args, outputs=None):
    """BASELINE configs[2] (the training step: the one path with a collective) as a sub-record of the default line, so a
    1 -> 8 GPU sweep carries a training-scaling curve next to the collective-free inference one."""
    from vmambair_b200.train_bench import run_train
    a = argparse.Namespace(**vars(args))
    a.warmup = 3
    t = run_train(a, build_net, ClockSampler, env_rank, dist_max, barrier, peaks, sample_clocks=False, outputs=outputs)
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "config", "e2e", "gpu_launches",
            "collective", "loss_last", "roofline")
    return {k: t[k] for k in keep}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="infer", choices=["infer", "train"])
    ap.add_argument("--net", default="light", choices=["light", "full"],
                    help="inference net: light = class-default MambaSISR6 [6,2,2,1]+6 (BASELINE configs[1]); full = the YAML's "
                         "[15,1,1,1]+15 (SURVEY.md 8d asks for both)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step sub-record of the default run")
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5],
                    help="1-based index into BASELINE.json configs: 2 = VmambaIR-light SRx4 inference (default, the metric's config), "
                         "4 = deraining 4 x 3x256x256, 5 = RealSR 2 x 3x128x128 per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last timed step as DIR/<name>.npy, float32 (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    outputs = {} if args.dump_outputs else None
    if args.impl == "reference":
        run_reference(args, outputs)
        if outputs:
            dump_outputs(outputs, args.dump_outputs)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path); use --impl reference for the CPU oracle")
    rank, local, world = env_rank()
    if world > 1:
        torch.cuda.set_device(local)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        if args.workload == "train":
            from vmambair_b200.train_bench import run_train
            out = run_train(args, build_net, ClockSampler, env_rank, dist_max, barrier, peaks, outputs=outputs)
        else:
            out = run_infer(args, outputs)
            if not args.no_train and args.config == 2:
                out["train"] = train_record(args, outputs)
        if rank == 0:
            print(json.dumps(out), flush=True)
            if outputs is not None:
                dump_outputs(outputs, args.dump_outputs)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
