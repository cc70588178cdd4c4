#!/usr/bin/env python
"""bench.py -- pose projections/s (forward + analytic d(dist)/d(pose) + step) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): a batch of 65 536 synthetic
21x4 quaternion poses PER GPU (weak scaling), random-init configs/amass.yaml weights (lrelu, "sensitised"
init so that d > 0, SURVEY 8d), one projection step x <- x - d * dd/dx per "step"
(/root/reference/experiments/sample_poses.py:71-74).  With N > 1 every step ends with the gather of the
projected poses that the north star puts at the end of a projection run (posendf_b200/dist.py::PeerGather: the
kernel's own write-back stores every projected tile into all peers' gathered buffers over NVLink, NCCL all-gather
as the fallback -- `config.gather` says which ran).

One JSON line on stdout (rank 0).  `value` = poses of all ranks / max-over-ranks device time, inputs resident in
HBM, L2 flushed between timed steps.  `e2e` = the same step from / to pinned HOST buffers with the copies (and, for
N > 1, the gather) inside the timed region.  `roofline` reports the kernel against the fp32-FMA pipe (the binding
one: 8 060 flop per compulsory HBM byte, SURVEY Appx C): nominal 148 SM x 128 lanes x 2 x max SM clock as `peak`,
the in-process FFMA2 micro-benchmark next to it; `roofline_hbm` is the north-star-mandated HBM fraction.
`configs` carries the other BASELINE.json configurations at this GPU count (C3 50-step projection + ONE gather,
C4 motion-denoise loop, C5 data-parallel train step).  `cpu_baseline` / `--impl reference` time the REFERENCE's own
PoseNDF (oracle/_ref, an unmodified copy made by oracle/make_ref.py) on the host cores -- the only places that
touch oracle/.

`--dump-outputs DIR` (rank 0) writes what the last timed step returned to its caller: the gathered projected poses
(DIR/projected_poses.npy, float32 [world*B, 21, 4]) and their distances (DIR/dist.npy, float32 [world*B, 1]).  Weights
and poses are seeded, so two builds run with the same arguments can be compared output for output.  Above
DUMP_BUDGET_BYTES the same fixed, seeded subset of poses is kept in both files (sorted pose order).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

BATCH_PER_GPU = 65536
FLOPS_PER_PROJECTION = 5_450_416      # SURVEY 8(d): 2*MAC, forward + input gradient
BYTES_PER_PROJECTION = 676            # 336 in + 336 out + 4 dist
WEIGHT_SEED, POSE_SEED = 1, 1234
DUMP_BUDGET_BYTES, DUMP_SAMPLE_SEED = 60 << 20, 0      # array bytes: the .npy files, headers included, stay under 64 MB
METRIC = "pose projections/s (fwd+grad+step)"
UNIT = "poses/s"
WORKLOAD = "configs[1]: 65 536-pose forward + d(dist)/d(pose) projection step per GPU, amass.yaml lrelu"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

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
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx, pw = [], set(), None, []
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2]); pw.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw) if pw else None)
        return out


def host_threads():
    """threads this process can really use: min(affinity mask, cgroup cpu quota) -- on the GPU box os.cpu_count()
    says 128 while the container's cgroup grants 16 CPUs; oversubscribing them makes torch ~10x slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


# ------------------------------------------------------------------------------------------------ reference arm
def reference_step_fn(threads):
    """One projection step of the reference on the host cores: the loop body of experiments/sample_poses.py:70-74
    (net(pose, train=False) -> gradient(pose, dist_pred) -> pose - dist*grad) on the reference's OWN PoseNDF module
    (oracle/_ref: unmodified copy, oracle/make_ref.py) with configs/amass.yaml and the bench's synthetic weights.
    Falls back to the oracle's torch port of the same operator sequence when oracle/_ref did not travel."""
    from posendf_b200 import synth
    torch.set_num_threads(threads)
    params = synth.make_params(WEIGHT_SEED)
    try:
        from oracle import make_ref
        PoseNDF, gradient, _ = make_ref.load_reference()
        net = PoseNDF(make_ref.amass_opt("cpu"))
        net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
        net.eval()

        def step(x):
            x = x.detach().requires_grad_(True)
            pred = net(x, train=False)
            g = gradient(x, pred["dist_pred"]).reshape(-1, 84)
            return (x - (pred["dist_pred"] * g).reshape(-1, 21, 4)).detach()

        return step, "reference", "reference PoseNDF (oracle/_ref, unmodified model/posendf.py + model/network/*)"
    except Exception as e:      # noqa: BLE001 -- the fallback is reported, never silent
        from oracle import posendf_torch as otorch
        from oracle.posendf_numpy import default_cfg
        tp = otorch.to_torch_params(params, torch.float32)
        cfg = default_cfg()
        return (lambda x: otorch.project_step(tp, x, cfg)[0]), "port", f"oracle torch port (oracle/_ref unavailable: {e})"


def cpu_reference_rate(batch, budget_s, threads):
    """best poses/s of the reference step over as many repetitions of a `batch`-pose step as fit in ~budget_s seconds
    (at least 2, at most 8)"""
    from posendf_b200 import synth
    step, kind, what = reference_step_fn(threads)
    x = torch.from_numpy(synth.make_poses(POSE_SEED, batch))
    step(x[: min(batch, 2048)])      # warm-up
    times = []
    t_start = time.perf_counter()
    while len(times) < 2 or (len(times) < 8 and time.perf_counter() - t_start < budget_s):
        t0 = time.perf_counter()
        step(x)
        times.append(time.perf_counter() - t0)
    return batch / min(times), times, kind, what


def run_reference(args, rank, world):
    """reference arm: the reference's CPU implementation on all host threads, the SAME configuration as our arm
    (65 536 poses per step).  Under torchrun rank 0 alone runs it."""
    if rank != 0:
        return
    from posendf_b200 import synth
    threads = host_threads()
    B = args.batch
    step, kind, what = reference_step_fn(threads)
    x = torch.from_numpy(synth.make_poses(POSE_SEED, B))
    for _ in range(max(1, min(args.warmup, 2))):
        step(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(x)
    dt = time.perf_counter() - t0
    rate = B * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "same_config": B == BATCH_PER_GPU,
                   "note": f"{what}; torch {torch.__version__} CPU, {threads} threads; ONE CPU process regardless of --gpus"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{args.steps} steps x {B} poses (forward + autograd grad + x - d*g)"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ other BASELINE configs
def _ev():
    return torch.cuda.Event(enable_timing=True)


def _max_over_ranks(ms, dev, world):
    import torch.distributed as dist
    t = torch.tensor([float(ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item()


def run_other_configs(eng, dev, rank, world, gather):
    """C3 / C4 / C5 of BASELINE.json at per-GPU shard sizes (weak scaling over the ranks of this launch); device time,
    max over ranks.  Returns the dict that goes under "configs" in the JSON line."""
    import torch.distributed as dist
    from posendf_b200 import PoseNDF, synth
    from posendf_b200.dist import DataParallelStep
    out = {}
    sync = (lambda: (dist.barrier() if world > 1 else None, torch.cuda.synchronize(dev)))

    # ---- C3: 50-step projection (experiments/sample_poses.py:70-74 with K = 50), 131 072 poses per GPU, ONE launch, then
    # ONE gather of the projected poses (no per-step communication)
    B3, K3 = 131072, 50
    x0 = torch.from_numpy(synth.make_poses(77 + rank, B3)).to(dev)
    g3 = gather(B3)
    x = g3.local_view()
    x.copy_(x0); g3.project_and_gather(eng, steps=2); sync()
    x.copy_(x0); a, b = _ev(), _ev()
    sync(); a.record(); g3.project_and_gather(eng, steps=K3); b.record(); sync()
    ms = _max_over_ranks(a.elapsed_time(b), dev, world)
    out["C3_projection_50_steps"] = {"poses_per_gpu": B3, "poses_total": B3 * world, "steps": K3, "ms": ms, "launches_per_gpu": 1,
                                     "pose_steps_per_s": world * B3 * K3 / ms * 1e3, "projected_poses_per_s": world * B3 / ms * 1e3,
                                     "gather": g3.kind + ", once after the 50 steps"}
    del g3, x, x0

    # ---- C4: motion denoise prior loop (experiments/motion_denoise.py:70-99), 128 sequences x 300 frames per GPU, 100 Adam steps
    S, T = 128, 300
    aa0 = torch.from_numpy(synth.make_axis_angle(2 + rank, S * T)).to(dev).reshape(S, T, 63).contiguous()
    aa = aa0.clone(); eng.denoise_prior_(aa, iterations=1, steps_per_iter=2); sync()
    aa = aa0.clone(); l0 = eng.launch_count(); a, b = _ev(), _ev()
    sync(); a.record(); eng.denoise_prior_(aa, iterations=2, steps_per_iter=50); b.record(); sync()
    ms = _max_over_ranks(a.elapsed_time(b), dev, world)
    out["C4_denoise_100_adam_steps"] = {"sequences_per_gpu": S, "frames": T, "steps": 100, "ms": ms,
                                        "kernel_launches_per_gpu": int(eng.launch_count() - l0),
                                        "graph_launches_per_gpu": 0 if eng.tile_for_batch(S * T) == 128 else 1,
                                        "note": ("tensor-core engine: ONE chain of 15 kernels per Adam step (the update of step t-1 in the "
                                                 "prologue of the first one) + the last update, plain launches (the host stays ahead)"
                                                 if eng.tile_for_batch(S * T) == 128 else
                                                 "two sequence groups = two parallel launch chains inside ONE CUDA graph"),
                                        "pose_steps_per_s": world * S * T * 100 / ms * 1e3, "sequences_per_s": world * S / ms * 1e3}
    del aa, aa0

    # ---- C5: data-parallel trainer step (model/train_posendf.py:93-99): 32 768 + 32 768 samples per GPU, dist + manifold +
    # Eikonal losses, gradient all-reduce, Adam(lr 1e-5, weight_decay 1e-4)
    B5 = 32768
    opt = {"train": {"device": str(dev), "loss_type": "l1", "batch_size": 4},
           "model": {"StrEnc": {"use": True, "act": "lrelu", "beta": 100},
                     "DFNet": {"in_dim": 126, "dims": [256, 512, 1024, 512, 256, 64], "act": "lrelu", "beta": 100}}}
    net = PoseNDF(opt)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_params(WEIGHT_SEED).items()})
    trainer = DataParallelStep(net, lr=1e-5, weight_decay=1e-4, weights=(1.0, 1.0, 1.0))
    tp = torch.from_numpy(synth.make_poses(11 + rank, B5, kind="noisy", sigma=0.25)).to(dev)
    tm = torch.from_numpy(synth.make_poses(211 + rank, B5)).to(dev)
    tgt = torch.from_numpy((synth.uniform01(411 + rank, B5) * 0.5).astype(np.float32)).to(dev)
    for _ in range(3):
        trainer.step(tp, tgt, tm)
    n5 = 5
    a, b = _ev(), _ev()
    sync(); a.record()
    for _ in range(n5):
        ld = trainer.step(tp, tgt, tm)
    b.record(); sync()
    ms = _max_over_ranks(a.elapsed_time(b) / n5, dev, world)
    out["C5_train_step"] = {"samples_per_gpu": B5, "manifold_samples_per_gpu": B5, "batch_total": world * B5, "ms_per_step": ms,
                            "samples_per_s": world * B5 / ms * 1e3, "optimizer": trainer.kind,
                            "losses_rank0": {k: float(v.detach()) for k, v in ld.items()}}
    return out


def dump_outputs(out_dir, arrays):
    """write {name: array, poses on axis 0} as out_dir/<name>.npy; above DUMP_BUDGET_BYTES every array keeps the same fixed,
    seeded subset of poses"""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    keep = DUMP_BUDGET_BYTES // sum(a.nbytes // n for a in arrays.values())
    rows = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(n, keep, replace=False)) if n > keep else slice(None)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows])


# ------------------------------------------------------------------------------------------------ main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="poses per GPU (default: the BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 legs")
    ap.add_argument("--gather", default="auto", choices=["auto", "peer", "nccl"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's projected poses and distances as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from posendf_b200 import synth
    from posendf_b200.dist import make_gather
    from posendf_b200.engine import Engine, fp32_peak_tflops

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch

    eng = Engine(device=local_rank)
    eng.set_weights_flat(synth.flatten_params(synth.make_params(WEIGHT_SEED)))
    poses_host = torch.from_numpy(synth.make_poses(POSE_SEED + rank, B)).pin_memory()
    x0 = poses_host.to(dev)
    gather = lambda n: make_gather(n, dev, prefer=args.gather)      # noqa: E731
    G = gather(B)                      # gathered (world*B, 21, 4) buffer; this rank's slice is where the kernel works in place
    x = G.local_view()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def step():
        G.project_and_gather(eng, steps=1)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # the clock sampler (an nvidia-smi process polling every 100 ms) starts BEFORE the warm-up: its start-up must not fall into
    # the timed region
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        x.copy_(x0)
        flush.fill_(0)
        step()
    sync_all()

    # ---- timed region: exactly K steps, device time per step, L2 flushed between steps
    ev = [(_ev(), _ev()) for _ in range(args.steps)]
    launches0 = eng.launch_count()
    sync_all()
    for i in range(args.steps):
        x.copy_(x0)
        flush.fill_(i & 0xFF)
        ev[i][0].record()
        step()
        ev[i][1].record()
    sync_all()
    launches = eng.launch_count() - launches0
    ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = _max_over_ranks(sum(ms), dev, world)
    if args.dump_outputs and rank == 0:      # before the e2e loop, which reuses x when N > 1
        dump_outputs(args.dump_outputs, {"projected_poses": G.poses.cpu().numpy(), "dist": G.dist.cpu().numpy()})

    # ---- kernel-only time (no gather) for the roofline, same flush discipline: the path the library picks for this batch
    # (tensor-core DFNet, "tile 128") and the fused fp32-FMA kernel (tile 32) next to it
    def kernel_only(tile):
        eng.set_tile_policy(tile)
        kms = []
        xk = x0.clone()
        for i in range(min(args.steps, 10) + 1):
            xk.copy_(x0)
            flush.fill_(i & 0xFF)
            a, b = _ev(), _ev()
            a.record(); eng.project_(xk, steps=1); b.record()
            torch.cuda.synchronize(dev)
            kms.append(a.elapsed_time(b))
        eng.set_tile_policy(0)
        return float(np.mean(kms[1:]))
    path_tile = eng.tile_for_batch(B)
    kernel_ms = kernel_only(0)
    ffma_ms = kernel_only(32) if path_tile == 128 else kernel_ms

    # ---- e2e: pinned HOST buffers in and out, copies (and for N > 1 the gather) inside the timed region
    out_host = torch.empty_like(poses_host).pin_memory()
    dist_host = torch.empty(B, 1).pin_memory()
    if world == 1:
        e2e_api = "pndf_project_host (pinned host buffers, chunked H2D/kernel/D2H overlap inside the library)"

        def e2e_step():
            eng.project_host(poses_host, steps=1, out=out_host, dist_out=dist_host)     # synchronous call
    else:
        e2e_api = ("pinned host shard -> H2D -> PoseNDF projection + gather of all ranks' projected poses (" + G.kind +
                   ") -> D2H of this rank's projected shard + distances")

        def e2e_step():
            x.copy_(poses_host, non_blocking=True)
            d = G.project_and_gather(eng, steps=1)
            out_host.copy_(x, non_blocking=True)
            dist_host.copy_(d, non_blocking=True)
            torch.cuda.synchronize(dev)
    for _ in range(2):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = _max_over_ranks(time.perf_counter() - t0, dev, world)
    e2e_rate = world * B * e2e_steps / e2e_s
    clocks = sampler.stop()      # sampled across the timed steps, the kernel-only loop and the e2e loop

    configs = None
    if not args.no_configs and B == BATCH_PER_GPU:
        configs = run_other_configs(eng, dev, rank, world, gather)

    if rank == 0:
        peaks, peak_src = measured_peaks()
        p_ffma = fp32_peak_tflops(local_rank, 0)
        p_ffma2 = max(fp32_peak_tflops(local_rank, 1), fp32_peak_tflops(local_rank, 5))   # two operand orders, best one
        sm_max = float(clocks.get("sm_max_mhz") or peaks.get("sm_max_mhz") or 1965.0)
        p_nominal = eng.num_sms() * 128 * 2 * sm_max * 1e6 / 1e12
        rate = world * B * args.steps / (total_ms * 1e-3)
        k_rate = B / (kernel_ms * 1e-3)
        ach_tf = B / (ffma_ms * 1e-3) * FLOPS_PER_PROJECTION / 1e12          # the fp32-FMA kernel
        ach_gbs = k_rate * BYTES_PER_PROJECTION / 1e9
        tc = path_tile == 128
        tf32_peak = float(peaks.get("bf16_tflops", 1590.0)) / 2.0            # dense tf32 = half the measured dense bf16 rate
        tc_alg_tf = k_rate * FLOPS_PER_PROJECTION / 1e12                     # algorithmic (fp32-equivalent) flops of the step
        traffic_tc, gemm_share = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic_tc.json")) as f:
                tj = json.load(f)
            traffic_tc, gemm_share = tj.get("dram_bytes_per_step"), tj.get("gemm_share")
        except Exception:
            pass
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "ms_steps_rank0": [round(t, 4) for t in ms],
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": world * B,
                       "weights": "random-init amass.yaml, sensitised (SURVEY 8d)",
                       "l2": "256 MiB flush write between timed steps", "parallelism": f"pose-sharded x{world}",
                       "gather": G.kind if world > 1 else "none (1 GPU)",
                       "path": ("tensor-core DFNet (3xTF32 tcgen05 GEMM chain, pndf_tc.cu)" if path_tile == 128
                                else f"fused fp32-FMA kernel, {path_tile}-pose tiles")},
            "roofline": ({"bound": "tensor", "achieved": 3.0 * tc_alg_tf, "peak": tf32_peak, "unit": "TFLOP/s",
                          "frac": 3.0 * tc_alg_tf / tf32_peak, "traffic": traffic_tc,
                          "kernel": "tc_gemm_kernel: 12 of the 15 launches of a step (6 forward + 6 reverse DFNet layers)"
                                    + (", %.0f %% of the step's device time in the ncu launch list (profiles/ncu_tc_path_r02.json)"
                                       % (100.0 * gemm_share) if gemm_share else ""),
                          "kernel_ms": kernel_ms, "achieved_fp32_equivalent": tc_alg_tf,
                          "gemm_kernels_only": ({"ms": kernel_ms * gemm_share, "achieved": 3.0 * tc_alg_tf / gemm_share,
                                                 "frac": 3.0 * tc_alg_tf / gemm_share / tf32_peak,
                                                 "note": "the step's CUDA-event time x the GEMM kernels' share of it in the ncu launch "
                                                         "list; all algorithmic flops of the step are GEMM flops"}
                                                if gemm_share else None),
                          "frac_algorithmic_of_bf16_peak": tc_alg_tf / float(peaks.get("bf16_tflops", 1590.0)),
                          "peak_source": peak_src + ": dense bf16 %.1f TFLOP/s (burst) / 2 = dense tf32; `achieved` counts the tf32 MMA "
                                         "flops actually issued = 3 x the algorithmic flops (3xTF32 split: hi*hi + lo*hi + hi*lo); the "
                                         "denominator is the whole step (encoder / head kernels included)" % float(peaks.get("bf16_tflops", 1590.0)),
                          "algorithmic_flops_per_pose": FLOPS_PER_PROJECTION} if tc else None),
            "roofline_fp32_path": {"bound": "fp32_fma", "achieved": ach_tf, "peak": p_nominal, "unit": "TFLOP/s", "frac": ach_tf / p_nominal,
                         "traffic": traffic, "kernel": "pndf_fused_kernel<1> (the fused fp32-FMA kernel, tile policy 32; what runs for "
                                                        "training / small batches)", "kernel_ms": ffma_ms,
                         "peak_source": "nominal fp32 FMA: %d SMs x 128 lanes x 2 x %.0f MHz (tensor cores unused: fp32 parity bar 1e-5)"
                                        % (eng.num_sms(), sm_max),
                         "peak_measured_ffma2": p_ffma2, "frac_of_measured": ach_tf / max(p_ffma, p_ffma2),
                         "peak_measured_source": "in-process micro-benchmark pndf_fp32_peak (scalar FFMA %.1f, packed FFMA2 %.1f TFLOP/s)"
                                                 % (p_ffma, p_ffma2),
                         "algorithmic_flops_per_pose": FLOPS_PER_PROJECTION},
            "roofline_hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": ach_gbs / peaks["hbm_gbs"], "peak_source": peak_src + " (of measured)",
                             "algorithmic_bytes_per_pose": BYTES_PER_PROJECTION,
                             "note": "north-star figure; the path is 8 060 flop/byte, i.e. FMA-bound not HBM-bound (SURVEY Appx C)"},
            "e2e": {"value": e2e_rate, "unit": UNIT, "h2d_bytes_per_step": B * 336, "d2h_bytes_per_step": B * 336 + B * 4,
                    "api": e2e_api},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if line["roofline"] is None:
            line["roofline"] = line["roofline_fp32_path"]
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            cpu_rate, times, kind, what = cpu_reference_rate(16384, 20.0, threads)
            line["cpu_baseline"] = {"value": cpu_rate, "unit": UNIT, "cores": threads, "kind": kind,
                                    "sample": f"{what}: {len(times)} x 16 384 poses of the same step (forward + autograd grad + "
                                              f"x-d*g), best of {len(times)}, {sum(times):.1f} s CPU, torch {torch.__version__}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
