"""bench.py — frames/s of the UniPose forward hot path on synthetic MPII-shaped input (BASELINE.json config 2:
MPII 384x384, 16 joints, batch 32 per GPU, fp16) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--precision fp16|bf16|fp32]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  A "step" is one forward pass of one batch (32 frames per GPU); the batch dimension
shards across ranks with no data-path collective (weak scaling).
  value        frames/s with the input resident in HBM (CUDA graph of the whole network, L2 flushed between steps)
  e2e          the same through the reference-facing call `model(input)` with the batch coming from pinned host
               memory and the heat-maps going back to pinned host memory every step
  parity       what was timed, checked: the heat-maps of the timed configuration against the CPU oracle on the first
               images (max-norm relative error, arg-max agreement on safe-margin joints, PCKh@0.5 of the timed
               heat-maps scored against the oracle's)
  parity_mode  the same network in the fp32-grade (bf16x3 split) mode that meets the 1e-3 north-star bound: its
               own ms/step, frames/s and error
  roofline     the WASP block alone (the graded block, SURVEY.md 8d)
  train        BASELINE.json configs[2] per-GPU shape (384x384, batch 32, bf16, fwd + MSE + bwd + NCCL gradient
               all-reduce + Adam): ms/step, frames/s and how much of the all-reduce is hidden under the backward
  cpu_baseline the reference's eager graph on the host cores (N=1 only)
`--impl reference` times the reference's own CPU eager path (oracle/_ref: the reference modules compiled to
byte-code; falls back to the oracle port when absent) on the host cores, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "frames/sec MPII 384x384 bs32 forward (UniPose ResNet-101+WASP+decoder)"
UNIT = "frames/s"
WASP_FLOPS_PER_IMG = 3.625e9        # SURVEY.md §8(d): 1.8125 GMAC nominal @24x24
WASP_MIN_BYTES_C2 = 91.4e6          # SURVEY.md §8(d): minimal fused bytes, batch 32, 2 B/elt
WASP_LAYERWISE_BYTES_C2 = 355.6e6   # SURVEY.md 8(d): layer-by-layer bytes of the block at config 2
# MMAC/img actually issued at 24x24 when whole-tile out-of-image taps are skipped and conv2 is folded:
# aspp1 302.0 + 339.7 * (0.25 + 0.44 + 0.69) + GAP 0.5 + conv1 (4 of 5 groups) 151.0
WASP_EXECUTED_FLOPS_PER_IMG_24 = 2.0 * (302.0 + 339.7 * 1.38 + 0.5 + 151.0) * 1e6
NET_FLOPS_PER_IMG = 68.1e9          # SURVEY.md §8(d): conv-only fwd @384^2
DUMP_MAX_BYTES = 64 * 10 ** 6


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("UNIPOSE_B200_BENCH_PRECISION", "fp16"),
                    choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=32, help="frames per GPU")
    ap.add_argument("--size", type=int, default=384)
    ap.add_argument("--joints", type=int, default=16)
    ap.add_argument("--cpu-batch", type=int, default=4, help="frames per CPU-baseline step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step sub-record")
    ap.add_argument("--no-parity-mode", action="store_true", help="skip the fp32-grade mode timing")
    ap.add_argument("--train-steps", type=int, default=6)
    ap.add_argument("--train-only", action="store_true", help="print only the training sub-record (tuning runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the heat-maps of the last timed step (rank 0) to DIR/heat.npy, fp32; above %d MB only "
                         "the first frames that fit" % (DUMP_MAX_BYTES // 10 ** 6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.train_only):
        ap.error("--dump-outputs needs the inference timing of --impl b200 (not --train-only)")
    return args


def dump_outputs(out_dir: str, heat) -> None:
    """Saves what a caller of the timed path receives (fp32 heat-maps [N, K+1, H/8, W/8]) for output-for-output
    comparisons of two builds: inputs and weights are seeded, so equal arguments give equal inputs."""
    import numpy as np
    per_frame = heat[0].numel() * 4
    heat = heat[:max(1, DUMP_MAX_BYTES // per_frame)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "heat.npy"), heat.detach().float().cpu().numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tflops_burst=p["bf16_tflops"], tflops_sustained=p["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        if self.ok:
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's eager path on the host cores
# ------------------------------------------------------------------------------------------------
def host_cpu_budget() -> int:
    """Cores this process may really use: scheduler affinity clamped by the cgroup CPU quota (an over-subscribed
    torch thread pool - e.g. 128 threads on a 16-core quota - is 10-50x slower than the right size)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def _cpu_forward_fn(args):
    """(callable(x) -> heat, kind, make_input): the compiled reference when oracle/_ref is present, else the port."""
    import torch
    from oracle import build_ref
    from oracle import unipose_oracle as O
    sd = O.synth_state_dict(args.joints, seed=0)
    if build_ref.have_ref():
        RefUnipose, _, _ = build_ref.import_reference()
        m = RefUnipose(dataset="MPII", num_classes=args.joints).eval()
        m.load_state_dict(sd, strict=True)
        return (lambda x: m(x)), "reference"
    return (lambda x: O.unipose_forward(x, sd)), "port"


def cpu_forward_fps(args, steps: int, warmup: int, budget_s: float = 60.0):
    """Frames/s of the CPU eager forward at the best thread count of a small sweep ({8,16,32,64,all} within the
    cgroup/affinity budget).  Returns (fps, sec/step, threads, kind, sweep)."""
    import torch
    from oracle import unipose_oracle as O
    fn, kind = _cpu_forward_fn(args)
    cores = host_cpu_budget()
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | {cores})
    probe = O.synth_input(1, args.size, args.size, seed=1)
    sweep = {}
    t_sweep0 = time.perf_counter()
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            fn(probe)                                  # warm-up (thread pool, oneDNN primitive cache)
            t0 = time.perf_counter()
            fn(probe)
            sweep[c] = time.perf_counter() - t0
            if time.perf_counter() - t_sweep0 > budget_s:
                break
        best = min(sweep, key=sweep.get)
        torch.set_num_threads(best)
        x = O.synth_input(args.cpu_batch, args.size, args.size, seed=0)
        for _ in range(warmup):
            fn(x)
        t0 = time.perf_counter()
        done = 0
        for _ in range(steps):
            fn(x)
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
    return args.cpu_batch * done / dt, dt / done, best, kind, {str(k): round(1.0 / v, 3) for k, v in sweep.items()}, done


def run_reference(args) -> int:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps = max(1, min(args.steps, 8))
    warmup = max(1, min(args.warmup, 2))
    fps, sec_per_step, threads, kind, sweep, done = cpu_forward_fps(args, steps, warmup, budget_s=90.0)
    what = ("the reference's own modules (oracle/_ref byte-code of /root/reference/model/*.py), torch CPU fp32 eager"
            if kind == "reference" else "oracle port of the reference eager graph, torch CPU fp32")
    sample = "%d steps of batch %d at %dx%d; %s; %d threads (best of sweep %s frames/s at batch 1)" % (
        done, args.cpu_batch, args.size, args.size, what, threads, sweep)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "MPII %dx%d inference, %d joints (BASELINE.json configs[1]), CPU sample batch %d" % (
            args.size, args.size, args.joints, args.cpu_batch), "host_cores_usable": host_cpu_budget()},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _timed_steps(fn, steps, flush):
    """Sum of per-step CUDA-event times (ms) of fn(), L2 flushed (untimed) before every step, and what the last
    step returned."""
    import torch
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        starts[i].record()
        out = fn()
        ends[i].record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in zip(starts, ends)), out


def parity_record(model, x_dev, heat_dev, precision, n_check=2):
    """The timed heat-maps against the CPU oracle on the first images of the timed batch."""
    import numpy as np
    import torch
    from oracle import evaluate_oracle as E
    from oracle import unipose_oracle as O
    torch.set_num_threads(min(host_cpu_budget(), 32))
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    with torch.no_grad():
        ref = O.unipose_forward(x_dev[:n_check].cpu(), sd).numpy()
    got = heat_dev[:n_check].detach().cpu().numpy()
    err = np.abs(got - ref)
    scale = float(np.abs(ref).max())
    max_rel = float(err.max() / scale)
    n, k = ref.shape[:2]
    fr, fg = ref.reshape(n, k, -1), got.reshape(n, k, -1)
    top2 = np.sort(fr, axis=2)[:, :, -2:]
    safe = (top2[..., 1] - top2[..., 0]) > 2.0 * err.max()
    agree = fr.argmax(2) == fg.argmax(2)
    acc = E.accuracy(got, ref, 0.2, 0.5, "MPII")
    return {"mode": precision, "vs": "CPU oracle (fp32) on the first %d images of the timed batch" % n_check,
            "max_rel": max_rel, "max_rel_def": "max|err| / max|ref|",
            "argmax_agree": float(agree.mean()), "argmax_agree_safe_margin": (float(agree[safe].mean()) if safe.any() else None),
            "safe_joint_frac": float(safe.mean()),
            "pckh": float(acc[2][0]), "pckh_def": "PCKh@0.5 of the timed heat-maps scored against the oracle's (1.0 = every joint within threshold)"}


def train_record(args, dev, rank, world):
    """configs[2] per-GPU shape: fwd + MSE + bwd + (NCCL all-reduce of the bucketed flat gradient) + Adam."""
    import warnings

    import torch
    import torch.distributed as dist

    from unipose_b200 import synth, train
    from unipose_b200.model.unipose import unipose
    B, S = args.batch, args.size
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = unipose(dataset="MPII", num_classes=args.joints, precision="bf16")
    synth.trained_like_init_(m, seed=0)
    m = m.cuda().train()
    torch.manual_seed(100 + rank)
    x = synth.mpii_like_input(B, S, S, seed=rank).to(dev)
    t = torch.rand(B, args.joints + 1, S // 8, S // 8, device=dev)
    ts = train.TrainStep(m)
    for _ in range(4):
        loss = ts.step(x, t)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.train_steps):
        loss = ts.step(x, t)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.train_steps
    stats = ts.comm_stats()
    if world > 1:
        chk = ts.flat_p.double().sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(float(hi - lo) == 0.0)
    else:
        same = True
    # what the collective costs: (a) all buckets back to back on an otherwise idle GPU, (b) the same steps with the
    # all-reduce switched off (ranks diverge from here on: measured last) -> exposed = full - compute_only
    ar_alone = ts.time_allreduce_alone()
    ts.comm_enabled = False
    for _ in range(2):
        ts.step(x, t)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0.record()
    for _ in range(args.train_steps):
        ts.step(x, t)
    e1.record()
    torch.cuda.synchronize()
    ms_nocomm = e0.elapsed_time(e1) / args.train_steps
    vals = torch.tensor([ms, ar_alone, ms_nocomm], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms, ar_alone, ms_nocomm = float(vals[0]), float(vals[1]), float(vals[2])
    exposed = max(0.0, ms - ms_nocomm)
    rec = {"workload": "MPII %dx%d training step, batch %d per GPU, bf16 compute / fp32 master (BASELINE.json configs[2])" % (S, S, B),
           "ms_per_step": ms, "frames_s": B * world / (ms * 1e-3), "n_gpus": world, "steps": args.train_steps,
           "loss": float(loss), "params_identical_across_ranks": same,
           "allreduce": {"bytes": int(ts.flat_g.numel() * 4), "buckets": stats.get("buckets"),
                         "bucket_mb": stats.get("bucket_mb"), "ms_alone": ar_alone,
                         "ms_per_step_without_allreduce": ms_nocomm, "exposed_ms": exposed,
                         "hidden_frac": (None if world == 1 or ar_alone <= 0 else max(0.0, min(1.0, 1.0 - exposed / ar_alone)))},
           "mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
    del ts, m
    torch.cuda.empty_cache()
    return rec


def run_b200(args) -> int:
    import warnings

    import torch
    import torch.distributed as dist

    from unipose_b200 import synth
    from unipose_b200.model.unipose import unipose

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.train_only:
        rec = train_record(args, dev, rank, world)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps({"train": rec}))
        return 0

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = unipose(dataset="MPII", num_classes=args.joints, precision=args.precision)
    synth.trained_like_init_(model, seed=0)
    model = model.cuda().eval()
    B, S = args.batch, args.size
    x_host = synth.mpii_like_input(B, S, S, seed=rank).pin_memory()
    x_dev = x_host.to(dev)
    plan = model.plan_for(x_dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # ---- kernel-resident number: inputs already in HBM ----
    for _ in range(max(args.warmup, 3)):
        model.forward_static(x_dev)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, heat_last = _timed_steps(lambda: model.forward_static(x_dev), args.steps, flush)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, heat_last)      # plan-owned buffer: saved before the next call overwrites it
    launches = plan.launches * args.steps
    heat_timed = model.forward_static(x_dev).clone()

    # ---- end to end through the public API `model(input)`: pinned host batch -> device -> model.forward -> heat-maps
    # back in pinned host memory, every step.  Two device input buffers: the H2D copy of step i+1 (copy stream)
    # overlaps the forward of step i.
    out_host = torch.empty((B, args.joints + 1, S // 8, S // 8), dtype=torch.float32).pin_memory()
    main = torch.cuda.current_stream(dev)
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    x_bufs = [torch.empty_like(x_dev) for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_heat = torch.cuda.Event()

    def e2e_step(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            if i >= 2:
                copy_stream.wait_event(ev_free[b])
            x_bufs[b].copy_(x_host, non_blocking=True)
            ev_ready[b].record(copy_stream)
        main.wait_event(ev_ready[b])
        heat = model(x_bufs[b])          # the reference-facing call (model/unipose.py:27)
        ev_free[b].record(main)
        # the result goes back to the host on its own stream (the next forward does not wait for PCIe); the copy of step
        # i is ordered before the copy of step i+1 on that stream, and the final barrier() synchronises the device
        ev_heat.record(main)
        d2h_stream.wait_event(ev_heat)
        with torch.cuda.stream(d2h_stream):
            out_host.copy_(heat, non_blocking=True)
        heat.record_stream(d2h_stream)

    for i in range(4):
        e2e_step(i)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        e2e_step(i + 4)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)

    # ---- the same end-to-end loop fed with raw uint8 HWC images (model.forward_uint8: the reference's (x-128)/256
    # normalisation fused into the stem's input packing) - a quarter of the host->device bytes, identical heat-maps
    u8_host = ((x_host * 256.0) + 128.0).round().clamp_(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().pin_memory()
    u8_bufs = [torch.empty(u8_host.shape, dtype=torch.uint8, device=dev) for _ in range(2)]

    def e2e_u8_step(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            if i >= 2:
                copy_stream.wait_event(ev_free[b])
            u8_bufs[b].copy_(u8_host, non_blocking=True)
            ev_ready[b].record(copy_stream)
        main.wait_event(ev_ready[b])
        heat = model.forward_uint8(u8_bufs[b])
        ev_free[b].record(main)
        ev_heat.record(main)
        d2h_stream.wait_event(ev_heat)
        with torch.cuda.stream(d2h_stream):
            out_host.copy_(heat, non_blocking=True)
        heat.record_stream(d2h_stream)

    for i in range(4):
        e2e_u8_step(i)
    barrier()
    same_bits = bool(torch.equal(model.forward_uint8(u8_bufs[0]), model(x_dev)))
    e0.record()
    for i in range(args.steps):
        e2e_u8_step(i + 4)
    e1.record()
    barrier()
    e2e_u8_ms = e0.elapsed_time(e1)

    # the host->device copy of one fp32 batch alone (same pinned buffer, same copy stream): when it takes as long as a
    # step, `e2e` is bound by the host link, not by the kernels (`e2e_uint8` moves a quarter of the bytes)
    barrier()
    h0 = torch.cuda.Event(enable_timing=True)
    h1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(copy_stream):
        h0.record(copy_stream)
        for i in range(8):
            x_bufs[i % 2].copy_(x_host, non_blocking=True)
        h1.record(copy_stream)
    barrier()
    h2d_ms = h0.elapsed_time(h1) / 8.0

    t = torch.tensor([dev_ms, e2e_ms, e2e_u8_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, e2e_u8_ms = float(t[0]), float(t[1]), float(t[2])

    peaks = measured_peaks()
    roofline = None
    if not args.no_roofline and rank == 0:
        roofline = wasp_roofline(model, args, dev, peaks)
        net_tf = NET_FLOPS_PER_IMG * B * args.steps / (dev_ms * 1e-3) / 1e12
        roofline["net_tflops_in_step"] = net_tf
        roofline["net_frac_of_sustained_peak"] = net_tf / peaks["tflops_sustained"]
        roofline["net_frac_of_burst_peak"] = net_tf / peaks["tflops_burst"]

    parity = None
    parity_mode = None
    if rank == 0:
        parity = parity_record(model, x_dev, heat_timed, args.precision)
        if not args.no_parity_mode and args.precision != "fp32":
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                m32 = unipose(dataset="MPII", num_classes=args.joints, precision="fp32")
            m32.load_state_dict(model.state_dict())
            m32 = m32.cuda().eval()
            for _ in range(3):
                m32.forward_static(x_dev)
            torch.cuda.synchronize()
            k32 = max(3, min(args.steps, 10))
            ms32 = _timed_steps(lambda: m32.forward_static(x_dev), k32, flush)[0] / k32
            h32 = m32.forward_static(x_dev).clone()
            p32 = parity_record(m32, x_dev, h32, "fp32")
            parity_mode = {"precision": "fp32 (bf16x3 split, fp32 accumulate)", "ms_per_step": ms32,
                           "frames_s": B / (ms32 * 1e-3), "steps": k32, "max_rel": p32["max_rel"],
                           "argmax_agree_safe_margin": p32["argmax_agree_safe_margin"], "pckh": p32["pckh"],
                           "meets_1e-3": bool(p32["max_rel"] < 1e-3)}
            del m32, h32
            torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps, sec, threads, kind, sweep, done = cpu_forward_fps(args, steps=3, warmup=1, budget_s=30.0)
        cpu = {"value": fps, "unit": UNIT, "cores": threads, "kind": kind,
               "sample": "%d steps of batch %d at %dx%d after 1 warm-up (%s, torch CPU fp32, %.2f s/step, %d threads = best "
                         "of sweep %s frames/s at batch 1; %d usable cores)" % (
                             done, args.cpu_batch, S, S, "reference modules from oracle/_ref" if kind == "reference"
                             else "oracle port", sec, threads, sweep, host_cpu_budget())}

    # free the inference plan before the training plan (15 GB of activations) is built
    del plan
    model._plans.clear()
    train_rec = None
    if not args.no_train:
        try:
            train_rec = train_record(args, dev, rank, world)
        except Exception as e:          # the inference line must survive a training-side failure
            train_rec = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    frames = B * world * args.steps
    line = {
        "metric": METRIC, "value": frames / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {"fp16": "f16", "bf16": "bf16", "fp32": "bf16x3 (fp32-grade)"}[args.precision],
        "data": "synthetic",
        "config": {"workload": "MPII %dx%d inference, %d joints, batch %d per GPU (BASELINE.json configs[1])" % (
            S, S, args.joints, B), "global_batch": B * world, "precision": args.precision, "parallelism": "dp%d" % world,
            "l2": "flushed between timed steps (256 MiB memset, untimed); per-step CUDA events summed",
            "cuda_graph": True, "e2e_call": "model(input) - unipose.forward of the nn.Module mirror"},
        "clocks": clocks,
        "e2e": {"value": frames / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": x_host.numel() * 4,
                "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": e2e_ms / args.steps,
                "h2d_alone_ms": h2d_ms, "h2d_gbs": x_host.numel() * 4 / (h2d_ms * 1e-3) / 1e9,
                "bound": "host link (the fp32 batch takes as long to arrive as a step takes to compute)"
                if h2d_ms > 0.9 * dev_ms / args.steps else "kernels"},
        "e2e_uint8": {"value": frames / (e2e_u8_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": u8_host.numel(),
                      "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": e2e_u8_ms / args.steps,
                      "call": "model.forward_uint8(images_u8_nhwc) - normalisation fused into the stem's input packing",
                      "same_bits_as_fp32_input": same_bits},
        "gpu_launches": launches,
    }
    if roofline is not None:
        line["roofline"] = roofline
    if parity is not None:
        line["parity"] = parity
    if parity_mode is not None:
        line["parity_mode"] = parity_mode
    if train_rec is not None:
        line["train"] = train_rec
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    return 0


def wasp_roofline(model, args, dev, peaks):
    """Times the WASP block alone (the graded block, SURVEY.md §8d) on a resident [B, 2048, S/16, S/16] input:
    nominal dense FLOPs (zero-padding taps counted) / CUDA-event time vs the measured bf16 tensor peak."""
    import torch

    from unipose_b200 import engine
    B, hw = args.batch, args.size // 16
    plan = engine.Plan(dev, args.precision)
    b = plan.builder
    x = b.act(B, hw, hw, 2048)
    x.t.copy_(torch.randn(x.t.shape, device=dev).clamp_min_(0) * (0.02 if x.t.shape[0] == 2 else 1.0))
    model.wasp._emit(b, x)
    plan.finalize([])
    for _ in range(3):
        plan.run()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    reps = 20
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        plan.graph.replay() if plan.graph is not None else plan._launch_all()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    ms = tot / reps
    flops = WASP_FLOPS_PER_IMG * (hw * hw / 576.0) * B
    achieved = flops / (ms * 1e-3) / 1e12
    t_roof_ms = max(flops / (peaks["tflops_burst"] * 1e12), WASP_MIN_BYTES_C2 / (peaks["hbm_gbs"] * 1e9)) * 1e3
    traffic = None
    for name in ("wasp_traffic_r2.json", "wasp_traffic_r1.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath) and B == 32 and hw == 24:
            traffic = json.load(open(tpath))["dram_bytes_per_block"]   # from the committed ncu capture of the same block
            break
    executed = WASP_EXECUTED_FLOPS_PER_IMG_24 * B if hw == 24 else None
    return {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
            "frac": achieved / peaks["tflops_burst"], "traffic": traffic, "peak_source": peaks["source"],
            "kernel": "WASP block = %d launches (%s)" % (plan.launches, ", ".join(sorted({n for n, f, s in plan.ops if f is not None}))),
            "wasp_ms": ms, "wasp_t_roof_ms": t_roof_ms, "wasp_roofline_frac": t_roof_ms / ms,
            "flops_convention": "nominal dense (zero taps counted, SURVEY.md 8d), %.1f GFLOP per block" % (flops / 1e9),
            # SURVEY.md 8(d): the layer-by-layer variant (every conv reads its input / writes its output: 355.6 MB at
            # config 2) and, reported separately and NOT used in `frac`, the work actually issued to the tensor
            # cores: out-of-image taps skipped and the shared conv2 folded into conv1's weights
            "wasp_t_roof_layerwise_ms": (max(flops / (peaks["tflops_burst"] * 1e12),
                                             WASP_LAYERWISE_BYTES_C2 / (peaks["hbm_gbs"] * 1e9)) * 1e3
                                         if (B == 32 and hw == 24) else None),
            "executed_gflop_estimate": (executed / 1e9 if executed else None),
            "executed_frac": (executed / (ms * 1e-3) / 1e12 / peaks["tflops_burst"] if executed else None)}


def main() -> int:
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
