#!/usr/bin/env python
"""bench.py — frustums/s forward of the B200 frustum hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload car|people|sunrgbd] [--batch 32] [--precision 0|1] [--dump-outputs DIR]

One "step" = one forward of the hot path (grouping -> PointNet -> FCN -> heads/decode) over one
batch of `--batch` synthetic frustums per GPU (default: cfgs/det_sample.yaml car, B=32 x 1024
points = BASELINE.json configs[1]).  Exactly `--steps` steps are timed per mode (resident, e2e),
in one region between two CUDA events.  `--dump-outputs DIR` writes what the last timed step
returned (rank 0) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared
output for output.  Weak scaling: every rank processes its own B frustums;
for N>1 the per-rank result block is all-gathered over NCCL inside the timed region (the only
exchange of the inference path, SURVEY.md section 8(e)).

Printed JSON (rank 0, one line): the base contract keys plus `roofline`, `cpu_baseline`,
`e2e`, `clocks`, `gpu_launches`, `hbm` (see DESIGN.md "Measurement").
`--impl reference` times the reference's own PyTorch path on the host CPUs (the oracle port:
/root/reference cannot travel to the GPU box and its CUDA op no longer compiles).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "frustums/sec fwd"
UNIT = "frustums/s"

# Algorithmic per-frustum figures (SURVEY.md section 8(d), BASELINE.md section 2)
ALGO = {
    "car": dict(bytes=32.0e3, gflop=2.977),
    "people": dict(bytes=61.7e3, gflop=7.469),
    "sunrgbd": dict(bytes=31.5e3, gflop=2.526),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock / throttle-reason sampling during the timed regions (B200_PROFILING.md clocks line).

    The timed regions last tens of milliseconds, far less than an `nvidia-smi` start-up, so the sampling is done
    in-process through NVML (`pynvml`, 1 ms period); `nvidia-smi -lms` is only the fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.sm, self.reasons, self.smax = [], set(), None
        self.nvml, self.h, self.run = None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ent = vis.split(",")[gpu_index].strip()
                phys = int(ent) if ent.isdigit() else None
            self.h = (pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None
                      else pynvml.nvmlDeviceGetHandleByUUID(ent))
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def start(self):
        if self.nvml is not None:
            self.run = True
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def sample_now(self):
        """One NVML sample (called by the polling thread)."""
        nv = self.nvml
        if nv is None:
            return
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for name, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                              ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                              ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                              ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)):
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _poll(self):
        # background polling only: NVML calls go through ctypes (GIL released), 2 ms period - no NVML call is
        # ever made from the issuing thread inside a timed region (VERDICT r1 weak #6)
        while self.run:
            self.sample_now()
            time.sleep(0.002)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.run = False
            self.t.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smax,
                    "sm_min_mhz": float(min(self.sm)) if self.sm else None,
                    "samples": len(self.sm), "source": "nvml", "reasons": sorted(self.reasons)}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "source": "nvidia-smi", "reasons": sorted(reasons)}


class _OutRing:
    """Result-block allocator handed to the engine (FrustumEngine.out_alloc): consecutive plans get
    consecutive slots of one buffer."""

    def __init__(self, slots):
        self.slots, self.buf, self.i = slots, None, 0

    def __call__(self, n, device):
        import torch
        if self.buf is None:
            self.n = n
            self.buf = torch.empty(self.slots * n, dtype=torch.float32, device=device)
        assert n == self.n and self.i < self.slots, "ring holds one result block per in-flight plan"
        v = self.buf[self.i * n: (self.i + 1) * n]
        self.i += 1
        return v


DUMP_LIMIT_BYTES = 64 << 20
# the 6-tuple PointNetDet.forward returns in eval mode (det_base.py:411)
OUTPUT_NAMES = ("cls_probs", "center", "heading", "size", "heading_probs", "size_probs")


def dump_outputs(path, arrays, seed=0):
    """Write {name: tensor/array} as path/<name>.npy (float64 stays float64, everything else float32).  Above
    DUMP_LIMIT_BYTES in all, the same seeded sample of leading-axis rows (frustums) is kept of every array."""
    arrays = {k: (v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = min(v.shape[0] for v in arrays.values())
        keep = np.sort(np.random.default_rng(seed).choice(n, max(1, n * DUMP_LIMIT_BYTES // total), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def host_threads():
    """Usable host threads: affinity mask, capped by the cgroup CPU quota when one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_reference_rate(workload, sample_B, iters, warm, seed=1234, min_seconds=0.0, budget_s=None):
    """frustums/s of the reference algorithm on host CPUs (oracle port, all host threads)."""
    import torch
    from frustum_convnet_b200 import config, synth
    from oracle import model as om
    cfg, w = config.load_workload(workload)
    n = host_threads()
    sd = om.to_torch_state(synth.make_state_dict(w["arch"], w["num_vec"], cfg.DATA.DATASET_NAME, seed=7))
    data = synth.make_frustums(workload, sample_B, seed=seed)
    mean = config.DATASET_INFO[cfg.DATA.DATASET_NAME].MEAN_SIZE_ARRAY
    run = lambda: om.pointnet_det_eval(data, sd, cfg.DATA.HEIGHT_HALF, w["arch"].nsample, mean)
    # "all the host threads it can use": intra-op scaling of small convolutions saturates early,
    # so probe a few thread counts (one forward each) and keep the fastest; report the one used.
    best = None
    for cand in sorted({n, max(1, n // 2), max(1, n // 4), min(n, 32), min(n, 16), min(n, 8)}, reverse=True):
        torch.set_num_threads(cand)
        run()
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, cand)
    n = best[1]
    torch.set_num_threads(n)
    if budget_s is not None and (iters + warm) * best[0] > budget_s and sample_B > 1:
        # keep the whole `--steps K --warmup W` run bounded: fewer frustums per step (never below one)
        sample_B = max(1, min(sample_B, int(sample_B * budget_s / ((iters + warm) * best[0]))))
        data = synth.make_frustums(workload, sample_B, seed=seed)
    for _ in range(warm):
        run()
    ts = []
    while len(ts) < iters or (sum(ts) < min_seconds and len(ts) < 400):
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
    return sample_B / float(np.median(ts)), float(np.sum(ts)), n, len(ts), sample_B


def workload_name(workload, B, points=None):
    from frustum_convnet_b200 import config, synth
    w = config.WORKLOADS[workload]
    N = points or synth._PRESETS[workload]["N"]
    return "%s cfgs/%s B=%d frustums/GPU x %d pts, T=%s, forward (eval)" % (
        workload, w["yaml"], B, N, list(synth.section_counts(workload)))


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample_B = min(args.batch, 8)
    t0 = time.perf_counter()
    rate, busy, n, _, sample_B = cpu_reference_rate(args.workload, sample_B, args.steps, max(args.warmup, 1),
                                                    budget_s=150.0)
    ms = 1e3 * sample_B / rate
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.batch) +
                               " [CPU arm: bounded sample of %d frustums per step]" % sample_B,
                   "batch_per_gpu": args.batch, "global_batch": args.batch, "parallelism": "dp1",
                   "reference_sample": "%d frustums per step (bounded CPU sample of the same workload)" % sample_B},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": n, "kind": "port",
                         "sample": "%d steps x %d frustums, oracle port of models/det_base.py on torch CPU fp32"
                                   % (args.steps, sample_B)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))


def _lib_call_adam(ts):
    """One fused Adam launch with a zero learning rate (phase timing only: parameters stay put)."""
    import torch
    from frustum_convnet_b200 import _lib
    _lib.call("fcn_adam_step", ts.flat.param.data_ptr(), ts.flat.grad.data_ptr(), ts.m.data_ptr(), ts.v.data_ptr(),
              ts.flat.numel, 0.0, 0.9, 0.999, 1e-8, 0.0, max(ts.step_count, 1), 1.0,
              torch.cuda.current_stream().cuda_stream)


def run_train(args, rank, local_rank, world):
    """Config 5 (BASELINE.json configs[4]): cfgs/refine_car.yaml TRAINING step on the hand-written kernels -
    forward + losses + backward + gradient all-reduce (flat bucket, NCCL over NVLink, overlapped with the
    PointNet backward) + fused Adam, B = --batch frustums per GPU (32 x 8 GPUs = 256)."""
    import torch
    import torch.distributed as dist
    from frustum_convnet_b200 import config, synth
    from frustum_convnet_b200.det_base import PointNetDet
    from frustum_convnet_b200.train_engine import TrainStep
    from frustum_convnet_b200 import train_path
    assert torch.cuda.is_available(), "bench.py --train needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, w = config.load_workload("refine_car")
    sd = synth.make_state_dict(w["arch"], 3, "KITTI", seed=7)

    def build():
        m = PointNetDet(3, num_vec=3)
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
        return m.to(dev).train()

    model = build()
    B = args.batch
    ts = TrainStep(model, lr=cfg.TRAIN.BASE_LR, weight_decay=cfg.TRAIN.WEIGHT_DECAY)
    npool = 64
    host_pool = [{k: torch.from_numpy(v).pin_memory() for k, v in
                  synth.make_frustums("refine_car", B, seed=1234 + rank + 1000 * i, with_labels=True).items()}
                 for i in range(npool)]
    dev_pool = [{k: v.to(dev) for k, v in d.items()} for d in host_pool]
    h2d_bytes = int(sum(v.numel() * v.element_size() for v in host_pool[0].values()))
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    stage = {k: torch.empty_like(v, device=dev) for k, v in host_pool[0].items()}

    def step_resident(i):
        return ts.step(dev_pool[i % npool])

    def step_e2e(i):
        for k, v in host_pool[i % npool].items():                 # H2D of this step's inputs + labels
            stage[k].copy_(v, non_blocking=True)
        losses, _ = ts.step(stage)
        loss_host.copy_(losses["total_loss"].detach().reshape(1), non_blocking=True)   # D2H of the step's loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 10)):
        step_resident(i)
    for i in range(max(args.warmup, 3)):
        step_e2e(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def region(fn):
        """Exactly `--steps` steps between two CUDA events -> (ms, what the last step returned)."""
        barrier()
        e0.record()
        for i in range(args.steps):
            out = fn(i)
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_e2e, _ = region(step_e2e)
    t_res, (losses, metrics) = region(step_resident)        # last: its final step's results are the dumped outputs
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {**losses, **metrics})
    t_regions = torch.tensor([t_res, t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_regions, op=dist.ReduceOp.MAX)
    ms_step, e2e_ms = (float(t) / args.steps for t in t_regions.cpu().numpy())
    value, e2e_value = world * B / (ms_step * 1e-3), world * B / (e2e_ms * 1e-3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- phase split of one step (CUDA events) and the PyTorch-autograd composition of the same branch (cuDNN, fp32)
    eng = list(ts.engines.values())[0]
    data = dev_pool[0]
    S = 4
    pc = data["point_cloud"][:, :3, :].contiguous()
    centers = [data["center_ref%d" % (i + 1)].contiguous() for i in range(S)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    acc = np.zeros(4)
    for it in range(23):
        if it == 3:
            acc[:] = 0.0          # the first iterations capture the single-stage backward graph
        ev[0].record()
        cls, reg = eng.forward(pc, centers, data["one_hot"])
        ev[1].record()
        _, _, dcls, dreg = ts._losses(eng, cls, reg, centers[1], data)
        ev[2].record()
        ts.flat.grad.zero_()
        eng.backward(dcls, dreg, update_running=False)
        ev[3].record()
        _lib_call_adam(ts)
        ev[4].record()
        torch.cuda.synchronize()
        acc += [ev[j].elapsed_time(ev[j + 1]) for j in range(4)]
    phases = {"forward_ms": acc[0] / 20, "losses_ms": acc[1] / 20, "backward_ms": acc[2] / 20,
              "adam_ms": acc[3] / 20, "loss_impl": ts.loss_impl,
              "note": "one step at a time on one stream (CUDA events); losses = fcn_det_loss (losses + dlogits + "
                      "metrics in one call) when loss_impl == 'kernel'"}
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref_model = build()
    ref_model.train_kernels = False
    opt = torch.optim.Adam(ref_model.parameters(), lr=cfg.TRAIN.BASE_LR, weight_decay=cfg.TRAIN.WEIGHT_DECAY)

    def torch_step(d):
        opt.zero_grad()
        l, _ = ref_model(d)
        l["total_loss"].backward()
        opt.step()

    for i in range(5):
        torch_step(dev_pool[i])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(20):
        torch_step(dev_pool[i % npool])
    torch.cuda.synchronize()
    autograd_ms = (time.perf_counter() - t0) / 20 * 1e3
    gflop_step = 3.0 * 0.240 * B                       # SURVEY 8(d): refine car fwd 0.240 GFLOP/frustum, step ~ 3x
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12         # nominal fp32 FMA peak of the B200 (no measured figure)
    line = {
        "metric": "frustums/sec train step (fwd+bwd+allreduce+Adam)", "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "refine_car cfgs/refine_car.yaml TRAIN step, B=%d frustums/GPU x 512 pts, T=%s"
                               % (B, list(eng.T)),
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": "dp%d" % world,
                   "optimizer": "Adam lr %g wd %g (fused, flat bucket)" % (cfg.TRAIN.BASE_LR, cfg.TRAIN.WEIGHT_DECAY),
                   "collective": "none (single GPU)" if world == 1 else
                                 "NCCL all_reduce of the flat fp32 gradient bucket (%.2f MB) in 2 pieces, the first "
                                 "overlapping the PointNet backward" % (ts.flat.numel * 4 / 1e6),
                   "l2": "inputs cycle through a %d-batch pool; every step rewrites ~0.4 GB of activations / "
                         "gradients (> 126 MB L2)" % npool,
                   "timing": "one %d-step region per mode (e2e, then resident)" % args.steps},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
        "gpu_launches": eng.kernel_launches_per_step() * args.steps,
        "launches_per_step": eng.kernel_launches_per_step(),
        "phases_ms": phases,
        "roofline": {"bound": "fp32", "kernel": "train step (all training kernels)", "achieved": gflop_step / ms_step,
                     "peak": fp32_peak, "unit": "TFLOP/s", "frac": gflop_step / ms_step / fp32_peak,
                     "peak_source": "nominal fp32 FMA (148 SMs x 128 lanes x 2 x 1.965 GHz)", "traffic": None},
        "cpu_baseline": None,
        "autograd_gpu_baseline": {"value": B / (autograd_ms * 1e-3), "unit": UNIT, "ms_per_step": autograd_ms,
                                  "kind": "same branch composed from PyTorch/cuDNN autograd ops on this GPU (fp32, "
                                          "train_kernels=False) + torch.optim.Adam, wall clock"},
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="car", choices=list(ALGO) + ["refine_car"])
    ap.add_argument("--train", action="store_true",
                    help="config 5: time the refine_car TRAINING step (fwd+bwd+all-reduce+Adam) on the hand-written kernels")
    ap.add_argument("--batch", type=int, default=32, help="frustums per GPU per step")
    ap.add_argument("--precision", type=int, default=int(os.environ.get("FCN_PRECISION", "1")),
                    help="1: TF32 tensor cores (tcgen05) — the arithmetic cuDNN uses by default; 0: fp32 FMA")
    ap.add_argument("--pool-mb", type=float, default=160.0, help="distinct input pool size (> L2)")
    ap.add_argument("--points", type=int, default=None,
                    help="points per frustum (default: the workload's yaml value; e.g. people at 512)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather-group", type=int, default=1, help="N>1, --exchange nccl: steps covered by one all-gather")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1 result exchange: peer = the heads epilogue stores every rank's rows into all ranks' "
                         "gather buffers over NVLink (no collective); nccl = all_gather_into_tensor per step")
    ap.add_argument("--streams", type=int, default=int(os.environ.get("FCN_STREAMS", "10")),
                    help="forwards in flight: steps are issued round-robin on this many CUDA streams")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32/float64, <= 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs times the GPU path; --impl reference has no GPU outputs")
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3)

    if args.train or args.workload == "refine_car":
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "no CPU arm for the training step: the reference "
                                  "train branch needs its CUDA grouping op (query_depth_point.py:23-24)"}))
            return
        run_train(args, rank, local_rank, world)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from frustum_convnet_b200 import config, synth

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, w = config.load_workload(args.workload)
    modname = "det_base_sunrgbd" if w["arch"].num_scales == 5 else "det_base"
    mod = __import__("frustum_convnet_b200." + modname, fromlist=["PointNetDet"])
    sd = synth.make_state_dict(w["arch"], w["num_vec"], cfg.DATA.DATASET_NAME, seed=7)
    model = mod.PointNetDet(3, num_vec=w["num_vec"])
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    model.precision = args.precision
    model = model.to(dev).eval()
    model.use_cuda_graph = True
    model.copy_outputs = False     # results are read from the engine's output block (D2H in e2e)
    model.freeze()                 # serving: weights are static, skip the per-call staleness scan
    B, S = args.batch, w["arch"].num_scales

    # ---- input pool larger than L2 (126 MB): distinct batches cycled through the timed loop
    one = synth.make_frustums(args.workload, B, seed=1234 + rank, N=args.points)
    keys = ["point_cloud"] + ["center_ref%d" % (i + 1) for i in range(S)] + ["one_hot"]
    step_in_bytes = int(sum(one[k].nbytes for k in keys))
    npool = max(2, int(np.ceil(args.pool_mb * 1e6 / step_in_bytes)))
    ngen = min(npool, 8)   # 8 seeded batches, the rest are per-frustum rotations of them
    base = [synth.make_frustums(args.workload, B, seed=1234 + rank + 1000 * i, N=args.points) for i in range(ngen)]
    T = [one["center_ref%d" % (i + 1)].shape[2] for i in range(S)]

    # `--streams` forwards in flight: step i runs on stream i % S with its own workspace + CUDA graph
    # (independent batches; the SM-starved FCN layers of one batch overlap the PointNet tiles of the next)
    nstream = max(1, args.streams)
    streams = [torch.cuda.Stream(device=dev) for _ in range(nstream)]
    eng = model.engine()
    peer = None
    if world > 1:
        n_out_blk = B * T[1] * (2 + 3 + 1 + 3 + eng.num_bins + eng.num_size)
        if args.exchange == "peer" and eng.use_mega:
            from frustum_convnet_b200.sharding import PeerResultExchange
            try:
                peer = PeerResultExchange(nstream, n_out_blk, dev)
            except Exception as e:   # no P2P mapping on this box: keep the measured path honest, say so
                sys.stderr.write("peer exchange unavailable (%r): falling back to NCCL all-gather\n" % (e,))
                peer = None
        if peer is not None:
            slot_i = [0]

            def peer_alloc(n, device):
                v = peer.local_block(slot_i[0])
                assert v.numel() == n
                slot_i[0] += 1
                return v
            eng.out_alloc = peer_alloc
        else:
            # NCCL path: the result blocks of all in-flight plans live in ONE ring, so that a group of
            # consecutive steps is all-gathered by a single collective
            ring = _OutRing(nstream)
            eng.out_alloc = ring
    plans = []
    for st in streams:
        with torch.cuda.stream(st):
            plans.append(eng.plan(B, one["point_cloud"].shape[2], T))
    eng.out_alloc = None
    if peer is not None:
        for k, pl in enumerate(plans):
            blocks, flags = peer.peer_targets(k)
            pl.set_peer_outputs(blocks, flags)
    plan = plans[0]
    # every pool entry is one packed block in the engine's input layout (one staging copy per step)
    host_pool, dev_pool, dev_flat_pool = [], [], []
    for i in range(npool):
        src = base[i % ngen]
        sh = (i // ngen) % B
        hflat, _ = plan.pack({k: np.roll(src[k], sh, axis=0) for k in keys}, pin=True)
        host_pool.append(hflat)
        dflat = hflat.to(dev)
        dviews = {k: dflat[off: off + ref.numel()].view(ref.shape)
                  for k, off, ref in zip(keys, plan._in_offs, [plan.in_pc] + plan.in_centers + [plan.in_onehot])}
        dev_pool.append(dviews)
        dev_flat_pool.append(dflat)
    # N>1: the per-rank result blocks are all-gathered (NCCL over NVLink) on ONE communication stream, in
    # step order on every rank (collectives of one communicator must not race on several streams).  One
    # collective covers `--gather-group` consecutive steps (default 1: measured on 2 GPUs, groups of 4 leave the
    # HBM-resident rate unchanged within noise and cost ~10 % of the e2e rate - bigger bubbles behind the D2H
    # copies); the streams of a group wait for "their" gather before overwriting their result blocks.
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    G = max(1, min(nstream, args.gather_group))
    ngroup = (nstream + G - 1) // G
    gather_done = [None] * ngroup
    if world > 1 and peer is None:
        n_out = plans[0].out_flat.numel()
        assert all(pl.out_flat.data_ptr() == ring.buf.data_ptr() + 4 * n_out * k for k, pl in enumerate(plans))
        group_src = [ring.buf[g * G * n_out: min(nstream, (g + 1) * G) * n_out] for g in range(ngroup)]
        gather_bufs = [torch.empty((world, src.numel()), dtype=torch.float32, device=dev) for src in group_src]
    n_gathers = [0]
    no_comm = os.environ.get("FCN_BENCH_NO_COMM") == "1" or peer is not None   # peer path: no collective to issue

    def gather(g):
        for k in range(g * G, min(nstream, (g + 1) * G)):
            comm_stream.wait_stream(streams[k])
        with torch.cuda.stream(comm_stream):
            dist.all_gather_into_tensor(gather_bufs[g], group_src[g])
            done = torch.cuda.Event()
            done.record(comm_stream)
        gather_done[g] = done
        n_gathers[0] += 1

    def after_step(i, last):
        """Issue the gather of step i's group when the group is complete (or the run ends)."""
        k = i % nstream
        if k % G == G - 1 or k == nstream - 1 or last:
            gather(k // G)

    in_views_res = [pl.input_views() for pl in plans]

    def step_resident(i, comm=True, last=False):
        # same call sequence as step_e2e below minus the PCIe legs: the step's packed input block (resident in
        # HBM, a different one every step) is copied device-to-device into the plan's input block, then the public
        # API runs on the plan's own views (so `e2e` differs from `value` by exactly the H2D + D2H copies)
        k = i % nstream
        with torch.cuda.stream(streams[k]):
            if world > 1 and gather_done[k // G] is not None:
                streams[k].wait_event(gather_done[k // G])
            plans[k].in_flat.copy_(dev_flat_pool[i % npool], non_blocking=True)
            out = model(in_views_res[k])
        if world > 1 and comm and not no_comm:
            after_step(i, last)
        return out

    def join_streams():
        cur = torch.cuda.current_stream()
        for st in streams:
            cur.wait_stream(st)
        if comm_stream is not None:
            cur.wait_stream(comm_stream)

    def fork_streams():
        cur = torch.cuda.current_stream()
        for st in streams:
            st.wait_stream(cur)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- e2e step: public API with HOST (pinned) buffers, H2D + D2H inside the timed region
    host_outs = [torch.empty(pl.out_flat.shape, dtype=torch.float32).pin_memory() for pl in plans]
    d2h_bytes = int(host_outs[0].numel() * 4)
    in_views = [pl.input_views() for pl in plans]

    def step_e2e(i, comm=True, last=False):
        k = i % nstream
        with torch.cuda.stream(streams[k]):
            if world > 1 and gather_done[k // G] is not None:
                streams[k].wait_event(gather_done[k // G])
            plans[k].in_flat.copy_(host_pool[i % npool], non_blocking=True)    # H2D of this step's inputs
            model(in_views[k])                                                 # public API, zero-copy staging
            host_outs[k].copy_(plans[k].out_flat, non_blocking=True)           # D2H of the 6-tuple block
        if world > 1 and comm and not no_comm:
            after_step(i, last)

    # ---- untimed pre-warm: graph capture + clock ramp (a FIXED step count without collectives, so that all
    # ranks issue identical NCCL sequences afterwards), then both step kinds WITH their collectives: NCCL's
    # lazy channel/proxy setup must not land in a timed region (>= 64 gathers before the first one)
    for j in range(512):
        step_resident(j, comm=False)
        if j % 64 == 63:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    nwarm = max(args.warmup, 64 if world > 1 else args.warmup)
    for i in range(nwarm):
        step_resident(i, last=(i == nwarm - 1))
    for i in range(nwarm):
        step_e2e(i, last=(i == nwarm - 1))
    barrier()

    # ---- timed regions.  ONE region per mode = EXACTLY `--steps` steps between two CUDA events, barrier +
    # synchronize on both sides; the max over ranks is taken.  The e2e region runs first, so that the last timed
    # step is a resident one: `value` is measured on that path and its last step's results are the dumped outputs.
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def region(fn):
        barrier()
        e0.record()
        fork_streams()
        for i in range(args.steps):
            out = fn(args.warmup + i, last=(i == args.steps - 1))
        join_streams()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_e2e, _ = region(step_e2e)
    t_res, last_out = region(step_resident)
    clocks = sampler.stop() if rank == 0 else None    # samples cover both timed regions
    if args.dump_outputs and rank == 0:   # before any later step overwrites the plan's output block
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, last_out)))
    t_regions = torch.tensor([t_res, t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_regions, op=dist.ReduceOp.MAX)
    t_regions = t_regions.cpu().numpy()
    ms_step = float(t_regions[0]) / args.steps
    value = world * B / (ms_step * 1e-3)
    e2e_ms_step = float(t_regions[1]) / args.steps
    e2e_value = world * B / (e2e_ms_step * 1e-3)
    spread = {"regions": 1, "steps_per_region": args.steps,
              "resident_ms_per_step": ms_step, "e2e_ms_per_step": e2e_ms_step,
              "device_seconds_timed": float(t_regions.sum() * 1e-3),
              "e2e_le_value": bool(e2e_value <= value * 1.02)}

    # host-side issue cost per step (queue empty, no waiting on the GPU): shows whether the loop is CPU-bound
    torch.cuda.synchronize()
    t_h = time.perf_counter()
    for i in range(32):
        step_resident(i, comm=False)
    host_us = (time.perf_counter() - t_h) / 32 * 1e6
    torch.cuda.synchronize()

    # ---- per-kernel timing of the eager launch sequence (CUDA events on the launching stream)
    kt = plan.time_kernels(dev_pool, iters=20) if rank == 0 else None

    # ---- latency of ONE forward at a time (single stream, graph replay): p10 / median / p90 over 100 calls
    latency = None
    if rank == 0:
        try:
            torch.cuda.synchronize()
            with torch.cuda.stream(streams[0]):
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                       for _ in range(100)]
                for j, (a, b) in enumerate(evs):
                    a.record()
                    model(dev_pool[j % npool])
                    b.record()
                    b.synchronize()
            ts = sorted(a.elapsed_time(b) for a, b in evs)
            latency = {"p10_ms": ts[10], "median_ms": ts[50], "p90_ms": ts[90],
                       "note": "one forward of %d frustums at a time, single stream, CUDA-graph replay" % B}
        except Exception as e:   # informative only: never lose the bench line over it
            latency = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    algo = dict(ALGO[args.workload])
    if args.points:   # non-default point count: 12 B per point more/less input per frustum (FLOPs are T x K bound)
        algo["bytes"] += 12.0 * (args.points - synth._PRESETS[args.workload]["N"])
    # dominant kernel = largest share of the step's SM time: launch duration x fraction of the SMs the kernel
    # occupies (the persistent FCN kernel deliberately runs on `mega_grid` CTAs - 24 of 148 SMs for this
    # workload - so that several forwards overlap; its wall time alone would overstate its share 6x)
    sm_total = torch.cuda.get_device_properties(dev).multi_processor_count
    for k in kt["kernels"]:
        if k["name"] == "fcn_mega":
            k["sms"] = min(sm_total, plan.mega_grid)
        k["sm_fraction"] = min(1.0, k.get("sms", sm_total) / sm_total)   # PointNet: clusters/CTAs of its balanced rounds
        k["sm_ms"] = k["ms"] * k["sm_fraction"]
    dom = max(kt["kernels"], key=lambda k: k["sm_ms"])
    traffic = None
    try:   # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        traffic = tj.get(dom["name"], {}).get(args.workload, {}).get("bytes")
    except Exception:
        pass
    tf32_peak = peaks["bf16_tflops"] / 2.0   # kind::tf32 runs at half the bf16 rate; burst figure (kernel timed alone)
    # a kernel that deliberately occupies a fraction of the SMs (the persistent FCN kernel) is measured against the
    # peak of THOSE SMs; `frac_of_whole_gpu` keeps the unnormalised figure
    roofline = {
        "bound": "tensor", "kernel": dom["name"], "achieved": dom["executed_tflops"], "peak": tf32_peak * dom["sm_fraction"],
        "unit": "TFLOP/s", "frac": dom["executed_tflops"] / (tf32_peak * dom["sm_fraction"]),
        "sm_fraction": dom["sm_fraction"], "frac_of_whole_gpu": dom["executed_tflops"] / tf32_peak,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops/2 (%s)" % peaks["source"],
        "ms_per_launch": dom["ms"], "executed_gflop_per_launch": dom["executed_gflop"],
        "nominal_gflop_per_launch": dom["nominal_gflop"], "traffic": traffic,
        "precision": "tf32-tcgen05" if args.precision == 1 else "fp32-simt",
    }
    # every tensor-core kernel of the step, same definitions (the two largest SM-time shares are close: see both)
    roofline["kernels"] = {
        k["name"]: {"ms_per_launch": round(k["ms"], 5), "sms": k.get("sms", sm_total),
                    "sm_time_share": round(k["sm_ms"] / sum(x["sm_ms"] for x in kt["kernels"]), 3),
                    "achieved_tflops": round(k["executed_tflops"], 1),
                    "frac": round(k["executed_tflops"] / (tf32_peak * k["sm_fraction"]), 3),
                    "frac_of_whole_gpu": round(k["executed_tflops"] / tf32_peak, 3)}
        for k in kt["kernels"] if k["executed_gflop"] > 0}
    hbm = {"achieved": value * algo["bytes"] / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
           "frac": value * algo["bytes"] / 1e9 / peaks["hbm_gbs"],
           "algorithmic_bytes_per_frustum": algo["bytes"],
           "note": "path is compute-bound by design (SURVEY.md 8(d)); HBM fraction is expected to be small"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32" if args.precision == 1 else "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, B, args.points),
            "batch_per_gpu": B, "global_batch": B * world, "parallelism": "dp%d" % world,
            "l2": "inputs cycle through a %d-batch pool (%.0f MB > 126 MB L2); weights/workspaces stay L2-resident"
                  % (npool, npool * step_in_bytes / 1e6),
            "cuda_graph": True, "precision": roofline["precision"], "streams_in_flight": nstream,
            "timing": "one %d-step region per mode (e2e, then resident)" % args.steps,
            "collective": ("none (single GPU)" if world == 1 else
                           "none: the heads epilogue of every forward stores its %d KB result block into all %d ranks' "
                           "gather buffers over NVLink peer memory (CUDA IPC) + one epoch flag per forward"
                           % (plans[0].out_flat.numel() * 4 // 1024, world) if peer is not None else
                           "NCCL all_gather of the per-rank result blocks, one per %d steps (%d issued in this run)"
                           % (G, n_gathers[0]))},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(plan.in_flat.numel() * 4),
                "d2h_bytes_per_step": d2h_bytes},
        "host_issue_us_per_step": host_us, "latency": latency, "timing": spread,
        "gpu_launches": kt["launches_per_step"] * args.steps,
        "launches_per_step": kt["launches_per_step"],
        "roofline": roofline, "hbm": hbm, "clocks": clocks,
        "achieved_tflops_nominal": value * algo["gflop"] / 1e3,
        "kernel_ms": {k["name"]: round(k["ms"], 5) for k in kt["kernels"]},
        "kernel_sm_ms": {k["name"]: round(k["sm_ms"], 5) for k in kt["kernels"]},
        "fcn_mega": ({"ctas": plan.mega_grid, "executed_tflops_on_its_sms": next(
            (k["executed_tflops"] / k["sm_fraction"] for k in kt["kernels"] if k["name"] == "fcn_mega"), None)}
            if plan.mega_args is not None else None),
        "unique_row_fraction": kt["unique_row_fraction"],
    }
    if world == 1 and not args.no_cpu_baseline:
        try:
            sample_B = min(B, 8)
            rate, busy, n, nf, sample_B = cpu_reference_rate(args.workload, sample_B, iters=5, warm=1,
                                                             min_seconds=12.0)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": n, "kind": "port",
                                    "sample": "%d forwards of %d frustums (%.1f s of CPU work), oracle port on "
                                              "torch CPU fp32" % (nf, sample_B, busy)}
        except Exception as e:   # the GPU measurement above must not be lost over the CPU leg
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
