#!/usr/bin/env python
"""Benchmark of the SMPL hot path: SMPL meshes/sec, forward+backward (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--mode fp32|bf16] [--dump-outputs DIR]

One "step" = one forward+backward pass of the batched SMPL layer over one batch of synthetic
(betas, pose, trans) with upstream gradients (dV, dJ): BASELINE.json configs[1] (B = 4096 bodies on
one B200), the same per-GPU batch on every rank for N > 1 (batch sharding, no communication).

Prints ONE JSON line (rank 0).  `value` = bodies processed by all ranks / max-over-ranks device
time with inputs resident in HBM; `e2e` = the same metric through the public module API with the
step's inputs copied from pinned host memory and the gradients copied back inside the timed region.
`--impl reference` times the reference's CPU path (the PyTorch-eager oracle port, all host threads)
on a bounded sample of the same workload.  `--dump-outputs DIR` writes what the last timed step returned
(rank 0) as DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "SMPL meshes/sec fwd+bwd"
UNIT = "meshes/s"
# algorithmic HBM bytes per mesh of the dominant (skinning) kernels, SURVEY.md section 8(d) / DESIGN.md
LBS_FWD_BYTES = 82680 + 1152 + 82680                 # v_posed in, A in, vertices out
LBS_BWD_BYTES = 82680 + 82680 + 1152 + 82680 + 1152  # dV in, v_posed in, A in, dv_posed out, dA out
KERNEL_BYTES = {"lbs_fwd": LBS_FWD_BYTES, "lbs_bwd": LBS_BWD_BYTES}
# tensor-pipe kernels: bf16 MMA FLOPs executed per mesh (fp32 mode = bf16x3 split: 3 products per fp32 product;
# K steps of 16: 3 for the constants+shape slab, 13 per pose product) and the fp32-equivalent algorithmic FLOPs
# of SURVEY.md section 8(d) (2 * 217 * 20670 per mesh, forward and backward-data alike)
ALGO_GEMM_FLOPS = 2 * 217 * 20670


def gemm_flops_per_mesh(kernel, mode, n_pad):
    if kernel == "blend_fwd_umma":
        ksteps = 3 + 13 * (3 if mode == "fp32" else 2)
        return 2.0 * 16 * ksteps * n_pad
    if kernel == "blend_bwd_umma":
        return 2.0 * 224 * n_pad * (3 if mode == "fp32" else 1)
    return None


def measured_tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["bf16_tflops"]), "measured burst (MEASURED_PEAKS.json)"
    return 1590.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    """sha256 over the CUDA sources: ncu-derived numbers committed under profiles/ are only quoted while the
    kernels they were captured from are the kernels being timed."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "soccerplayershapepose_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(csrc, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic():
    """DRAM bytes per launch from the committed `ncu --set full` capture (scripts/ncu_to_profiles.py); {} when the
    capture is missing or was taken from other kernel sources (stale)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    d = json.load(open(p))
    return d if d.get("kernel_source_hash") == kernel_source_hash() else {}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_inputs(B, seed, device):
    from soccerplayershapepose_b200.synthetic_inputs import make_smpl_inputs, make_upstream_grads
    x = make_smpl_inputs(B, seed)
    dV, dJ = make_upstream_grads(B, seed)
    return [t.to(device) for t in (x["betas"], x["rotmats"], x["trans"], dV, dJ)]


DUMP_BODIES = 512              # 512 bodies' vertices are 42 MB: a dump stays under 64 MB at any batch
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs, B):
    """Write the per-body outputs of one step as float32 DIR/<name>.npy, all of them for the same bodies: every body
    when B <= DUMP_BODIES, else a fixed sample of DUMP_BODIES bodies drawn with seed 0 (in ascending order)."""
    if B <= DUMP_BODIES:
        idx = torch.arange(B)
    else:
        idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:DUMP_BODIES].sort().values
    arrays = {name: t.detach()[idx.to(t.device)].float().cpu().numpy() for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md): an in-process
    NVML polling thread (~1 kHz; the timed region is tens of milliseconds, too short for
    `nvidia-smi -lms`), falling back to one nvidia-smi query when NVML is unavailable."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake": 0x80}

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:  # noqa: BLE001
            self.h = None

    def _poll(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((sm, rs))
            except Exception:  # noqa: BLE001
                break
            time.sleep(0.001)

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def stop(self):
        if self.h is None:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20)
                sm, mx = (float(x) for x in out.stdout.strip().split(","))
                return {"sm_mhz": sm, "sm_max_mhz": mx, "reasons": [], "samples": 1, "how": "nvidia-smi after the region"}
            except Exception:  # noqa: BLE001
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        sms = [s for s, _ in self.samples]
        mask = 0
        for _, r in self.samples:
            mask |= int(r)
        try:
            mx = self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            mx = None
        return {"sm_mhz": statistics.median(sms) if sms else None, "sm_max_mhz": mx,
                "reasons": sorted(k for k, bit in self.REASONS.items() if mask & bit), "samples": len(sms),
                "how": "NVML polled during the timed region"}


def timing_report(lib):
    buf = ctypes.create_string_buffer(1 << 16)
    lib.b200smpl_timing_report(buf, 1 << 16)
    out = {}
    for ln in buf.value.decode().splitlines():
        name, n, ms = ln.split()
        out[name] = (int(n), float(ms))
    return out


def cpu_reference_best(steps, warmup, batches, budget_seconds):
    """The CPU arm at its best batch: a short probe of each candidate batch, then the timed run at the winner."""
    probe = {}
    for b in batches:
        probe[b] = cpu_reference_run(2, 1, b)[0]
    best = max(probe, key=probe.get)
    val, ms, n, threads = cpu_reference_run(steps, warmup, best, min_seconds=budget_seconds)
    return val, ms, n, threads, best, {str(k): round(v, 1) for k, v in probe.items()}


_CPU_MODEL = {}


def cpu_reference_run(steps, warmup, sample_B, min_seconds=0.0):
    """The reference's CPU path: PyTorch-eager restatement (oracle/) of models/smpl_official.py on
    the host cores, forward + backward, fp32, all threads."""
    from oracle.smpl_oracle import SMPLOracle, batch_rodrigues
    from soccerplayershapepose_b200.model_io import make_synthetic_smpl
    torch.set_num_threads(os.cpu_count() or 1)
    if "orc" not in _CPU_MODEL:
        _CPU_MODEL["orc"] = SMPLOracle(make_synthetic_smpl(1234), dtype=torch.float32)
    orc = _CPU_MODEL["orc"]
    g = torch.Generator().manual_seed(0)
    betas = torch.randn(sample_B, 10, generator=g)
    pose = torch.randn(sample_B, 72, generator=g) * 0.3
    rot = batch_rodrigues(pose.reshape(-1, 3)).reshape(sample_B, 24, 3, 3)
    trans = torch.rand(sample_B, 3, generator=g) * 2 - 1
    dV = torch.randn(sample_B, 6890, 3, generator=g)
    dJ = torch.randn(sample_B, 90, 3, generator=g)

    def step():
        b, r, t = (x.clone().requires_grad_(True) for x in (betas, rot, trans))
        out = orc.forward_flat(b, r, t, pose2rot=False)
        torch.autograd.backward([out.vertices, out.joints], [dV, dJ])
        return b.grad

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    n = 0
    while n < steps or (time.perf_counter() - t0) < min_seconds:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return sample_B * n / dt, dt / n * 1e3, n, torch.get_num_threads()


def eager_gpu_reference_run(dev, B=4096, iters=5, warmup=3):
    """SURVEY.md section 8d: the same PyTorch-eager restatement run on the GPU (what the reference's own
    torch path does on a CUDA device) -- reported inside `cpu_baseline` as a second comparison point."""
    from oracle.smpl_oracle import SMPLOracle, batch_rodrigues
    from soccerplayershapepose_b200.model_io import make_synthetic_smpl
    orc = SMPLOracle(make_synthetic_smpl(1234), dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev).manual_seed(0)
    kw = dict(generator=g, device=dev)
    betas = torch.randn(B, 10, **kw)
    rot = batch_rodrigues((torch.randn(B, 72, **kw) * 0.3).reshape(-1, 3)).reshape(B, 24, 3, 3)
    trans = torch.rand(B, 3, **kw) * 2 - 1
    dV, dJ = torch.randn(B, 6890, 3, **kw), torch.randn(B, 90, 3, **kw)

    def step():
        b, r, t = (x.clone().requires_grad_(True) for x in (betas, rot, trans))
        out = orc.forward_flat(b, r, t, pose2rot=False)
        torch.autograd.backward([out.vertices, out.joints], [dV, dJ])

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    return {"value": B / ms * 1e3, "unit": UNIT, "sample": "oracle port (PyTorch eager) on the GPU, fwd+bwd at batch %d, "
            "%d iterations, %.2f ms each" % (B, iters, ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--batch-per-gpu", type=int, default=4096)
    ap.add_argument("--global-batch", type=int, default=0,
                    help="fixed total batch split evenly over the GPUs (BASELINE.json configs[3]: 65536): strong scaling")
    ap.add_argument("--model", default="compact", choices=["compact", "wide"],
                    help="sparsity statistics of the synthetic model (model_io.make_synthetic_smpl)")
    ap.add_argument("--slab", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0, help="CPU-arm batch per step; 0 = best of 64 / 256 / 1024")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sustain-seconds", type=float, default=2.0,
                    help="extra leg: the same step repeated for this long with NVML clocks (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained / small-batch / forward-only legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned on rank 0 (vertices, joints and the "
                         "gradients of betas, rotation matrices and translation; float32, at most %d bodies) as "
                         "DIR/<name>.npy" % DUMP_BODIES)
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        raise SystemExit("--dump-outputs writes the outputs of the timed device path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    B = args.batch_per_gpu
    strong = args.global_batch > 0
    if strong:
        if args.global_batch % world:
            raise SystemExit("--global-batch must divide evenly over the GPUs")
        B = args.global_batch // world
    cpu_batches = [args.cpu_sample] if args.cpu_sample > 0 else [64, 256, 1024]

    config = {"workload": "BASELINE.json configs[%d]: batched SMPL forward+backward, batch %d per GPU, neutral-model "
                          "shapes (6890 verts, 24 joints, 10 betas, 90 output joints), synthetic model seed 1234 (%s "
                          "sparsity statistics)" % (3 if strong else 1, B, args.model),
              "batch_per_gpu": B, "global_batch": B * world, "mode": args.mode,
              "parallelism": "batch-sharded x%d, no communication" % world,
              "l2": "inputs larger than L2 (dV alone is %.0f MB per step)" % (B * 82680 / 1e6),
              "cpu_arm": "--impl reference / cpu_baseline time bounded samples of this workload on the host cores: "
                         "one forward+backward per step at the best of batch %s (probed in the run)" % cpu_batches}

    if args.impl == "reference":
        if rank != 0:
            return 0
        val, ms, n, threads, best, probe = cpu_reference_best(args.steps, args.warmup, cpu_batches, 0.0)
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong" if strong else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                                 "sample": "oracle port (PyTorch eager CPU) fwd+bwd, batch %d per step (NOT the GPU "
                                           "arm's %d); probe meshes/s per batch: %s" % (best, B, probe)},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the SMPL path has no CPU fallback")
    import torch.distributed as dist
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from soccerplayershapepose_b200 import _lib
    from soccerplayershapepose_b200.model_io import make_synthetic_smpl
    from soccerplayershapepose_b200.smpl import SMPLLayer
    lib = _lib.load()
    model = make_synthetic_smpl(1234, statistics=args.model)
    layer = SMPLLayer(model, mode=args.mode, slab_bodies=args.slab).to(dev)
    eng = layer._engine(dev)
    mode = _lib.MODES[args.mode]
    betas, rot, trans, dV, dJ = make_inputs(B, seed=rank, device=dev)

    def step():
        """One forward + backward; returns what a caller of this path receives."""
        v, j, _, saved = eng.forward(betas, rot, trans, None, mode=mode, slab=args.slab, save=True)
        g_betas, g_rot, g_trans, _ = eng.backward(betas, rot, trans, None, None, dV, dJ, None, mode=mode,
                                                  slab=args.slab, saved=saved)
        return {"vertices": v, "joints": j, "grad_betas": g_betas, "grad_rotmats": g_rot.view(B, 24, 3, 3),
                "grad_trans": g_trans}

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # warm-up and timed steps alike hold one step's outputs while the next runs: the same allocations in both
    for _ in range(warmup):
        last = step()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.b200smpl_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    sync_all()
    launches = lib.b200smpl_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, B)
    del last
    from soccerplayershapepose_b200 import sharding
    ms_total = sharding.max_over_ranks(ms_total, dev)           # the slowest rank decides
    value = sharding.aggregate_throughput(B, world, args.steps, ms_total)

    # ---- per-kernel device times over the same K steps (events on the launching stream) ----
    lib.b200smpl_timing_enable(1)
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize(dev)
    lib.b200smpl_timing_enable(0)
    kt = timing_report(lib)
    peak, peak_src = measured_peaks()
    tpeak, tpeak_src = measured_tensor_peak()
    step_ms_timed = sum(ms for _, ms in kt.values()) / args.steps
    traffic = ncu_traffic()
    n_pad = int(eng.info.num_blend_rows_padded)

    def kernel_roofline(k):
        n_launch, ms = kt[k]
        per_launch_ms = ms / n_launch
        bodies_per_launch = B * args.steps / n_launch
        tr = traffic.get(k) if (traffic.get("batch") == bodies_per_launch and args.mode == "fp32") else None
        common = {"kernel": k, "avg_launch_ms": per_launch_ms, "share_of_step": ms / args.steps / step_ms_timed,
                  "traffic": tr}
        if k in KERNEL_BYTES:
            achieved = KERNEL_BYTES[k] * bodies_per_launch / (per_launch_ms / 1e3) / 1e9
            return dict(common, bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                        peak_source=peak_src, bytes_per_mesh=KERNEL_BYTES[k])
        fl = gemm_flops_per_mesh(k, args.mode, n_pad)
        if fl is not None:
            achieved = fl * bodies_per_launch / (per_launch_ms / 1e3) / 1e12
            algo = ALGO_GEMM_FLOPS * bodies_per_launch / (per_launch_ms / 1e3) / 1e12
            return dict(common, bound="tensor", achieved=achieved, peak=tpeak, unit="TFLOP/s", frac=achieved / tpeak,
                        peak_source=tpeak_src, flops_per_mesh=fl,
                        note="achieved = bf16 MMA FLOPs executed (bf16x3 split in fp32 mode); fp32-equivalent "
                             "algorithmic rate %.1f TFLOP/s" % algo)
        return None

    dom = max(kt, key=lambda k: kt[k][1], default=None)
    roofline = kernel_roofline(dom) if dom is not None else None
    if roofline is not None:
        roofline["kernels_ms_per_step"] = {k: v[1] / args.steps for k, v in sorted(kt.items())}
        roofline["others"] = {k: {kk: vv for kk, vv in r.items() if kk in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
                              for k in ("lbs_fwd", "lbs_bwd", "blend_fwd_umma", "blend_bwd_umma") if k in kt and k != dom
                              for r in [kernel_roofline(k)] if r is not None}

    # ---- end to end through the public module API, host buffers in, gradients out ----
    # Every step copies ITS inputs from pinned host memory and ITS gradients back to pinned host memory; as in any
    # input pipeline the copies run on their own streams (double-buffered), so the H2D of step i+1 and the D2H of
    # step i-1 overlap the kernels of step i.  The timed region ends when the last step's gradients are on the host.
    hb, hr, ht = (x.cpu().pin_memory() for x in (betas, rot, trans))
    cur = torch.cuda.current_stream(dev)
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_in = [[torch.empty_like(x, device=dev) for x in (hb, hr, ht)] for _ in range(2)]
    h_out = [[torch.empty((B, 10)).pin_memory(), torch.empty((B, 24, 3, 3)).pin_memory(), torch.empty((B, 3)).pin_memory()]
             for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_used = [torch.cuda.Event() for _ in range(2)]
    ev_grad = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        k = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_used[k])                    # the step that read this slot has finished with it
            for dst, src in zip(d_in[k], (hb, hr, ht)):
                dst.copy_(src, non_blocking=True)
            ev_in[k].record(s_in)

    def e2e_run(n):
        for k in range(2):
            ev_used[k].record(cur)
            ev_out[k].record(s_out)
        prefetch(0)
        for i in range(n):
            k = i & 1
            if i + 1 < n:
                prefetch(i + 1)
            cur.wait_event(ev_in[k])
            b, r, tt = (x.detach().requires_grad_(True) for x in d_in[k])
            v, j = layer(b, r, tt)
            torch.autograd.backward([v, j], [dV, dJ])
            ev_used[k].record(cur)
            ev_grad[k].record(cur)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_grad[k])
                ev_out[k].synchronize()                    # the host buffers of this slot were consumed two steps ago
                for dst, src in zip(h_out[k], (b.grad, r.grad, tt.grad)):
                    dst.copy_(src, non_blocking=True)
                    src.record_stream(s_out)
                ev_out[k].record(s_out)
        s_out.synchronize()                                # the last step's result is on the host
        cur.synchronize()

    e2e_run(4)
    sync_all()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    sync_all()
    e2e_val = B * world * args.steps / sharding.max_over_ranks(time.perf_counter() - t0, dev)
    io_bytes = B * (10 + 216 + 3) * 4

    extras = {}
    if not args.no_extras and rank == 0 and world == 1:
        # ---- sustained leg: the same step back to back for >= 2 s, clocks polled (the headline is a 12 ms burst) ----
        if args.sustain_seconds > 0:
            n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / (ms_total / args.steps)) + 1)
            samp = ClockSampler(local_rank)
            torch.cuda.synchronize(dev)
            samp.start()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(n_sus):
                step()
            s1.record()
            torch.cuda.synchronize(dev)
            sus_ms = s0.elapsed_time(s1)
            extras["sustained"] = {"seconds": sus_ms / 1e3, "steps": n_sus, "ms_per_step": sus_ms / n_sus,
                                   "value": B * n_sus / (sus_ms / 1e3), "unit": UNIT, "clocks": samp.stop()}

        # ---- forward only on the device (no products kept for a backward: the fused blend + skinning kernel) ----
        def fwd_device():
            eng.forward(betas, rot, trans, None, mode=mode, slab=args.slab)
        for _ in range(3):
            fwd_device()
        torch.cuda.synchronize(dev)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            fwd_device()
        f1.record()
        torch.cuda.synchronize(dev)
        fwd_ms = f0.elapsed_time(f1) / args.steps
        lib.b200smpl_timing_enable(1)
        for _ in range(args.steps):
            fwd_device()
        torch.cuda.synchronize(dev)
        lib.b200smpl_timing_enable(0)
        fkt = timing_report(lib)
        fwd_bytes = 82680 + 90 * 12 + (10 + 216 + 3) * 4          # vertices + joints out, inputs in: the fused lower bound
        extras["forward_only_device"] = {
            "ms_per_step": fwd_ms, "value": B / (fwd_ms / 1e3), "unit": "meshes/s (forward only)",
            "kernels_ms_per_step": {k: v[1] / args.steps for k, v in sorted(fkt.items())},
            "roofline": {"bound": "hbm", "achieved": B * fwd_bytes / (fwd_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": B * fwd_bytes / (fwd_ms / 1e3) / 1e9 / peak, "bytes_per_mesh": fwd_bytes,
                         "note": "algorithmic bytes of the fully fused forward (SURVEY.md section 8d); v_posed stays on "
                                 "chip (csrc/fused_fwd.cu), joints still read their virtual rows from HBM"}}

        # ---- small batches (the reference's own regime: SMPL(batch_size=1), player_recon.py:147) ----
        def timed(fn, n=50):
            for _ in range(5):
                fn()
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b) / n

        small = {}
        for sb in (1, 64):
            bs, rs, ts, dVs, dJs = betas[:sb], rot[:sb], trans[:sb], dV[:sb].contiguous(), dJ[:sb].contiguous()

            def fwd_only():
                eng.forward(bs, rs, ts, None, mode=mode)

            def fwd_bwd():
                sv = eng.forward(bs, rs, ts, None, mode=mode, save=True)[3]
                eng.backward(bs, rs, ts, None, None, dVs, dJs, None, mode=mode, saved=sv)

            small[str(sb)] = {"forward_ms": timed(fwd_only), "forward_backward_ms": timed(fwd_bwd)}
        extras["small_batch_latency"] = small

        # ---- forward-only e2e, vertices copied to the host every step (predict_3D.py:139-155) ----
        # inputs from pinned host memory, vertices + joints to pinned host memory on a copy stream (double-buffered);
        # this leg is PCIe-bound: its roofline is the measured D2H copy rate of the same bytes
        hv = [torch.empty((B, 6890, 3)).pin_memory() for _ in range(2)]
        hj = [torch.empty((B, 90, 3)).pin_memory() for _ in range(2)]
        dv_out = [torch.empty((B, 6890, 3), device=dev) for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_copied = [torch.cuda.Event() for _ in range(2)]

        def fwd_e2e(n):
            for k in range(2):
                ev_copied[k].record(s_out)
            prefetch(0)
            for i in range(n):
                k = i & 1
                if i + 1 < n:
                    prefetch(i + 1)
                cur.wait_event(ev_in[k])
                cur.wait_event(ev_copied[k])                   # the slot's previous vertices have left the device
                with torch.no_grad():
                    v, j = layer(*d_in[k])
                dv_out[k].copy_(v)                              # keeps the step's output alive in a fixed slot
                ev_used[k].record(cur)
                ev_done[k].record(cur)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_done[k])
                    hv[k].copy_(dv_out[k], non_blocking=True)
                    hj[k].copy_(j, non_blocking=True)
                    j.record_stream(s_out)
                    ev_copied[k].record(s_out)
            s_out.synchronize()
            cur.synchronize()

        for k in range(2):
            ev_used[k].record(cur)
        fwd_e2e(4)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fwd_e2e(args.steps)
        torch.cuda.synchronize(dev)
        fwd_val = B * args.steps / (time.perf_counter() - t0)
        d2h_bytes = B * (6890 + 90) * 12
        torch.cuda.synchronize(dev)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            hv[0].copy_(dv_out[0], non_blocking=True)
        c1.record()
        torch.cuda.synchronize(dev)
        d2h_gbs = 5 * B * 6890 * 12 / (c0.elapsed_time(c1) / 1e3) / 1e9
        extras["e2e_forward_vertices_to_host"] = {
            "value": fwd_val, "unit": "meshes/s (forward only)", "h2d_bytes_per_step": io_bytes,
            "d2h_bytes_per_step": d2h_bytes,
            "roofline": {"bound": "pcie d2h", "achieved": fwd_val * (d2h_bytes / B) / 1e9, "peak": d2h_gbs, "unit": "GB/s",
                         "frac": fwd_val * (d2h_bytes / B) / 1e9 / d2h_gbs,
                         "peak_source": "pinned D2H copy of one step's vertices, measured in this run"}}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        val, ms, n, threads, best, probe = cpu_reference_best(5, 3, cpu_batches, 10.0)
        cpu_baseline = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": "oracle port (PyTorch eager CPU, fp32) fwd+bwd at batch %d (best of %s: %s meshes/s), "
                                  "%d iterations, %.1f ms each" % (best, cpu_batches, probe, n, ms)}
        try:
            cpu_baseline["torch_eager_gpu"] = eager_gpu_reference_run(dev, B=B)
        except Exception as e:  # a comparison point only: never fail the bench line on it
            cpu_baseline["torch_eager_gpu"] = {"unavailable": repr(e)[:200]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": "f32 (bf16x3 split on tcgen05, fp32 accumulate)" if args.mode == "fp32" else "bf16-GEMM / f32",
                "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline}
        if cpu_baseline is not None:
            line["vs_cpu_baseline"] = {"device": value / cpu_baseline["value"], "e2e": e2e_val / cpu_baseline["value"],
                                       "note": "vs_baseline stays null: BASELINE.md holds no published number"}
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
