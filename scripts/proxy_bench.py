#!/usr/bin/env python
"""The proxy-representation kernel (csrc/proxy.cu) on one GPU: 512 x 512 uint8 masks + 17 keypoints -> 18 x 256 x 256
fp32, both layouts, B in {64, 256, 1024}.

  python scripts/proxy_bench.py [--out profiles/r06_proxy_b200.json] [--iters 50]

Per batch and layout: kernel time by CUDA events (mean over --iters launches after warm-up), the bytes the kernel
must write over that time, and the same for a plain `zero_()` of the same output buffer measured in the same run
(the fill rate the kernel is compared with).  Outputs are 302 MB to 4.8 GB, well past the 126 MB L2.  Then the
host -> device copy of one 256-crop step's inputs from pinned memory with ordinary `copy_(non_blocking=True)`: the raw
inputs (masks, keypoints, vis) against prebuilt fp32 proxies.  The card's name and power limit are read in the same
run and written with the numbers."""
import argparse, json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from soccerplayershapepose_b200 import ops          # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--iters", type=int, default=50)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("proxy_bench needs a CUDA device")
dev = torch.device("cuda", 0)
IN, S, K = 512, 256, 17


def card():
    info = {"name": torch.cuda.get_device_name(dev), "power_limit_w": "not read"}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:                     # noqa: BLE001  (the number is then reported as not read)
        info["power_limit_w"] = "not read ({})".format(type(e).__name__)
    return info


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def inputs(B, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    masks = (torch.rand(B, IN, IN, device=dev, generator=g) > 0.5).to(torch.uint8)
    kp = torch.rand(B, K, 2, device=dev, generator=g) * IN
    vis = torch.rand(B, K, device=dev, generator=g) > 0.1
    return masks, kp, vis


rec = {"workload": "proxy representation 512 -> 256, K = 17 (18 channels), fp32 output", "card": card(), "kernel": []}
for B in (64, 256, 1024):
    masks, kp, vis = inputs(B)
    for cl in (False, True):
        out = torch.empty(B, 1 + K, S, S, device=dev,
                          memory_format=torch.channels_last if cl else torch.contiguous_format)
        nbytes = out.numel() * 4
        ms_k = timed(lambda: ops.proxy_representation(masks, kp, vis, S, channels_last=cl, out=out), args.iters)
        ms_z = timed(lambda: out.zero_(), args.iters)
        ms_k2 = timed(lambda: ops.proxy_representation(masks, kp, vis, S, channels_last=cl, out=out), args.iters)
        ms_k = min(ms_k, ms_k2)                  # the kernel before and after the fill, the better of the two
        line = {"B": B, "layout": "NHWC" if cl else "NCHW", "out_bytes": nbytes,
                "in_bytes": masks.numel() + kp.numel() * 4 + vis.numel(), "kernel_ms": ms_k,
                "kernel_write_GBps": nbytes / ms_k / 1e6, "zero_ms": ms_z, "zero_GBps": nbytes / ms_z / 1e6,
                "fraction_of_fill": ms_z / ms_k}
        rec["kernel"].append(line)
        print(json.dumps(line), flush=True)
        del out
    del masks, kp, vis
    torch.cuda.empty_cache()

# host -> device for one 256-crop step: raw inputs against prebuilt fp32 proxies, from pinned memory
B = 256
raw_h = [torch.zeros(B, IN, IN, dtype=torch.uint8).pin_memory(), torch.zeros(B, K, 2).pin_memory(),
         torch.zeros(B, K, dtype=torch.uint8).pin_memory()]
raw_d = [t.to(dev) for t in raw_h]
prox_h = torch.zeros(B, 1 + K, S, S).pin_memory()
prox_d = torch.empty(B, 1 + K, S, S, device=dev)


def copy_raw():
    for d, h in zip(raw_d, raw_h):
        d.copy_(h, non_blocking=True)


h2d = {"batch": B, "raw_bytes": sum(t.numel() * t.element_size() for t in raw_h),
       "proxy_bytes": prox_h.numel() * 4,
       "raw_ms": timed(copy_raw, 20), "proxy_ms": timed(lambda: prox_d.copy_(prox_h, non_blocking=True), 20)}
h2d["saved_ms_per_step"] = h2d["proxy_ms"] - h2d["raw_ms"]
h2d["raw_GBps"] = h2d["raw_bytes"] / h2d["raw_ms"] / 1e6
h2d["proxy_GBps"] = h2d["proxy_bytes"] / h2d["proxy_ms"] / 1e6
rec["h2d_one_step"] = h2d
print(json.dumps({"h2d_one_step": h2d, "card": rec["card"]}), flush=True)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
