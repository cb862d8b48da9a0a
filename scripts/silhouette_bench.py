"""Timings of the silhouette rasteriser (csrc/silhouette.cu) on the GPU; writes profiles/r03_silhouette_<tag>.json.

Device-event timings after warm-up of: the render forward, forward + backward and the fused loss at
B in {64, 1024}, S in {256, 512}, sigma in {0, 1}; the same soft render restated in fp32 PyTorch eager on the GPU
(oracle/silhouette_oracle.py: every (face, pixel) pair inside the face's grown box, autograd backward) at B = 64;
a BatchedFitter iteration with and without the silhouette term at 1024 players.  Face-pixel pairs are counted from
the kernels' bins (32 x 8 tiles met by each face's grown box, 256 pixels each).  The card's name and power limit are
read in the same run.  Bodies: 64 distinct posed synthetic bodies, repeated down the batch.

    python scripts/silhouette_bench.py [--tag b200] [--quick]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import silhouette_oracle as SO  # noqa: E402
from oracle import smpl_oracle as O  # noqa: E402
from soccerplayershapepose_b200 import config, ops  # noqa: E402
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch  # noqa: E402
from soccerplayershapepose_b200.fitting import BatchedFitter  # noqa: E402
from soccerplayershapepose_b200.model_io import make_synthetic_smpl  # noqa: E402
from soccerplayershapepose_b200.smpl import SMPL  # noqa: E402

DEV = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, warm=3, reps=10):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bodies(smpl, B, seed=0):
    g = torch.Generator().manual_seed(seed)
    P = min(B, 64)
    betas = torch.randn(P, 10, generator=g)
    pose = torch.randn(P, 72, generator=g) * 0.3
    cam = torch.stack([torch.rand(P, generator=g) * 0.6 + 0.6, torch.rand(P, generator=g) * 0.4 - 0.2,
                       torch.rand(P, generator=g) * 0.4 - 0.2], 1).to(DEV)
    with torch.no_grad():
        v = smpl(betas=betas.to(DEV), body_pose=pose[:, 3:].to(DEV), global_orient=pose[:, :3].to(DEV)).vertices
    t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, 512)
    rep = (B + P - 1) // P
    return v.repeat(rep, 1, 1)[:B].contiguous(), t.repeat(rep, 1)[:B].contiguous()


def pairs_from_bins(v, t, faces, S, f, sigma):
    """Face-pixel pairs the kernels evaluate: sum over kept faces of (32x8 tiles met by the grown box) x 256."""
    tri, kept, _ = SO.face_table(v, t, faces, f, S)
    pad = (math.sqrt(SO.cutoff_d2(sigma)) if sigma > 0 else 0.0) + 1e-2
    lo, hi = tri.min(2).values, tri.max(2).values
    c0 = torch.floor((lo[..., 0] - pad - 0.5) / 32).clamp(min=0)
    c1 = torch.floor((hi[..., 0] + pad - 0.5) / 32).clamp(max=(S - 1) // 32)
    r0 = torch.floor((lo[..., 1] - pad - 0.5) / 8).clamp(min=0)
    r1 = torch.floor((hi[..., 1] + pad - 0.5) / 8).clamp(max=(S - 1) // 8)
    n = ((c1 - c0 + 1).clamp(min=0) * (r1 - r0 + 1).clamp(min=0)) * kept
    return float(n.sum()) * 256


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    ap.add_argument("--out", default=None, help="output path (default profiles/r03_silhouette_<tag>.json)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "silhouette_bench needs a CUDA device"
    smpl = SMPL(model_data=make_synthetic_smpl(1234)).to(DEV)
    faces = smpl.faces_int32(DEV)
    res = {"card": card(), "render": [], "eager": [], "fitter": []}
    Bs, Ss = ([8], [64]) if a.quick else ([64, 1024], [256, 512])
    for B in Bs:
        v, t = bodies(smpl, B)
        for S in Ss:
            f = config.FOCAL_LENGTH * S / 512
            for sigma in (0.0, 1.0):
                row = {"B": B, "S": S, "sigma": sigma}
                row["fwd_ms"] = timed(lambda: ops.render_silhouettes(v, faces, t, S, f, sigma))
                pairs = pairs_from_bins(v[:64], t[:64], faces, S, f, sigma) * (B / min(B, 64))
                row["pairs_per_call"] = pairs
                row["fwd_pairs_per_s"] = pairs / (row["fwd_ms"] * 1e-3)
                if sigma > 0:
                    vv = v.clone().requires_grad_(True)
                    g = torch.randn(B, S, S, device=DEV)

                    def fb():
                        vv.grad = None
                        ops.render_silhouettes(vv, faces, t, S, f, sigma).backward(g)
                    row["fwd_bwd_ms"] = timed(fb)
                    target = ops.render_silhouettes(v * 1.02, faces, t, S, f, 0.0) > 0.5
                    lpb = torch.zeros(B, device=DEV)
                    row["fused_loss_ms"] = timed(lambda: ops.silhouette_loss(v, faces, t, target, S, f, sigma, 1.0, lpb))
                res["render"].append(row)
                print(json.dumps(row), flush=True)
    # fp32 eager restatement on the GPU (soft, forward + autograd backward), against the kernels at the same B
    Be = 8 if a.quick else 64
    v, t = bodies(smpl, Be)
    for S in Ss:
        f = config.FOCAL_LENGTH * S / 512
        vv = v.clone().requires_grad_(True)
        g = torch.randn(Be, S, S, device=DEV)

        def eager():
            vv.grad = None
            SO.render(vv, faces, t, S, f, 1.0).backward(g)
        torch.cuda.reset_peak_memory_stats()
        row = {"B": Be, "S": S, "sigma": 1.0, "eager_fwd_bwd_ms": timed(eager, warm=1, reps=3),
               "eager_peak_gb": torch.cuda.max_memory_allocated() / 1e9}
        target = ops.render_silhouettes(v * 1.02, faces, t, S, f, 0.0) > 0.5
        lpb = torch.zeros(Be, device=DEV)
        row["fused_loss_ms"] = timed(lambda: ops.silhouette_loss(v, faces, t, target, S, f, 1.0, 1.0, lpb))
        row["speedup_fused_vs_eager"] = row["eager_fwd_bwd_ms"] / row["fused_loss_ms"]
        res["eager"].append(row)
        print(json.dumps(row), flush=True)
    # one BatchedFitter iteration with and without the silhouette term
    P = 16 if a.quick else 1024
    g = torch.Generator().manual_seed(3)
    betas = torch.randn(P, 10, generator=g) * 0.8
    rot = O.batch_rodrigues((torch.randn(P, 72, generator=g) * 0.25).reshape(-1, 3)).reshape(P, 24, 3, 3).float()
    cam = torch.stack([0.6 + 0.6 * torch.rand(P, generator=g), 0.4 * torch.rand(P, generator=g) - 0.2,
                       0.4 * torch.rand(P, generator=g) - 0.2], 1)
    label = torch.rand(P, 17, 2, generator=g) * 512
    d = lambda x: x.to(DEV)  # noqa: E731
    for S in ([64] if a.quick else [64, 128, 256]):
        for w in (0.0, 1.0):
            fitter = BatchedFitter(smpl, lr=1e-3, silhouette_weight=w, silhouette_wh=S, graph_iterations=20)
            sil = torch.rand(P, S, S, generator=g).to(DEV) > 0.5 if w > 0 else None
            iters = 41
            fitter.fit(d(rot), d(betas), d(cam), d(label), iterations=iters, silhouettes=sil)    # capture
            ms = timed(lambda: fitter.fit(d(rot), d(betas), d(cam), d(label), iterations=40, silhouettes=sil),
                       warm=1, reps=3)
            row = {"players": P, "silhouette_wh": S, "silhouette_weight": w, "ms_per_iteration": ms / 40}
            res["fitter"].append(row)
            print(json.dumps(row), flush=True)
    out = a.out or os.path.join(ROOT, "profiles", "r03_silhouette_{}.json".format(a.tag))
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
