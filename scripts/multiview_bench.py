#!/usr/bin/env python
"""Multi-view fitting (the reference's multi_view_optimization, PlayerReconstruction/player_recon.py:1568-1999, at
its own schedule: 3 rounds x 2 phases x 50 epochs, global_var.py:79 / player_recon.py:1720) for P synthetic players
seen from V views: multiview_bench.py [P] [V] [epochs] [out.json].  Times the CUDA-graph path and the eager path.

--silhouette-weight W (> 0) adds the silhouette term at --sil-res S pixels and blur --sil-sigma s, with the hard
renders of the true parameters per view as targets; the line then also carries the mean IoU of the start and of the
result.  The card's name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ClockSampler                                                  # noqa: E402
from soccerplayershapepose_b200 import config, ops                              # noqa: E402
from soccerplayershapepose_b200.fitting import MultiViewFitter                  # noqa: E402
from soccerplayershapepose_b200.model_io import make_synthetic_smpl             # noqa: E402
from soccerplayershapepose_b200.smpl import SMPL                                # noqa: E402
from soccerplayershapepose_b200.synthetic_inputs import axis_angle_to_rotmat    # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("P", type=int, nargs="?", default=1024)
ap.add_argument("V", type=int, nargs="?", default=4)
ap.add_argument("epochs", type=int, nargs="?", default=50)
ap.add_argument("out_path", nargs="?", default=None)
ap.add_argument("--silhouette-weight", type=float, default=0.0)
ap.add_argument("--sil-res", type=int, default=256)
ap.add_argument("--sil-sigma", type=float, default=1.0)
a = ap.parse_args()
P, V, epochs, out_path = a.P, a.V, a.epochs, a.out_path
use_sil = a.silhouette_weight > 0.0
dev = torch.device("cuda", 0)
smpl = SMPL(model_data=make_synthetic_smpl(1234), mode="fp32").to(dev)
g = torch.Generator().manual_seed(0)
betas_t = torch.randn(P, 10, generator=g) * 0.8
bp_aa = torch.randn(P, 69, generator=g) * 0.25
go_aa = torch.randn(P, V, 3, generator=g) * 0.6
cam_t = torch.stack([0.6 + 0.6 * torch.rand(P, V, generator=g), 0.4 * torch.rand(P, V, generator=g) - 0.2,
                     0.4 * torch.rand(P, V, generator=g) - 0.2], -1)
rm = lambda aa: axis_angle_to_rotmat(aa.double().reshape(-1, 3)).float()   # noqa: E731
bp_t, go_t = rm(bp_aa).reshape(P, 23, 3, 3), rm(go_aa).reshape(P, V, 3, 3)
label = torch.empty(P, V, 17, 2, device=dev)
sil = torch.empty(P, V, a.sil_res, a.sil_res, dtype=torch.bool, device=dev) if use_sil else None
with torch.no_grad():
    for v in range(V):
        o = smpl(betas=betas_t.to(dev), body_pose=bp_t.to(dev), global_orient=go_t[:, v:v + 1].to(dev), pose2rot=False,
                 return_verts=use_sil)
        label[:, v] = ops.orthographic_project(o.joints, cam_t[:, v].to(dev), 512.0)[:, config.SMPL_TO_KPRCNN_MAP, :]
        if use_sil:
            sil[:, v] = smpl.render_silhouettes(o.vertices, cam_t[:, v].to(dev), img_wh=a.sil_res, sigma=0.0) > 0.5
betas0 = (betas_t + 0.5 * torch.randn(P, 10, generator=g)).to(dev)
bp0 = rm(bp_aa + 0.15 * torch.randn(P, 69, generator=g)).reshape(P, 23, 3, 3).to(dev)
go0 = rm(go_aa + 0.1 * torch.randn(P, V, 3, generator=g)).reshape(P, V, 3, 3).to(dev)
cam0 = (cam_t + 0.05 * torch.randn(P, V, 3, generator=g)).to(dev)
sil_kw = dict(silhouette_weight=a.silhouette_weight, silhouette_sigma=a.sil_sigma, silhouette_wh=a.sil_res)
res = {}
for use_graph in (True, False):
    fitter = MultiViewFitter(smpl, lr=1e-3, rounds=3, use_cuda_graph=use_graph, **sil_kw)
    fitter.fit(bp0, betas0, go0, cam0, label, iterations=2, silhouettes=sil)   # warm-up: allocations, captures
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    r = fitter.fit(bp0, betas0, go0, cam0, label, iterations=epochs, silhouettes=sil)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    res["graph" if use_graph else "eager"] = (dt, sampler.stop(), r["initial_loss"].mean().item(), r["best_loss"].mean().item(),
                                              r["silhouette_iou"].mean().item() if use_sil else None)
steps = 3 * 2 * epochs * V
loss = "joints2D loss" + (" + %g x silhouette term (S = %d, sigma = %g, targets: hard renders of the truth)"
                          % (a.silhouette_weight, a.sil_res, a.sil_sigma) if use_sil else "")
line = {"workload": "multi-view fitting: %d players x %d views, 3 rounds x 2 phases x %d epochs (one Adam step per view and "
                    "epoch + a validation pass), lr 1e-3, %s, %s SMPL path"
                    % (P, V, epochs, loss, "full-vertex" if use_sil else "joints-only"),
        "seconds_cuda_graph": res["graph"][0], "seconds_eager": res["eager"][0], "view_steps": steps,
        "us_per_view_step_incl_validation": res["graph"][0] / steps * 1e6,
        "player_view_steps_per_s": P * steps / res["graph"][0], "clocks": res["graph"][1],
        "mean_loss_first_epoch": res["graph"][2], "mean_loss_best": res["graph"][3],
        "eager_mean_loss_best": res["eager"][3]}
if use_sil:
    line["mean_iou_initial"] = fitter.silhouette_iou(bp0, betas0, go0, cam0, sil).mean().item()
    line["mean_iou_best"] = res["graph"][4]
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True)
line["card"] = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}
print(json.dumps(line))
if out_path:
    json.dump(line, open(out_path, "w"), indent=1)
