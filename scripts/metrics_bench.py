#!/usr/bin/env python
"""The reconstruction-error kernel (csrc/metrics.cu) and regressor.validation_step on one GPU.

  python scripts/metrics_bench.py [--out profiles/r07_metrics_b200.json] [--iters 50]

Kernel: B in {256, 1024, 4096} distinct posed bodies of the synthetic SMPL model (6890 vertices, the 14 LSP joints of
90) with noisy, rotated predictions; CUDA events, mean over --iters launches after warm-up.  The working set is 42 MB
at B = 256 and 169 / 677 MB at the larger sizes (above the 126 MB L2), so at those sizes each call reads from HBM.
The algorithmic bytes per body are 2 V 12 + 2 14 12 (each point read once); the read rate is compared with a
`copy_` of the same number of bytes timed in the same run.  In the same run, two other ways to get the same numbers:
the reference's path (device -> host copy + the float64 numpy transcription of utils/eval_utils.py) and a torch-eager
restatement on the GPU with batched torch.linalg.svd.  Then validation_step against train_step for the head-only
regressor (512-d features, 256 crops, fused loss).  The card's name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import metrics_oracle as M                                  # noqa: E402
from soccerplayershapepose_b200 import config, ops, regressor          # noqa: E402
from soccerplayershapepose_b200.model_io import make_synthetic_smpl    # noqa: E402
from soccerplayershapepose_b200.smpl import SMPL                        # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--iters", type=int, default=50)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("metrics_bench needs a CUDA device")
dev = torch.device("cuda", 0)
J14 = torch.tensor(config.ALL_JOINTS_TO_J14_MAP, dtype=torch.int32, device=dev)


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


smpl = SMPL(model_data=make_synthetic_smpl(1234), mode="fp32").to(dev)


def bodies(B, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    betas = torch.randn(B, 10, device=dev, generator=g)
    pose = torch.randn(B, 72, device=dev, generator=g) * 0.3
    transl = (torch.rand(B, 3, device=dev, generator=g) - 0.5) * 20
    with torch.no_grad():
        t = smpl(betas=betas, body_pose=pose[:, 3:], global_orient=pose[:, :3], transl=transl)
        dpose = pose + torch.randn(B, 72, device=dev, generator=g) * 0.1
        p = smpl(betas=betas + 0.3 * torch.randn(B, 10, device=dev, generator=g), body_pose=dpose[:, 3:],
                 global_orient=dpose[:, :3], transl=transl + 0.05)
    return p.vertices, t.vertices, p.joints, t.joints


def torch_eager(pv, tv, pj, tj):
    """The definition restated in eager torch on the GPU (fp32, batched SVD): what a user would write without the
    kernel."""
    def one(P, Q):
        mp, mq = P.mean(1, keepdim=True), Q.mean(1, keepdim=True)
        X, Y = P - mp, Q - mq
        e = (P - Q).norm(dim=-1).mean(1)
        rp, rq = X.pow(2).sum((1, 2)).div(P.shape[1]).sqrt(), Y.pow(2).sum((1, 2)).div(P.shape[1]).sqrt()
        esc = (X * (rq / rp)[:, None, None] - Y).norm(dim=-1).mean(1)
        K = X.transpose(1, 2) @ Y
        U, _, Vh = torch.linalg.svd(K)
        V = Vh.transpose(1, 2)
        d = torch.linalg.det(V @ U.transpose(1, 2))
        D = torch.diag_embed(torch.stack([torch.ones_like(d), torch.ones_like(d), d], 1))
        R = V @ D @ U.transpose(1, 2)
        s = torch.diagonal(R @ K, dim1=1, dim2=2).sum(1) / X.pow(2).sum((1, 2))
        epa = (s[:, None, None] * X @ R.transpose(1, 2) - Y).norm(dim=-1).mean(1)
        return torch.stack([e, esc, epa], 1)
    jl = J14.long()
    return torch.cat([one(pv, tv), one(pj[:, jl], tj[:, jl])], 1)


def reference_path(pv, tv, pj, tj):
    """The tracker's path: the meshes to the host, then the float64 numpy transcription of the reference."""
    h = [t.cpu().numpy() for t in (pv, tv, pj, tj)]
    m = np.asarray(config.ALL_JOINTS_TO_J14_MAP)
    return np.concatenate([M.reference_errors(h[0], h[1]), M.reference_errors(h[2][:, m], h[3][:, m])], 1)


rec = {"workload": "reconstruction errors, 6890 vertices + 14 of 90 joints per body, fp32 inputs",
       "card": card(), "kernel": []}
for B in (256, 1024, 4096):
    pv, tv, pj, tj = bodies(B, B)
    V = pv.shape[1]
    nbytes = B * (2 * V * 12 + 2 * 14 * 12)
    src = torch.empty(nbytes // 4, device=dev)
    dst = torch.empty_like(src)
    run = lambda: ops.reconstruction_errors(pv, tv, pj, tj, J14)      # noqa: E731
    ms_k = timed(run, args.iters)
    ms_c = timed(lambda: dst.copy_(src), args.iters)
    ms_k = min(ms_k, timed(run, args.iters))    # the kernel before and after the copy, the better of the two
    ms_t = timed(lambda: torch_eager(pv, tv, pj, tj), max(5, args.iters // 5))
    got = run().double().cpu().numpy()
    eager_diff = float(np.nanmax(np.abs(torch_eager(pv, tv, pj, tj).double().cpu().numpy() - got)))
    line = {"B": B, "bytes": nbytes, "kernel_ms": ms_k, "kernel_read_GBps": nbytes / ms_k / 1e6,
            "copy_ms": ms_c, "copy_GBps": nbytes / ms_c / 1e6, "fraction_of_copy": ms_c / ms_k,
            "torch_eager_ms": ms_t, "torch_eager_max_abs_diff_m": eager_diff}
    if B == 256:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ref = reference_path(pv, tv, pj, tj)
        line["reference_path_ms"] = (time.perf_counter() - t0) * 1e3
        line["reference_max_abs_diff_m"] = float(np.abs(ref - got).max())
    rec["kernel"].append(line)
    print(json.dumps(line), flush=True)
    del pv, tv, pj, tj, src, dst
    torch.cuda.empty_cache()

# validation_step against train_step: head-only regressor, 512-d features, 256 crops, fused five-term loss
B = 256
torch.manual_seed(0)
head = regressor.IEFModule().to(dev)
crit = regressor.MultiTaskLoss(("verts", "joints2D", "joints3D", "shape_params", "pose_params")).to(dev)
opt = torch.optim.Adam(list(head.parameters()) + list(crit.parameters()), lr=1e-4)
g = torch.Generator(device=dev).manual_seed(1)
feats = torch.randn(B, 512, device=dev, generator=g)
pv, tv, pj, tj = bodies(B, 7)
rot = ops.batch_rodrigues(torch.randn(B * 24, 3, device=dev, generator=g) * 0.3).view(B, 24, 3, 3)
labels = {"verts": tv, "joints2D": torch.rand(B, 17, 2, device=dev, generator=g) * 256,
          "joints3D": tj[:, config.ALL_JOINTS_TO_COCO_MAP], "shape_params": torch.randn(B, 10, device=dev, generator=g),
          "pose_params_rot_matrices": rot}
g6, _ = regressor.gpu_ops()
sums = torch.zeros(7, device=dev)


def val():
    _, errors = regressor.validation_step(head, crit, smpl, feats, labels, g6, None, fused_loss=True)
    sums.add_(errors.sum(0))


step = {"batch": B, "features": 512,
        "train_step_ms": timed(lambda: regressor.train_step(head, crit, opt, smpl, feats, labels, g6, None,
                                                             fused_loss=True), 20),
        "validation_step_ms": timed(val, 20)}
step["train_step_ms_after"] = timed(lambda: regressor.train_step(head, crit, opt, smpl, feats, labels, g6, None,
                                                                  fused_loss=True), 20)
rec["steps"] = step
print(json.dumps({"steps": step, "card": rec["card"]}), flush=True)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
