#!/usr/bin/env python
"""BASELINE.json configs[4]: regressor training step -- crops -> ResNet-18 encoder -> IEF head -> SMPL -> multi-task
loss (verts, joints2D, joints3D, shape, pose) -> backward -> gradient all-reduce -> Adam, batch 256 crops per step
per GPU, data-parallel over NCCL when launched under torchrun.  One CUDA graph per step.

  python scripts/regressor_bench.py [--steps 50] [--batch 256] [--input encoder|features] [--res 256]
                                    [--loss fused|eager] [--no-overlap] [--eager]
                                    [--silhouette-weight W [--sil-res S] [--sil-sigma SIGMA]]
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/regressor_bench.py ...

--input encoder (default): the reference's SingleInputRegressor (models/regressor.py: ResNet-18 over 18 x res x res
proxy inputs + IEFModule([512,512])), 11.9 M parameters = 47.6 MB all-reduced per step.  BASELINE.json says 224x224
crops; the reference's regressor input is 18x256x256 (config.REGRESSOR_IMG_WH, PyTorch3DTest.py:241): --res picks.
--input features: synthetic 512-d features into IEFModule([1024,1024]) (the round-1 head-only configuration).
--silhouette-weight W > 0 adds the silhouette term (initial weight W; PyTorch3DTest.py:1084-1087) at S x S pixels:
the targets are the hard silhouettes of the label bodies; the fused loss runs ops.silhouette_term, the eager loss
renders the soft silhouettes first.
Prints one JSON line (rank 0)."""
import argparse, json, os, sys
import torch
import torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from soccerplayershapepose_b200 import config, ops, regressor, sharding          # noqa: E402
from soccerplayershapepose_b200.model_io import make_synthetic_smpl             # noqa: E402
from soccerplayershapepose_b200.smpl import SMPL                                # noqa: E402
from soccerplayershapepose_b200.synthetic_inputs import make_smpl_inputs        # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--input", default="encoder", choices=["encoder", "features"])
ap.add_argument("--res", type=int, default=256)
ap.add_argument("--loss", default="fused", choices=["fused", "eager"])
ap.add_argument("--no-overlap", action="store_true", help="one all-reduce after the backward instead of bucketed overlap")
ap.add_argument("--eager", action="store_true", help="no CUDA graph: eager step (DistributedDataParallel when N > 1)")
ap.add_argument("--amp", action="store_true", help="run the (library, cuDNN) encoder under bf16 autocast; the head, the SMPL "
                                                   "layer and the loss stay fp32")
ap.add_argument("--silhouette-weight", type=float, default=0.0, help="> 0: add the silhouette term at this weight")
ap.add_argument("--sil-res", type=int, default=config.REGRESSOR_IMG_WH, help="silhouette resolution S")
ap.add_argument("--sil-sigma", type=float, default=1.0, help="soft silhouette blur (px^2)")
args = ap.parse_args()
steps, B = args.steps, args.batch
rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
dev = torch.device("cuda", local)
torch.cuda.set_device(dev)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
smpl = SMPL(model_data=make_synthetic_smpl(1234), mode="fp32").to(dev)
torch.manual_seed(0)
if args.input == "encoder":
    head = regressor.SingleInputRegressor(resnet_in_channels=18).to(dev).to(memory_format=torch.channels_last)
    if args.amp:
        enc_fwd = head.image_encoder.forward

        def amp_forward(x):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = enc_fwd(x)
            return y.float()
        head.image_encoder.forward = amp_forward
    feats = torch.randn(B, 18, args.res, args.res, device=dev).contiguous(memory_format=torch.channels_last)
else:
    head = regressor.IEFModule((1024, 1024), in_features=512).to(dev)
    feats = torch.randn(B, 512, device=dev)
sil = args.silhouette_weight > 0
crit = regressor.MultiTaskLoss(("verts", "joints2D", "joints3D", "shape_params", "pose_params") + (("silhouette",) if sil else ()),
                               {"verts": 1.0, "joints2D": 0.1, "joints3D": 1.0, "shape_params": 0.1, "pose_params": 0.1,
                                "silhouette": args.silhouette_weight},
                               faces=smpl.faces_int32(dev) if sil else None, silhouette_sigma=args.sil_sigma,
                               silhouette_wh=args.sil_res).to(dev)
fused = args.loss == "fused"
r6, proj = regressor.gpu_ops()
render = regressor.gpu_silhouette_renderer(smpl.faces_int32(dev), args.sil_res, args.sil_sigma) if sil else None


class Step(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.head, self.crit = head, crit

    def forward(self, f, labels):
        out = regressor.predict(self.head, smpl, f, r6, None if fused else proj,
                                render_silhouettes=None if fused else render)
        return (self.crit.forward_fused(labels, out) if fused else self.crit(labels, out))[0]


x = make_smpl_inputs(B, rank)
rot, betas = x["rotmats"].to(dev), x["betas"].to(dev)
cam = torch.tensor([0.9, 0.0, 0.0], device=dev).repeat(B, 1)
with torch.no_grad():
    t = smpl(betas=betas, body_pose=rot[:, 1:], global_orient=rot[:, :1], pose2rot=False)
    labels = {"verts": t.vertices, "joints3D": t.joints[:, config.ALL_JOINTS_TO_COCO_MAP, :].contiguous(), "shape_params": betas,
              "pose_params_rot_matrices": rot,
              "joints2D": ops.orthographic_project(t.joints, cam, 512.0)[:, config.SMPL_TO_KPRCNN_MAP, :].contiguous()}
    if sil:
        labels["silhouette"] = smpl.render_silhouettes(t.vertices, cam, img_wh=args.sil_res, sigma=0.0) > 0.5

if args.eager:
    model = Step()
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local])
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = model(feats, labels)
        loss.backward()
        opt.step()
        return loss
else:
    gstep = regressor.GraphedTrainStep(head, crit, smpl, feats, labels, r6, proj, lr=1e-4, world_size=world,
                                       fused_loss=fused, overlap=not args.no_overlap, render_silhouettes=render)

    def step():
        return gstep(feats, labels)

for _ in range(5):
    l0 = step().clone()
torch.cuda.synchronize()
if world > 1:
    dist.barrier()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
    l1 = step()
e1.record()
torch.cuda.synchronize()
ms = sharding.max_over_ranks(e0.elapsed_time(e1), dev)
nparams = sum(p.numel() for p in list(head.parameters()) + list(crit.parameters()))
if rank == 0:
    what = ("18x%dx%d crops -> ResNet-18%s -> IEF head (512,512)" % (args.res, args.res, " (bf16 autocast)" if args.amp else " (fp32/TF32 cuDNN)")
            if args.input == "encoder"
            else "512-d features -> IEF head (1024,1024)")
    terms = "5-term" if not sil else "6-term (+ silhouette at %dx%d, sigma %g, weight %g)" % (
        args.sil_res, args.sil_res, args.sil_sigma, args.silhouette_weight)
    print(json.dumps({"workload": "BASELINE.json configs[4]: regressor step: %s -> SMPL -> %s multi-task loss (%s kernels), "
                                  "batch %d per GPU x %d GPU(s), %s" % (what, terms, args.loss, B, world,
                                                                       "eager" if args.eager else "one CUDA graph per step"),
                      "ms_per_step": ms / steps, "crops_per_s": B * world * steps / (ms / 1e3),
                      "allreduced_params": nparams if world > 1 else 0, "allreduced_mb": nparams * 4 / 1e6 if world > 1 else 0,
                      "allreduce": "none" if world == 1 else ("DistributedDataParallel" if args.eager else
                                                              ("one flat all-reduce after the backward" if args.no_overlap
                                                               else "8 MB buckets on a side stream, overlapped with the backward (forked inside the graph)")),
                      "loss_first": float(l0), "loss_last": float(l1)}))
if world > 1:
    torch.cuda.synchronize()
    dist.barrier()
    if not args.eager:
        # a process group whose collectives are referenced by a live CUDA graph can block in its destructor:
        # everything is flushed and synchronised, leave without running it
        sys.stdout.flush()
        os._exit(0)
    dist.destroy_process_group()
