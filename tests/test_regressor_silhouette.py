"""The silhouette term of the regressor's multi-task loss on the CPU: the fp64 oracles stand in for the SMPL and
silhouette kernels (S = 32, bodies about 26 px tall at cam [0.9, 0, 0])."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import silhouette_oracle as SO
from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import config, regressor
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch

LOSSES = ("verts", "joints2D", "joints3D", "shape_params", "pose_params", "silhouette")
WEIGHTS = {"verts": 1.0, "joints2D": 0.1, "joints3D": 1.0, "shape_params": 0.1, "pose_params": 0.1,
           "silhouette": 0.5}
S, SIGMA, PROJ = 32, 1.0, 512.0


class _OracleSMPL:
    def __init__(self, model, dtype):
        self.orc = O.SMPLOracle(model, dtype=dtype)

    def __call__(self, body_pose, global_orient, betas, pose2rot=False, return_verts=True):
        return self.orc.forward(betas, body_pose, global_orient, None, pose2rot)


def _focal():
    return config.FOCAL_LENGTH * S / PROJ


def _oracle_renderer(faces, sigma=SIGMA):
    """render_silhouettes(verts, cam) for predict: the camera of SMPL.render_silhouettes through the fp64 oracle."""
    faces = torch.as_tensor(faces)

    def render(verts, cam):
        t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, PROJ)
        return SO.render(verts, faces, t, S, _focal(), sigma)
    return render


def _cpu_ops():
    return O.rot6d_to_rotmat, (lambda joints, cam: O.undo_keypoint_normalisation(O.orthographic_project(joints, cam), 512))


def _batch(model, B, seed, dtype=torch.float32):
    """Features and labels, the silhouette label being the hard silhouette of the label body at cam [0.9, 0, 0]."""
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, 64, generator=g)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
    cam = torch.tensor([0.9, 0.0, 0.0]).repeat(B, 1)
    betas, rot, cam = betas.double(), rot.double(), cam.double()
    out = O.SMPLOracle(model, dtype=torch.float64).forward(betas, rot[:, 1:], rot[:, :1], None, False)
    j2d = O.undo_keypoint_normalisation(O.orthographic_project(out.joints, cam), 512)[:, config.SMPL_TO_KPRCNN_MAP, :]
    sil = _oracle_renderer(model["faces"], 0.0)(out.vertices, cam)
    labels = {"joints2D": j2d, "verts": out.vertices, "shape_params": betas, "pose_params_rot_matrices": rot,
              "joints3D": out.joints[:, config.ALL_JOINTS_TO_COCO_MAP, :], "silhouette": sil}
    return feats.to(dtype), {k: v.to(dtype) for k, v in labels.items()}


def _make(model, losses=LOSSES, seed=0, dtype=torch.float64):
    """Head whose output starts near the mean parameters (camera [0.9, 0, 0]), so the bodies lie in the image."""
    torch.manual_seed(seed)
    head = regressor.IEFModule((48, 48), in_features=64).to(dtype)
    with torch.no_grad():
        head.fc3.weight.mul_(0.05)
    crit = regressor.MultiTaskLoss(losses, WEIGHTS, faces=model["faces"], silhouette_sigma=SIGMA,
                                   silhouette_wh=S, proj_wh=PROJ).to(dtype)
    return head, crit


def test_kendall_form_and_log_var_init(synthetic_model):
    _, crit = _make(synthetic_model, ("silhouette",))
    assert abs(crit.silhouette_log_var.item() + np.log(0.5 + 1e-6)) < 1e-6
    assert set(crit.state_dict()) == {"silhouette_log_var"}
    assert crit.silhouette_faces.dtype == torch.int32 and crit.silhouette_faces.shape == (13776, 3)
    g = torch.Generator().manual_seed(2)
    alpha = torch.rand(3, S, S, generator=g, dtype=torch.float64)
    target = torch.rand(3, S, S, generator=g, dtype=torch.float64)
    with torch.no_grad():
        crit.silhouette_log_var.fill_(0.3)
    loss, parts = crit({"silhouette": target}, {"silhouettes": alpha})
    L = ((alpha - (target >= 0.5).double()) ** 2).mean()
    assert torch.allclose(loss, L * math.exp(-0.3) + 0.3, rtol=1e-12)
    assert torch.allclose(parts["silhouette"], L * math.exp(-0.3), rtol=1e-12)
    # integer and boolean masks: non-zero is inside
    loss_u8, _ = crit({"silhouette": (target >= 0.5).to(torch.uint8) * 7}, {"silhouettes": alpha})
    assert torch.allclose(loss_u8, loss, rtol=1e-12)


def test_eager_term_equals_oracle_loss(synthetic_model):
    B = 3
    head, crit = _make(synthetic_model, ("silhouette",))
    with torch.no_grad():
        crit.silhouette_log_var.zero_()
    feats, labels = _batch(synthetic_model, B, 1, torch.float64)
    r6, proj = _cpu_ops()
    out = regressor.predict(head, _OracleSMPL(synthetic_model, torch.float64), feats, r6, proj,
                            render_silhouettes=_oracle_renderer(synthetic_model["faces"]))
    assert out["silhouettes"].shape == (B, S, S)
    loss, parts = crit(labels, out)
    t = convert_weak_perspective_to_camera_translation_torch(out["cam"], config.FOCAL_LENGTH, PROJ)
    ref = SO.loss(out["verts"], torch.as_tensor(synthetic_model["faces"]), t, labels["silhouette"], S, _focal(), SIGMA,
                  1.0).mean()
    assert 1e-3 < float(ref) < 0.5                   # the bodies overlap their labels but not exactly
    assert torch.allclose(loss, ref, rtol=1e-12) and torch.allclose(parts["silhouette"], ref, rtol=1e-12)


def test_train_step_with_the_term_reduces_the_loss(synthetic_model):
    head, crit = _make(synthetic_model, ("joints2D", "silhouette"), dtype=torch.float32)
    feats, labels = _batch(synthetic_model, 4, 3)
    smpl = _OracleSMPL(synthetic_model, torch.float32)
    r6, proj = _cpu_ops()
    render = _oracle_renderer(synthetic_model["faces"])
    opt = torch.optim.Adam(list(head.parameters()) + list(crit.parameters()), lr=1e-3)

    def sil_part():
        with torch.no_grad():
            out = regressor.predict(head, smpl, feats, r6, proj, render_silhouettes=render)
            return float(crit(labels, out)[1]["silhouette"] * torch.exp(crit.silhouette_log_var))

    l0 = sil_part()
    losses = [float(regressor.train_step(head, crit, opt, smpl, feats, labels, r6, proj, render_silhouettes=render))
              for _ in range(5)]
    assert losses[-1] < losses[0]
    assert sil_part() < l0


def test_missing_faces_and_wrong_target_shape_raise(synthetic_model):
    with pytest.raises(ValueError):
        regressor.MultiTaskLoss(("verts", "silhouette"))
    with pytest.raises(ValueError):
        regressor.MultiTaskLoss(("silhouette",), faces=np.zeros((4, 2), np.int64))
    regressor.MultiTaskLoss(("verts",))                 # faces are only needed with the term
    _, crit = _make(synthetic_model, ("silhouette",))
    alpha = torch.rand(2, S, S, dtype=torch.float64)
    for bad in (torch.zeros(2, S, S + 1), torch.zeros(3, S, S), torch.zeros(2, S * S)):
        with pytest.raises(ValueError):
            crit({"silhouette": bad.double()}, {"silhouettes": alpha})
    with pytest.raises(ValueError):
        crit({"silhouette": torch.zeros(2, S, S)}, {"verts": torch.zeros(2, 6890, 3)})   # no renderer given


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _ddp_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from soccerplayershapepose_b200.model_io import make_synthetic_smpl
        from soccerplayershapepose_b200 import sharding
        torch.set_num_threads(2)
        model = make_synthetic_smpl(1234)
        head, crit = _make(model)

        class Both(torch.nn.Module):
            def __init__(self):
                super().__init__()
                self.head, self.crit = head, crit

            def forward(self, feats, labels, smpl, r6, proj, render):
                outputs = regressor.predict(self.head, smpl, feats, r6, proj, render_silhouettes=render)
                return self.crit(labels, outputs)[0]

        ddp = torch.nn.parallel.DistributedDataParallel(Both())
        feats, labels = _batch(model, 4, 5, torch.float64)
        f = sharding.shard(feats, rank, world)
        lab = {k: sharding.shard(v, rank, world) for k, v in labels.items()}
        r6, proj = _cpu_ops()
        loss = ddp(f, lab, _OracleSMPL(model, torch.float64), r6, proj, _oracle_renderer(model["faces"]))
        loss.backward()
        if rank == 0:
            np.savez(os.path.join(out_dir, "g.npz"), fc3=head.fc3.weight.grad.numpy(), fc1=head.fc1.weight.grad.numpy(),
                     lv=crit.silhouette_log_var.grad.numpy())
    finally:
        dist.destroy_process_group()


def test_data_parallel_gradients_with_the_term_match_full_batch(tmp_path, synthetic_model):
    mp.spawn(_ddp_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "g.npz"))
    head, crit = _make(synthetic_model)
    feats, labels = _batch(synthetic_model, 4, 5, torch.float64)
    r6, proj = _cpu_ops()
    outputs = regressor.predict(head, _OracleSMPL(synthetic_model, torch.float64), feats, r6, proj,
                                render_silhouettes=_oracle_renderer(synthetic_model["faces"]))
    crit(labels, outputs)[0].backward()
    assert float(crit.silhouette_log_var.grad.abs()) > 0.0
    np.testing.assert_allclose(got["fc3"], head.fc3.weight.grad.numpy(), rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(got["fc1"], head.fc1.weight.grad.numpy(), rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(got["lv"], crit.silhouette_log_var.grad.numpy(), rtol=1e-9)
