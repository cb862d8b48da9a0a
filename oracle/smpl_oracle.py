"""CPU oracle for the batched SMPL hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this module, and only as the checker / reported baseline.  The product
(`soccerplayershapepose_b200/`) never imports it and has no CPU fallback.

What it restates
----------------
The reference's hot path is `models/smpl_official.py:27-41` (in tree, 41 lines) on top of the
third-party PyPI package **smplx** (unpinned, `PlayerReconstruction/requirements.txt:6`;
`from smplx.body_models import SMPLOutput` implies >= 0.1.21).  smplx is NOT in the reference
tree, NOT installed in the build container and cannot be installed (no network), and the
licensed SMPL model files are absent too.  So:

* The smplx arithmetic (`smplx/lbs.py`: blend_shapes, vertices2joints, batch_rodrigues,
  transform_mat, batch_rigid_transform, lbs; `smplx/body_models.py::SMPL.forward`;
  `smplx/vertex_joint_selector.py`) is restated from its published algorithm as recorded in
  SURVEY.md Appendix A.  **PARITY UNPINNED** for this part: the reference holds no test or
  golden vector for it and the package cannot be executed here.  It is anchored on the
  reference's call sites (`models/smpl_official.py:29-41`, `player_recon.py:1207-1210`,
  `predict/predict_3D.py:139-148`) and on self-consistency / invariance properties
  (tests/test_oracle.py).
* The in-tree functions (`utils/cam_utils.py:5-85`, `utils/joints2d_utils.py:5-10`,
  `utils/rigid_transform_utils.py:27-41`, `losses/multi_task_loss.py:97-113`,
  `config.py:15-16,29-38`) ARE pinned: `tests/golden/make_golden_from_reference.py` imports the
  reference files themselves in the build container and freezes input/output vectors in
  `tests/golden/intree_golden.npz`; tests/test_oracle.py checks this oracle against them.

Everything is plain PyTorch eager on CPU, dtype-generic (fp32 = the reference's arithmetic,
fp64 = the high-precision checker), differentiable through torch autograd.
"""
from __future__ import annotations

from typing import Dict, NamedTuple, Optional

import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------
# smplx/lbs.py (SURVEY.md Appendix A.1)
# ----------------------------------------------------------------------------------------------
def blend_shapes(betas: torch.Tensor, shape_disps: torch.Tensor) -> torch.Tensor:
    """smplx.lbs.blend_shapes: einsum('bl,mkl->bmk').  betas (B,L), shape_disps (V,3,L)."""
    return torch.einsum("bl,mkl->bmk", [betas, shape_disps])


def vertices2joints(J_regressor: torch.Tensor, vertices: torch.Tensor) -> torch.Tensor:
    """smplx.lbs.vertices2joints: einsum('bik,ji->bjk').  Used at models/smpl_official.py:30-32."""
    return torch.einsum("bik,ji->bjk", [vertices, J_regressor])


def batch_rodrigues(rot_vecs: torch.Tensor) -> torch.Tensor:
    """smplx.lbs.batch_rodrigues (N,3)->(N,3,3).  Quirk kept: 1e-8 is added to every component
    before the norm; the direction divides the *un-shifted* vector by that norm."""
    n = rot_vecs.shape[0]
    dtype, device = rot_vecs.dtype, rot_vecs.device
    angle = torch.norm(rot_vecs + 1e-8, dim=1, keepdim=True)
    rot_dir = rot_vecs / angle
    cos = torch.unsqueeze(torch.cos(angle), dim=1)
    sin = torch.unsqueeze(torch.sin(angle), dim=1)
    rx, ry, rz = torch.split(rot_dir, 1, dim=1)
    zeros = torch.zeros((n, 1), dtype=dtype, device=device)
    K = torch.cat([zeros, -rz, ry, rz, zeros, -rx, -ry, rx, zeros], dim=1).view((n, 3, 3))
    ident = torch.eye(3, dtype=dtype, device=device).unsqueeze(dim=0)
    return ident + sin * K + (1 - cos) * torch.bmm(K, K)


def transform_mat(R: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """smplx.lbs.transform_mat: [[R, t], [0, 1]] for R (N,3,3), t (N,3,1)."""
    return torch.cat([F.pad(R, [0, 0, 0, 1]), F.pad(t, [0, 0, 0, 1], value=1)], dim=2)


def batch_rigid_transform(rot_mats: torch.Tensor, joints: torch.Tensor, parents: torch.Tensor):
    """smplx.lbs.batch_rigid_transform: sequential chain in parent order.
    Returns posed joints (B,J,3) and A = G - pad(G . [J;0]) (B,J,4,4)."""
    joints = torch.unsqueeze(joints, dim=-1)
    rel_joints = joints.clone()
    rel_joints[:, 1:] -= joints[:, parents[1:]]
    transforms_mat = transform_mat(rot_mats.reshape(-1, 3, 3),
                                   rel_joints.reshape(-1, 3, 1)).reshape(-1, joints.shape[1], 4, 4)
    transform_chain = [transforms_mat[:, 0]]
    for i in range(1, parents.shape[0]):
        transform_chain.append(torch.matmul(transform_chain[int(parents[i])], transforms_mat[:, i]))
    transforms = torch.stack(transform_chain, dim=1)
    posed_joints = transforms[:, :, :3, 3]
    joints_homogen = F.pad(joints, [0, 0, 0, 1])
    rel_transforms = transforms - F.pad(torch.matmul(transforms, joints_homogen), [3, 0, 0, 0, 0, 0, 0, 0])
    return posed_joints, rel_transforms


def lbs(betas, pose, v_template, shapedirs, posedirs, J_regressor, parents, lbs_weights, pose2rot=True):
    """smplx.lbs.lbs.  pose is (B,72) axis-angle when pose2rot else (B,24,3,3) rotation matrices.
    Returns (vertices (B,V,3), posed chain joints (B,24,3))."""
    batch_size = max(betas.shape[0], pose.shape[0])
    dtype, device = betas.dtype, betas.device
    v_shaped = v_template + blend_shapes(betas, shapedirs)
    J = vertices2joints(J_regressor, v_shaped)
    ident = torch.eye(3, dtype=dtype, device=device)
    if pose2rot:
        rot_mats = batch_rodrigues(pose.reshape(-1, 3)).view([batch_size, -1, 3, 3])
        pose_feature = (rot_mats[:, 1:, :, :] - ident).view([batch_size, -1])
        pose_offsets = torch.matmul(pose_feature, posedirs).view(batch_size, -1, 3)
    else:
        pose_feature = pose[:, 1:].view(batch_size, -1, 3, 3) - ident
        rot_mats = pose.view(batch_size, -1, 3, 3)
        pose_offsets = torch.matmul(pose_feature.view(batch_size, -1), posedirs).view(batch_size, -1, 3)
    v_posed = pose_offsets + v_shaped
    J_transformed, A = batch_rigid_transform(rot_mats, J, parents)
    W = lbs_weights.unsqueeze(dim=0).expand([batch_size, -1, -1])
    num_joints = J_regressor.shape[0]
    T = torch.matmul(W, A.view(batch_size, num_joints, 16)).view(batch_size, -1, 4, 4)
    homogen_coord = torch.ones([batch_size, v_posed.shape[1], 1], dtype=dtype, device=device)
    v_posed_homo = torch.cat([v_posed, homogen_coord], dim=2)
    v_homo = torch.matmul(T, torch.unsqueeze(v_posed_homo, dim=-1))
    verts = v_homo[:, :, :3, 0]
    return verts, J_transformed


# ----------------------------------------------------------------------------------------------
# smplx/body_models.py::SMPL.forward + vertex_joint_selector + models/smpl_official.py:27-41
# ----------------------------------------------------------------------------------------------
class OracleOutput(NamedTuple):
    vertices: torch.Tensor     # (B, 6890, 3)
    joints: torch.Tensor       # (B, 90, 3)
    full_pose: torch.Tensor    # (B, 24, 3, 3) or (B, 72)


class SMPLOracle:
    """The reference's `models.smpl_official.SMPL` (smplx.SMPL + 3 extra joint regressors),
    restated.  `model` is the dict produced by `soccerplayershapepose_b200.model_io`."""

    def __init__(self, model: Dict[str, np.ndarray], dtype=torch.float32, device="cpu"):
        t = lambda a: torch.as_tensor(np.asarray(a), dtype=dtype, device=device)  # noqa: E731
        self.dtype, self.device = dtype, device
        self.v_template = t(model["v_template"])
        self.shapedirs = t(model["shapedirs"])
        self.posedirs = t(model["posedirs"])
        self.J_regressor = t(model["J_regressor"])
        self.lbs_weights = t(model["lbs_weights"])
        self.parents = torch.as_tensor(np.asarray(model["parents"]), dtype=torch.long, device=device)
        self.extra_joints_idxs = torch.as_tensor(np.asarray(model["extra_joints_idxs"]), dtype=torch.long,
                                                 device=device)
        self.J_regressor_extra = t(model["J_regressor_extra"])
        self.J_regressor_cocoplus = t(model["J_regressor_cocoplus"])
        self.J_regressor_h36m = t(model["J_regressor_h36m"])
        self.faces = np.asarray(model["faces"])

    def smplx_forward(self, betas, body_pose, global_orient, transl=None, pose2rot=True):
        """smplx.SMPL.forward (SURVEY.md Appendix A.2): 45 joints."""
        full_pose = torch.cat([global_orient, body_pose], dim=1)
        batch_size = max(betas.shape[0], global_orient.shape[0], body_pose.shape[0])
        if betas.shape[0] != batch_size:
            num_repeats = int(batch_size / betas.shape[0])
            betas = betas.expand(num_repeats, -1)
        vertices, joints = lbs(betas, full_pose, self.v_template, self.shapedirs, self.posedirs,
                               self.J_regressor, self.parents, self.lbs_weights, pose2rot=pose2rot)
        # VertexJointSelector (SURVEY.md Appendix A.3)
        extra = torch.index_select(vertices, 1, self.extra_joints_idxs)
        joints = torch.cat([joints, extra], dim=1)
        if transl is not None:
            joints = joints + transl.unsqueeze(dim=1)
            vertices = vertices + transl.unsqueeze(dim=1)
        return vertices, joints, full_pose

    def forward(self, betas, body_pose, global_orient, transl=None, pose2rot=True) -> OracleOutput:
        """models/smpl_official.py:27-41: + extra(9), cocoplus(19), h36m(17) -> 90 joints."""
        vertices, joints, full_pose = self.smplx_forward(betas, body_pose, global_orient, transl, pose2rot)
        extra_joints = vertices2joints(self.J_regressor_extra, vertices)
        cocoplus_joints = vertices2joints(self.J_regressor_cocoplus, vertices)
        h36m_joints = vertices2joints(self.J_regressor_h36m, vertices)
        all_joints = torch.cat([joints, extra_joints, cocoplus_joints, h36m_joints], dim=1)
        return OracleOutput(vertices, all_joints, full_pose)

    __call__ = forward

    def forward_flat(self, betas, pose, trans=None, pose2rot=False) -> OracleOutput:
        """north_star positional surface forward(betas, pose, trans): pose is (B,24,3,3)
        rotation matrices (pose2rot=False) or (B,72) axis-angle (pose2rot=True)."""
        if pose2rot:
            pose = pose.reshape(pose.shape[0], -1)
            return self.forward(betas, pose[:, 3:], pose[:, :3], trans, True)
        pose = pose.reshape(pose.shape[0], -1, 3, 3)
        return self.forward(betas, pose[:, 1:], pose[:, :1], trans, False)


# ----------------------------------------------------------------------------------------------
# in-tree projection / conversion helpers (pinned against the reference files, see module doc)
# ----------------------------------------------------------------------------------------------
def orthographic_project(points3D: torch.Tensor, cam_params: torch.Tensor) -> torch.Tensor:
    """utils/cam_utils.py:5-26: u = s (x + tx), v = s (y + ty); cam = [s, tx, ty]."""
    s = cam_params[:, 0].unsqueeze(1)
    u = s * (points3D[:, :, 0] + cam_params[:, 1].unsqueeze(1))
    v = s * (points3D[:, :, 1] + cam_params[:, 2].unsqueeze(1))
    return torch.stack([u, v], dim=-1)


def weak_perspective_to_translation(cam_wp: torch.Tensor, focal_length: float, resolution: float) -> torch.Tensor:
    """utils/cam_utils.py:28-34: [tx, ty, 2 f / (res * s + 1e-9)]."""
    tz = 2 * focal_length / (resolution * cam_wp[:, 0] + 1e-9)
    return torch.stack([cam_wp[:, 1], cam_wp[:, 2], tz], dim=-1)


def translation_to_weak_perspective(translation: torch.Tensor, focal_length: float, resolution: float) -> torch.Tensor:
    """utils/cam_utils.py:36-42."""
    s = 2 * focal_length / (resolution * translation[:, 2] + 1e-9)
    return torch.stack([s, translation[:, 0], translation[:, 1]], dim=-1)


def intrinsics_matrix(img_width: float, img_height: float, focal_length: float) -> np.ndarray:
    """utils/cam_utils.py:44-52."""
    return np.array([[focal_length, 0.0, img_width / 2.0],
                     [0.0, focal_length, img_height / 2.0],
                     [0.0, 0.0, 1.0]])


def perspective_project(points, rotation, translation, cam_K=None, focal_length=None, img_wh=None):
    """utils/cam_utils.py:54-85: X' = R X + t ; X'/z ; K . ; drop last row."""
    if cam_K is None:
        K = torch.as_tensor(intrinsics_matrix(img_wh, img_wh, focal_length).astype(np.float32))
        cam_K = K[None].expand(points.shape[0], -1, -1).to(points.device).to(points.dtype)
    points = torch.einsum("bij,bkj->bki", rotation, points) + translation.unsqueeze(1)
    projected = points / points[:, :, -1].unsqueeze(-1)
    projected = torch.einsum("bij,bkj->bki", cam_K, projected)
    return projected[:, :, :-1]


def undo_keypoint_normalisation(normalised_keypoints: torch.Tensor, img_wh: float) -> torch.Tensor:
    """utils/joints2d_utils.py:5-10: [-1,1] -> pixels."""
    return (normalised_keypoints + 1) * (img_wh / 2.0)


def rot6d_to_rotmat(x: torch.Tensor) -> torch.Tensor:
    """utils/rigid_transform_utils.py:27-41 (Zhou et al.): view(-1,3,2); Gram-Schmidt; columns."""
    x = x.reshape(-1, 3, 2)
    a1, a2 = x[:, :, 0], x[:, :, 1]
    b1 = F.normalize(a1)
    b2 = F.normalize(a2 - torch.einsum("bi,bi->b", b1, a2).unsqueeze(-1) * b1)
    b3 = torch.cross(b1, b2, dim=1)
    return torch.stack((b1, b2, b3), dim=-1)


def joints2d_loss(pred_pixels: torch.Tensor, label_pixels: torch.Tensor, log_var: torch.Tensor,
                  img_wh: float = 256.0, vis: Optional[torch.Tensor] = None) -> torch.Tensor:
    """losses/multi_task_loss.py:97-113: optional vis mask, both sides 2x/wh - 1, MSE(mean),
    * exp(-log_var) + log_var."""
    if vis is not None:
        label_pixels = label_pixels[vis, :]
        pred_pixels = pred_pixels[vis, :]
    label = (2.0 * label_pixels) / img_wh - 1.0
    pred = (2.0 * pred_pixels) / img_wh - 1.0
    mse = torch.mean((pred - label) ** 2)
    return mse * torch.exp(-log_var) + log_var


def fit_loss_per_player(pred_pixels: torch.Tensor, label_pixels: torch.Tensor, log_var: float, betas: torch.Tensor,
                        shape_weight: float, img_wh: float = 256.0, vis: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-player loss of the fitting loop (B,): `joints2d_loss` applied to ONE player (pred/label (B,K,2) pixels, vis
    (B,K) bool or None) + shape_weight * mean(betas^2).  A player with no visible keypoint has mean 0 (loss =
    log_var + shape term), where `joints2d_loss` would return NaN."""
    w = torch.ones(pred_pixels.shape[:2], dtype=pred_pixels.dtype, device=pred_pixels.device) if vis is None \
        else vis.to(pred_pixels.dtype)
    d = ((2.0 * pred_pixels) / img_wh - 1.0) - ((2.0 * label_pixels) / img_wh - 1.0)
    sq = (d * d).sum(-1) * w
    count = 2.0 * w.sum(1)
    mse = sq.sum(1) / count.clamp(min=1.0)          # an empty sum over a zero count stays 0
    return mse * float(np.exp(-log_var)) + log_var + shape_weight * (betas * betas).mean(1)


def init_log_var(weight: float, eps: float = 1e-6) -> float:
    """losses/multi_task_loss.py:38: log_var0 = -log(w + eps)."""
    return float(-np.log(weight + eps))
