"""Drop-in for the reference's `models.smpl_official.SMPL` (models/smpl_official.py:10-41), i.e.
smplx.SMPL + the extra / COCO-plus / H36M joint regressors, backed by libb200smpl.so.

Call surface kept (SURVEY.md section 8b):
    smpl = SMPL(model_path, batch_size=1).to(device)
    out = smpl(body_pose=R[:, 1:], global_orient=R[:, :1], betas=b, pose2rot=False)
    out.vertices (B,6890,3)  out.joints (B,90,3)  smpl.faces (numpy)
plus the north_star positional form `SMPLLayer.forward(betas, pose, trans) -> (vertices, joints)`.
Buffers carry the smplx names so `state_dict()` is interchangeable.  The module must live on a
CUDA device: there is no CPU implementation.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple, Union

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .engine import SMPLEngine, SMPLFunction
from .model_io import load_smpl_model, validate_model


class SMPLOutput(dict):
    """Stand-in for smplx.body_models.SMPLOutput (models/smpl_official.py:4,35-40): attribute and
    dict access to vertices, joints, full_pose, betas, global_orient, body_pose."""

    def __init__(self, vertices=None, joints=None, full_pose=None, betas=None, global_orient=None,
                 body_pose=None, **extra):
        super().__init__(vertices=vertices, joints=joints, full_pose=full_pose, betas=betas,
                         global_orient=global_orient, body_pose=body_pose, **extra)

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


class VertexJointSelector(nn.Module):
    """Holder of smplx's picked-vertex joint ids under smplx's own name
    (`vertex_joint_selector.extra_joints_idxs`, SURVEY.md Appendix A.3); the picking itself happens in the kernels."""

    def __init__(self, extra_joints_idxs):
        super().__init__()
        self.register_buffer("extra_joints_idxs", torch.tensor(np.asarray(extra_joints_idxs), dtype=torch.long))


class SMPL(nn.Module):
    NUM_BODY_JOINTS = 23

    def __init__(self, model_path: Union[str, Dict[str, np.ndarray], None] = None, batch_size: int = 1,
                 gender: str = "neutral", mode: str = "fp32", slab_bodies: int = 0,
                 model_data: Optional[Dict[str, np.ndarray]] = None, dtype=torch.float32, **kwargs):
        """`model_path`: file / directory as smplx accepts, or pass the arrays via `model_data`
        (e.g. `model_io.make_synthetic_smpl()`).  `mode`: 'fp32' (bf16x3 tensor-core split),
        'bf16' (bf16-GEMM mode) or 'fp32_simt' (verification)."""
        super().__init__()
        if dtype != torch.float32:
            raise TypeError("the SMPL layer computes in float32")
        if isinstance(model_path, dict) and model_data is None:
            model_data, model_path = model_path, None
        if model_data is None:
            if model_path is None:
                raise ValueError("model_path or model_data is required")
            model_data = load_smpl_model(model_path, gender=gender,
                                         extra_regressor_paths=kwargs.get("extra_regressor_paths"))
        validate_model(model_data)
        self.batch_size = batch_size
        self.mode = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
        self.slab_bodies = int(slab_bodies)
        self.faces = np.asarray(model_data["faces"])
        f32 = lambda k: torch.tensor(np.asarray(model_data[k]), dtype=torch.float32)  # noqa: E731
        # smplx buffer names (SURVEY.md section 8 row a12) + models/smpl_official.py:20-25
        self.register_buffer("faces_tensor", torch.tensor(self.faces.astype(np.int64), dtype=torch.long))
        self.register_buffer("v_template", f32("v_template"))
        self.register_buffer("shapedirs", f32("shapedirs"))
        self.register_buffer("posedirs", f32("posedirs"))
        self.register_buffer("J_regressor", f32("J_regressor"))
        self.register_buffer("lbs_weights", f32("lbs_weights"))
        self.register_buffer("parents", torch.tensor(np.asarray(model_data["parents"]), dtype=torch.long))
        # smplx keeps the picked-vertex ids in a submodule: state_dict key `vertex_joint_selector.extra_joints_idxs`
        self.vertex_joint_selector = VertexJointSelector(model_data["extra_joints_idxs"])
        for k in ("J_regressor_extra", "J_regressor_cocoplus", "J_regressor_h36m"):
            self.register_buffer(k, f32(k))
        nb = self.shapedirs.shape[-1]
        # smplx default parameters (zeros)
        self.betas = nn.Parameter(torch.zeros(batch_size, nb))
        self.global_orient = nn.Parameter(torch.zeros(batch_size, 3))
        self.body_pose = nn.Parameter(torch.zeros(batch_size, self.NUM_BODY_JOINTS * 3))
        self.transl = nn.Parameter(torch.zeros(batch_size, 3))
        # identity + version 0 = "still the untouched zero default" (kept outside nn.Module's parameter registry)
        object.__setattr__(self, "_transl_default", self.transl)
        self._engines: Dict[torch.device, Tuple[tuple, SMPLEngine]] = {}

    # the tensors the packed device model is built from; any change to them (load_state_dict, in-place edit,
    # re-assignment) must reach the kernels, so the engine is keyed on their identity and version
    _MODEL_BUFFERS = ("v_template", "shapedirs", "posedirs", "J_regressor", "lbs_weights", "parents",
                      "J_regressor_extra", "J_regressor_cocoplus", "J_regressor_h36m")

    @property
    def extra_joints_idxs(self) -> torch.Tensor:
        return self.vertex_joint_selector.extra_joints_idxs

    def _model_tensors(self) -> Dict[str, torch.Tensor]:
        d = {k: getattr(self, k) for k in self._MODEL_BUFFERS}
        d["extra_joints_idxs"] = self.vertex_joint_selector.extra_joints_idxs
        return d

    # one packed handle per device the module has been moved to, rebuilt when a model buffer changes
    def _engine(self, device: torch.device) -> SMPLEngine:
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("b200 SMPL runs on CUDA only (module is on {}); call .to('cuda')".format(device))
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        tensors = self._model_tensors()
        key = tuple((id(t), t._version) for t in tensors.values())
        hit = self._engines.get(device)
        if hit is not None and hit[0] == key:
            return hit[1]
        model = {k: t.detach().cpu().numpy() for k, t in tensors.items()}
        validate_model(model)
        eng = SMPLEngine(model, device)
        self._engines[device] = (key, eng)
        return eng

    def _transl_is_untouched_default(self) -> bool:
        """True while self.transl is the zeros Parameter created in __init__ (never assigned, loaded, stepped or
        edited in place): adding it is the identity, so the call may skip it.  `.to(device)` keeps identity and
        version, so a moved module still qualifies."""
        t = self.transl
        return t is self._transl_default and t._version == 0

    @staticmethod
    def _expand(t: torch.Tensor, B: int) -> torch.Tensor:
        if t.shape[0] == B:
            return t
        if B % t.shape[0] != 0:
            raise ValueError("cannot broadcast batch {} to {}".format(t.shape[0], B))
        return t.expand(B // t.shape[0], *t.shape[1:]) if t.shape[0] == 1 else t.repeat(B // t.shape[0],
                                                                                      *([1] * (t.dim() - 1)))

    def forward(self, betas=None, body_pose=None, global_orient=None, transl=None, return_verts=True,
                return_full_pose=False, pose2rot=True, cam=None, **kwargs) -> SMPLOutput:
        """smplx.SMPL.forward keywords (SURVEY.md Appendix A.2) + `cam` (B,3) weak-perspective
        [s,tx,ty]: when given, the output also carries `joints2d` = orthographic_project_torch(
        joints, cam) (utils/cam_utils.py:5-26) computed in the same pass."""
        device = self.v_template.device
        eng = self._engine(device)
        apply_default_transl = transl is None
        global_orient = global_orient if global_orient is not None else self.global_orient
        body_pose = body_pose if body_pose is not None else self.body_pose
        betas = betas if betas is not None else self.betas
        transl = transl if transl is not None else self.transl
        B = max(betas.shape[0], global_orient.shape[0], body_pose.shape[0])
        if pose2rot:
            go = self._expand(global_orient.reshape(global_orient.shape[0], -1), B)
            bp = self._expand(body_pose.reshape(body_pose.shape[0], -1), B)
            full_pose = torch.cat([go, bp], dim=1)                           # (B, 72)
        else:
            go = self._expand(global_orient.reshape(global_orient.shape[0], -1, 3, 3), B)
            bp = self._expand(body_pose.reshape(body_pose.shape[0], -1, 3, 3), B)
            full_pose = torch.cat([go, bp], dim=1)                           # (B, 24, 3, 3)
        betas_b = self._expand(betas, B)
        # smplx always adds transl (argument or its own Parameter).  The only case skipped here is the untouched
        # zeros default outside of training (no gradient can be asked for it): adding zeros is the identity.
        if apply_default_transl and self._transl_is_untouched_default() and not (
                self.transl.requires_grad and torch.is_grad_enabled()):
            tr = None
        else:
            tr = self._expand(transl, B)
        verts, joints, j2d = SMPLFunction.apply(eng, betas_b.float().contiguous(), full_pose.float().contiguous(),
                                                None if tr is None else tr.float().contiguous(),
                                                None if cam is None else cam.float().contiguous(),
                                                bool(pose2rot), self.mode, bool(return_verts), self.slab_bodies)
        out = SMPLOutput(vertices=verts if return_verts else None, joints=joints,
                         full_pose=full_pose if return_full_pose else None, betas=betas,
                         global_orient=global_orient, body_pose=body_pose)
        if cam is not None:
            out["joints2d"] = j2d
        return out


    def silhouette_inputs(self, vertices: torch.Tensor, cam_wp: torch.Tensor, proj_wh: float = 512.0) -> Dict:
        """Hand-off to a differentiable rasteriser in the layout the reference feeds its neural renderer
        (player_recon.py:288-289, 686-697): `vertices` (B,6890,3) fp32 contiguous as the skinning kernel wrote them,
        `faces` (B,13776,3) float (the int32 topology cast to float and repeated per body), `t` (B,1,3) camera
        translation from the weak-perspective camera (cam_utils.py:44-52).  No copy of the vertices is made."""
        from . import config
        from .cam_utils import convert_weak_perspective_to_camera_translation_torch
        B = vertices.shape[0]
        faces = torch.from_numpy(self.faces.astype(np.int32)).float().to(vertices.device)
        t = convert_weak_perspective_to_camera_translation_torch(cam_wp, config.FOCAL_LENGTH, proj_wh)
        return {"vertices": vertices.contiguous(), "faces": faces[None].expand(B, -1, -1), "t": t.unsqueeze(1)}

    def faces_int32(self, device: torch.device) -> torch.Tensor:
        """The model's faces (F,3) as int32 on `device`, uploaded once per device."""
        device = torch.device(device)
        cache = self.__dict__.setdefault("_faces_dev", {})
        f = cache.get(device)
        if f is None:
            f = torch.from_numpy(np.ascontiguousarray(self.faces, dtype=np.int32)).to(device)
            cache[device] = f
        return f

    def render_silhouettes(self, vertices: torch.Tensor, cam_wp: torch.Tensor, img_wh: int = 256, sigma: float = 0.0,
                           proj_wh: float = 512.0, focal_length: Optional[float] = None) -> torch.Tensor:
        """Silhouettes (B, img_wh, img_wh) of posed meshes (ops.render_silhouettes) with the camera translation
        built as `silhouette_inputs` builds it from the weak-perspective camera [s, tx, ty] of the `proj_wh`-pixel
        crop: t = [tx, ty, 2 f / (proj_wh s)], f = config.FOCAL_LENGTH.  The render focal length defaults to
        f * img_wh / proj_wh, so the image frames the same view as that crop at any resolution (img_wh = proj_wh
        renders at f itself).  sigma == 0: binary; sigma > 0: soft, differentiable into `vertices` (and through
        SMPLFunction into betas / pose) and `cam_wp`."""
        from . import config, ops
        from .cam_utils import convert_weak_perspective_to_camera_translation_torch
        t = convert_weak_perspective_to_camera_translation_torch(cam_wp, config.FOCAL_LENGTH, proj_wh)
        f = config.FOCAL_LENGTH * float(img_wh) / float(proj_wh) if focal_length is None else float(focal_length)
        return ops.render_silhouettes(vertices, self.faces_int32(vertices.device), t.contiguous(), img_wh,
                                      focal_length=f, sigma=sigma)


class SMPLLayer(SMPL):
    """north_star surface: forward(betas, pose, trans) -> (vertices, joints).
    pose: (B,24,3,3) rotation matrices, or (B,72) axis-angle (detected from the shape)."""

    def forward(self, betas, pose, trans=None, cam=None):  # type: ignore[override]
        eng = self._engine(self.v_template.device)
        B = betas.shape[0]
        axis_angle = pose.dim() == 2 and pose.shape[1] == 72
        verts, joints, j2d = SMPLFunction.apply(eng, betas.contiguous(), pose.contiguous(),
                                                None if trans is None else trans.contiguous(),
                                                None if cam is None else cam.contiguous(), axis_angle, self.mode,
                                                True, self.slab_bodies)
        if cam is not None:
            return verts, joints, j2d
        return verts, joints
