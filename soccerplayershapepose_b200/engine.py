"""Host-side engine: owns one packed model handle per device and drives the C-ABI.

PyTorch is used for device memory (outputs, scratch), streams and autograd plumbing only; all
arithmetic of the SMPL path runs in libb200smpl.so.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import BackwardArgs, ForwardArgs, ModelDesc, ModelInfo


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _as_f32c(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a), dtype=np.float32)


class SMPLEngine:
    """A packed SMPL model on one CUDA device (or host-only with device=None, for CPU tests of the
    packing logic).  Thread-compatible: calls take the current stream of the tensors' device."""

    def __init__(self, model: Dict[str, np.ndarray], device: Optional[torch.device] = None):
        self.lib = _lib.load()
        v_template = _as_f32c(model["v_template"])
        shapedirs = _as_f32c(model["shapedirs"])
        posedirs = _as_f32c(model["posedirs"])
        J_regressor = _as_f32c(model["J_regressor"])
        lbs_weights = _as_f32c(model["lbs_weights"])
        parents = np.ascontiguousarray(np.asarray(model["parents"]), dtype=np.int64)
        vj = np.ascontiguousarray(np.asarray(model.get("extra_joints_idxs", np.zeros(0))), dtype=np.int64)
        regs = [_as_f32c(model[k]) for k in ("J_regressor_extra", "J_regressor_cocoplus", "J_regressor_h36m")
                if k in model]
        V = v_template.shape[0]
        reg = np.ascontiguousarray(np.concatenate(regs, 0)) if regs else np.zeros((0, V), np.float32)
        if shapedirs.shape[:2] != (V, 3) or posedirs.shape != (207, 3 * V) or lbs_weights.shape != (V, 24):
            raise ValueError("SMPL model arrays have inconsistent shapes")
        keep = [v_template, shapedirs, posedirs, J_regressor, lbs_weights, parents, vj, reg]
        desc = ModelDesc(
            num_verts=V, num_joints=J_regressor.shape[0], num_betas=shapedirs.shape[2],
            num_vertex_joints=len(vj), num_regressed_joints=reg.shape[0], reserved0=0,
            v_template=v_template.ctypes.data, shapedirs=shapedirs.ctypes.data, posedirs=posedirs.ctypes.data,
            J_regressor=J_regressor.ctypes.data, lbs_weights=lbs_weights.ctypes.data, parents=parents.ctypes.data,
            vertex_joint_ids=vj.ctypes.data if len(vj) else None,
            joint_regressors=reg.ctypes.data if reg.shape[0] else None)
        if device is None:
            dev_index = -1
            self.device = None
        else:
            self.device = torch.device(device)
            if self.device.type != "cuda":
                raise RuntimeError("SMPLEngine needs a CUDA device: the SMPL path has no CPU implementation")
            dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
            self.device = torch.device("cuda", dev_index)
        handle = ctypes.c_void_p()
        _lib.check(self.lib.b200smpl_model_create(ctypes.byref(desc), dev_index, ctypes.byref(handle)),
                   "b200smpl_model_create")
        del keep
        self.handle = handle
        info = ModelInfo()
        _lib.check(self.lib.b200smpl_model_get_info(self.handle, ctypes.byref(info)), "b200smpl_model_get_info")
        self.info = info
        self.num_verts = info.num_verts
        self.num_joints_out = info.num_joints_out
        self.num_betas = info.num_betas
        self._ws: Dict[Tuple, torch.Tensor] = {}

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.b200smpl_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---- test hook -------------------------------------------------------------------------
    def debug_array(self, name: str, dtype) -> np.ndarray:
        data, nbytes = ctypes.c_void_p(), ctypes.c_size_t()
        _lib.check(self.lib.b200smpl_model_debug_array(self.handle, name.encode(), ctypes.byref(data),
                                                       ctypes.byref(nbytes)), "b200smpl_model_debug_array")
        if nbytes.value == 0:                 # an empty table (a model without virtual joint rows) has no address
            return np.zeros(0, dtype=dtype)
        buf = (ctypes.c_uint8 * nbytes.value).from_address(data.value)
        return np.frombuffer(buf, dtype=dtype).copy()

    # ---- helpers ---------------------------------------------------------------------------
    def _check_in(self, t: Optional[torch.Tensor], shape, name: str) -> Optional[torch.Tensor]:
        if t is None:
            return None
        if not isinstance(t, torch.Tensor):
            raise TypeError("{} must be a torch.Tensor".format(name))
        if t.device != self.device:
            raise RuntimeError("{} is on {} but the SMPL model lives on {}".format(name, t.device, self.device))
        if t.dtype != torch.float32:
            raise TypeError("{} must be float32, got {}".format(name, t.dtype))
        if tuple(t.shape) != tuple(shape):
            raise ValueError("{} has shape {}, expected {}".format(name, tuple(t.shape), tuple(shape)))
        return t.contiguous()

    def _workspace(self, kind: str, B: int, mode: int, slab: int) -> torch.Tensor:
        fn = (self.lib.b200smpl_forward_workspace_bytes if kind == "fwd"
              else self.lib.b200smpl_backward_workspace_bytes)
        nbytes = int(fn(self.handle, B, mode, slab))
        key = (kind, torch.cuda.current_stream(self.device).cuda_stream)
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    # ---- forward / backward through the C-ABI -----------------------------------------------
    def forward(self, betas: torch.Tensor, pose: torch.Tensor, transl: Optional[torch.Tensor] = None,
                cam: Optional[torch.Tensor] = None, *, axis_angle: bool = False, mode: int = _lib.MODE_FP32,
                want_vertices: bool = True, slab: int = 0, save: bool = False,
                saved_buffer: Optional[torch.Tensor] = None):
        """betas (B,nb); pose (B,24,3,3) or (B,72); transl (B,3)|None; cam (B,3)|None.
        Returns vertices (B,V,3)|None, joints (B,NJ,3), joints2d (B,NJ,2)|None (and, with save=True,
        the opaque saved-for-backward buffer as a 4th element)."""
        if self.device is None:
            raise RuntimeError("host-only SMPLEngine: no CUDA device (there is no CPU fallback)")
        B = int(betas.shape[0])
        betas = self._check_in(betas, (B, self.num_betas), "betas")
        pose = self._check_in(pose.reshape(B, -1), (B, 72 if axis_angle else 216), "pose")
        transl = self._check_in(transl, (B, 3), "transl")
        cam = self._check_in(cam, (B, 3), "cam")
        dev = self.device
        verts = torch.empty((B, self.num_verts, 3), dtype=torch.float32, device=dev) if want_vertices else None
        joints = torch.empty((B, self.num_joints_out, 3), dtype=torch.float32, device=dev)
        j2d = torch.empty((B, self.num_joints_out, 2), dtype=torch.float32, device=dev) if cam is not None else None
        with torch.cuda.device(dev):
            ws = self._workspace("fwd", B, mode, slab)
            saved = None
            if save:
                nsaved = int(self.lib.b200smpl_saved_bytes(self.handle, B, slab))
                if saved_buffer is not None and saved_buffer.numel() >= nsaved and saved_buffer.dtype == torch.uint8:
                    saved = saved_buffer                      # caller-owned (e.g. the fitting loop reuses one)
                else:
                    saved = torch.empty(nsaved, dtype=torch.uint8, device=dev)
            args = ForwardArgs(batch=B, mode=mode, pose_is_axis_angle=int(axis_angle), slab_bodies=slab,
                               betas=_ptr(betas), pose=_ptr(pose), transl=_ptr(transl), cam=_ptr(cam),
                               vertices=_ptr(verts), joints=_ptr(joints), joints2d=_ptr(j2d),
                               workspace=_ptr(ws), workspace_bytes=ws.numel(),
                               saved=_ptr(saved), saved_bytes=0 if saved is None else saved.numel())
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.b200smpl_forward(self.handle, ctypes.byref(args), ctypes.c_void_p(stream)),
                       "b200smpl_forward")
        if save:
            # a joints-only forward blends (and keeps) only the virtual joint rows: such a buffer cannot serve a
            # backward with vertex gradients
            saved._b200_joints_only = not want_vertices
            return verts, joints, j2d, saved
        return verts, joints, j2d

    def backward(self, betas, pose, transl, cam, joints, grad_vertices, grad_joints, grad_joints2d, *,
                 axis_angle: bool = False, mode: int = _lib.MODE_FP32, slab: int = 0,
                 need_transl: bool = True, need_cam: bool = True, saved: Optional[torch.Tensor] = None):
        """Returns (grad_betas, grad_pose, grad_transl|None, grad_cam|None)."""
        B = int(betas.shape[0])
        dev = self.device
        betas = self._check_in(betas, (B, self.num_betas), "betas")
        pose = self._check_in(pose.reshape(B, -1), (B, 72 if axis_angle else 216), "pose")
        transl = self._check_in(transl, (B, 3), "transl")
        cam = self._check_in(cam, (B, 3), "cam")
        gv = self._check_in(grad_vertices, (B, self.num_verts, 3), "grad_vertices")
        gj = self._check_in(grad_joints, (B, self.num_joints_out, 3), "grad_joints")
        g2 = self._check_in(grad_joints2d, (B, self.num_joints_out, 2), "grad_joints2d")
        joints = self._check_in(joints, (B, self.num_joints_out, 3), "joints") if g2 is not None else None
        if gv is not None and saved is not None and getattr(saved, "_b200_joints_only", False):
            raise RuntimeError("grad_vertices given with a saved buffer of a joints-only forward (it holds no vertex rows)")
        g_betas = torch.empty((B, self.num_betas), dtype=torch.float32, device=dev)
        g_pose = torch.empty((B, 72 if axis_angle else 216), dtype=torch.float32, device=dev)
        g_transl = torch.empty((B, 3), dtype=torch.float32, device=dev) if need_transl else None
        g_cam = torch.empty((B, 3), dtype=torch.float32, device=dev) if (need_cam and cam is not None) else None
        with torch.cuda.device(dev):
            ws = self._workspace("bwd", B, mode, slab)
            args = BackwardArgs(batch=B, mode=mode, pose_is_axis_angle=int(axis_angle), slab_bodies=slab,
                                betas=_ptr(betas), pose=_ptr(pose), transl=_ptr(transl), cam=_ptr(cam),
                                joints=_ptr(joints), grad_vertices=_ptr(gv), grad_joints=_ptr(gj),
                                grad_joints2d=_ptr(g2), grad_betas=_ptr(g_betas), grad_pose=_ptr(g_pose),
                                grad_transl=_ptr(g_transl), grad_cam=_ptr(g_cam),
                                workspace=_ptr(ws), workspace_bytes=ws.numel(),
                                saved=_ptr(saved), saved_bytes=0 if saved is None else saved.numel())
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.b200smpl_backward(self.handle, ctypes.byref(args), ctypes.c_void_p(stream)),
                       "b200smpl_backward")
        return g_betas, g_pose, g_transl, g_cam


class SMPLFunction(torch.autograd.Function):
    """autograd bridge: forward/backward are single C-ABI calls; nothing but the inputs (and the
    joints when a camera is attached) is saved -- the backward recomputes on the tensor cores."""

    @staticmethod
    def forward(ctx, engine: SMPLEngine, betas, pose, transl, cam, axis_angle: bool, mode: int,
                want_vertices: bool, slab: int):
        need_grad = any(t is not None and t.requires_grad for t in (betas, pose, transl, cam))
        out = engine.forward(betas, pose, transl, cam, axis_angle=axis_angle, mode=mode,
                             want_vertices=want_vertices, slab=slab, save=need_grad)
        verts, joints, j2d = out[:3]
        ctx.saved_blend = out[3] if len(out) > 3 else None   # ~93 KB / body: spares the backward the pose stage and a GEMM
        # (joints-only calls keep it too; only the joint rows of the blend output are computed and filled)
        ctx.set_materialize_grads(False)      # unused outputs arrive as None -> their kernels are skipped
        ctx.engine, ctx.axis_angle, ctx.mode, ctx.slab = engine, axis_angle, mode, slab
        ctx.pose_shape = pose.shape
        ctx.has_transl, ctx.has_cam = transl is not None, cam is not None
        ctx.save_for_backward(betas, pose, transl, cam, joints if cam is not None else None)
        outs = (verts if want_vertices else betas.new_zeros(0), joints, j2d if j2d is not None else betas.new_zeros(0))
        if not want_vertices:
            ctx.mark_non_differentiable(outs[0])
        if j2d is None:
            ctx.mark_non_differentiable(outs[2])
        ctx.want_vertices = want_vertices
        return outs

    @staticmethod
    def backward(ctx, g_verts, g_joints, g_j2d):
        betas, pose, transl, cam, joints = ctx.saved_tensors
        eng = ctx.engine
        gv = g_verts.contiguous() if (ctx.want_vertices and g_verts is not None) else None
        gj = g_joints.contiguous() if g_joints is not None else None
        g2 = g_j2d.contiguous() if (ctx.has_cam and g_j2d is not None) else None
        gb, gp, gt, gc = eng.backward(betas, pose, transl, cam, joints, gv, gj, g2, axis_angle=ctx.axis_angle,
                                      mode=ctx.mode, slab=ctx.slab, need_transl=ctx.has_transl,
                                      need_cam=ctx.has_cam, saved=ctx.saved_blend)
        ctx.saved_blend = None
        return (None, gb, gp.reshape(ctx.pose_shape), gt if ctx.has_transl else None,
                gc if ctx.has_cam else None, None, None, None, None)
