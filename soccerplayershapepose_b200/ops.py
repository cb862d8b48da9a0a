"""The small in-tree helpers of the SMPL path as autograd Functions over the C-ABI kernels
(SURVEY.md section 8 rows a13-a18).  CUDA float32 tensors only -- no CPU path."""
from __future__ import annotations

import ctypes
import weakref
from typing import Optional

import torch

from . import _lib, config


def _stream(t: torch.Tensor) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _req(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError("{} must be a CUDA tensor: the b200 SMPL ops have no CPU implementation".format(name))
    if t.dtype != torch.float32:
        raise TypeError("{} must be float32".format(name))
    return t.contiguous()


class _Rot6d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _req(x, "x").reshape(-1, 6)
        n = x.shape[0]
        out = torch.empty((n, 3, 3), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200smpl_rot6d_to_rotmat(x.data_ptr(), out.data_ptr(), n, _stream(x)), "rot6d")
        ctx.save_for_backward(x)
        return out

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = g.contiguous()
        gx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200smpl_rot6d_to_rotmat_backward(x.data_ptr(), g.data_ptr(), gx.data_ptr(),
                                                                     x.shape[0], _stream(x)), "rot6d_bwd")
        return gx


def rot6d_to_rotmat(x: torch.Tensor) -> torch.Tensor:
    """utils/rigid_transform_utils.py:27-41: (B,6k) -> (B*k,3,3); gradient flows to the input's shape."""
    return _Rot6d.apply(x.reshape(-1, 6))


class _Rodrigues(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rot_vecs):
        x = _req(rot_vecs, "rot_vecs").reshape(-1, 3)
        n = x.shape[0]
        out = torch.empty((n, 3, 3), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200smpl_batch_rodrigues(x.data_ptr(), out.data_ptr(), n, _stream(x)), "batch_rodrigues")
        ctx.save_for_backward(x)
        return out

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = g.contiguous()
        gx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200smpl_batch_rodrigues_backward(x.data_ptr(), g.data_ptr(), gx.data_ptr(),
                                                                     x.shape[0], _stream(x)), "batch_rodrigues_bwd")
        return gx


def batch_rodrigues(rot_vecs: torch.Tensor, epsilon: float = 1e-8) -> torch.Tensor:
    """smplx.lbs.batch_rodrigues (reference call sites: player_recon.py:201,655, hmr.py:207): (N,3) axis-angle ->
    (N,3,3), with the library's `angle = ||r + 1e-8||`; differentiable.  Only the default epsilon is implemented."""
    if epsilon != 1e-8:
        raise ValueError("batch_rodrigues: only epsilon=1e-8 (the smplx default) is implemented")
    return _Rodrigues.apply(rot_vecs.reshape(-1, 3))


class _Ortho(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pts, cam, pixel_wh):
        pts, cam = _req(pts, "points3D"), _req(cam, "cam_params")
        B, N = pts.shape[0], pts.shape[1]
        out = torch.empty((B, N, 2), dtype=torch.float32, device=pts.device)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_orthographic_project(pts.data_ptr(), cam.data_ptr(), out.data_ptr(), B, N,
                                                                 float(pixel_wh), _stream(pts)), "ortho")
        ctx.save_for_backward(pts, cam)
        ctx.pixel_wh = float(pixel_wh)
        return out

    @staticmethod
    def backward(ctx, g):
        pts, cam = ctx.saved_tensors
        g = g.contiguous()
        B, N = pts.shape[0], pts.shape[1]
        gp = torch.empty_like(pts) if ctx.needs_input_grad[0] else None
        gc = torch.empty_like(cam) if ctx.needs_input_grad[1] else None
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_orthographic_project_backward(
                pts.data_ptr(), cam.data_ptr(), g.data_ptr(), None if gp is None else gp.data_ptr(),
                None if gc is None else gc.data_ptr(), B, N, ctx.pixel_wh, _stream(pts)), "ortho_bwd")
        return gp, gc, None


def orthographic_project(points3D: torch.Tensor, cam_params: torch.Tensor, pixel_wh: float = 0.0) -> torch.Tensor:
    """utils/cam_utils.py:5-26; pixel_wh>0 fuses utils/joints2d_utils.py:5-10 behind it."""
    return _Ortho.apply(points3D, cam_params, pixel_wh)


class _Persp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pts, rot, trans, focal, wh):
        pts, rot, trans = _req(pts, "points"), _req(rot, "rotation"), _req(trans, "translation")
        B, N = pts.shape[0], pts.shape[1]
        out = torch.empty((B, N, 2), dtype=torch.float32, device=pts.device)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_perspective_project(pts.data_ptr(), rot.data_ptr(), trans.data_ptr(),
                                                                out.data_ptr(), B, N, float(focal), float(wh),
                                                                _stream(pts)), "persp")
        ctx.save_for_backward(pts, rot, trans)
        ctx.focal, ctx.wh = float(focal), float(wh)
        return out

    @staticmethod
    def backward(ctx, g):
        pts, rot, trans = ctx.saved_tensors
        g = g.contiguous()
        B, N = pts.shape[0], pts.shape[1]
        gp, gr, gt = torch.empty_like(pts), torch.empty_like(rot), torch.empty_like(trans)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_perspective_project_backward(
                pts.data_ptr(), rot.data_ptr(), trans.data_ptr(), g.data_ptr(), gp.data_ptr(), gr.data_ptr(),
                gt.data_ptr(), B, N, ctx.focal, ctx.wh, _stream(pts)), "persp_bwd")
        return gp, gr, gt, None, None


class _PerspK(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pts, rot, trans, cam_K):
        pts, rot, trans, cam_K = _req(pts, "points"), _req(rot, "rotation"), _req(trans, "translation"), _req(cam_K, "cam_K")
        B, N = pts.shape[0], pts.shape[1]
        batched = cam_K.dim() == 3
        if tuple(cam_K.shape) not in ((3, 3), (B, 3, 3)):
            raise ValueError("cam_K has shape {}, expected (3, 3) or ({}, 3, 3)".format(tuple(cam_K.shape), B))
        out = torch.empty((B, N, 2), dtype=torch.float32, device=pts.device)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_perspective_project_camk(
                pts.data_ptr(), rot.data_ptr(), trans.data_ptr(), cam_K.data_ptr(), int(batched), out.data_ptr(), B, N,
                _stream(pts)), "persp_camk")
        ctx.save_for_backward(pts, rot, trans, cam_K)
        ctx.batched = batched
        return out

    @staticmethod
    def backward(ctx, g):
        pts, rot, trans, cam_K = ctx.saved_tensors
        g = g.contiguous()
        B, N = pts.shape[0], pts.shape[1]
        gp, gr, gt = torch.empty_like(pts), torch.empty_like(rot), torch.empty_like(trans)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().b200smpl_perspective_project_camk_backward(
                pts.data_ptr(), rot.data_ptr(), trans.data_ptr(), cam_K.data_ptr(), int(ctx.batched), g.data_ptr(),
                gp.data_ptr(), gr.data_ptr(), gt.data_ptr(), B, N, _stream(pts)), "persp_camk_bwd")
        return gp, gr, gt, None


def perspective_project_camk(points, rotation, translation, cam_K) -> torch.Tensor:
    """utils/cam_utils.py:54-85 with an explicit intrinsics matrix cam_K (B,3,3) or (3,3); cam_K gets no gradient."""
    return _PerspK.apply(points, rotation, translation, cam_K)


def perspective_project(points, rotation, translation, focal_length: float, img_wh: float) -> torch.Tensor:
    """utils/cam_utils.py:54-85 with the (focal_length, img_wh) intrinsics form used at
    player_recon.py:685-688."""
    return _Persp.apply(points, rotation, translation, focal_length, img_wh)


_JOINT_MAP_OK = {}


def _checked_joint_map(joint_map: torch.Tensor, device: torch.device, nj: int) -> torch.Tensor:
    """The loss kernel reads the map as int32 and indexes joints / grad_joints with it unchecked: convert integer
    maps to int32 and check the range once per (tensor, version) -- the range check is a host read, so it is cached
    and skipped inside a CUDA-graph capture."""
    if not isinstance(joint_map, torch.Tensor) or joint_map.device != device:
        raise RuntimeError("joint_map must be a tensor on {}".format(device))
    key = (joint_map.data_ptr(), joint_map.numel(), joint_map._version, str(joint_map.dtype), nj)
    hit = _JOINT_MAP_OK.get(key)
    if hit is not None and hit[0]() is joint_map:             # the very tensor that was checked, unmodified since
        return hit[1]
    if joint_map.dtype not in (torch.int32, torch.int64, torch.int16, torch.uint8, torch.int8):
        raise TypeError("joint_map must be an integer tensor, got {}".format(joint_map.dtype))
    m32 = joint_map.to(torch.int32).contiguous().view(-1)
    if torch.cuda.is_current_stream_capturing():
        return m32                                            # unchecked (and uncached) inside a capture
    if m32.numel() and (int(m32.min()) < 0 or int(m32.max()) >= nj):
        raise IndexError("joint_map entries must lie in [0, {})".format(nj))
    if len(_JOINT_MAP_OK) > 64:
        _JOINT_MAP_OK.clear()
    _JOINT_MAP_OK[key] = (weakref.ref(joint_map), m32)
    return m32


class _J2dLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, joints, cam, joint_map, label, vis, proj_wh, norm_wh, log_var):
        joints, cam, label = _req(joints, "joints"), _req(cam, "cam"), _req(label, "label")
        B, NJ = joints.shape[0], joints.shape[1]
        nmap = joint_map.numel()
        joint_map = _checked_joint_map(joint_map, joints.device, NJ)
        if tuple(cam.shape) != (B, 3):
            raise ValueError("cam has shape {}, expected {}".format(tuple(cam.shape), (B, 3)))
        if tuple(label.shape) != (B, nmap, 2):
            raise ValueError("label has shape {}, expected {}".format(tuple(label.shape), (B, nmap, 2)))
        if vis is not None and tuple(vis.shape) != (B, nmap):
            raise ValueError("vis has shape {}, expected {}".format(tuple(vis.shape), (B, nmap)))
        loss = torch.zeros(2, dtype=torch.float32, device=joints.device)
        gj = torch.empty_like(joints)
        gc = torch.empty_like(cam)
        visu8 = None if vis is None else vis.to(torch.uint8).contiguous()
        with torch.cuda.device(joints.device):
            _lib.check(_lib.load().b200smpl_joints2d_loss(
                joints.data_ptr(), cam.data_ptr(), joint_map.data_ptr(), label.data_ptr(),
                None if visu8 is None else visu8.data_ptr(), B, NJ, nmap, float(proj_wh), float(norm_wh),
                float(log_var), loss.data_ptr(), gj.data_ptr(), gc.data_ptr(), _stream(joints)), "joints2d_loss")
        ctx.save_for_backward(gj, gc)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        gj, gc = ctx.saved_tensors
        return gj * g, gc * g, None, None, None, None, None, None


def joints2d_loss(joints: torch.Tensor, cam: torch.Tensor, joint_map: torch.Tensor, label_pixels: torch.Tensor,
                  vis: Optional[torch.Tensor] = None, proj_wh: float = 512.0, norm_wh: float = 256.0,
                  log_var: float = 0.0) -> torch.Tensor:
    """Fused reprojection loss: orthographic_project_torch(joints, cam)[:, joint_map] ->
    undo_keypoint_normalisation(., proj_wh) -> joints2D term of the multi-task loss
    (losses/multi_task_loss.py:97-113) with a fixed log-variance.  joint_map: integer CUDA tensor with entries in
    [0, NJ) (converted to int32; a repeated joint accumulates its gradient)."""
    return _J2dLoss.apply(joints, cam, joint_map, label_pixels, vis, proj_wh, norm_wh, log_var)


class _MultiTaskLoss(torch.autograd.Function):
    """loss, parts = f(log_var[5], verts, joints, cam, shape, pose | labels, maps): two launches forward (one
    reduction pass + finalise), one launch backward; the upstream gradient and the log-variances are read on the
    device, so the whole thing sits inside a CUDA graph."""

    @staticmethod
    def forward(ctx, log_var, verts, joints, cam, shape, pose, verts_label, map2d, label2d, vis, map3d, label3d,
                shape_label, pose_label, proj_wh, norm_wh):
        dev = log_var.device
        f = lambda t, n: None if t is None else _req(t, n)   # noqa: E731
        log_var = _req(log_var, "log_var")
        verts, joints, cam = f(verts, "verts"), f(joints, "joints"), f(cam, "cam")
        shape, pose = f(shape, "shape"), f(pose, "pose")
        verts_label, label2d, label3d = f(verts_label, "verts_label"), f(label2d, "label2d"), f(label3d, "label3d")
        shape_label, pose_label = f(shape_label, "shape_label"), f(pose_label, "pose_label")
        ref = joints if joints is not None else (verts if verts is not None else (shape if shape is not None else pose))
        if ref is None:
            raise ValueError("multitask_loss needs at least one term")
        B = ref.shape[0]
        NJ = 0 if joints is None else joints.shape[1]
        if map2d is not None:
            map2d = _checked_joint_map(map2d, dev, NJ)
        if map3d is not None:
            map3d = _checked_joint_map(map3d, dev, NJ)
        n2 = 0 if map2d is None else map2d.numel()
        n3 = 0 if map3d is None else map3d.numel()

        def chk(t, shp, name):
            if t is not None and tuple(t.shape) != tuple(shp):
                raise ValueError("{} has shape {}, expected {}".format(name, tuple(t.shape), tuple(shp)))
        if log_var.numel() != 5:
            raise ValueError("log_var must hold 5 values (verts, joints2D, joints3D, shape, pose)")
        V = 0 if verts is None else verts.shape[1]
        chk(verts, (B, V, 3), "verts"); chk(verts_label, (B, V, 3), "verts_label")
        chk(cam, (B, 3), "cam"); chk(label2d, (B, n2, 2), "label2d"); chk(label3d, (B, n3, 3), "label3d")
        if (verts is None) != (verts_label is None) or (shape is None) != (shape_label is None) or \
                (pose is None) != (pose_label is None):
            raise ValueError("a prediction and its label must be given together")
        pose2 = None if pose is None else pose.reshape(B, -1)
        pose_label2 = None if pose_label is None else pose_label.reshape(B, -1)
        if shape is not None:
            chk(shape_label, tuple(shape.shape), "shape_label")
        if pose2 is not None:
            chk(pose_label2, tuple(pose2.shape), "pose_label")
        visu8 = None
        if vis is not None:
            chk(vis, (B, n2), "vis")
            visu8 = vis.to(torch.uint8).contiguous()
        p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        scratch = torch.empty(16, dtype=torch.float32, device=dev)
        out = torch.empty(11, dtype=torch.float32, device=dev)
        args = _lib.MultiTaskLossArgs(
            batch=B, num_verts=V, num_joints=NJ, nmap2d=n2, nmap3d=n3, num_betas=0 if shape is None else shape.shape[1],
            pose_cols=0 if pose2 is None else pose2.shape[1], reserved0=0, proj_wh=float(proj_wh), norm_wh=float(norm_wh),
            verts=p(verts), verts_label=p(verts_label), joints=p(joints), cam=p(cam), map2d=p(map2d), label2d=p(label2d),
            vis=p(visu8), map3d=p(map3d), label3d=p(label3d), shape=p(shape), shape_label=p(shape_label), pose=p(pose2),
            pose_label=p(pose_label2), log_var=p(log_var), scratch=p(scratch))
        with torch.cuda.device(dev):
            _lib.check(_lib.load().b200smpl_multitask_loss(ctypes.byref(args), out.data_ptr(), _stream(log_var)),
                       "multitask_loss")
        ctx.args = args
        ctx.keep = (log_var, verts, joints, cam, shape, pose2, verts_label, map2d, label2d, visu8, map3d, label3d,
                    shape_label, pose_label2, scratch, out)          # the raw pointers in `args` stay valid
        ctx.pose_shape = None if pose is None else pose.shape
        parts = out[1:6]
        ctx.mark_non_differentiable(parts)
        return out[0], parts

    @staticmethod
    def backward(ctx, g_loss, _g_parts):
        (log_var, verts, joints, cam, shape, pose2, _vl, _m2, _l2, _vis, _m3, _l3, _sl, _pl, _scratch, out) = ctx.keep
        need = ctx.needs_input_grad
        g = g_loss.contiguous().float()
        mk = lambda t, on: torch.empty_like(t) if (t is not None and on) else None   # noqa: E731
        gv, gj, gc = mk(verts, need[1]), mk(joints, need[2]), mk(cam, need[3])
        gs, gp = mk(shape, need[4]), mk(pose2, need[5])
        p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        with torch.cuda.device(g.device):
            _lib.check(_lib.load().b200smpl_multitask_loss_backward(
                ctypes.byref(ctx.args), g.data_ptr(), p(gv), p(gj), p(gc), p(gs), p(gp), _stream(g)),
                "multitask_loss_backward")
        glv = out[6:11] * g if need[0] else None
        if gp is not None:
            gp = gp.reshape(ctx.pose_shape)
        return (glv, gv, gj, gc, gs, gp) + (None,) * 10


def multitask_loss(log_var: torch.Tensor, *, verts=None, verts_label=None, joints=None, cam=None, map2d=None,
                   label2d=None, vis=None, map3d=None, label3d=None, shape=None, shape_label=None, pose=None,
                   pose_label=None, proj_wh: float = 512.0, norm_wh: float = 256.0):
    """Fused HomoscedasticUncertaintyWeightedMultiTaskLoss (losses/multi_task_loss.py:92-130 without the silhouette
    term, which regressor.MultiTaskLoss adds with `silhouette_term`): `log_var` (5,) = log-variances of (verts, joints2D, joints3D, shape_params, pose_params); a term is
    evaluated when its prediction (its joint map for the joint terms) is given.  Returns (loss, parts (5,))."""
    return _MultiTaskLoss.apply(log_var, verts, joints, cam, shape, pose, verts_label, map2d, label2d, vis, map3d,
                                label3d, shape_label, pose_label, proj_wh, norm_wh)


# ---- silhouettes (DESIGN.md section 11) ------------------------------------------------------------------------------
_FACES_I32 = {}


def _faces_int32(faces: torch.Tensor, device: torch.device, V: int) -> torch.Tensor:
    """(F,3) integer faces as contiguous int32 on `device`, range-checked once per (tensor, version) like the joint
    maps (the kernels drop a face with an out-of-range index, but a wrong topology should fail loudly)."""
    if not isinstance(faces, torch.Tensor):
        faces = torch.as_tensor(faces)
    if faces.dim() != 2 or faces.shape[1] != 3:
        raise ValueError("faces has shape {}, expected (F, 3)".format(tuple(faces.shape)))
    if faces.dtype.is_floating_point or faces.dtype == torch.bool:
        raise TypeError("faces must be an integer tensor, got {}".format(faces.dtype))
    key = (faces.data_ptr(), faces.numel(), faces._version, str(faces.dtype), str(faces.device), str(device), V)
    hit = _FACES_I32.get(key)
    if hit is not None and hit[0]() is faces:
        return hit[1]
    f32 = faces.to(device=device, dtype=torch.int32).contiguous()
    if torch.cuda.is_current_stream_capturing():
        return f32
    if f32.numel() and (int(f32.min()) < 0 or int(f32.max()) >= V):
        raise IndexError("faces entries must lie in [0, {})".format(V))
    if len(_FACES_I32) > 64:
        _FACES_I32.clear()
    _FACES_I32[key] = (weakref.ref(faces), f32)
    return f32


def silhouette_args(vertices: torch.Tensor, faces32: torch.Tensor, cam_t: torch.Tensor, img_wh: int,
                    focal_length: float, sigma: float) -> "_lib.SilhouetteArgs":
    """The C-ABI argument struct over caller-owned device tensors (kept alive by the caller)."""
    B, V = vertices.shape[0], vertices.shape[1]
    if vertices.dim() != 3 or vertices.shape[2] != 3:
        raise ValueError("vertices has shape {}, expected (B, V, 3)".format(tuple(vertices.shape)))
    if tuple(cam_t.shape) != (B, 3):
        raise ValueError("cam_t has shape {}, expected {}".format(tuple(cam_t.shape), (B, 3)))
    if cam_t.device != vertices.device or faces32.device != vertices.device:
        raise RuntimeError("vertices, faces and cam_t must be on the same device")
    if int(img_wh) < 1 or not float(sigma) >= 0.0:
        raise ValueError("need img_wh >= 1 and sigma >= 0")
    return _lib.SilhouetteArgs(batch=B, num_verts=V, num_faces=faces32.shape[0], img_wh=int(img_wh),
                               focal_length=float(focal_length), sigma=float(sigma), vertices=vertices.data_ptr(),
                               cam_t=cam_t.data_ptr(), faces=faces32.data_ptr(), workspace=None, workspace_bytes=0)


class _Silhouette(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vertices, cam_t, faces32, img_wh, focal_length, sigma):
        vertices, cam_t = _req(vertices, "vertices"), _req(cam_t, "cam_t")
        args = silhouette_args(vertices, faces32, cam_t, img_wh, focal_length, sigma)
        B, S = vertices.shape[0], int(img_wh)
        alpha = torch.empty((B, S, S), dtype=torch.float32, device=vertices.device)
        with torch.cuda.device(vertices.device):
            _lib.check(_lib.load().b200smpl_silhouette_render(ctypes.byref(args), alpha.data_ptr(), _stream(vertices)),
                       "silhouette_render")
        ctx.save_for_backward(vertices, cam_t, faces32)
        ctx.img_wh, ctx.focal_length, ctx.sigma = S, float(focal_length), float(sigma)
        if sigma == 0.0:
            ctx.mark_non_differentiable(alpha)
        return alpha

    @staticmethod
    def backward(ctx, g):
        vertices, cam_t, faces32 = ctx.saved_tensors
        args = silhouette_args(vertices, faces32, cam_t, ctx.img_wh, ctx.focal_length, ctx.sigma)
        g = g.contiguous().float()
        gv = torch.empty_like(vertices)
        gt = torch.empty_like(cam_t)
        with torch.cuda.device(vertices.device):
            _lib.check(_lib.load().b200smpl_silhouette_render_backward(
                ctypes.byref(args), g.data_ptr(), gv.data_ptr(), gt.data_ptr(), _stream(vertices)),
                "silhouette_render_backward")
        return gv, gt, None, None, None, None


def render_silhouettes(vertices: torch.Tensor, faces, cam_t: torch.Tensor, img_wh: int,
                       focal_length: float = config.FOCAL_LENGTH, sigma: float = 0.0) -> torch.Tensor:
    """Silhouettes (B, S, S) of the meshes `vertices` (B,V,3) / `faces` (F,3) seen through the camera of the
    reference's neural-renderer call nmr(vertices, faces, t) (player_recon.py:1226-1229): R = I, translation `cam_t`
    (B,3), K = [[f,0,S/2],[0,f,S/2],[0,0,1]], S = img_wh.  Element [i, j] is the pixel centred at (j + 0.5, i + 0.5)
    with u = f (x+tx)/(z+tz) + S/2 and v likewise -- what cam_utils.perspective_project_torch returns -- and no
    vertical flip (the orientation of the reference's renderer could not be checked; use torch.flip if a caller
    needs the other one).  sigma == 0: binary coverage, no gradient (a backward raises ValueError).  sigma > 0 (px^2):
    the SoftRas / SoftSilhouetteShader soft silhouette, differentiable w.r.t. `vertices` and `cam_t`."""
    vertices = _req(vertices, "vertices")
    faces32 = _faces_int32(faces, vertices.device, vertices.shape[1])
    return _Silhouette.apply(vertices, cam_t, faces32, int(img_wh), float(focal_length), float(sigma))


def silhouette_loss(vertices: torch.Tensor, faces, cam_t: torch.Tensor, target: torch.Tensor, img_wh: int,
                    focal_length: float = config.FOCAL_LENGTH, sigma: float = 1.0, weight: float = 1.0,
                    loss_per_body: Optional[torch.Tensor] = None):
    """Fused silhouette term of the fitting loop (one kernel; the image is never written):
    loss_per_body[b] += weight * mean over the S^2 pixels of (alpha_b - target_b)^2, target (B,S,S) mask.  Returns
    (loss_per_body, grad_vertices, grad_cam_t) -- plain tensors, no autograd.  The form of the reference's silhouette
    loss term (losses/multi_task_loss.py:132-144) could not be read; this squared error is the stated definition."""
    vertices, cam_t = _req(vertices, "vertices"), _req(cam_t, "cam_t")
    B = vertices.shape[0]
    faces32 = _faces_int32(faces, vertices.device, vertices.shape[1])
    args = silhouette_args(vertices, faces32, cam_t, img_wh, focal_length, sigma)
    S = int(img_wh)
    if tuple(target.shape) != (B, S, S):
        raise ValueError("target has shape {}, expected {}".format(tuple(target.shape), (B, S, S)))
    tgt = target.to(device=vertices.device, dtype=torch.uint8).contiguous()
    if loss_per_body is None:
        loss_per_body = torch.zeros(B, dtype=torch.float32, device=vertices.device)
    gv = torch.empty_like(vertices)
    gt = torch.empty_like(cam_t)
    with torch.cuda.device(vertices.device):
        _lib.check(_lib.load().b200smpl_silhouette_loss(ctypes.byref(args), tgt.data_ptr(), float(weight),
                                                        loss_per_body.data_ptr(), gv.data_ptr(), gt.data_ptr(),
                                                        _stream(vertices)), "silhouette_loss")
    return loss_per_body, gv, gt


def _binary_target(target: torch.Tensor, B: int, S: int, device: torch.device) -> torch.Tensor:
    """(B,S,S) mask as contiguous uint8 on `device`: floating point `>= 0.5`, other dtypes non-zero (as
    `silhouette_iou` reads masks).  Plain tensor ops, so a CUDA graph can capture it."""
    if tuple(target.shape) != (B, S, S):
        raise ValueError("target has shape {}, expected {}".format(tuple(target.shape), (B, S, S)))
    mask = target >= 0.5 if target.dtype.is_floating_point else target != 0
    return mask.to(device=device, dtype=torch.uint8).contiguous()


def silhouette_loss_value(vertices: torch.Tensor, faces, cam_t: torch.Tensor, target: torch.Tensor, img_wh: int,
                          focal_length: float = config.FOCAL_LENGTH, sigma: float = 1.0, weight: float = 1.0,
                          loss_per_body: Optional[torch.Tensor] = None) -> torch.Tensor:
    """loss_per_body[b] += weight * mean over the S^2 pixels of (alpha_b - target_b)^2 without the gradient: one
    kernel that neither writes the image nor runs the backward (validation and no-grad passes).  sigma == 0 scores
    the hard silhouette.  Returns loss_per_body (B,), a plain tensor."""
    vertices, cam_t = _req(vertices, "vertices"), _req(cam_t, "cam_t")
    B, S = vertices.shape[0], int(img_wh)
    faces32 = _faces_int32(faces, vertices.device, vertices.shape[1])
    args = silhouette_args(vertices, faces32, cam_t, S, focal_length, sigma)
    tgt = _binary_target(target, B, S, vertices.device)
    if loss_per_body is None:
        loss_per_body = torch.zeros(B, dtype=torch.float32, device=vertices.device)
    elif (tuple(loss_per_body.shape) != (B,) or loss_per_body.dtype != torch.float32
          or loss_per_body.device != vertices.device or not loss_per_body.is_contiguous()):
        raise ValueError("loss_per_body must be a contiguous float32 ({},) tensor on the device of vertices".format(B))
    with torch.cuda.device(vertices.device):
        _lib.check(_lib.load().b200smpl_silhouette_loss_value(ctypes.byref(args), tgt.data_ptr(), float(weight),
                                                              loss_per_body.data_ptr(), _stream(vertices)),
                   "silhouette_loss_value")
    return loss_per_body


class _SilhouetteTerm(torch.autograd.Function):
    """Batch mean of the per-body silhouette loss through the fused loss kernel: its forward keeps the gradients of
    the term, its backward scales them by the upstream gradient on the device (no host read: graph-capturable)."""

    @staticmethod
    def forward(ctx, vertices, cam_t, faces32, tgt, img_wh, focal_length, sigma):
        args = silhouette_args(vertices, faces32, cam_t, img_wh, focal_length, sigma)
        B = vertices.shape[0]
        loss = torch.zeros(B, dtype=torch.float32, device=vertices.device)
        gv, gt = torch.empty_like(vertices), torch.empty_like(cam_t)
        with torch.cuda.device(vertices.device):
            _lib.check(_lib.load().b200smpl_silhouette_loss(ctypes.byref(args), tgt.data_ptr(), 1.0 / B,
                                                            loss.data_ptr(), gv.data_ptr(), gt.data_ptr(),
                                                            _stream(vertices)), "silhouette_loss")
        ctx.save_for_backward(gv, gt)
        return loss.sum()

    @staticmethod
    def backward(ctx, g):
        gv, gt = ctx.saved_tensors
        return gv * g, gt * g, None, None, None, None, None


def silhouette_term(vertices: torch.Tensor, faces, cam_t: torch.Tensor, target: torch.Tensor, img_wh: int,
                    focal_length: float = config.FOCAL_LENGTH, sigma: float = 1.0) -> torch.Tensor:
    """Scalar silhouette term: the batch mean of the per-body mean over the S^2 pixels of (alpha - target)^2,
    differentiable w.r.t. `vertices` and `cam_t` (sigma > 0).  When a gradient is needed the fused loss kernel runs
    and keeps it; otherwise (no_grad, or no input requires a gradient) only the gradient-free value kernel runs.
    target (B,S,S): floating point `>= 0.5` or non-zero is inside."""
    vertices, cam_t = _req(vertices, "vertices"), _req(cam_t, "cam_t")
    B, S = vertices.shape[0], int(img_wh)
    faces32 = _faces_int32(faces, vertices.device, vertices.shape[1])
    tgt = _binary_target(target, B, S, vertices.device)
    if torch.is_grad_enabled() and (vertices.requires_grad or cam_t.requires_grad):
        return _SilhouetteTerm.apply(vertices, cam_t, faces32, tgt, S, float(focal_length), float(sigma))
    return silhouette_loss_value(vertices, faces32, cam_t, tgt, S, focal_length, sigma, 1.0 / B).sum()


def silhouette_iou(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """IoU per body of compute_silh_error_metrics (metrics/silhouettes_joints_metrics.py:5-37) on masks
    `alpha >= 0.5`: (B,S,S) x (B,S,S) -> (B,).  A metric, not on the hot path: plain torch ops.  An empty union
    gives IoU 1."""
    p = pred >= 0.5 if pred.dtype.is_floating_point else pred.bool()
    t = target >= 0.5 if target.dtype.is_floating_point else target.bool()
    inter = (p & t).flatten(1).sum(1).double()
    union = (p | t).flatten(1).sum(1).double()
    return torch.where(union > 0, inter / union.clamp(min=1), torch.ones_like(union)).float()
