"""Batched per-player SMPL fitting on 2D keypoints (SURVEY.md section 8f.1; BASELINE.json configs[2]).

Restates the optimisation loop of the reference's `single_view_optimization`
(PlayerReconstruction/player_recon.py:1172-1294) for a batch of independent players:

  * parameters, as there: global orientation and body pose as raw rotation matrices (`pose2rot=False`),
    weak-perspective camera `[s, tx, ty]` and betas; the hands / feet joints of the body pose (body_pose[:, 6:8]
    and body_pose[:, 21:], player_recon.py:1175-1177, 1202-1206) stay at their initial value;
  * loss per player: joints2D term of the multi-task loss on the 17 COCO joints, after
    `orthographic_project_torch` and `undo_keypoint_normalisation` (player_recon.py:1217-1221,
    losses/multi_task_loss.py:97-113), optionally plus a shape prior `shape_weight * mean(betas^2)`
    (BASELINE.json asks for one; the reference loop has none -- default 0 reproduces the reference);
    optionally plus a silhouette term `silhouette_weight * mean over pixels of (alpha - target)^2` on the soft
    silhouette of the posed mesh (player_recon.py:1226-1229 renders it with the neural renderer; here the
    rasteriser of csrc/silhouette.cu, DESIGN.md section 11) when `fit(..., silhouettes=...)` is given;
  * optimiser: `torch.optim.Adam(params, lr)` arithmetic (player_recon.py:1199), elementwise, so a batch of
    players with a summed loss is exactly a set of independent per-player optimisations;
  * the best iterate per player is kept (player_recon.py:1254-1266) -- here on the device, by loss value,
    instead of a host round trip per iteration;
  * results under the reference's `.npz` keys (player_recon.py:1293-1294): body_pose, global_orient, betas,
    translation (`convert_weak_perspective_to_camera_translation`, cam_utils.py:44-52).

Without silhouettes only the joints are computed (virtual rows of the blend GEMM, no vertex is skinned).  One
iteration = 7 kernel launches through the C-ABI (the backward reuses the forward's transforms and blend rows); after
one eager iteration, twenty consecutive iterations are captured in one CUDA graph (kept, with its state buffers, for
later calls of the same shape) and replayed.  With silhouettes an iteration is the full-vertex forward, fit_loss, the
fused silhouette loss (forward, loss and backward in one kernel), the backward with vertex and joint gradients and
fit_update, with the camera-translation gradient chained into the camera's Adam step; it is captured the same way.
CUDA float32 only: there is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import torch

from . import _lib, config
from .cam_utils import convert_weak_perspective_to_camera_translation_torch
from .smpl import SMPL

FROZEN_FULL_JOINTS = (7, 8, 22, 23)       # body_pose[:, 6:8] and body_pose[:, 21:] in full-pose numbering


def _target_masks(silhouettes: torch.Tensor, shape: tuple, dev: torch.device) -> torch.Tensor:
    """The fitters' target masks: `silhouettes` of the given shape as bool on `dev`, non-zero is inside."""
    if tuple(silhouettes.shape) != shape:
        raise ValueError("silhouettes has shape {}, expected {}".format(tuple(silhouettes.shape), shape))
    return silhouettes.to(device=dev) != 0


class BatchedFitter:
    def __init__(self, smpl: SMPL, lr: float = 1e-3, shape_weight: float = 0.0, joints2d_log_var: float = 0.0,
                 proj_wh: float = 512.0, norm_wh: float = float(config.REGRESSOR_IMG_WH),
                 betas: tuple = (0.9, 0.999), eps: float = 1e-8, use_cuda_graph: bool = True,
                 frozen_joints=FROZEN_FULL_JOINTS, mode: Optional[str] = None, graph_iterations: int = 20,
                 silhouette_weight: float = 0.0, silhouette_sigma: float = 1.0, silhouette_wh: int = 256):
        """silhouette_weight > 0 adds the silhouette term to the loss of every player when `fit` receives target
        silhouettes (silhouette_wh x silhouette_wh masks); silhouette_sigma (px^2 at that resolution) is the blur of
        the soft silhouette (SMPL.render_silhouettes frames the image like the `proj_wh` crop)."""
        dev = next(smpl.buffers()).device
        if dev.type != "cuda":
            raise RuntimeError("BatchedFitter needs the SMPL module on a CUDA device (no CPU path)")
        self.smpl, self.dev = smpl, dev
        self.eng = smpl._engine(dev)
        self.mode = _lib.MODES[mode] if mode is not None else smpl.mode
        self.lib = _lib.load()
        self.lr, self.shape_weight, self.log_var = float(lr), float(shape_weight), float(joints2d_log_var)
        self.proj_wh, self.norm_wh = float(proj_wh), float(norm_wh)
        self.b1, self.b2, self.eps = float(betas[0]), float(betas[1]), float(eps)
        self.use_graph = use_cuda_graph
        self.graph_iterations = max(2, int(graph_iterations) // 2 * 2)   # even: the step counter's parity repeats per replay
        self.jmap = torch.tensor(config.SMPL_TO_KPRCNN_MAP, dtype=torch.int32, device=dev)
        frozen = torch.zeros(24, 9, dtype=torch.uint8)
        for j in frozen_joints:
            frozen[j] = 1
        self.frozen_rot = frozen.reshape(-1).to(dev)
        self.sil_weight, self.sil_sigma, self.sil_wh = float(silhouette_weight), float(silhouette_sigma), int(silhouette_wh)
        if self.sil_weight > 0.0 and not self.sil_sigma > 0.0:
            raise ValueError("the silhouette term needs silhouette_sigma > 0 (the hard silhouette has no gradient)")
        self.faces = smpl.faces_int32(dev)
        self._cache = {}
        self._state = None
        self._parity = 0

    # ---- one iteration: every call below is one C-ABI entry point on the current stream ----------------
    def _iteration(self, st: Dict[str, torch.Tensor]) -> None:
        lib, B = self.lib, st["rot"].shape[0]
        stream = ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)
        sil = "sil" in st
        # the transforms and the virtual rows of the blend output are kept for the backward (no recomputation)
        verts, joints, _, saved = self.eng.forward(st["betas"], st["rot"], None, None, axis_angle=False, mode=self.mode,
                                                   want_vertices=sil, save=True, saved_buffer=st.get("saved"))
        st["saved"] = saved
        vis = st.get("vis")
        _lib.check(lib.b200smpl_fit_loss(
            joints.data_ptr(), st["cam"].data_ptr(), self.jmap.data_ptr(), st["label"].data_ptr(),
            None if vis is None else vis.data_ptr(), st["betas"].data_ptr(), B, joints.shape[1], self.jmap.numel(),
            st["betas"].shape[1], self.proj_wh, self.norm_wh, self.log_var, self.shape_weight, st["loss"].data_ptr(),
            st["gj"].data_ptr(), st["gcam"].data_ptr(), st["gbetas_prior"].data_ptr(), stream), "fit_loss")
        cam_extra = self._silhouette_term(verts, st["cam"], st["sil"], st["loss"], st["gv"], st["t"], st["gt"],
                                          st["gcam_sil"], stream) if sil else None
        gb, gp, _, _ = self.eng.backward(st["betas"], st["rot"], None, None, None, st["gv"] if sil else None, st["gj"],
                                         None, axis_angle=False, mode=self.mode, need_transl=False, need_cam=False,
                                         saved=saved)
        # best-iterate bookkeeping + the Adam step of the three parameter tensors: one launch
        groups = (_lib.FitGroup * 3)()
        for k, (name, grad, extra, frozen) in enumerate((("rot", gp, None, self.frozen_rot),
                                                         ("betas", gb, st["gbetas_prior"], None),
                                                         ("cam", st["gcam"], cam_extra, None))):
            p = st[name]
            groups[k] = _lib.FitGroup(p.data_ptr(), grad.data_ptr(), None if extra is None else extra.data_ptr(),
                                      st["m_" + name].data_ptr(), st["v_" + name].data_ptr(), st["best_" + name].data_ptr(),
                                      None if frozen is None else frozen.data_ptr(), p.numel() // B)
        _lib.check(lib.b200smpl_fit_update(ctypes.cast(groups, ctypes.c_void_p), 3, st["loss"].data_ptr(),
                                           st["best_loss"].data_ptr(), st["best_iter"].data_ptr(), st["first_loss"].data_ptr(),
                                           st["step"].data_ptr(), self._parity, B, self.lr, self.b1, self.b2, self.eps, stream),
                   "fit_update")
        self._parity ^= 1

    # ---- the silhouette term on caller-owned buffers (this fitter's iteration and MultiViewFitter's view steps) -----
    def _silhouette_args(self, verts: torch.Tensor, cam: torch.Tensor, t: torch.Tensor):
        """Writes t = [tx, ty, 2 f / (proj_wh s + 1e-9)] (cam_utils.py:44-52) of the weak-perspective `cam` (B,3) into
        `t` and returns the rasteriser's arguments for `verts` seen through it, with proj_wh s + 1e-9."""
        from .ops import silhouette_args
        f = config.FOCAL_LENGTH
        den = self.proj_wh * cam[:, 0] + 1e-9
        t[:, :2] = cam[:, 1:]
        t[:, 2] = (2 * f) / den
        return silhouette_args(verts, self.faces, t, self.sil_wh, f * self.sil_wh / self.proj_wh, self.sil_sigma), den

    def _silhouette_term(self, verts: torch.Tensor, cam: torch.Tensor, target: torch.Tensor, loss: torch.Tensor,
                         gv: torch.Tensor, t: torch.Tensor, gt: torch.Tensor, gcam: torch.Tensor, stream) -> torch.Tensor:
        """Adds `silhouette_weight * mean((alpha - target)^2)` to `loss` (B,), writes d loss / d vertices to `gv` and
        returns d loss / d cam chained through t (`gcam`, the camera's extra gradient); `t`, `gt` are (B,3) scratch."""
        args, den = self._silhouette_args(verts, cam, t)
        _lib.check(self.lib.b200smpl_silhouette_loss(ctypes.byref(args), target.data_ptr(), self.sil_weight,
                                                     loss.data_ptr(), gv.data_ptr(), gt.data_ptr(), stream),
                   "silhouette_loss")
        gcam[:, 0] = -gt[:, 2] * (2 * config.FOCAL_LENGTH * self.proj_wh) / (den * den)
        gcam[:, 1:] = gt[:, :2]
        return gcam

    def _silhouette_value(self, verts: torch.Tensor, cam: torch.Tensor, target: torch.Tensor, loss: torch.Tensor,
                          t: torch.Tensor, stream) -> None:
        """Adds the same term to `loss` without its gradient (b200smpl_silhouette_loss_value: validation passes)."""
        args, _ = self._silhouette_args(verts, cam, t)
        _lib.check(self.lib.b200smpl_silhouette_loss_value(ctypes.byref(args), target.data_ptr(), self.sil_weight,
                                                           loss.data_ptr(), stream), "silhouette_loss_value")

    def silhouette_iou(self, rotmats: torch.Tensor, betas: torch.Tensor, cam: torch.Tensor,
                       silhouettes: torch.Tensor) -> torch.Tensor:
        """IoU (B,) of the binary silhouettes of the given parameters against `silhouettes` (ops.silhouette_iou)."""
        from .ops import silhouette_iou
        B = rotmats.shape[0]
        verts, _, _ = self.eng.forward(betas.float().contiguous(), rotmats.float().reshape(B, 216).contiguous(), None,
                                       None, axis_angle=False, mode=self.mode)
        alpha = self.smpl.render_silhouettes(verts, cam.float(), img_wh=silhouettes.shape[-1], sigma=0.0,
                                             proj_wh=self.proj_wh)
        return silhouette_iou(alpha, silhouettes.to(alpha.device))

    def fit(self, rotmats: torch.Tensor, betas: torch.Tensor, cam: torch.Tensor, keypoints2d: torch.Tensor,
            vis: Optional[torch.Tensor] = None, iterations: int = 200,
            silhouettes: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """rotmats (B,24,3,3) initial pose, betas (B,10), cam (B,3) weak-perspective [s,tx,ty], keypoints2d
        (B,17,2) target COCO keypoints in pixels of the `proj_wh` image, vis (B,17) bool or None.
        silhouettes (B, silhouette_wh, silhouette_wh) target masks or None: with silhouette_weight > 0 the loss gains
        the silhouette term; either way the result then carries `silhouette_iou` of the best iterate."""
        dev = self.dev
        B = rotmats.shape[0]
        f32 = dict(dtype=torch.float32, device=dev)
        use_sil = silhouettes is not None and self.sil_weight > 0.0
        masks = None if silhouettes is None else _target_masks(silhouettes, (B, self.sil_wh, self.sil_wh), dev)
        # the state buffers (and the graph captured over them) are kept per problem shape and reused by later calls
        key = (B, int(betas.shape[1]), vis is not None) + (("sil",) if use_sil else ())
        cached = self._cache.get(key)
        if cached is None:
            st = {"rot": torch.empty((B, 216), **f32), "betas": torch.empty((B, betas.shape[1]), **f32),
                  "cam": torch.empty((B, 3), **f32), "label": torch.empty((B, self.jmap.numel(), 2), **f32)}
            if vis is not None:
                st["vis"] = torch.empty((B, self.jmap.numel()), dtype=torch.uint8, device=dev)
            for name in ("rot", "betas", "cam"):
                st["m_" + name] = torch.empty_like(st[name])
                st["v_" + name] = torch.empty_like(st[name])
                st["best_" + name] = torch.empty_like(st[name])
            st["loss"] = torch.empty(B, **f32)
            st["first_loss"] = torch.empty(B, **f32)
            st["best_loss"] = torch.empty(B, **f32)
            st["best_iter"] = torch.empty(B, dtype=torch.int32, device=dev)
            st["improved"] = torch.empty(B, dtype=torch.uint8, device=dev)
            st["step"] = torch.empty(2, dtype=torch.int32, device=dev)
            st["gj"] = torch.empty((B, self.eng.num_joints_out, 3), **f32)
            st["gcam"] = torch.empty((B, 3), **f32)
            st["gbetas_prior"] = torch.empty((B, betas.shape[1]), **f32)
            if use_sil:
                st["sil"] = torch.empty((B, self.sil_wh, self.sil_wh), dtype=torch.uint8, device=dev)
                st["gv"] = torch.empty((B, self.eng.num_verts, 3), **f32)
                for name in ("t", "gt", "gcam_sil"):
                    st[name] = torch.empty((B, 3), **f32)
            cached = {"st": st, "graph": None, "per": 0}
            self._cache[key] = cached
        st = cached["st"]
        st["rot"].copy_(rotmats.to(**f32).reshape(B, 216))
        st["betas"].copy_(betas.to(**f32))
        st["cam"].copy_(cam.to(**f32))
        st["label"].copy_(keypoints2d.to(**f32))
        if vis is not None:
            st["vis"].copy_(vis.to(device=dev, dtype=torch.uint8))
        if use_sil:
            st["sil"].copy_(masks)
        for name in ("rot", "betas", "cam"):
            st["m_" + name].zero_()
            st["v_" + name].zero_()
            st["best_" + name].copy_(st[name])
        for name in ("loss", "first_loss", "best_iter", "improved", "step", "gj", "gcam", "gbetas_prior"):
            st[name].zero_()
        st["best_loss"].fill_(float("inf"))
        self._parity = 0                                      # the double-buffered step counter starts at step[0]
        left = iterations
        if self.use_graph and cached["graph"] is not None:
            # later calls of a known shape: replays only (the graph was captured after one eager iteration, i.e. its
            # first iteration reads step[1]; from a zeroed counter either slot is a valid start)
            per = cached["per"]
            for _ in range(left // per):
                cached["graph"].replay()
            if left // per:
                self._parity = 1
            left = left % per
        elif left > 0:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._iteration(st)                           # eager: allocations, attribute set-up
            torch.cuda.current_stream(dev).wait_stream(side)
            left -= 1
            per = self.graph_iterations
            if self.use_graph and left >= per:                # shorter fits stay eager: a capture costs more than it saves
                # one graph = `per` consecutive iterations (consecutive replays of a one-iteration graph leave a
                # launch gap between iterations); the capture itself does not execute
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    for _ in range(per):
                        self._iteration(st)
                cached["graph"], cached["per"] = graph, per
                for _ in range(left // per):
                    graph.replay()
                left = left % per
        for _ in range(left):
            self._iteration(st)
        first_loss = st["first_loss"].clone() if iterations > 0 else None
        best_rot = st["best_rot"].reshape(B, 24, 3, 3)
        out = {"body_pose": best_rot[:, 1:].contiguous(), "global_orient": best_rot[:, :1].contiguous(),
               "betas": st["best_betas"].clone(), "cam": st["best_cam"].clone(),
               "translation": convert_weak_perspective_to_camera_translation_torch(
                   st["best_cam"], config.FOCAL_LENGTH, self.proj_wh),
               "best_loss": st["best_loss"].clone(), "best_iter": st["best_iter"].clone(), "initial_loss": first_loss,
               "final_rotmats": st["rot"].reshape(B, 24, 3, 3).clone(), "final_betas": st["betas"].clone(),
               "final_cam": st["cam"].clone(), "last_loss": st["loss"].clone()}
        if silhouettes is not None:
            out["silhouette_iou"] = self.silhouette_iou(best_rot, st["best_betas"], st["best_cam"], silhouettes)
        self._state = st
        return out


class MultiViewFitter:
    """Batched restatement of the reference's `multi_view_optimization`
    (PlayerReconstruction/player_recon.py:1568-1999) for P independent players seen from V views each.

    Per player, as there: body pose and betas are shared by the views, global orientation and weak-perspective
    camera are per view.  `rounds` (3, player_recon.py:1721) times: phase A optimises the per-view cameras and
    global orientations with a fresh Adam (:1734-1740), phase B the body pose -- hands / feet joints frozen
    (:1706-1708, 1723-1732) -- and the betas with another fresh Adam (:1863-1869).  An epoch walks the views in a
    shuffled order with ONE optimiser step per view (:1746-1749, 1813-1814); because the per-view parameters are
    stacked tensors, a step on view v also moves the other views by their Adam momentum (zero gradient), exactly as
    `optim.Adam([cam_wp_mult, global_orient_mult])` does.  After the training pass every view is evaluated again
    (the `is_train = False` pass) and the parameters of the epoch are kept when the summed validation loss is the
    best the player has seen in any phase so far (:1823-1838, 1938-1954); each phase ends by restoring its
    parameters to their best epoch (:1846-1847, 1961-1962).  The loss of a view is the joints2D term, plus, with
    `fit(..., silhouettes=masks)` and silhouette_weight > 0, the silhouette term of `BatchedFitter` on that view's
    mask, seen through that view's camera.  Differences, stated: model selection uses the summed validation loss
    instead of the metrics tracker's joints2D / silhouette metrics, and the shuffled view order of an epoch is shared
    by all players of the batch (the reference shuffles per player).

    Every step is the C-ABI sequence of `BatchedFitter` (joints-only forward, fused loss, backward, fused Adam; with
    the silhouette term the full-vertex forward, fit_loss, the fused silhouette loss and the backward with vertex
    gradients); the glue between steps (slice copies, the per-epoch comparison) is a handful of tiny elementwise torch
    ops.  The validation pass adds the silhouette term through the gradient-free value kernel.
    """

    def __init__(self, smpl: SMPL, lr: float = 1e-3, rounds: int = 3, shape_weight: float = 0.0,
                 joints2d_log_var: float = 0.0, proj_wh: float = 512.0, norm_wh: float = float(config.REGRESSOR_IMG_WH),
                 betas: tuple = (0.9, 0.999), eps: float = 1e-8, mode: Optional[str] = None,
                 use_cuda_graph: bool = True, silhouette_weight: float = 0.0, silhouette_sigma: float = 1.0,
                 silhouette_wh: int = 256):
        """silhouette_weight, silhouette_sigma and silhouette_wh: as in `BatchedFitter`."""
        self.base = BatchedFitter(smpl, lr=lr, shape_weight=shape_weight, joints2d_log_var=joints2d_log_var,
                                  proj_wh=proj_wh, norm_wh=norm_wh, betas=betas, eps=eps, use_cuda_graph=False, mode=mode,
                                  silhouette_weight=silhouette_weight, silhouette_sigma=silhouette_sigma,
                                  silhouette_wh=silhouette_wh)
        self.rounds = int(rounds)
        self.use_graph = bool(use_cuda_graph)
        dev = self.base.dev
        frozen = torch.zeros(23, 9, dtype=torch.uint8)
        for j in (6, 7, 21, 22):                     # body_pose[:, 6:8] and body_pose[:, 21:]
            frozen[j] = 1
        self.frozen_bp = frozen.reshape(-1).to(dev)
        self._inc = torch.tensor([0, 1], dtype=torch.int32, device=dev)
        self._cache = {}

    # one Adam step of `p` (rows, cols) through the C-ABI; `step` holds [committed, current]
    def _adam(self, p, g, extra, m, v, step, frozen, never):
        b = self.base
        _lib.check(b.lib.b200smpl_fit_adam_step(
            p.data_ptr(), g.data_ptr(), None if extra is None else extra.data_ptr(), m.data_ptr(), v.data_ptr(),
            p.data_ptr(), never.data_ptr(), None if frozen is None else frozen.data_ptr(), step.data_ptr(), 0,
            p.shape[0], p.shape[1], b.lr, b.b1, b.b2, b.eps,
            ctypes.c_void_p(torch.cuda.current_stream(b.dev).cuda_stream)), "fit_adam_step")

    def _loss(self, st, v, need_grad):
        """Forward of view v with the current parameters; fills st['loss'] (and the gradients, with the silhouette
        term's camera gradient or None).  The training pass keeps the forward's transforms and blend rows for its
        backward (no pose stage / blend GEMM recomputation)."""
        b = self.base
        sil = "sil" in st
        st["rot"][:, :9] = st["go"][v]
        if need_grad:
            verts, joints, _, saved = b.eng.forward(st["betas"], st["rot"], None, None, axis_angle=False, mode=b.mode,
                                                    want_vertices=sil, save=True, saved_buffer=st.get("saved"))
            st["saved"] = saved
        else:
            verts, joints, _ = b.eng.forward(st["betas"], st["rot"], None, None, axis_angle=False, mode=b.mode,
                                             want_vertices=sil)
        vis = st.get("vis")
        stream = ctypes.c_void_p(torch.cuda.current_stream(b.dev).cuda_stream)
        P = st["rot"].shape[0]
        _lib.check(b.lib.b200smpl_fit_loss(
            joints.data_ptr(), st["cam"][v].data_ptr(), b.jmap.data_ptr(), st["label"][v].data_ptr(),
            None if vis is None else vis[v].data_ptr(), st["betas"].data_ptr(), P, joints.shape[1], b.jmap.numel(),
            st["betas"].shape[1], b.proj_wh, b.norm_wh, b.log_var, b.shape_weight, st["loss"].data_ptr(),
            st["gj"].data_ptr(), st["gcam"].data_ptr(), st["gbetas_prior"].data_ptr(), stream), "fit_loss")
        if not need_grad:
            if sil:
                b._silhouette_value(verts, st["cam"][v], st["sil"][v], st["loss"], st["t"], stream)
            return None
        cam_extra = b._silhouette_term(verts, st["cam"][v], st["sil"][v], st["loss"], st["gv"], st["t"], st["gt"],
                                       st["gcam_sil"], stream) if sil else None
        gb, gp, _, _ = b.eng.backward(st["betas"], st["rot"], None, None, None, st["gv"] if sil else None, st["gj"],
                                      None, axis_angle=False, mode=b.mode, need_transl=False, need_cam=False,
                                      saved=st["saved"])
        return gb, gp, cam_extra

    # ---- static state + the two kinds of work units (one optimiser step on one view; one validation pass) --------
    def _state(self, P, V, nb, has_vis, use_sil):
        key = (P, V, nb, has_vis) + (("sil",) if use_sil else ())
        c = self._cache.get(key)
        if c is not None:
            return c
        b = self.base
        dev = b.dev
        f32 = dict(dtype=torch.float32, device=dev)
        st = {"go": torch.empty((V, P, 9), **f32), "cam": torch.empty((V, P, 3), **f32),
              "label": torch.empty((V, P, b.jmap.numel(), 2), **f32), "bp": torch.empty((P, 207), **f32),
              "betas": torch.empty((P, nb), **f32), "rot": torch.empty((P, 216), **f32), "loss": torch.zeros(P, **f32),
              "gj": torch.zeros((P, b.eng.num_joints_out, 3), **f32), "gcam": torch.zeros((P, 3), **f32),
              "gbetas_prior": torch.zeros((P, nb), **f32)}
        if has_vis:
            st["vis"] = torch.empty((V, P, b.jmap.numel()), dtype=torch.uint8, device=dev)
        if use_sil:
            st["sil"] = torch.empty((V, P, b.sil_wh, b.sil_wh), dtype=torch.uint8, device=dev)
            st["gv"] = torch.empty((P, b.eng.num_verts, 3), **f32)
            for name in ("t", "gt", "gcam_sil"):
                st[name] = torch.empty((P, 3), **f32)
        c = {"st": st,
             # dense per-view gradients: all zero except the slice of the view being stepped (written before the
             # Adam launch, cleared after it) -- the other views move by their momentum only, as under
             # optim.Adam([cam_wp_mult, global_orient_mult]) in the reference
             "g_go": torch.zeros((V, P, 9), **f32), "g_cam": torch.zeros((V, P, 3), **f32), "g_bp": torch.zeros((P, 207), **f32),
             "mom": {k: (torch.zeros_like(st[k]), torch.zeros_like(st[k])) for k in ("go", "cam", "bp", "betas")},
             "step": torch.zeros(2, dtype=torch.int32, device=dev),
             "never": torch.zeros(V * P, dtype=torch.uint8, device=dev),
             "val": torch.zeros(P, **f32), "best_metric": torch.empty(P, **f32),
             "best": {k: torch.empty_like(st[k]) for k in ("go", "cam", "bp", "betas")},
             "final": {k: torch.empty_like(st[k]) for k in ("go", "cam", "bp", "betas")},
             "graphs": {}, "warm": set()}
        self._cache[key] = c
        return c

    def _view_step(self, c, phase, v):
        st, step, mom, never = c["st"], c["step"], c["mom"], c["never"]
        V, P = st["go"].shape[0], st["go"].shape[1]
        gb, gp, cam_extra = self._loss(st, v, need_grad=True)
        step += self._inc
        if phase == "A":                                        # per-view camera and global orientation
            g_go, g_cam = c["g_go"], c["g_cam"]
            g_go[v] = gp[:, :9]
            g_cam[v] = st["gcam"]
            if cam_extra is not None:                           # the silhouette's pull through t
                g_cam[v].add_(cam_extra)
            self._adam(st["go"].view(V * P, 9), g_go.view(V * P, 9), None, mom["go"][0].view(V * P, 9),
                       mom["go"][1].view(V * P, 9), step, None, never)
            self._adam(st["cam"].view(V * P, 3), g_cam.view(V * P, 3), None, mom["cam"][0].view(V * P, 3),
                       mom["cam"][1].view(V * P, 3), step, None, never)
            g_go[v].zero_()
            g_cam[v].zero_()
        else:                                                   # shared body pose (hands / feet frozen) and betas
            c["g_bp"].copy_(gp[:, 9:])
            self._adam(st["bp"], c["g_bp"], None, mom["bp"][0], mom["bp"][1], step, self.frozen_bp, never)
            self._adam(st["betas"], gb, st["gbetas_prior"], mom["betas"][0], mom["betas"][1], step, None, never)
            st["rot"][:, 9:] = st["bp"]

    def _validate(self, c, phase):
        st, val, best_metric = c["st"], c["val"], c["best_metric"]
        V, P = st["go"].shape[0], st["go"].shape[1]
        val.zero_()
        for v in range(V):
            self._loss(st, v, need_grad=False)
            val += st["loss"]
        improved = val < best_metric
        best_metric.copy_(torch.where(improved, val, best_metric))
        phase_keys = ("go", "cam") if phase == "A" else ("bp", "betas")
        for k in ("go", "cam", "bp", "betas"):
            mask = improved.view(1, P, 1) if k in ("go", "cam") else improved.view(P, 1)
            c["final"][k].copy_(torch.where(mask, st[k], c["final"][k]))
            if k in phase_keys:
                c["best"][k].copy_(torch.where(mask, st[k], c["best"][k]))

    def _run(self, c, name, fn):
        """One work unit: eager the first time (allocations, attribute set-up), then captured once and replayed."""
        if not self.use_graph:
            fn()
            return
        g = c["graphs"].get(name)
        if g is not None:
            g.replay()
            return
        dev = self.base.dev
        if name not in c["warm"]:
            c["warm"].add(name)
            fn()
            return
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(dev)
        with torch.cuda.graph(g):
            fn()
        c["graphs"][name] = g
        g.replay()                                              # the capture itself does not execute

    def fit(self, body_pose: torch.Tensor, betas: torch.Tensor, global_orient: torch.Tensor, cam: torch.Tensor,
            keypoints2d: torch.Tensor, vis: Optional[torch.Tensor] = None, iterations: int = 10,
            view_orders=None, seed: int = 0, silhouettes: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """body_pose (P,23,3,3) and betas (P,10) shared by the views; global_orient (P,V,3,3), cam (P,V,3),
        keypoints2d (P,V,17,2) [, vis (P,V,17)] per view.  `iterations` epochs per phase.  `view_orders`: optional
        list (one per epoch, in execution order: round 0 phase A, round 0 phase B, ...) of view permutations.
        silhouettes (P, V, silhouette_wh, silhouette_wh) target masks or None: with silhouette_weight > 0 every view's
        loss, in the steps and in the validation passes, gains the silhouette term; either way the result then carries
        `silhouette_iou` (P,V) of the returned parameters.

        With `use_cuda_graph` the work units -- (phase, view) optimiser steps and the two validation passes -- are
        captured once per problem shape over static state buffers and replayed: an epoch is V + 1 graph launches
        whatever its view order, instead of ~12 V eager C-ABI / torch calls."""
        b = self.base
        dev = b.dev
        f32 = dict(dtype=torch.float32, device=dev)
        P, V = global_orient.shape[0], global_orient.shape[1]
        use_sil = silhouettes is not None and b.sil_weight > 0.0
        masks = None if silhouettes is None else _target_masks(silhouettes, (P, V, b.sil_wh, b.sil_wh), dev)
        c = self._state(P, V, int(betas.shape[1]), vis is not None, use_sil)
        st = c["st"]
        if use_sil:
            st["sil"].copy_(masks.transpose(0, 1))
        st["go"].copy_(global_orient.to(**f32).reshape(P, V, 9).transpose(0, 1))
        st["cam"].copy_(cam.to(**f32).transpose(0, 1))
        st["label"].copy_(keypoints2d.to(**f32).transpose(0, 1))
        st["bp"].copy_(body_pose.to(**f32).reshape(P, 207))
        st["betas"].copy_(betas.to(**f32))
        if vis is not None:
            st["vis"].copy_(vis.to(device=dev, dtype=torch.uint8).transpose(0, 1))
        st["rot"][:, 9:] = st["bp"]
        for k in ("g_go", "g_cam", "g_bp"):
            c[k].zero_()
        c["best_metric"].fill_(float("inf"))
        for k in ("go", "cam", "bp", "betas"):
            c["best"][k].copy_(st[k])                           # per-phase restore points
            c["final"][k].copy_(st[k])                          # everything at the best epoch
        mom, step, best, final = c["mom"], c["step"], c["best"], c["final"]
        gen = torch.Generator().manual_seed(seed)
        first_val = None
        epoch_no = 0

        def order():
            nonlocal epoch_no
            o = list(view_orders[epoch_no]) if view_orders is not None else torch.randperm(V, generator=gen).tolist()
            epoch_no += 1
            return o

        for _ in range(self.rounds):
            for phase, keys in (("A", ("go", "cam")), ("B", ("bp", "betas"))):
                for k in keys:                                  # a fresh Adam per phase (:1734-1740, :1863-1869)
                    mom[k][0].zero_(); mom[k][1].zero_()
                step.zero_()
                for _e in range(iterations):
                    for v in order():
                        self._run(c, (phase, v), lambda: self._view_step(c, phase, v))
                    self._run(c, ("val", phase), lambda: self._validate(c, phase))
                    if first_val is None:
                        first_val = c["val"].clone()
                for k in keys:                                  # the phase ends at its best epoch (:1846-1847, :1961-1962)
                    st[k].copy_(best[k])
                st["rot"][:, 9:] = st["bp"]

        go = final["go"].transpose(0, 1).reshape(P, V, 3, 3).contiguous()
        cam_out = final["cam"].transpose(0, 1).contiguous()
        out = {"body_pose": final["bp"].reshape(P, 23, 3, 3).clone(), "betas": final["betas"].clone(), "global_orient": go,
               "cam": cam_out,
               "translation": convert_weak_perspective_to_camera_translation_torch(
                   cam_out.reshape(P * V, 3), config.FOCAL_LENGTH, b.proj_wh).reshape(P, V, 3),
               "best_loss": c["best_metric"].clone(), "initial_loss": first_val,
               "last": {"body_pose": st["bp"].reshape(P, 23, 3, 3).clone(), "betas": st["betas"].clone(),
                        "global_orient": st["go"].transpose(0, 1).reshape(P, V, 3, 3).clone(),
                        "cam": st["cam"].transpose(0, 1).clone()}}
        if silhouettes is not None:
            out["silhouette_iou"] = self.silhouette_iou(out["body_pose"], out["betas"], go, cam_out, silhouettes)
        return out

    def silhouette_iou(self, body_pose: torch.Tensor, betas: torch.Tensor, global_orient: torch.Tensor,
                       cam: torch.Tensor, silhouettes: torch.Tensor) -> torch.Tensor:
        """IoU (P,V) of the binary silhouette of every view against `silhouettes` (P,V,S,S), shapes as in `fit`
        (`BatchedFitter.silhouette_iou` per view)."""
        return torch.stack([self.base.silhouette_iou(torch.cat([global_orient[:, v:v + 1], body_pose], 1), betas,
                                                     cam[:, v], silhouettes[:, v])
                            for v in range(global_orient.shape[1])], 1)
