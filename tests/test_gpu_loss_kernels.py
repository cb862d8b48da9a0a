"""GPU tests of the kernels that turn SMPL outputs into losses and parameter updates: the fitters' fit_loss /
fit_mark_best / fit_adam_step (csrc/fit.cu), the regressor's multi-task loss (csrc/loss.cu) and the small helpers of
csrc/aux_ops.cu (joints2D loss, projections, rot6d, Rodrigues).  Every output is compared with an fp64 autograd
reference on the GPU, at the settings where a dropped factor, a loop that loses its stride or a miscounted mask would
show: log-variances away from 0, the shape prior on, proj_wh != 2 norm_wh, random visibility masks, joint maps longer
than a warp with repeated joints, random upstream gradients, and sizes that take every per-thread and grid-stride
loop past its first pass."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, ops, regressor

pytestmark = pytest.mark.gpu

F64 = torch.float64
GUARD = 64                 # floats of guard band on each side of an output buffer
SENTINEL = -12345.5
ADAM = dict(lr=1e-2, beta1=0.9, beta2=0.999, eps=1e-8)
ADAM_ATOL = 2e-6           # as test_fit_update_matches_torch_adam


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _p(t):
    return None if t is None else t.data_ptr()


def _rel(a, b):
    """max |a - b| over max |b| (a: the kernel's fp32 output, b: the fp64 reference)."""
    return (a.double() - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _guarded(shape, dev):
    """(full buffer, view of `shape` inside it) with GUARD elements of SENTINEL on each side."""
    n = int(np.prod(shape))
    full = torch.full((n + 2 * GUARD,), SENTINEL, device=dev)
    return full, full[GUARD:GUARD + n].view(shape)


def _guards_intact(full):
    return bool((full[:GUARD] == SENTINEL).all()) and bool((full[-GUARD:] == SENTINEL).all())


def _joint_map(kind, nj, gen):
    """'coco': the 17-entry COCO map (folded onto nj joints); 'm45' / 'm70': random maps longer than a warp, with
    repeated joints (so the kernels' atomic accumulation into one joint is exercised)."""
    if kind == "coco":
        m = [j % nj for j in config.SMPL_TO_KPRCNN_MAP]
    else:
        n = int(kind[1:])
        m = torch.randint(0, nj, (n,), generator=gen).tolist()
        m[1] = m[0]                                          # at least one repeat
        m[-1] = m[n // 2]
    return torch.tensor(m, dtype=torch.int32)


def _cams(B, gen):
    return torch.stack([torch.rand(B, generator=gen) * 0.6 + 0.6, torch.rand(B, generator=gen) * 0.4 - 0.2,
                        torch.rand(B, generator=gen) * 0.4 - 0.2], 1)


def _vis(kind, B, nmap, gen):
    """None, a random mask, or a random mask with body 0 fully hidden and body 1 seeing a single keypoint."""
    if kind == "none":
        return None
    v = torch.rand(B, nmap, generator=gen) > 0.35
    if kind == "edge":
        v[0] = False
        if B > 1:
            v[1] = False
            v[1, nmap // 3] = True
    return v


def _pixels(joints, cam, jmap, proj_wh):
    return O.undo_keypoint_normalisation(O.orthographic_project(joints, cam)[:, jmap.long()], proj_wh)


# ---------------------------------------------------------------------------------------------------------------------
# b200smpl_fit_loss
# ---------------------------------------------------------------------------------------------------------------------
FIT_CASES = [  # B, nj, map, nb, vis, log_var, shape_weight, grad_betas
    (1, 90, "coco", 10, "none", -0.7, 0.05, True),
    (3, 24, "m45", 1, "random", 0.9, 0.3, True),
    (4, 90, "m70", 16, "random", -0.7, 0.05, False),
    (5, 90, "coco", 10, "edge", 0.9, 0.3, True),
    (5, 24, "m70", 10, "edge", -0.7, 0.3, True),
    (1023, 90, "m45", 10, "random", 0.9, 0.05, True),
    (4099, 24, "m70", 16, "edge", -0.7, 0.3, True),
    (4099, 90, "coco", 1, "random", 0.9, 0.05, False),
]


def _fit_loss_call(lib, dev, t, B, nj, nmap, nb, proj_wh, norm_wh, lv, sw, out):
    rc = lib.b200smpl_fit_loss(t["joints"].data_ptr(), t["cam"].data_ptr(), t["jmap"].data_ptr(), t["label"].data_ptr(),
                               _p(t["vis"]), t["betas"].data_ptr(), B, nj, nmap, nb, proj_wh, norm_wh, lv, sw,
                               out["loss"].data_ptr(), out["gj"].data_ptr(), out["gcam"].data_ptr(), _p(out["gb"]),
                               _stream(dev))
    _lib.check(rc, "fit_loss")


@pytest.mark.parametrize("B,nj,kind,nb,vis_kind,lv,sw,with_gb", FIT_CASES)
def test_fit_loss_matches_fp64_per_player_loss(lib, dev, B, nj, kind, nb, vis_kind, lv, sw, with_gb):
    """loss_per_body, grad_joints, grad_cam and grad_betas against fp64 autograd of the per-player loss: ragged
    four-warp CTAs, maps longer than a warp with repeats, one hidden and one single-keypoint player, guard bands
    around every output, and two calls bit for bit."""
    gen = torch.Generator().manual_seed(B * 131 + nj + nb)
    proj_wh, norm_wh = 480.0, 200.0                          # proj_wh != 2 norm_wh: both scales matter
    jmap = _joint_map(kind, nj, gen)
    nmap = jmap.numel()
    joints = torch.randn(B, nj, 3, generator=gen) * 0.5
    cam = _cams(B, gen)
    label = torch.rand(B, nmap, 2, generator=gen) * proj_wh
    betas = torch.randn(B, nb, generator=gen)
    vis = _vis(vis_kind, B, nmap, gen)
    t = {"joints": joints.to(dev), "cam": cam.to(dev), "jmap": jmap.to(dev), "label": label.to(dev),
         "betas": betas.to(dev), "vis": None if vis is None else vis.to(torch.uint8).to(dev)}
    bufs, out = {}, {}
    for name, shape in (("loss", (B,)), ("gj", (B, nj, 3)), ("gcam", (B, 3)), ("gb", (B, nb))):
        if name == "gb" and not with_gb:
            out[name] = None
            continue
        bufs[name], out[name] = _guarded(shape, dev)
    _fit_loss_call(lib, dev, t, B, nj, nmap, nb, proj_wh, norm_wh, lv, sw, out)
    torch.cuda.synchronize()
    first = {k: v.clone() for k, v in out.items() if v is not None}

    j64 = joints.to(dev, F64).requires_grad_(True)
    c64 = cam.to(dev, F64).requires_grad_(True)
    b64 = betas.to(dev, F64).requires_grad_(True)
    ref = O.fit_loss_per_player(_pixels(j64, c64, jmap.to(dev), proj_wh), label.to(dev, F64), lv, b64, sw, norm_wh,
                                None if vis is None else vis.to(dev))
    ref.sum().backward()
    assert _rel(out["loss"], ref.detach()) < 1e-5
    assert _rel(out["gj"], j64.grad) < 1e-5
    assert _rel(out["gcam"], c64.grad) < 1e-5
    if with_gb:
        assert _rel(out["gb"], b64.grad) < 1e-5
    if vis_kind == "edge":                                   # nothing visible: mean 0, no keypoint gradient
        shape0 = sw * (betas[0].double() ** 2).mean().item()
        assert abs(out["loss"][0].item() - (lv + shape0)) < 1e-6 * max(1.0, abs(lv + shape0))
        assert out["gj"][0].abs().max().item() == 0.0 and out["gcam"][0].abs().max().item() == 0.0
        assert out["gcam"][1].abs().max().item() > 0.0
    for k, full in bufs.items():
        assert _guards_intact(full), k

    _fit_loss_call(lib, dev, t, B, nj, nmap, nb, proj_wh, norm_wh, lv, sw, out)
    torch.cuda.synchronize()
    for k, v in first.items():
        assert torch.equal(out[k], v), k


# ---------------------------------------------------------------------------------------------------------------------
# b200smpl_fit_mark_best
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [5, 300])
def test_fit_mark_best_matches_host_restatement(lib, dev, B):
    """improved = loss < best_loss (strict: a tie does not improve, nor does a NaN loss), best_loss / best_iter
    updated where it does, step[1] = step[0] + 1 with step[0] untouched; bodies past the first 256-thread CTA."""
    gen = torch.Generator().manual_seed(B)
    best_loss = torch.full((B,), float("inf"), device=dev)
    best_iter = torch.full((B,), -1, dtype=torch.int32, device=dev)
    improved = torch.full((B,), 7, dtype=torch.uint8, device=dev)
    step = torch.tensor([4, 0], dtype=torch.int32, device=dev)
    want_best = torch.full((B,), float("inf"), dtype=torch.float32)
    want_iter = torch.full((B,), -1, dtype=torch.int32)
    for it in range(4):
        loss = torch.rand(B, generator=gen) + (0.5 if it == 2 else 0.0)
        if it > 0:
            loss[::3] = want_best[::3]                       # ties
            loss[1::7] = float("nan")
        t = int(step[0].item()) + 1
        _lib.check(lib.b200smpl_fit_mark_best(loss.to(dev).data_ptr(), best_loss.data_ptr(), best_iter.data_ptr(),
                                              improved.data_ptr(), step.data_ptr(), B, _stream(dev)), "fit_mark_best")
        torch.cuda.synchronize()
        imp = loss < want_best
        want_best = torch.where(imp, loss, want_best)
        want_iter = torch.where(imp, torch.full_like(want_iter, t), want_iter)
        assert torch.equal(improved.cpu(), imp.to(torch.uint8)), it
        assert torch.equal(best_loss.cpu(), want_best), it
        assert torch.equal(best_iter.cpu(), want_iter), it
        assert step.tolist() == [t - 1, t], it
        if it > 0:
            assert not imp[::3].any() and not imp[1::7].any()
            if B > 100:
                assert imp.any() and not imp.all()
        step[0] = t                                          # what the committing Adam call of the iteration does


# ---------------------------------------------------------------------------------------------------------------------
# b200smpl_fit_adam_step
# ---------------------------------------------------------------------------------------------------------------------
ADAM_CASES = [  # P, cols, aliased best (MultiViewFitter._adam), commit_step, frozen columns, grad_extra
    (37, 216, False, 1, True, True),
    (4096, 216, False, 1, True, True),        # 884 736 elements: three passes of the capped grid
    (4096, 216, True, 0, True, False),
    (1500, 207, False, 0, False, True),       # 310 500 elements: a short second pass
    (1, 3, True, 1, False, False),
]


@pytest.mark.parametrize("P,cols,aliased,commit,with_frozen,with_extra", ADAM_CASES)
def test_fit_adam_step_matches_torch_adam(lib, dev, P, cols, aliased, commit, with_frozen, with_extra):
    """Three steps against torch.optim.Adam in fp64: frozen columns, grad_extra, improved flags (best-iterate copy
    before the update), best == params aliasing as MultiViewFitter calls it, and the step counter protocol: the
    kernel's bias corrections use step[1]; commit_step = 1 copies it to step[0], commit_step = 0 leaves step[0]."""
    gen = torch.Generator().manual_seed(P + cols)
    p = torch.randn(P, cols, generator=gen).to(dev)
    ref = p.double().clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=ADAM["lr"], betas=(ADAM["beta1"], ADAM["beta2"]), eps=ADAM["eps"])
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    best = p if aliased else torch.full_like(p, SENTINEL)
    want_best = None if aliased else best.clone()
    frozen = (torch.rand(cols, generator=gen) < 0.25).to(torch.uint8).to(dev) if with_frozen else None
    step = torch.zeros(2, dtype=torch.int32, device=dev)
    for it in range(1, 4):
        g = torch.randn(P, cols, generator=gen).to(dev)
        extra = torch.randn(P, cols, generator=gen).to(dev) if with_extra else None
        imp = (torch.rand(P, generator=gen) < 0.5).to(torch.uint8).to(dev)
        if aliased:
            imp.zero_()                                      # MultiViewFitter passes its all-zero `never` flags
        step[1] = it if commit else step[1] + 1              # fit_mark_best / MultiViewFitter's `step += [0, 1]`
        before = step[0].item()
        x = p.clone()                                        # the parameters that produced this iteration's loss
        _lib.check(lib.b200smpl_fit_adam_step(p.data_ptr(), g.data_ptr(), _p(extra), m.data_ptr(), v.data_ptr(),
                                              best.data_ptr(), imp.data_ptr(), _p(frozen), step.data_ptr(), commit, P,
                                              cols, ADAM["lr"], ADAM["beta1"], ADAM["beta2"], ADAM["eps"],
                                              _stream(dev)), "fit_adam_step")
        torch.cuda.synchronize()
        assert step.tolist() == ([it, it] if commit else [before, it]), it
        if not aliased:
            sel = imp.bool()
            want_best[sel] = x[sel]                          # copied bit for bit before the update
        gr = g.double() + (0.0 if extra is None else extra.double())
        if frozen is not None:
            gr[:, frozen.bool()] = 0.0
        ref.grad = gr
        opt.step()
        st = opt.state[ref]
        assert torch.allclose(p.double(), ref.detach(), atol=ADAM_ATOL), (it, (p.double() - ref.detach()).abs().max())
        assert torch.allclose(m.double(), st["exp_avg"], atol=ADAM_ATOL), it
        assert torch.allclose(v.double(), st["exp_avg_sq"], atol=ADAM_ATOL, rtol=1e-5), it
        if not aliased:
            assert torch.equal(best, want_best), it
    if frozen is not None:
        fz = frozen.bool()
        assert fz.any() and (m[:, fz] == 0).all() and (v[:, fz] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# joints2d_loss
# ---------------------------------------------------------------------------------------------------------------------
J2D_CASES = [  # B, map, vis, log_var
    (1, "m45", "random", -0.7),
    (37, "m70", "random", 0.9),
    (37, "coco", "none", -0.7),
    (16000, "coco", "random", 0.9),           # 272 000 (body, keypoint) pairs: count_vis past its 1024-CTA grid
    (16000, "m45", "random", -0.7),
]


@pytest.mark.parametrize("B,kind,vis_kind,lv", J2D_CASES)
def test_joints2d_loss_matches_fp64(dev, B, kind, vis_kind, lv):
    """ops.joints2d_loss value and both gradients (random upstream gradient) against fp64 autograd of
    O.joints2d_loss: exp(-log_var) weighting, log_var added once per batch, maps longer than a warp with repeats."""
    gen = torch.Generator().manual_seed(B + len(kind))
    proj_wh, norm_wh, nj = 480.0, 200.0, 90
    jmap = _joint_map(kind, nj, gen)
    nmap = jmap.numel()
    joints = torch.randn(B, nj, 3, generator=gen) * 0.5
    cam = _cams(B, gen)
    label = torch.rand(B, nmap, 2, generator=gen) * proj_wh
    vis = _vis(vis_kind, B, nmap, gen)
    up = 0.5 + torch.rand((), generator=gen).item()
    j = joints.to(dev).requires_grad_(True)
    c = cam.to(dev).requires_grad_(True)
    loss = ops.joints2d_loss(j, c, jmap.to(dev), label.to(dev), None if vis is None else vis.to(dev),
                             proj_wh=proj_wh, norm_wh=norm_wh, log_var=lv)
    (up * loss).backward()
    j64 = joints.to(dev, F64).requires_grad_(True)
    c64 = cam.to(dev, F64).requires_grad_(True)
    ref = O.joints2d_loss(_pixels(j64, c64, jmap.to(dev), proj_wh), label.to(dev, F64),
                          torch.tensor(lv, dtype=F64, device=dev), norm_wh, None if vis is None else vis.to(dev))
    (up * ref).backward()
    # the loss is one fp32 atomicAdd per body: at 16 000 bodies the rounding of the running sum alone nears 1e-5
    rtol = 1e-5 if B < 1000 else 4e-5
    assert abs(loss.item() - ref.item()) < rtol * max(1.0, abs(ref.item()))
    assert _rel(j.grad, j64.grad) < 1e-5
    assert _rel(c.grad, c64.grad) < 1e-5


def test_joints2d_loss_with_nothing_visible(dev):
    """An all-hidden batch: the kernel's mean counts as 0, so the loss is log_var and the gradients are zero (the
    reference's mean over an empty selection is NaN)."""
    B, nj, lv = 37, 90, 0.9
    gen = torch.Generator().manual_seed(2)
    jmap = _joint_map("m45", nj, gen)
    joints = (torch.randn(B, nj, 3, generator=gen) * 0.5).to(dev).requires_grad_(True)
    cam = _cams(B, gen).to(dev).requires_grad_(True)
    label = (torch.rand(B, jmap.numel(), 2, generator=gen) * 512).to(dev)
    vis = torch.zeros(B, jmap.numel(), dtype=torch.bool, device=dev)
    loss = ops.joints2d_loss(joints, cam, jmap.to(dev), label, vis, proj_wh=512.0, norm_wh=256.0, log_var=lv)
    loss.backward()
    assert loss.item() == np.float32(lv)
    assert joints.grad.abs().max().item() == 0.0 and cam.grad.abs().max().item() == 0.0
    ref = O.joints2d_loss(_pixels(joints.detach().double(), cam.detach().double(), jmap.to(dev), 512.0),
                          label.double(), torch.tensor(lv, dtype=F64), 256.0, vis)
    assert torch.isnan(ref)


# ---------------------------------------------------------------------------------------------------------------------
# multi-task loss
# ---------------------------------------------------------------------------------------------------------------------
TERMS = ("verts", "joints2D", "joints3D", "shape_params", "pose_params")
MTL_LOG_VARS = {"verts": -0.7, "joints2D": 0.9, "joints3D": 0.4, "shape_params": -0.3, "pose_params": 0.6}


@pytest.mark.parametrize("B,V", [(64, 6890), (256, 6890), (255, 6889)])
def test_multitask_loss_matches_fp64(dev, B, V):
    """ops.multitask_loss: the loss, the five parts, d/d log_var and every gradient against regressor.MultiTaskLoss
    in fp64, each term alone and all five together; vertex counts that take mtl_reduce / mtl_grad through several
    grid-stride passes, with an even (B V 3) and an odd one; a 2D map longer than a warp with repeats that shares
    joints with the 3D map; an upstream gradient != 1 read from the device."""
    proj_wh, norm_wh = 480.0, float(config.REGRESSOR_IMG_WH)
    nj = 90
    for k, terms in enumerate([(t,) for t in TERMS] + [TERMS]):
        gen = torch.Generator().manual_seed(B * 10 + V + k)    # fresh data per run: no stale buffer can pass
        map2d = _joint_map("m45", nj, gen)
        map3d = torch.tensor(config.ALL_JOINTS_TO_COCO_MAP, dtype=torch.int32)
        x = {"verts": torch.randn(B, V, 3, generator=gen) * 0.3, "joints": torch.randn(B, nj, 3, generator=gen) * 0.5,
             "cam": _cams(B, gen), "shape_params": torch.randn(B, 10, generator=gen),
             "pose_params_rot_matrices": torch.randn(B, 24, 3, 3, generator=gen) * 0.5}
        lab = {"verts": x["verts"] + 0.05 * torch.randn(B, V, 3, generator=gen),
               "joints2D": torch.rand(B, map2d.numel(), 2, generator=gen) * proj_wh,
               "joints3D": torch.randn(B, map3d.numel(), 3, generator=gen) * 0.5,
               "shape_params": torch.randn(B, 10, generator=gen),
               "pose_params_rot_matrices": torch.randn(B, 24, 3, 3, generator=gen) * 0.5,
               "vis": torch.rand(B, map2d.numel(), generator=gen) > 0.3}
        up = 0.5 + torch.rand((), generator=gen).item()
        lv = torch.tensor([MTL_LOG_VARS[t] if t in terms else 0.0 for t in TERMS], device=dev).requires_grad_(True)
        leaves = {n: x[n].to(dev).requires_grad_(True) for n in x}
        d = {n: t.to(dev) for n, t in lab.items()}
        kw = {}
        if "verts" in terms:
            kw.update(verts=leaves["verts"], verts_label=d["verts"])
        if "joints2D" in terms:
            kw.update(joints=leaves["joints"], cam=leaves["cam"], map2d=map2d.to(dev), label2d=d["joints2D"], vis=d["vis"])
        if "joints3D" in terms:
            kw.update(joints=leaves["joints"], map3d=map3d.to(dev), label3d=d["joints3D"])
        if "shape_params" in terms:
            kw.update(shape=leaves["shape_params"], shape_label=d["shape_params"])
        if "pose_params" in terms:
            kw.update(pose=leaves["pose_params_rot_matrices"], pose_label=d["pose_params_rot_matrices"])
        loss, parts = ops.multitask_loss(lv, proj_wh=proj_wh, norm_wh=norm_wh, **kw)
        (up * loss).backward()

        crit = regressor.MultiTaskLoss(terms).double().to(dev)
        with torch.no_grad():
            for t in terms:
                getattr(crit, t + "_log_var").fill_(MTL_LOG_VARS[t])
        l64 = {n: x[n].to(dev, F64).requires_grad_(True) for n in x}
        o64 = dict(l64)
        o64["joints2D"] = _pixels(l64["joints"], l64["cam"], map2d.to(dev), proj_wh)
        o64["joints3D"] = l64["joints"][:, map3d.long().to(dev)]
        lab64 = {n: (t.to(dev, F64) if t.dtype.is_floating_point else t.to(dev)) for n, t in lab.items()}
        ref, parts64 = crit(lab64, o64)
        (up * ref).backward()
        assert abs(loss.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item())), terms
        for i, t in enumerate(TERMS):
            if t not in terms:
                assert parts[i].item() == 0.0 and lv.grad[i].item() == 0.0, (terms, t)
                continue
            assert abs(parts[i].item() - parts64[t].item()) < 1e-5 * max(1e-3, abs(parts64[t].item())), (terms, t)
            g64 = getattr(crit, t + "_log_var").grad
            assert abs(lv.grad[i].item() - g64.item()) < 1e-5 * max(1.0, abs(g64.item())), (terms, t)
        for n in x:
            g64 = l64[n].grad
            if g64 is None:
                assert leaves[n].grad is None, (terms, n)
                continue
            assert _rel(leaves[n].grad, g64) < 1e-5, (terms, n, _rel(leaves[n].grad, g64))


def test_multitask_loss_with_nothing_visible_is_nan(dev):
    """The multi-task loss keeps the reference's rule: a 2D term with no visible keypoint is the mean of an empty
    selection, NaN (unlike fit_loss / joints2d_loss, which count that mean as 0)."""
    B, nj = 8, 90
    gen = torch.Generator().manual_seed(4)
    map2d = torch.tensor(config.SMPL_TO_KPRCNN_MAP, dtype=torch.int32, device=dev)
    lv = torch.tensor([0.0, 0.9, 0.0, 0.0, 0.0], device=dev)
    loss, parts = ops.multitask_loss(lv, joints=(torch.randn(B, nj, 3, generator=gen) * 0.5).to(dev),
                                     cam=_cams(B, gen).to(dev), map2d=map2d,
                                     label2d=(torch.rand(B, 17, 2, generator=gen) * 512).to(dev),
                                     vis=torch.zeros(B, 17, dtype=torch.bool, device=dev))
    assert torch.isnan(loss) and torch.isnan(parts[1])


# ---------------------------------------------------------------------------------------------------------------------
# projections
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [(1, 1), (1, 127), (300, 129), (300, 6890), (1, 6890), (300, 1)]


def _rotations(B, gen):
    return O.batch_rodrigues((torch.randn(B, 3, generator=gen, dtype=F64) * 0.6)).float()


@pytest.mark.parametrize("B,N", SIZES)
def test_orthographic_project_matches_fp64(lib, dev, B, N):
    """Forward and backward (random upstream gradient) at pixel_wh 0 and 512, point counts below, at and above the
    128 threads of a body's CTA; the C-ABI backward with each gradient output NULL in turn writes the other one bit
    for bit as the full call does."""
    gen = torch.Generator().manual_seed(B * 7 + N)
    pts = torch.randn(B, N, 3, generator=gen) * 0.5
    cam = _cams(B, gen)
    w = torch.randn(B, N, 2, generator=gen)
    for pixel_wh in (0.0, 512.0):
        p = pts.to(dev).requires_grad_(True)
        c = cam.to(dev).requires_grad_(True)
        out = ops.orthographic_project(p, c, pixel_wh)
        (out * w.to(dev)).sum().backward()
        p64 = pts.to(dev, F64).requires_grad_(True)
        c64 = cam.to(dev, F64).requires_grad_(True)
        ref = O.orthographic_project(p64, c64)
        if pixel_wh > 0:
            ref = O.undo_keypoint_normalisation(ref, pixel_wh)
        (ref * w.to(dev, F64)).sum().backward()
        assert _rel(out.detach(), ref.detach()) < 1e-5
        assert _rel(p.grad, p64.grad) < 1e-5
        assert _rel(c.grad, c64.grad) < 1e-5
        # NULL outputs through the C-ABI
        wd = w.to(dev)
        full = [torch.full((B, N, 3), SENTINEL, device=dev), torch.full((B, 3), SENTINEL, device=dev)]
        _lib.check(lib.b200smpl_orthographic_project_backward(p.data_ptr(), c.data_ptr(), wd.data_ptr(),
                                                              full[0].data_ptr(), full[1].data_ptr(), B, N, pixel_wh,
                                                              _stream(dev)), "ortho_bwd")
        for drop in range(2):
            part = [torch.full_like(t, SENTINEL) for t in full]
            ptrs = [None if k == drop else part[k].data_ptr() for k in range(2)]
            _lib.check(lib.b200smpl_orthographic_project_backward(p.data_ptr(), c.data_ptr(), wd.data_ptr(), *ptrs,
                                                                  B, N, pixel_wh, _stream(dev)), "ortho_bwd")
            torch.cuda.synchronize()
            for k in range(2):
                assert torch.equal(part[k], full[k]) if k != drop else (part[k] == SENTINEL).all(), (drop, k)


def _persp_call(lib, dev, form, pts, rot, tr, K, f, wh, gout, outs):
    B, N = pts.shape[0], pts.shape[1]
    if form == "focal":
        return lib.b200smpl_perspective_project_backward(pts.data_ptr(), rot.data_ptr(), tr.data_ptr(), gout.data_ptr(),
                                                         *[_p(o) for o in outs], B, N, f, wh, _stream(dev))
    return lib.b200smpl_perspective_project_camk_backward(pts.data_ptr(), rot.data_ptr(), tr.data_ptr(), K.data_ptr(),
                                                          int(form == "batched"), gout.data_ptr(),
                                                          *[_p(o) for o in outs], B, N, _stream(dev))


@pytest.mark.parametrize("B,N", SIZES)
def test_perspective_project_matches_fp64(lib, dev, B, N):
    """Both perspective forms -- (focal_length, img_wh), one shared cam_K, a per-body cam_K -- forward and backward
    (random upstream gradient) against fp64 autograd; the C-ABI backward with each of its three outputs NULL in turn
    writes the others bit for bit as the full call does."""
    gen = torch.Generator().manual_seed(B * 11 + N)
    f, wh = 5000.0, 512.0
    pts = torch.randn(B, N, 3, generator=gen) * 0.5
    rot = _rotations(B, gen)
    tr = torch.cat([torch.randn(B, 2, generator=gen) * 0.2, 8.0 + 4.0 * torch.rand(B, 1, generator=gen)], 1)
    Kb = torch.zeros(B, 3, 3)
    Kb[:, 0, 0] = 4000.0 + 2000.0 * torch.rand(B, generator=gen)
    Kb[:, 1, 1] = 4000.0 + 2000.0 * torch.rand(B, generator=gen)
    Kb[:, 0, 1] = 10.0 * torch.randn(B, generator=gen)        # a skew term: K[0][1] reaches the v gradient
    Kb[:, 0, 2] = 200.0 + 100.0 * torch.rand(B, generator=gen)
    Kb[:, 1, 2] = 200.0 + 100.0 * torch.rand(B, generator=gen)
    Kb[:, 2, 2] = 1.0
    w = torch.randn(B, N, 2, generator=gen)
    for form in ("focal", "shared", "batched"):
        K = None if form == "focal" else (Kb[0] if form == "shared" else Kb)
        p, r, t = (a.to(dev).requires_grad_(True) for a in (pts, rot, tr))
        if form == "focal":
            out = ops.perspective_project(p, r, t, f, wh)
        else:
            out = ops.perspective_project_camk(p, r, t, K.to(dev))
        (out * w.to(dev)).sum().backward()
        p64, r64, t64 = (a.to(dev, F64).requires_grad_(True) for a in (pts, rot, tr))
        if form == "focal":
            ref = O.perspective_project(p64, r64, t64, focal_length=f, img_wh=wh)
        else:
            ref = O.perspective_project(p64, r64, t64, cam_K=K.expand(B, 3, 3).to(dev, F64))
        (ref * w.to(dev, F64)).sum().backward()
        assert _rel(out.detach(), ref.detach()) < 1e-5, form
        assert _rel(p.grad, p64.grad) < 1e-5, form
        assert _rel(r.grad, r64.grad) < 1e-5, form
        assert _rel(t.grad, t64.grad) < 1e-5, form
        Kd = None if K is None else K.to(dev).contiguous()
        wd = w.to(dev)
        shapes = [(B, N, 3), (B, 3, 3), (B, 3)]
        full = [torch.full(s, SENTINEL, device=dev) for s in shapes]
        _lib.check(_persp_call(lib, dev, form, p, r, t, Kd, f, wh, wd, full), "persp_bwd")
        for drop in range(3):
            part = [None if k == drop else torch.full(s, SENTINEL, device=dev) for k, s in enumerate(shapes)]
            _lib.check(_persp_call(lib, dev, form, p, r, t, Kd, f, wh, wd, part), "persp_bwd")
            torch.cuda.synchronize()
            for k in range(3):
                if k != drop:
                    assert torch.equal(part[k], full[k]), (form, drop, k)


# ---------------------------------------------------------------------------------------------------------------------
# rot6d and Rodrigues
# ---------------------------------------------------------------------------------------------------------------------
def test_rot6d_at_a_million_rotations(dev):
    """n = 10^6: forward and backward (random upstream gradient) against fp64 where the Gram-Schmidt is well
    conditioned; zero and parallel columns give finite output and gradients."""
    n = 1_000_000
    gen = torch.Generator().manual_seed(6)
    x = torch.randn(n, 6, generator=gen)
    deg = torch.tensor([[0, 0, 0, 0, 0, 0],                   # both columns zero
                        [0, 1, 0, 2, 0, 3],                   # first column zero
                        [1, 0, 2, 0, 3, 0],                   # second column zero
                        [1, 2, 2, 4, 3, 6],                   # parallel
                        [1, -3, -2, 6, 0.5, -1.5]], dtype=torch.float32)   # antiparallel
    x[:deg.shape[0]] = deg
    w = torch.randn(n, 3, 3, generator=gen)
    xd = x.to(dev).requires_grad_(True)
    R = ops.rot6d_to_rotmat(xd)
    (R * w.to(dev)).sum().backward()
    assert torch.isfinite(R).all() and torch.isfinite(xd.grad).all()
    a = x.view(n, 3, 2).double()
    n1, n2 = a[:, :, 0].norm(dim=1), a[:, :, 1].norm(dim=1)
    sin = torch.cross(a[:, :, 0], a[:, :, 1], dim=1).norm(dim=1) / (n1 * n2).clamp(min=1e-30)
    ok = ((n1 > 0.2) & (n2 > 0.2) & (sin > 0.2)).to(dev)
    assert ok.sum().item() > 0.9 * n
    x64 = x.to(dev, F64).requires_grad_(True)
    R64 = O.rot6d_to_rotmat(x64)
    (R64 * w.to(dev, F64)).sum().backward()
    assert _rel(R.detach()[ok], R64.detach()[ok]) < 1e-5
    assert _rel(xd.grad[ok], x64.grad[ok]) < 1e-5


def test_batch_rodrigues_at_a_million_rotations(dev):
    """n = 10^6: forward and backward (random upstream gradient) against fp64 away from the zero vector, where
    smplx's 1e-8 angle offset makes fp32 and fp64 legitimately differ; the zero vector gives finite output."""
    n = 1_000_000
    gen = torch.Generator().manual_seed(8)
    r = torch.randn(n, 3, generator=gen) * 0.8
    r[0] = 0.0
    w = torch.randn(n, 3, 3, generator=gen)
    rd = r.to(dev).requires_grad_(True)
    R = ops.batch_rodrigues(rd)
    (R * w.to(dev)).sum().backward()
    assert torch.isfinite(R).all() and torch.isfinite(rd.grad).all()
    ok = (r.norm(dim=1) > 0.05).to(dev)
    r64 = r.to(dev, F64).requires_grad_(True)
    R64 = O.batch_rodrigues(r64)
    (R64 * w.to(dev, F64)).sum().backward()
    assert _rel(R.detach()[ok], R64.detach()[ok]) < 1e-5
    assert _rel(rd.grad[ok], r64.grad[ok]) < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# argument checks: refused with B200SMPL_ERR_INVALID, before any launch or write
# ---------------------------------------------------------------------------------------------------------------------
def _refused(lib, dev, call, outs, argsets):
    """call(*args) for every argument set must return ERR_INVALID, launch nothing and leave `outs` unchanged."""
    torch.cuda.synchronize()
    before = [o.clone() for o in outs]
    n0 = lib.b200smpl_launch_count()
    for args in argsets:
        assert call(*args) == _lib.ERR_INVALID, args
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0
    for o, b in zip(outs, before):
        assert torch.equal(o, b)


def _sweep(base, nulls, bad):
    """Argument sets: each pointer of `nulls` (indices into base) replaced by None, then each (index, value) of bad."""
    out = []
    for i in nulls:
        a = list(base)
        a[i] = None
        out.append(a)
    for i, v in bad:
        a = list(base)
        a[i] = v
        out.append(a)
    return out


def test_argument_checks_refuse_without_launch_or_write(lib, dev):
    B, nj, nmap, nb = 4, 24, 17, 10
    f32 = dict(device=dev)
    joints, cam = torch.zeros(B, nj, 3, **f32), torch.zeros(B, 3, **f32)
    jmap = torch.zeros(nmap, dtype=torch.int32, device=dev)
    label, betas = torch.zeros(B, nmap, 2, **f32), torch.zeros(B, nb, **f32)
    vis = torch.ones(B, nmap, dtype=torch.uint8, device=dev)
    loss = torch.full((B,), SENTINEL, **f32)
    gj, gcam, gb = (torch.full(s, SENTINEL, **f32) for s in ((B, nj, 3), (B, 3), (B, nb)))
    st = _stream(dev)
    P = lambda t: t.data_ptr()   # noqa: E731

    # fit_loss: joints cam map label vis betas B nj nmap nb proj norm lv sw loss gj gcam gb stream
    base = [P(joints), P(cam), P(jmap), P(label), P(vis), P(betas), B, nj, nmap, nb, 512.0, 256.0, 0.0, 0.0,
            P(loss), P(gj), P(gcam), P(gb), st]
    _refused(lib, dev, lib.b200smpl_fit_loss, [loss, gj, gcam, gb],
             _sweep(base, [0, 1, 2, 3, 5, 14, 15, 16], [(6, 0), (7, 0), (8, 0), (9, 0), (6, -1), (9, -3)]))

    # joints2d_loss: joints cam map label vis B nj nmap proj norm lv loss gj gcam stream
    loss2 = torch.full((2,), SENTINEL, **f32)
    base = [P(joints), P(cam), P(jmap), P(label), P(vis), B, nj, nmap, 512.0, 256.0, 0.0, P(loss2), P(gj), P(gcam), st]
    _refused(lib, dev, lib.b200smpl_joints2d_loss, [loss2, gj, gcam],
             _sweep(base, [0, 1, 2, 3, 11], [(5, 0), (6, 0), (7, 0), (6, -2)]))

    # fit_mark_best: loss best_loss best_iter improved step B stream
    best_loss, best_iter = torch.full((B,), SENTINEL, **f32), torch.full((B,), 5, dtype=torch.int32, device=dev)
    improved, step = torch.full((B,), 9, dtype=torch.uint8, device=dev), torch.tensor([3, 3], dtype=torch.int32, device=dev)
    base = [P(loss), P(best_loss), P(best_iter), P(improved), P(step), B, st]
    _refused(lib, dev, lib.b200smpl_fit_mark_best, [best_loss, best_iter, improved, step],
             _sweep(base, [0, 1, 2, 3, 4], [(5, 0), (5, -1)]))

    # fit_adam_step: params grad extra m v best improved frozen step commit B cols lr b1 b2 eps stream
    prm, m, v, best = (torch.full((B, 9), SENTINEL, **f32) for _ in range(4))
    base = [P(prm), P(gj), None, P(m), P(v), P(best), P(improved), None, P(step), 1, B, 9, 1e-3, 0.9, 0.999, 1e-8, st]
    _refused(lib, dev, lib.b200smpl_fit_adam_step, [prm, m, v, best, step],
             _sweep(base, [0, 1, 3, 4, 5, 6, 8], [(10, 0), (11, 0), (10, -1)]))

    # projections: points cam out B n pixel_wh stream / the backward with both gradient outputs
    pts, out2 = torch.zeros(B, 5, 3, **f32), torch.full((B, 5, 2), SENTINEL, **f32)
    gpts = torch.full((B, 5, 3), SENTINEL, **f32)
    _refused(lib, dev, lib.b200smpl_orthographic_project, [out2],
             _sweep([P(pts), P(cam), P(out2), B, 5, 0.0, st], [0, 1, 2], [(3, 0), (4, 0)]))
    _refused(lib, dev, lib.b200smpl_orthographic_project_backward, [gpts, gcam],
             _sweep([P(pts), P(cam), P(out2), P(gpts), P(gcam), B, 5, 0.0, st], [0, 1, 2], [(5, 0), (6, 0)]))
    rot, K = torch.zeros(B, 3, 3, **f32), torch.zeros(3, 3, **f32)
    grot = torch.full((B, 3, 3), SENTINEL, **f32)
    _refused(lib, dev, lib.b200smpl_perspective_project, [out2],
             _sweep([P(pts), P(rot), P(cam), P(out2), B, 5, 5000.0, 512.0, st], [0, 1, 2, 3], [(4, 0), (5, 0)]))
    _refused(lib, dev, lib.b200smpl_perspective_project_camk, [out2],
             _sweep([P(pts), P(rot), P(cam), P(K), 0, P(out2), B, 5, st], [0, 1, 2, 3, 5], [(6, 0), (7, 0)]))
    _refused(lib, dev, lib.b200smpl_perspective_project_backward, [gpts, grot, gcam],
             _sweep([P(pts), P(rot), P(cam), P(out2), P(gpts), P(grot), P(gcam), B, 5, 5000.0, 512.0, st],
                    [0, 1, 2, 3], [(7, 0), (8, 0)]))
    _refused(lib, dev, lib.b200smpl_perspective_project_camk_backward, [gpts, grot, gcam],
             _sweep([P(pts), P(rot), P(cam), P(K), 0, P(out2), P(gpts), P(grot), P(gcam), B, 5, st],
                    [0, 1, 2, 3, 5], [(9, 0), (10, 0)]))

    # rot6d / Rodrigues: x out n stream, x grad_out grad_x n stream
    x6, R9 = torch.zeros(B, 6, **f32), torch.full((B, 3, 3), SENTINEL, **f32)
    g6 = torch.full((B, 6), SENTINEL, **f32)
    for fwd, bwd in ((lib.b200smpl_rot6d_to_rotmat, lib.b200smpl_rot6d_to_rotmat_backward),
                     (lib.b200smpl_batch_rodrigues, lib.b200smpl_batch_rodrigues_backward)):
        _refused(lib, dev, fwd, [R9], _sweep([P(x6), P(R9), B, st], [0, 1], [(2, -1)]))
        _refused(lib, dev, bwd, [g6], _sweep([P(x6), P(R9), P(g6), B, st], [0, 1, 2], [(3, -1)]))

    # multi-task loss: the argument struct and out / the backward's 8-byte aligned grad_verts
    V = 6
    verts, vlab = torch.zeros(B, V, 3, **f32), torch.zeros(B, V, 3, **f32)
    lv, scratch = torch.zeros(5, **f32), torch.full((16,), SENTINEL, **f32)
    out11 = torch.full((11,), SENTINEL, **f32)
    gverts = torch.full((B * V * 3 + 1,), SENTINEL, **f32)
    good = dict(batch=B, num_verts=V, num_joints=nj, nmap2d=nmap, nmap3d=nmap, num_betas=nb, pose_cols=0, reserved0=0,
                proj_wh=512.0, norm_wh=256.0, verts=P(verts), verts_label=P(vlab), joints=P(joints), cam=P(cam),
                map2d=P(jmap), label2d=P(label), vis=P(vis), map3d=P(jmap), label3d=P(joints), shape=P(betas),
                shape_label=P(betas), pose=None, pose_label=None, log_var=P(lv), scratch=P(scratch))
    bad_args = [dict(batch=0), dict(log_var=None), dict(scratch=None), dict(verts_label=None), dict(shape=None),
                dict(pose=P(betas)), dict(joints=None), dict(cam=None), dict(label2d=None), dict(label3d=None),
                dict(verts=P(verts) + 4)]
    structs = [_lib.MultiTaskLossArgs(**dict(good, **b)) for b in bad_args]
    _refused(lib, dev, lambda a, o: lib.b200smpl_multitask_loss(ctypes.byref(a) if a is not None else None, o, st),
             [scratch, out11], [(a, P(out11)) for a in structs] + [(_lib.MultiTaskLossArgs(**good), None), (None, P(out11))])
    bwd_outs = [gverts, gj, gcam, gb]
    _refused(lib, dev, lambda a, gv: lib.b200smpl_multitask_loss_backward(
        ctypes.byref(a) if a is not None else None, P(lv), gv, P(gj), P(gcam), P(gb), None, st), bwd_outs,
        [(a, P(gverts)) for a in structs] + [(_lib.MultiTaskLossArgs(**good), P(gverts) + 4), (None, P(gverts))])
