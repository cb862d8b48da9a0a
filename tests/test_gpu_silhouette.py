"""GPU tests of the silhouette rasteriser (csrc/silhouette.cu) against the fp64 oracle (oracle/silhouette_oracle.py),
through ops / SMPL into the SMPL backward, and of the silhouette term of BatchedFitter."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import silhouette_oracle as SO
from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, ops
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch
from soccerplayershapepose_b200.fitting import FROZEN_FULL_JOINTS, BatchedFitter
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


def _bodies(B, seed):
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    cam = torch.stack([torch.rand(B, generator=g) * 0.6 + 0.6, torch.rand(B, generator=g) * 0.4 - 0.2,
                       torch.rand(B, generator=g) * 0.4 - 0.2], 1)
    return betas, pose, cam


def _posed(smpl, B, seed):
    """Posed vertices (B,6890,3) on the device, camera translation (B,3) and the render focal length per size."""
    betas, pose, cam = _bodies(B, seed)
    out = smpl(betas=betas.to(DEV), body_pose=pose[:, 3:].to(DEV), global_orient=pose[:, :3].to(DEV))
    t = convert_weak_perspective_to_camera_translation_torch(cam.to(DEV), config.FOCAL_LENGTH, 512)
    return out.vertices.detach().contiguous(), t.contiguous(), cam


def _focal(S):
    return config.FOCAL_LENGTH * S / 512


def _ambiguous(v, t, faces, S, sigma):
    """Pixels near a face whose kept / dropped status fp32 may decide differently from fp64 (|area| < 1e-4 px^2):
    excluded from the soft comparisons.  They must be rare (at S = 64, 1.7 % of the pixels lie near one)."""
    tri, kept, area = SO.face_table(v.double().cpu(), t.double().cpu(), faces.cpu(), _focal(S), S)
    mask = torch.zeros(v.shape[0], S, S, dtype=torch.bool)
    rad = np.sqrt(SO.cutoff_d2(sigma)) + 1.0
    for b, f in zip(*torch.nonzero(area.abs() < 1e-4, as_tuple=True)):
        lo, hi = tri[b, f].min(0).values.tolist(), tri[b, f].max(0).values.tolist()
        c0, c1 = int(max(0, np.floor(lo[0] - rad))), int(min(S, np.ceil(hi[0] + rad)))
        r0, r1 = int(max(0, np.floor(lo[1] - rad))), int(min(S, np.ceil(hi[1] + rad)))
        mask[b, r0:r1, c0:c1] = True
    assert mask.float().mean() < 0.05
    return mask


@pytest.mark.parametrize("S", [64, 256])
def test_hard_mask_matches_oracle(smpl, S):
    v, t, _ = _posed(smpl, 5, 10 + S)
    faces = smpl.faces_int32(DEV)
    a = ops.render_silhouettes(v, faces, t, S, _focal(S), 0.0)
    ref = SO.render(v.double().cpu(), faces.cpu(), t.double().cpu(), S, _focal(S), 0.0)
    assert a.shape == (5, S, S) and a.dtype == torch.float32
    assert float(ref.sum()) > 100 and set(np.unique(a.cpu().numpy())) <= {0.0, 1.0}
    bad = torch.nonzero(a.cpu().double() != ref)
    for b in range(5):
        sel = bad[bad[:, 0] == b]
        if len(sel):
            d = SO.edge_distance(v.double().cpu(), faces.cpu(), t.double().cpu(), S, _focal(S), b, sel[:, 1], sel[:, 2])
            assert float(d.max()) < 1e-3, (b, float(d.max()))


@pytest.mark.parametrize("S,sigma", [(64, 1.0), (256, 1.0), (256, 4.0)])
def test_soft_alpha_matches_oracle(smpl, S, sigma):
    v, t, _ = _posed(smpl, 5, 20 + S)
    faces = smpl.faces_int32(DEV)
    a = ops.render_silhouettes(v, faces, t, S, _focal(S), sigma).cpu().double()
    ref = SO.render(v.double().cpu(), faces.cpu(), t.double().cpu(), S, _focal(S), sigma)
    amb = _ambiguous(v, t, faces, S, sigma)
    err = (a - ref).abs()
    assert float(err[~amb].max()) < 1e-4, float(err[~amb].max())


@pytest.mark.parametrize("S,sigma", [(64, 1.0), (256, 2.0)])
def test_gradients_match_oracle(smpl, S, sigma):
    v, t, _ = _posed(smpl, 5, 30 + S)
    faces = smpl.faces_int32(DEV)
    g = torch.randn(5, S, S, generator=torch.Generator().manual_seed(S))
    g[_ambiguous(v, t, faces, S, sigma)] = 0.0
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    (ops.render_silhouettes(vv, faces, tt, S, _focal(S), sigma) * g.to(DEV)).sum().backward()
    v64, t64 = v.double().cpu().requires_grad_(True), t.double().cpu().requires_grad_(True)
    (SO.render(v64, faces.cpu(), t64, S, _focal(S), sigma) * g.double()).sum().backward()
    for got, want in ((vv.grad, v64.grad), (tt.grad, t64.grad)):
        rel = float((got.cpu().double() - want).abs().max() / want.abs().max())
        assert rel < 1e-3, rel


def test_end_to_end_into_betas_and_pose(smpl, synthetic_model):
    B, S, sigma = 3, 64, 1.0
    betas, pose, cam = _bodies(B, 40)
    w = torch.randn(B, S, S, generator=torch.Generator().manual_seed(41))
    b_, p_, c_ = (x.to(DEV).requires_grad_(True) for x in (betas, pose, cam))
    out = smpl(betas=b_, body_pose=p_[:, 3:], global_orient=p_[:, :3])
    alpha = smpl.render_silhouettes(out.vertices, c_, img_wh=S, sigma=sigma)
    (alpha * w.to(DEV)).sum().backward()
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    b64, p64, c64 = (x.double().requires_grad_(True) for x in (betas, pose, cam))
    verts = orc.forward_flat(b64, p64, None, pose2rot=True).vertices
    t64 = convert_weak_perspective_to_camera_translation_torch(c64, config.FOCAL_LENGTH, 512)
    faces = torch.from_numpy(smpl.faces.astype(np.int64))
    a64 = SO.render(verts, faces, t64, S, _focal(S), sigma)
    assert float((alpha.detach().cpu().double() - a64.detach()).abs().max()) < 1e-3
    (a64 * w.double()).sum().backward()
    for got, want in ((b_.grad, b64.grad), (p_.grad, p64.grad), (c_.grad, c64.grad)):
        rel = float((got.cpu().double() - want).abs().max() / want.abs().max())
        assert rel < 2e-3, rel


@pytest.mark.parametrize("S", [64, 256])
def test_fused_loss_matches_render_loss_backward(smpl, S):
    sigma, weight = 1.0, 3.0
    v, t, _ = _posed(smpl, 5, 50 + S)
    faces = smpl.faces_int32(DEV)
    target = ops.render_silhouettes(v * 1.02, faces, t, S, _focal(S), 0.0) > 0.5
    base = torch.rand(5, device=DEV)
    loss, gv, gt = ops.silhouette_loss(v, faces, t, target, S, _focal(S), sigma, weight, loss_per_body=base.clone())
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    a = ops.render_silhouettes(vv, faces, tt, S, _focal(S), sigma)
    ref = weight * ((a - target.float()) ** 2).mean(dim=(1, 2))
    ref.sum().backward()
    assert torch.allclose(loss - base, ref.detach(), rtol=1e-5, atol=1e-7)
    for got, want in ((gv, vv.grad), (gt, tt.grad)):
        assert float((got - want).abs().max() / want.abs().max()) < 1e-5


def test_results_do_not_depend_on_batch_position(smpl):
    S, sigma = 128, 1.0
    v, t, _ = _posed(smpl, 5, 60)
    faces = smpl.faces_int32(DEV)
    g = torch.randn(5, S, S, generator=torch.Generator().manual_seed(61)).to(DEV)
    perm = torch.tensor([3, 0, 4, 1, 2], device=DEV)
    for sg in (0.0, sigma):
        a = ops.render_silhouettes(v, faces, t, S, _focal(S), sg)
        ap = ops.render_silhouettes(v[perm].contiguous(), faces, t[perm].contiguous(), S, _focal(S), sg)
        a1 = ops.render_silhouettes(v[2:3].contiguous(), faces, t[2:3].contiguous(), S, _focal(S), sg)
        assert torch.equal(a[perm], ap) and torch.equal(a[2:3], a1)
    outs = []
    for vv, tt, gg in ((v, t, g), (v[perm].contiguous(), t[perm].contiguous(), g[perm].contiguous())):
        vv, tt = vv.clone().requires_grad_(True), tt.clone().requires_grad_(True)
        (ops.render_silhouettes(vv, faces, tt, S, _focal(S), sigma) * gg).sum().backward()
        outs.append((vv.grad, tt.grad))
    for x, y in zip(outs[0], outs[1]):
        assert float((x[perm] - y).abs().max()) <= 1e-6 * float(x.abs().max())


def test_no_write_outside_caller_buffers(smpl):
    """Every output of the three entry points lies between two sentinel-filled guard bands, at a ragged size."""
    B, S, sigma = 3, 72, 1.0
    v, t, _ = _posed(smpl, B, 70)
    faces = smpl.faces_int32(DEV)
    GUARD = 4096
    bands = []

    def guarded(n, dtype=torch.float32):
        item = torch.empty((), dtype=dtype).element_size()
        pad = (-(n * item)) % 512
        raw = torch.full((GUARD + n * item + pad + GUARD,), 0xA5, dtype=torch.uint8, device=DEV)
        bands.append((raw, GUARD, GUARD + n * item))
        return raw[GUARD:GUARD + n * item].view(dtype)

    args = ops.silhouette_args(v, faces, t, S, _focal(S), sigma)
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    alpha = guarded(B * S * S)
    _lib.check(lib.b200smpl_silhouette_render(ctypes.byref(args), alpha.data_ptr(), st), "render")
    ga = torch.randn(B * S * S, device=DEV)
    gv, gt = guarded(B * 6890 * 3), guarded(B * 3)
    _lib.check(lib.b200smpl_silhouette_render_backward(ctypes.byref(args), ga.data_ptr(), gv.data_ptr(), gt.data_ptr(),
                                                       st), "render_backward")
    target = (alpha.view(B, S, S) > 0.5).to(torch.uint8).flip(2).contiguous()
    loss, gv2, gt2 = guarded(B), guarded(B * 6890 * 3), guarded(B * 3)
    loss.zero_()
    _lib.check(lib.b200smpl_silhouette_loss(ctypes.byref(args), target.data_ptr(), 1.0, loss.data_ptr(), gv2.data_ptr(),
                                            gt2.data_ptr(), st), "loss")
    args0 = ops.silhouette_args(v, faces, t, S, _focal(S), 0.0)
    alpha0 = guarded(B * S * S)
    _lib.check(lib.b200smpl_silhouette_render(ctypes.byref(args0), alpha0.data_ptr(), st), "render hard")
    torch.cuda.synchronize()
    assert float(alpha.max()) > 0.5 and float(loss.min()) > 0.0 and float(gv2.abs().max()) > 0.0
    for raw, lo, hi in bands:
        assert bool((raw[:lo] == 0xA5).all()) and bool((raw[hi:] == 0xA5).all())


def test_hard_mode_refuses_backward(smpl):
    v, t, _ = _posed(smpl, 2, 80)
    vv = v.clone().requires_grad_(True)
    a = ops.render_silhouettes(vv, smpl.faces_int32(DEV), t, 64, _focal(64), 0.0)
    assert not a.requires_grad
    args = ops.silhouette_args(v, smpl.faces_int32(DEV), t, 64, _focal(64), 0.0)
    g = torch.zeros(2, 64, 64, device=DEV)
    gv, gt = torch.empty_like(v), torch.empty_like(t)
    with pytest.raises(ValueError):
        _lib.check(_lib.load().b200smpl_silhouette_render_backward(ctypes.byref(args), g.data_ptr(), gv.data_ptr(),
                                                                   gt.data_ptr(), None), "render_backward")
    with pytest.raises(ValueError):
        ops.silhouette_loss(v, smpl.faces_int32(DEV), t, g > 0, 64, _focal(64), sigma=0.0)


def test_saturated_overlap_matches_oracle():
    """Two large overlapping faces and a small sigma: deep inside both, 1 - D_f underflows in fp32.  Gradients stay
    finite and agree with the fp64 oracle."""
    S, sigma = 64, 0.05
    pix = torch.tensor([[4, 4], [60, 4], [4, 60], [8, 6], [58, 12], [10, 58]], dtype=torch.float64)
    v = torch.cat([pix - S / 2.0, torch.zeros(6, 1, dtype=torch.float64)], 1)[None]
    t = torch.tensor([[0.0, 0.0, 1.0]], dtype=torch.float64)
    faces = torch.tensor([[0, 1, 2], [3, 4, 5]], dtype=torch.int32)
    g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    vv, tt = v.float().to(DEV).requires_grad_(True), t.float().to(DEV).requires_grad_(True)
    a = ops.render_silhouettes(vv, faces.to(DEV), tt, S, 1.0, sigma)
    (a * g.float().to(DEV)).sum().backward()
    v64, t64 = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    a64 = SO.render(v64, faces, t64, S, 1.0, sigma)
    (a64 * g).sum().backward()
    assert float((a.detach().cpu().double() - a64.detach()).abs().max()) < 1e-4
    for got, want in ((vv.grad, v64.grad), (tt.grad, t64.grad)):
        assert torch.isfinite(got).all()
        assert float((got.cpu().double() - want).abs().max() / want.abs().max()) < 1e-3


# ---- the fitter's silhouette term ------------------------------------------------------------------------------
def _fit_problem(smpl, B, S, seed):
    g = torch.Generator().manual_seed(seed)
    betas_t = torch.randn(B, 10, generator=g) * 0.8
    pose_t = torch.randn(B, 72, generator=g) * 0.25
    cam_t = torch.stack([0.6 + 0.6 * torch.rand(B, generator=g), 0.4 * torch.rand(B, generator=g) - 0.2,
                         0.4 * torch.rand(B, generator=g) - 0.2], 1)
    rot_t = O.batch_rodrigues(pose_t.reshape(-1, 3)).reshape(B, 24, 3, 3).float()
    betas0 = betas_t + 0.5 * torch.randn(B, 10, generator=g)
    rot0 = O.batch_rodrigues((pose_t + 0.15 * torch.randn(B, 72, generator=g)).reshape(-1, 3)).reshape(B, 24, 3, 3).float()
    cam0 = cam_t + 0.05 * torch.randn(B, 3, generator=g)
    d = lambda x: x.to(DEV)  # noqa: E731
    out = smpl(betas=d(betas_t), body_pose=d(rot_t)[:, 1:], global_orient=d(rot_t)[:, :1], pose2rot=False)
    label = ops.orthographic_project(out.joints, d(cam_t), 512.0)[:, config.SMPL_TO_KPRCNN_MAP].detach()
    sil = smpl.render_silhouettes(out.vertices.detach(), d(cam_t), img_wh=S, sigma=0.0) > 0.5
    return d(rot0), d(betas0), d(cam0), label.contiguous(), sil


def test_fitter_with_silhouettes_matches_eager_restatement(smpl):
    B, S, iters, lr, w, sigma = 8, 64, 5, 2e-3, 2.0, 1.0
    rot0, betas0, cam0, label, sil = _fit_problem(smpl, B, S, 1)
    fitter = BatchedFitter(smpl, lr=lr, silhouette_weight=w, silhouette_sigma=sigma, silhouette_wh=S,
                           use_cuda_graph=True, graph_iterations=2)
    res = fitter.fit(rot0, betas0, cam0, label, iterations=iters, silhouettes=sil)
    # eager restatement: autograd through SMPLFunction, ops.joints2d_loss per player, ops.render_silhouettes, Adam
    rot, betas, cam = (x.clone().requires_grad_(True) for x in (rot0, betas0, cam0))
    opt = torch.optim.Adam([rot, betas, cam], lr=lr)
    jmap = torch.tensor(config.SMPL_TO_KPRCNN_MAP, device=DEV)
    losses = []
    for _ in range(iters):
        out = smpl(betas=betas, body_pose=rot[:, 1:], global_orient=rot[:, :1], pose2rot=False)
        lj = torch.stack([ops.joints2d_loss(out.joints[b:b + 1], cam[b:b + 1], jmap, label[b:b + 1]) for b in range(B)])
        a = smpl.render_silhouettes(out.vertices, cam, img_wh=S, sigma=sigma)
        loss_b = lj + w * ((a - sil.float()) ** 2).mean(dim=(1, 2))
        losses.append(loss_b.detach())
        opt.zero_grad()
        loss_b.sum().backward()
        rot.grad[:, list(FROZEN_FULL_JOINTS)] = 0.0
        opt.step()
    torch.cuda.synchronize()
    assert torch.allclose(res["initial_loss"], losses[0], rtol=1e-4)
    assert torch.allclose(res["last_loss"], losses[-1], rtol=1e-3)
    for got, want in ((res["final_rotmats"], rot.detach()), (res["final_betas"], betas.detach()),
                      (res["final_cam"], cam.detach())):
        diff = (got.reshape(want.shape) - want).abs()
        assert diff.median().item() < 1e-5 and diff.max().item() < 2 * lr * iters
    assert res["silhouette_iou"].shape == (B,)


def test_fitter_silhouette_raises_iou(smpl):
    B, S = 8, 64
    rot0, betas0, cam0, label, sil = _fit_problem(smpl, B, S, 2)
    fitter = BatchedFitter(smpl, lr=1e-2, silhouette_weight=5.0, silhouette_sigma=1.0, silhouette_wh=S)
    iou0 = fitter.silhouette_iou(rot0, betas0, cam0, sil)
    res = fitter.fit(rot0, betas0, cam0, label, iterations=60, silhouettes=sil)
    torch.cuda.synchronize()
    assert float(res["silhouette_iou"].mean()) > float(iou0.mean())
    assert (res["best_loss"] < res["initial_loss"]).all()


def test_fit_without_silhouettes_is_unchanged(smpl):
    """The joints-only path: a fitter configured for silhouettes but called without them, and one given silhouettes
    at weight 0, run the plain fitter's launches.  The first loss comes from the (bit-deterministic) forward and is
    equal bit for bit; everything after a backward carries the backward's fp32 RED order (run-to-run ~1e-7)."""
    B, S = 6, 64
    rot0, betas0, cam0, label, sil = _fit_problem(smpl, B, S, 3)
    plain = BatchedFitter(smpl, lr=2e-3, graph_iterations=4).fit(rot0, betas0, cam0, label, iterations=9)
    conf = BatchedFitter(smpl, lr=2e-3, graph_iterations=4, silhouette_weight=3.0, silhouette_wh=S)
    a = conf.fit(rot0, betas0, cam0, label, iterations=9)
    b = BatchedFitter(smpl, lr=2e-3, graph_iterations=4, silhouette_wh=S).fit(rot0, betas0, cam0, label, iterations=9,
                                                                              silhouettes=sil)
    for other in (a, b):
        assert set(plain) <= set(other) and torch.equal(plain["initial_loss"], other["initial_loss"])
        assert torch.equal(plain["best_iter"], other["best_iter"])
        for k, x in plain.items():
            assert torch.allclose(x.float(), other[k].float(), rtol=1e-4, atol=1e-5), k
    assert "silhouette_iou" not in a and b["silhouette_iou"].shape == (B,)
