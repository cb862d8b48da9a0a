"""GPU tests of the silhouette term in MultiViewFitter: against the multi-view loop restated with autograd (the SMPL
module, SMPL.render_silhouettes with sigma > 0, torch.optim.Adam over stacked per-view tensors), the kernels its steps
and validation passes launch, the IoU it reaches, and the joints-only loop it leaves unchanged."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, ops
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch
from soccerplayershapepose_b200.fitting import MultiViewFitter
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
FROZEN_BP = [6, 7, 21, 22]                  # body_pose[:, 6:8] and body_pose[:, 21:]


@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


def _problem(smpl, P, V, S, seed):
    """Truth and a perturbed start for P players x V views; keypoint labels and hard-rendered masks (P,V,S,S) of the
    truth per view."""
    g = torch.Generator().manual_seed(seed)
    betas_t = torch.randn(P, 10, generator=g) * 0.8
    bp_aa = torch.randn(P, 69, generator=g) * 0.25
    go_aa = torch.randn(P, V, 3, generator=g) * 0.6
    cam_t = torch.stack([0.6 + 0.6 * torch.rand(P, V, generator=g), 0.4 * torch.rand(P, V, generator=g) - 0.2,
                         0.4 * torch.rand(P, V, generator=g) - 0.2], -1)
    rm = lambda aa: O.batch_rodrigues(aa.double().reshape(-1, 3)).float()  # noqa: E731
    bp_t, go_t = rm(bp_aa).reshape(P, 23, 3, 3).to(DEV), rm(go_aa).reshape(P, V, 3, 3).to(DEV)
    label = torch.empty(P, V, 17, 2, device=DEV)
    sil = torch.empty(P, V, S, S, dtype=torch.bool, device=DEV)
    with torch.no_grad():
        for v in range(V):
            out = smpl(betas=betas_t.to(DEV), body_pose=bp_t, global_orient=go_t[:, v:v + 1], pose2rot=False)
            label[:, v] = ops.orthographic_project(out.joints, cam_t[:, v].to(DEV), 512.0)[:, config.SMPL_TO_KPRCNN_MAP]
            sil[:, v] = smpl.render_silhouettes(out.vertices, cam_t[:, v].to(DEV), img_wh=S, sigma=0.0) > 0.5
    betas0 = (betas_t + 0.5 * torch.randn(P, 10, generator=g)).to(DEV)
    bp0 = rm(bp_aa + 0.15 * torch.randn(P, 69, generator=g)).reshape(P, 23, 3, 3).to(DEV)
    go0 = rm(go_aa + 0.1 * torch.randn(P, V, 3, generator=g)).reshape(P, V, 3, 3).to(DEV)
    cam0 = (cam_t + 0.05 * torch.randn(P, V, 3, generator=g)).to(DEV)
    return bp0, betas0, go0, cam0, label, sil


def _orders(V, n, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.permutation(V).tolist() for _ in range(n)]


def _ref_multiview(smpl, bp0, betas0, go0, cam0, label, sil, iters, lr, rounds, orders, w, sigma):
    """The loop of test_gpu_fitting._ref_multiview restated in fp32 autograd with the silhouette term: per view the
    joints2D loss per player plus w * mean((alpha - target)^2) of the soft silhouette; stacked per-view tensors under
    one Adam per phase, a validation pass per epoch, per-phase restore to the best epoch, global best kept."""
    P, V = go0.shape[0], go0.shape[1]
    S = sil.shape[-1]
    go = go0.transpose(0, 1).contiguous().clone()          # (V,P,3,3)
    cam = cam0.transpose(0, 1).contiguous().clone()        # (V,P,3)
    bp, betas = bp0.clone(), betas0.clone()
    lab, tgt = label.transpose(0, 1), sil.transpose(0, 1).float()
    jmap = torch.tensor(config.SMPL_TO_KPRCNN_MAP, device=DEV)

    def loss_view(v):
        out = smpl(betas=betas, body_pose=bp, global_orient=go[v][:, None], pose2rot=False)
        lj = torch.stack([ops.joints2d_loss(out.joints[p:p + 1], cam[v][p:p + 1], jmap, lab[v][p:p + 1])
                          for p in range(P)])
        a = smpl.render_silhouettes(out.vertices, cam[v], img_wh=S, sigma=sigma)
        return lj + w * ((a - tgt[v]) ** 2).mean(dim=(1, 2))

    best_metric = torch.full((P,), float("inf"), device=DEV)
    best = {"go": go.clone(), "cam": cam.clone(), "bp": bp.clone(), "betas": betas.clone()}
    final = {k: t.clone() for k, t in best.items()}
    e, first_val = 0, None
    for _ in range(rounds):
        for phase in ("A", "B"):
            params = {"A": {"cam": cam, "go": go}, "B": {"bp": bp, "betas": betas}}[phase]
            for t in params.values():
                t.requires_grad_(True)
            opt = torch.optim.Adam(list(params.values()), lr=lr)
            for _e in range(iters):
                for v in orders[e]:
                    opt.zero_grad()
                    loss_view(v).sum().backward()
                    if phase == "B":
                        bp.grad[:, FROZEN_BP] = 0.0
                    opt.step()
                e += 1
                with torch.no_grad():
                    val = sum(loss_view(v) for v in range(V))
                    if first_val is None:
                        first_val = val.clone()
                    imp = val < best_metric
                    best_metric = torch.where(imp, val, best_metric)
                    cur = {"go": go, "cam": cam, "bp": bp, "betas": betas}
                    for k in cur:
                        for d_ in [final[k]] + ([best[k]] if k in params else []):
                            if k in ("go", "cam"):
                                d_[:, imp] = cur[k].detach()[:, imp]
                            else:
                                d_[imp] = cur[k].detach()[imp]
            for t in params.values():
                t.requires_grad_(False)
            with torch.no_grad():
                for k in params:
                    params[k].copy_(best[k])
    return {"final": final, "best_metric": best_metric, "first_val": first_val,
            "last": {"go": go, "cam": cam, "bp": bp, "betas": betas}}


@pytest.mark.parametrize("use_graph", [True, False])
def test_multiview_silhouette_matches_autograd_restatement(smpl, use_graph):
    P, V, S, iters, rounds, lr, w, sigma = 3, 2, 64, 3, 2, 2e-3, 2.0, 1.0
    bp0, betas0, go0, cam0, label, sil = _problem(smpl, P, V, S, 11)
    orders = _orders(V, rounds * 2 * iters)
    ref = _ref_multiview(smpl, bp0, betas0, go0, cam0, label, sil, iters, lr, rounds, orders, w, sigma)
    fitter = MultiViewFitter(smpl, lr=lr, rounds=rounds, use_cuda_graph=use_graph, silhouette_weight=w,
                             silhouette_sigma=sigma, silhouette_wh=S)
    res = fitter.fit(bp0, betas0, go0, cam0, label, iterations=iters, view_orders=orders, silhouettes=sil)
    torch.cuda.synchronize()
    if use_graph:                                       # replays only, from re-initialised state buffers
        assert len(fitter._cache[(P, V, 10, False, "sil")]["graphs"]) == 2 * V + 2
        again = fitter.fit(bp0, betas0, go0, cam0, label, iterations=iters, view_orders=orders, silhouettes=sil)
        for k in ("body_pose", "betas", "global_orient", "cam", "best_loss", "silhouette_iou"):
            assert (again[k] - res[k]).abs().max().item() < 1e-5, k
    np.testing.assert_allclose(res["initial_loss"].cpu().numpy(), ref["first_val"].cpu().numpy(), rtol=2e-3)
    np.testing.assert_allclose(res["best_loss"].cpu().numpy(), ref["best_metric"].cpu().numpy(), rtol=5e-3)
    nsteps = rounds * iters * V
    pairs = ((res["body_pose"].reshape(P, 207), ref["final"]["bp"].reshape(P, 207)),
             (res["betas"], ref["final"]["betas"]),
             (res["global_orient"].reshape(P, V, 9), ref["final"]["go"].transpose(0, 1).reshape(P, V, 9)),
             (res["cam"], ref["final"]["cam"].transpose(0, 1)),
             (res["last"]["body_pose"].reshape(P, 207), ref["last"]["bp"].reshape(P, 207)),
             (res["last"]["global_orient"].reshape(P, V, 9), ref["last"]["go"].transpose(0, 1).reshape(P, V, 9)),
             (res["last"]["cam"], ref["last"]["cam"].transpose(0, 1)))
    for got, want in pairs:
        diff = (got - want.detach()).abs()
        assert diff.median().item() < 2e-5 and diff.max().item() < 2 * lr * nsteps
        assert torch.quantile(diff.flatten(), 0.99).item() < 3e-3
    assert (res["best_loss"] < res["initial_loss"]).all()


def _kernels(fn):
    """Kernel launches by name while `fn` runs (b200smpl_timing_*; eager launches only)."""
    lib = _lib.load()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.b200smpl_timing_report(buf, 1 << 16)               # drop earlier records
    lib.b200smpl_timing_enable(1)
    try:
        out = fn()
        torch.cuda.synchronize()
    finally:
        lib.b200smpl_timing_enable(0)
    lib.b200smpl_timing_report(buf, 1 << 16)
    counts = {}
    for line in buf.value.decode().splitlines():
        name, n, _ms = line.split()
        counts[name] = int(n)
    return out, counts


def test_validation_runs_the_value_kernel(smpl):
    """Eager fit: one fused sil_loss per view step, V sil_loss_value per validation pass, no sil_bwd, and V sil_fwd
    (the IoU of the result).  The best loss is the summed validation loss of the returned parameters: fit_loss plus
    ops.silhouette_loss_value per view, recomputed here."""
    P, V, S, iters, rounds, w, sigma = 3, 2, 32, 2, 1, 2.0, 1.0
    bp0, betas0, go0, cam0, label, sil = _problem(smpl, P, V, S, 12)
    fitter = MultiViewFitter(smpl, lr=5e-3, rounds=rounds, use_cuda_graph=False, silhouette_weight=w,
                             silhouette_sigma=sigma, silhouette_wh=S)
    res, k = _kernels(lambda: fitter.fit(bp0, betas0, go0, cam0, label, iterations=iters, silhouettes=sil))
    epochs = rounds * 2 * iters
    assert k.get("sil_loss") == epochs * V and k.get("sil_loss_value") == epochs * V
    assert "sil_bwd" not in k and k.get("sil_fwd") == V
    jmap = torch.tensor(config.SMPL_TO_KPRCNN_MAP, device=DEV)
    want = torch.zeros(P, device=DEV)
    with torch.no_grad():
        for v in range(V):
            out = smpl(betas=res["betas"], body_pose=res["body_pose"], global_orient=res["global_orient"][:, v:v + 1],
                       pose2rot=False)
            cam = res["cam"][:, v].contiguous()
            want += torch.stack([ops.joints2d_loss(out.joints[p:p + 1], cam[p:p + 1], jmap, label[p:p + 1, v])
                                 for p in range(P)])
            t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, 512.0).contiguous()
            ops.silhouette_loss_value(out.vertices, smpl.faces_int32(DEV), t, sil[:, v], S,
                                      config.FOCAL_LENGTH * S / 512.0, sigma, w, loss_per_body=want)
    assert torch.allclose(res["best_loss"], want, rtol=1e-5, atol=1e-7), (res["best_loss"], want)


def test_silhouette_term_raises_iou_and_keeps_frozen_joints(smpl):
    """Targets are hard renders of the truth: with the term the returned parameters overlap them better than the
    start does.  Hands and feet of the shared body pose never move; the result keeps the reference's keys."""
    P, V, S = 4, 2, 64
    bp0, betas0, go0, cam0, label, sil = _problem(smpl, P, V, S, 13)
    fitter = MultiViewFitter(smpl, lr=1e-2, rounds=3, silhouette_weight=5.0, silhouette_sigma=1.0, silhouette_wh=S)
    iou0 = fitter.silhouette_iou(bp0, betas0, go0, cam0, sil)
    res = fitter.fit(bp0, betas0, go0, cam0, label, iterations=10, silhouettes=sil)
    torch.cuda.synchronize()
    assert iou0.shape == (P, V) and res["silhouette_iou"].shape == (P, V)
    assert float(res["silhouette_iou"].mean()) > float(iou0.mean())
    assert (res["best_loss"] < res["initial_loss"]).all()
    for bp in (res["body_pose"], res["last"]["body_pose"]):
        assert torch.equal(bp[:, FROZEN_BP], bp0[:, FROZEN_BP])
    shapes = {"body_pose": (P, 23, 3, 3), "betas": (P, 10), "global_orient": (P, V, 3, 3), "cam": (P, V, 3),
              "translation": (P, V, 3), "best_loss": (P,), "initial_loss": (P,)}
    for k, shp in shapes.items():
        assert tuple(res[k].shape) == shp, k


def test_joints_only_fit_is_unchanged(smpl):
    """A fitter built with the silhouette options but called without masks, and one given masks at weight 0, run the
    plain fitter's loop: the same launches (plus, with masks, the IoU evaluation of the result), the same state key
    and graphs.  The first loss comes from the bit-deterministic forward and is equal bit for bit; everything after a
    backward carries the backward's fp32 RED order (run-to-run ~1e-7)."""
    P, V, S, iters, rounds, lr = 3, 2, 32, 3, 2, 2e-3
    bp0, betas0, go0, cam0, label, sil = _problem(smpl, P, V, S, 14)
    orders = _orders(V, rounds * 2 * iters, seed=1)
    lib = _lib.load()

    def run(fitter, **kw):
        torch.cuda.synchronize()
        n0 = lib.b200smpl_launch_count()
        r = fitter.fit(bp0, betas0, go0, cam0, label, iterations=iters, view_orders=orders, **kw)
        torch.cuda.synchronize()
        return r, lib.b200smpl_launch_count() - n0

    fitters = [MultiViewFitter(smpl, lr=lr, rounds=rounds),
               MultiViewFitter(smpl, lr=lr, rounds=rounds, silhouette_weight=3.0, silhouette_wh=S),
               MultiViewFitter(smpl, lr=lr, rounds=rounds, silhouette_wh=S)]
    plain, n_plain = run(fitters[0])
    conf, n_conf = run(fitters[1])
    zero, n_zero = run(fitters[2], silhouettes=sil)
    n0 = lib.b200smpl_launch_count()
    fitters[2].silhouette_iou(zero["body_pose"], zero["betas"], zero["global_orient"], zero["cam"], sil)
    n_iou = lib.b200smpl_launch_count() - n0
    assert n_conf == n_plain and n_zero == n_plain + n_iou
    for f in fitters:
        assert list(f._cache) == [(P, V, 10, False)] and len(f._cache[(P, V, 10, False)]["graphs"]) == 2 * V + 2
    assert "silhouette_iou" not in plain and "silhouette_iou" not in conf and zero["silhouette_iou"].shape == (P, V)
    for other in (conf, zero):
        assert torch.equal(plain["initial_loss"], other["initial_loss"])
        for k in ("body_pose", "betas", "global_orient", "cam", "translation", "best_loss"):
            assert torch.allclose(plain[k], other[k], rtol=1e-4, atol=1e-5), k


def test_silhouette_errors(smpl):
    P, V, S = 2, 2, 32
    bp0, betas0, go0, cam0, label, sil = _problem(smpl, P, V, S, 15)
    fitter = MultiViewFitter(smpl, silhouette_weight=1.0, silhouette_wh=S)
    for bad in (sil[:, :, :, :-1], sil.reshape(P * V, S, S), sil.transpose(0, 1)[:1]):
        with pytest.raises(ValueError):
            fitter.fit(bp0, betas0, go0, cam0, label, iterations=1, silhouettes=bad)
    with pytest.raises(ValueError):
        MultiViewFitter(smpl, silhouette_weight=1.0, silhouette_sigma=0.0)
