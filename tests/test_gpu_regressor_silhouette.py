"""GPU tests of the gradient-free silhouette loss kernel (sil_loss_value), ops.silhouette_term and the silhouette term
of the regressor's multi-task loss, against the fp64 oracles (oracle/silhouette_oracle.py, oracle/smpl_oracle.py)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import silhouette_oracle as SO
from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, ops, regressor
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
NDISTINCT = 5


@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


@pytest.fixture(scope="module")
def faces(smpl):
    return smpl.faces_int32(DEV)


def _focal(S):
    return config.FOCAL_LENGTH * S / 512


def _posed(smpl, B, seed):
    """Posed vertices (B,6890,3) and camera translations (B,3) of min(B, NDISTINCT) random bodies, repeated in
    batch order (body b is body b % NDISTINCT)."""
    n = min(B, NDISTINCT)
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(n, 10, generator=g)
    pose = torch.randn(n, 72, generator=g) * 0.3
    cam = torch.stack([torch.rand(n, generator=g) * 0.6 + 0.6, torch.rand(n, generator=g) * 0.4 - 0.2,
                       torch.rand(n, generator=g) * 0.4 - 0.2], 1)
    out = smpl(betas=betas.to(DEV), body_pose=pose[:, 3:].to(DEV), global_orient=pose[:, :3].to(DEV))
    t = convert_weak_perspective_to_camera_translation_torch(cam.to(DEV), config.FOCAL_LENGTH, 512)
    idx = torch.arange(B, device=DEV) % n
    return out.vertices.detach()[idx].contiguous(), t[idx].contiguous()


def _target(v, faces, t, S):
    """Hard silhouettes of slightly larger bodies, as uint8 masks."""
    return (ops.render_silhouettes(v * 1.03, faces, t, S, _focal(S), 0.0) > 0.5).to(torch.uint8)


def _ambiguous(v, t, faces, S, sigma, limit=0.05):
    """Pixels near a face whose kept / dropped status fp32 may decide differently from fp64 (|area| < 1e-4 px^2).
    They must be fewer than `limit` of the image."""
    tri, _, area = SO.face_table(v.double(), t.double(), faces, _focal(S), S)
    mask = torch.zeros(v.shape[0], S, S, dtype=torch.bool, device=v.device)
    rad = np.sqrt(SO.cutoff_d2(sigma)) + 1.0 if sigma > 0 else 1.0
    for b, k in torch.nonzero(area.abs() < 1e-4).tolist():
        lo, hi = tri[b, k].min(0).values.tolist(), tri[b, k].max(0).values.tolist()
        c0, c1 = (int(np.clip(x, 0, S)) for x in (np.floor(lo[0] - rad), np.ceil(hi[0] + rad)))
        r0, r1 = (int(np.clip(x, 0, S)) for x in (np.floor(lo[1] - rad), np.ceil(hi[1] + rad)))
        mask[b, r0:r1, c0:c1] = True
    assert float(mask.float().mean()) < limit
    return mask


def _value(v, faces, t, target, S, sigma, weight=1.0, base=None):
    return ops.silhouette_loss_value(v, faces, t, target, S, _focal(S), sigma, weight,
                                     loss_per_body=None if base is None else base.clone())


# ---- the value kernel ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [33, 64, 256])
@pytest.mark.parametrize("B", [1, 5, 37, 300])
def test_value_kernel_matches_oracle(smpl, faces, B, S):
    """Soft and hard loss per body against the fp64 oracle; B = 1 and 5 split a body's bands over a cluster, 300 is
    more than two waves.  Hard: every pixel where kernel and oracle differ lies within 1e-3 px of an edge.  Soft:
    the oracle's alpha, with the kernel's render on the few pixels fp32 cannot decide like fp64, within the fused
    loss's bounds."""
    v, t = _posed(smpl, B, 100 + S)
    target = _target(v, faces, t, S)
    n = min(B, NDISTINCT)
    v1, t1, tg1 = v[:n], t[:n], target[:n].double()
    # hard
    got = _value(v, faces, t, target, S, 0.0)
    a_fwd = ops.render_silhouettes(v1, faces, t1, S, _focal(S), 0.0).double()
    ref = SO.render(v1.double(), faces, t1.double(), S, _focal(S), 0.0)
    bad = torch.nonzero(a_fwd != ref)
    for b in bad[:, 0].unique().tolist():
        sel = bad[bad[:, 0] == b]
        d = SO.edge_distance(v1.double(), faces, t1.double(), S, _focal(S), b, sel[:, 1], sel[:, 2])
        assert float(d.max()) < 1e-3
    exact = ((a_fwd - tg1) ** 2).mean(dim=(1, 2))          # the coverage of sil_fwd at sigma = 0
    assert float(exact.max()) > 0.0
    for b in range(B):
        assert abs(float(got[b]) - float(exact[b % n])) <= 1e-6 * float(exact[b % n])
    nmis = torch.zeros(n, dtype=torch.float64, device=DEV).index_add_(0, bad[:, 0], torch.ones(len(bad), device=DEV,
                                                                                                dtype=torch.float64))
    ref_h = ((ref - tg1) ** 2).mean(dim=(1, 2))
    assert bool(((got[:n].double() - ref_h).abs() <= nmis / S ** 2 + 1e-6 * ref_h).all())
    # soft
    sigma = 1.0
    got = _value(v, faces, t, target, S, sigma)
    a = ops.render_silhouettes(v1, faces, t1, S, _focal(S), sigma).double()
    ref = SO.render(v1.double(), faces, t1.double(), S, _focal(S), sigma)
    # at S = 33 and 64 a body is 25 to 50 px tall, so the pixels near its degenerate faces are a larger share
    amb = _ambiguous(v1, t1, faces, S, sigma, limit=0.05 if S >= 256 else 0.25)
    ref = torch.where(amb, a, ref)
    ref_s = ((ref - tg1) ** 2).mean(dim=(1, 2))
    for b in range(B):
        assert abs(float(got[b]) - float(ref_s[b % n])) <= 1e-5 * float(ref_s[b % n]) + 1e-7, (b, float(got[b]))


@pytest.mark.parametrize("S", [64, 256])
@pytest.mark.parametrize("B", [1, 5, 300])
def test_value_kernel_matches_fused_loss(smpl, faces, B, S):
    v, t = _posed(smpl, B, 200 + S)
    target = _target(v, faces, t, S)
    for sigma in (0.5, 2.0):
        got = _value(v, faces, t, target, S, sigma, weight=2.5)
        fused, _, _ = ops.silhouette_loss(v, faces, t, target, S, _focal(S), sigma, 2.5)
        assert float(fused.min()) > 0.0
        assert float(((got - fused).abs() / fused).max()) <= 1e-6


@pytest.mark.parametrize("B", [1, 5, 300])
def test_value_kernel_is_deterministic(smpl, faces, B):
    """Bitwise the same from run to run and across batch positions (every copy of a body in the batch)."""
    S = 256
    v, t = _posed(smpl, B, 300)
    target = _target(v, faces, t, S)
    n = min(B, NDISTINCT)
    for sigma in (0.0, 1.0):
        a = _value(v, faces, t, target, S, sigma)
        for _ in range(3):
            assert torch.equal(_value(v, faces, t, target, S, sigma), a)
        for b in range(B):
            assert torch.equal(a[b], a[b % n])
        if B > 1:
            perm = torch.randperm(B, generator=torch.Generator().manual_seed(1)).to(DEV)
            ap = _value(v[perm].contiguous(), faces, t[perm].contiguous(), target[perm].contiguous(), S, sigma)
            assert torch.equal(ap, a[perm])


def test_value_kernel_adds_and_writes_nothing_else(smpl, faces):
    B, S, GUARD = 5, 72, 4096
    v, t = _posed(smpl, B, 400)
    target = _target(v, faces, t, S)
    raw = torch.full((GUARD + 4 * B + GUARD,), 0xA5, dtype=torch.uint8, device=DEV)
    loss = raw[GUARD:GUARD + 4 * B].view(torch.float32)
    base = torch.rand(B, device=DEV) + 1.0
    loss.copy_(base)
    for sigma in (0.0, 1.0):
        before = loss.clone()
        args = ops.silhouette_args(v, faces, t, S, _focal(S), sigma)
        _lib.check(_lib.load().b200smpl_silhouette_loss_value(
            ctypes.byref(args), target.data_ptr(), 0.75, loss.data_ptr(),
            ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)), "silhouette_loss_value")
        alone = _value(v, faces, t, target, S, sigma, 0.75)
        torch.cuda.synchronize()
        assert float(alone.min()) > 0.0
        assert torch.allclose(loss, before + alone, rtol=1e-6, atol=0.0)
    assert bool((raw[:GUARD] == 0xA5).all()) and bool((raw[GUARD + 4 * B:] == 0xA5).all())


def test_value_kernel_argument_checks():
    """Each bad argument gives B200SMPL_ERR_INVALID without launching a kernel or writing loss_per_body."""
    lib = _lib.load()
    S, B = 16, 2
    p = torch.tensor([[2.0, 2.0], [14.0, 3.0], [5.0, 13.0]], dtype=torch.float64)
    v = torch.cat([p - S / 2.0, torch.zeros(3, 1, dtype=torch.float64)], 1)[None].float().to(DEV)
    v = v.expand(B, 3, 3).contiguous()
    t = torch.tensor([[0.0, 0.0, 1.0]], device=DEV).expand(B, 3).contiguous()
    fc = torch.tensor([[0, 1, 2]], dtype=torch.int32, device=DEV)
    target = torch.ones(B, S, S, dtype=torch.uint8, device=DEV)
    loss = torch.full((B,), 7.0, device=DEV)

    def args(**kw):
        a = dict(batch=B, num_verts=3, num_faces=1, img_wh=S, focal_length=1.0, sigma=1.0, vertices=v.data_ptr(),
                 cam_t=t.data_ptr(), faces=fc.data_ptr(), workspace=None, workspace_bytes=0)
        a.update(kw)
        return ctypes.byref(_lib.SilhouetteArgs(**a))

    def call(p, target_p=target.data_ptr(), loss_p=loss.data_ptr(), weight=1.0):
        return lambda: lib.b200smpl_silhouette_loss_value(p, target_p, weight, loss_p, None)

    bad = [args(batch=0), args(num_verts=2), args(num_verts=65536), args(num_faces=0), args(img_wh=0),
           args(img_wh=16385), args(sigma=float("nan")), args(sigma=-1.0), args(sigma=float("inf")),
           args(focal_length=0.0), args(focal_length=float("inf")), args(focal_length=float("nan")),
           args(vertices=None), args(cam_t=None), args(faces=None), None]
    cases = [call(p) for p in bad] + [call(args(), target_p=None), call(args(), loss_p=None),
                                      call(args(), weight=float("nan")), call(args(), weight=float("inf"))]
    torch.cuda.synchronize()
    n0 = lib.b200smpl_launch_count()
    for i, c in enumerate(cases):
        rc = c()
        assert rc == _lib.ERR_INVALID, (i, rc)
        with pytest.raises(ValueError):
            _lib.check(rc, "case {}".format(i))
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 and bool((loss == 7.0).all())
    for sg in (0.0, 1.0):                               # valid arguments launch, hard mode included
        _lib.check(call(args(sigma=sg))(), "loss_value")
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 + 2 and float(loss.min()) > 7.0


# ---- ops.silhouette_term ---------------------------------------------------------------------------------------
def _kernels(fn):
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


@pytest.mark.parametrize("B", [5, 300])
def test_silhouette_term_launches_one_kernel(smpl, faces, B):
    S, sigma = 128, 1.0
    v, t = _posed(smpl, B, 500)
    target = _target(v, faces, t, S).float()
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    with_grad, k1 = _kernels(lambda: ops.silhouette_term(vv, faces, tt, target, S, _focal(S), sigma))
    assert k1.get("sil_loss") == 1 and "sil_loss_value" not in k1 and "sil_fwd" not in k1
    assert with_grad.requires_grad
    with torch.no_grad():
        no_grad, k2 = _kernels(lambda: ops.silhouette_term(vv, faces, tt, target, S, _focal(S), sigma))
    assert {k: n for k, n in k2.items() if k.startswith("sil")} == {"sil_loss_value": 1}
    plain, k3 = _kernels(lambda: ops.silhouette_term(v, faces, t, target, S, _focal(S), sigma))
    assert {k: n for k, n in k3.items() if k.startswith("sil")} == {"sil_loss_value": 1}
    for x in (no_grad, plain):
        assert not x.requires_grad and abs(x.item() - with_grad.item()) <= 1e-6 * with_grad.item()


@pytest.mark.parametrize("S", [64, 256])
def test_silhouette_term_gradients(smpl, faces, S):
    """Under a non-unit upstream gradient, against render + render_backward + autograd."""
    B, sigma, up = 5, 1.0, -2.75
    v, t = _posed(smpl, B, 600 + S)
    target = _target(v, faces, t, S)
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    term = ops.silhouette_term(vv, faces, tt, target.bool(), S, _focal(S), sigma)
    (up * term).backward()
    v2, t2 = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    a = ops.render_silhouettes(v2, faces, t2, S, _focal(S), sigma)
    ref = ((a - target.float()) ** 2).mean(dim=(1, 2)).mean()
    (up * ref).backward()
    assert abs(float(term) - float(ref)) <= 1e-5 * float(ref)
    for got, want in ((vv.grad, v2.grad), (tt.grad, t2.grad)):
        assert float(want.abs().max()) > 0.0
        assert float((got - want).abs().max() / want.abs().max()) < 1e-5


# ---- the criterion ---------------------------------------------------------------------------------------------
LOSSES = ("verts", "joints2D", "joints3D", "shape_params", "pose_params")
WEIGHTS = {"verts": 1.0, "joints2D": 0.1, "joints3D": 1.0, "shape_params": 0.1, "pose_params": 0.1,
           "silhouette": 0.5}


class _OracleSMPL:
    def __init__(self, model, dtype):
        self.orc = O.SMPLOracle(model, dtype=dtype)

    def __call__(self, body_pose, global_orient, betas, pose2rot=False, return_verts=True):
        return self.orc.forward(betas, body_pose, global_orient, None, pose2rot)


def _cpu_ops():
    return O.rot6d_to_rotmat, (lambda joints, cam: O.undo_keypoint_normalisation(O.orthographic_project(joints, cam), 512))


def _batch(model, B, seed, S):
    """Features and labels (float32, CPU); the silhouette label is the hard silhouette of the label body."""
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, 64, generator=g)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
    cam = torch.tensor([0.9, 0.0, 0.0]).repeat(B, 1)
    betas, rot, cam = betas.double(), rot.double(), cam.double()
    out = O.SMPLOracle(model, dtype=torch.float64).forward(betas, rot[:, 1:], rot[:, :1], None, False)
    j2d = O.undo_keypoint_normalisation(O.orthographic_project(out.joints, cam), 512)[:, config.SMPL_TO_KPRCNN_MAP, :]
    t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, 512)
    sil = SO.render(out.vertices.to(DEV), torch.as_tensor(model["faces"]).to(DEV), t.to(DEV), S, _focal(S), 0.0)
    labels = {"joints2D": j2d, "verts": out.vertices, "shape_params": betas, "pose_params_rot_matrices": rot,
              "joints3D": out.joints[:, config.ALL_JOINTS_TO_COCO_MAP, :], "silhouette": sil.cpu()}
    return feats, {k: v.float() for k, v in labels.items()}


def _make(model, losses, S, dtype=torch.float32, seed=0):
    torch.manual_seed(seed)
    head = regressor.IEFModule((48, 48), in_features=64).to(dtype)
    with torch.no_grad():
        head.fc3.weight.mul_(0.05)                      # the camera starts near [0.9, 0, 0]: bodies in the image
    crit = regressor.MultiTaskLoss(losses, WEIGHTS, faces=model["faces"], silhouette_sigma=1.0, silhouette_wh=S)
    return head, crit.to(dtype)


@pytest.mark.parametrize("S", [64, 256])
def test_fused_and_eager_criteria_agree(smpl, synthetic_model, S):
    B = 7
    feats, labels = _batch(synthetic_model, B, 11, S)
    lab = {k: v.to(DEV) for k, v in labels.items()}
    g6, gproj = regressor.gpu_ops()
    render = regressor.gpu_silhouette_renderer(smpl.faces_int32(DEV), S, 1.0)
    head, crit_f = _make(synthetic_model, LOSSES + ("silhouette",), S)
    head, crit_f = head.to(DEV), crit_f.to(DEV)
    crit_e = regressor.MultiTaskLoss(LOSSES + ("silhouette",), WEIGHTS, faces=synthetic_model["faces"],
                                     silhouette_wh=S).to(DEV)
    with torch.no_grad():
        for c in (crit_f, crit_e):
            c.silhouette_log_var.fill_(0.4)
    out = regressor.predict(head, smpl, feats.to(DEV), g6, gproj)
    leaves = {k: out[k].detach().clone().requires_grad_(True) for k in ("verts", "joints", "cam", "shape_params",
                                                                        "pose_params_rot_matrices")}
    loss_f, parts_f = crit_f.forward_fused(lab, leaves)
    (1.5 * loss_f).backward()
    le = {k: v.detach().clone().requires_grad_(True) for k, v in leaves.items()}
    oe = dict(le)
    oe["joints2D"] = ops.orthographic_project(le["joints"], le["cam"], 512.0)[:, config.SMPL_TO_KPRCNN_MAP]
    oe["joints3D"] = le["joints"][:, config.ALL_JOINTS_TO_COCO_MAP]
    oe["silhouettes"] = render(le["verts"], le["cam"])
    loss_e, parts_e = crit_e(lab, oe)
    (1.5 * loss_e).backward()
    assert 1e-3 < float(parts_f["silhouette"]) < 1.0
    assert abs(loss_f.item() - loss_e.item()) < 1e-5 * max(1.0, abs(loss_e.item()))
    assert set(parts_f) == set(parts_e)
    for n in parts_e:
        assert abs(parts_f[n].item() - parts_e[n].item()) < 1e-5 * max(1e-3, abs(parts_e[n].item())), n
        g, ge = getattr(crit_f, n + "_log_var").grad, getattr(crit_e, n + "_log_var").grad
        assert abs(g.item() - ge.item()) < 1e-5 * max(1.0, abs(ge.item())), n
    for k in ("verts", "cam"):
        want = le[k].grad
        assert float((leaves[k].grad - want).abs().max()) < 1e-4 * float(want.abs().max()), k


@pytest.mark.parametrize("S", [64, 256])
def test_criteria_match_oracle_gradients(smpl, synthetic_model, S):
    """Fused and eager criteria with the silhouette term against fp64 oracle SMPL + oracle silhouettes: the loss and
    the gradients of the head's parameters and of its camera output."""
    B = 5
    feats, labels = _batch(synthetic_model, B, 21, S)
    faces_cpu = torch.as_tensor(synthetic_model["faces"])
    head64, crit64 = _make(synthetic_model, ("silhouette",), S, torch.float64)
    r6, proj = _cpu_ops()

    def render64(verts, cam):
        t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, 512)
        return SO.render(verts.to(DEV), faces_cpu.to(DEV), t.to(DEV), S, _focal(S), 1.0).cpu()

    out64 = regressor.predict(head64, _OracleSMPL(synthetic_model, torch.float64), feats.double(), r6, proj,
                              render_silhouettes=render64)
    out64["cam"].retain_grad()
    loss64 = crit64({k: v.double() for k, v in labels.items()}, out64)[0]
    loss64.backward()
    g6, gproj = regressor.gpu_ops()
    lab = {k: v.to(DEV) for k, v in labels.items()}
    for fused in (True, False):
        head, crit = _make(synthetic_model, ("silhouette",), S)
        head, crit = head.to(DEV), crit.to(DEV)
        render = regressor.gpu_silhouette_renderer(smpl.faces_int32(DEV), S, 1.0)
        out = regressor.predict(head, smpl, feats.to(DEV), g6, None if fused else gproj,
                                render_silhouettes=None if fused else render)
        out["cam"].retain_grad()
        loss = (crit.forward_fused(lab, out) if fused else crit(lab, out))[0]
        loss.backward()
        assert abs(loss.item() - loss64.item()) < 1e-4 * abs(loss64.item()), fused
        for got, want in [(getattr(head, n).weight.grad, getattr(head64, n).weight.grad) for n in ("fc1", "fc3")] + \
                [(out["cam"].grad, out64["cam"].grad), (crit.silhouette_log_var.grad, crit64.silhouette_log_var.grad)]:
            assert float(want.abs().max()) > 0.0
            rel = float((got.cpu().double() - want).abs().max() / want.abs().max())
            assert rel < 2e-3, (fused, rel)


def test_graphed_step_with_the_term_matches_eager_steps(smpl, synthetic_model):
    """The captured step with the eager criterion and the injected renderer follows the eager `train_step`."""
    S = 64
    feats, labels = _batch(synthetic_model, 6, 9, S)
    feats, labels = feats.to(DEV), {k: v.to(DEV) for k, v in labels.items()}
    g6, gproj = regressor.gpu_ops()
    render = regressor.gpu_silhouette_renderer(smpl.faces_int32(DEV), S, 1.0)
    losses = LOSSES + ("silhouette",)
    head_a, crit_a = (m.to(DEV) for m in _make(synthetic_model, losses, S))
    head_b, crit_b = (m.to(DEV) for m in _make(synthetic_model, losses, S))
    head_b.load_state_dict(head_a.state_dict())
    crit_b.load_state_dict(crit_a.state_dict())
    lr, warm, n = 1e-3, 2, 3
    opt = torch.optim.Adam(list(head_a.parameters()) + list(crit_a.parameters()), lr=lr)
    eager = [regressor.train_step(head_a, crit_a, opt, smpl, feats, labels, g6, gproj, render_silhouettes=render).item()
             for _ in range(warm + n)]
    gs = regressor.GraphedTrainStep(head_b, crit_b, smpl, feats, labels, g6, gproj, lr=lr, warmup=warm,
                                    render_silhouettes=render)
    assert "silhouette" in gs.labels
    graphed = [gs(feats, labels).item() for _ in range(n)]
    np.testing.assert_allclose(graphed, eager[warm:], rtol=2e-4)
    for pa, pb in zip(list(head_a.parameters()) + [crit_a.silhouette_log_var],
                      list(head_b.parameters()) + [crit_b.silhouette_log_var]):
        assert (pa - pb).abs().max().item() < 2e-5


def test_graphed_step_with_the_term_fused_and_encoder(smpl, synthetic_model):
    """The captured step with the fused loss kernels, the silhouette term and the ResNet-18 encoder follows the eager
    step with the eager loss."""
    S, B = 64, 4
    _, labels = _batch(synthetic_model, B, 13, S)
    labels = {k: v.to(DEV) for k, v in labels.items()}
    crops = torch.randn(B, 18, 64, 64, generator=torch.Generator().manual_seed(1)).to(DEV)
    g6, gproj = regressor.gpu_ops()
    render = regressor.gpu_silhouette_renderer(smpl.faces_int32(DEV), S, 1.0)
    torch.manual_seed(0)
    net_a = regressor.SingleInputRegressor(18).to(DEV)
    net_b = regressor.SingleInputRegressor(18).to(DEV)
    with torch.no_grad():
        net_a.ief_module.fc3.weight.mul_(0.05)
    net_b.load_state_dict(net_a.state_dict())
    losses = LOSSES + ("silhouette",)
    crit_a = regressor.MultiTaskLoss(losses, WEIGHTS, faces=synthetic_model["faces"], silhouette_wh=S).to(DEV)
    crit_b = regressor.MultiTaskLoss(losses, WEIGHTS, faces=synthetic_model["faces"], silhouette_wh=S).to(DEV)
    lr, warm, n = 1e-4, 2, 3
    opt = torch.optim.Adam(list(net_a.parameters()) + list(crit_a.parameters()), lr=lr)
    eager = [regressor.train_step(net_a, crit_a, opt, smpl, crops, labels, g6, gproj, render_silhouettes=render).item()
             for _ in range(warm + n)]
    gs = regressor.GraphedTrainStep(net_b, crit_b, smpl, crops, labels, g6, None, lr=lr, warmup=warm, fused_loss=True)
    graphed = [gs(crops, labels).item() for _ in range(n)]
    np.testing.assert_allclose(graphed, eager[warm:], rtol=2e-3)


def test_criterion_without_the_term_makes_the_same_launches(smpl, synthetic_model):
    """Without "silhouette" a step makes the same library launches whether or not a renderer and faces are given;
    with it, the fused step adds exactly sil_loss and the eager step sil_fwd + sil_bwd."""
    S = 64
    lib = _lib.load()
    feats, labels = _batch(synthetic_model, 4, 31, S)
    feats, labels = feats.to(DEV), {k: v.to(DEV) for k, v in labels.items()}
    g6, gproj = regressor.gpu_ops()
    render = regressor.gpu_silhouette_renderer(smpl.faces_int32(DEV), S, 1.0)

    def launches(crit, fused, **kw):
        head, _ = _make(synthetic_model, LOSSES, S)
        head, crit = head.to(DEV), crit.to(DEV)
        opt = torch.optim.Adam(list(head.parameters()) + list(crit.parameters()), lr=1e-4)
        regressor.train_step(head, crit, opt, smpl, feats, labels, g6, gproj, fused_loss=fused, **kw)   # warm
        torch.cuda.synchronize()
        n0 = lib.b200smpl_launch_count()
        regressor.train_step(head, crit, opt, smpl, feats, labels, g6, gproj, fused_loss=fused, **kw)
        torch.cuda.synchronize()
        return lib.b200smpl_launch_count() - n0

    for fused in (True, False):
        plain = launches(regressor.MultiTaskLoss(LOSSES, WEIGHTS), fused)
        assert plain > 0
        assert launches(regressor.MultiTaskLoss(LOSSES, WEIGHTS, faces=synthetic_model["faces"], silhouette_wh=S),
                        fused, render_silhouettes=render) == plain
        sil = launches(regressor.MultiTaskLoss(LOSSES + ("silhouette",), WEIGHTS, faces=synthetic_model["faces"],
                                               silhouette_wh=S), fused, render_silhouettes=render)
        assert sil == plain + (1 if fused else 2), (fused, plain, sil)
