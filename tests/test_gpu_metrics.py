"""GPU tests of the reconstruction-error kernel (csrc/metrics.cu, ops.reconstruction_errors) and of
regressor.validation_step against the fp64 oracle (oracle/metrics_oracle.py)."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

from oracle import metrics_oracle as M
from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, ops, regressor
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
J14 = config.ALL_JOINTS_TO_J14_MAP


@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


def _similar(X, rng, kind):
    """A prediction for target X (N, 3) float64: noisy, rigid, similarity, mirrored or identical."""
    R = Rotation.random(random_state=int(rng.integers(1 << 30))).as_matrix()
    t = rng.standard_normal(3) * 3
    if kind == "noise":
        return X + 0.02 * rng.standard_normal(X.shape)
    if kind == "rigid":
        return X @ R.T + t
    if kind == "similarity":
        return 0.8 * X @ R.T + t + 0.005 * rng.standard_normal(X.shape)
    if kind == "mirrored":
        c = X.mean(0)
        return (X - c) * np.array([1.0, 1.0, -1.0]) + c + 0.01 * rng.standard_normal(X.shape)
    return X.copy()


KINDS = ("noise", "rigid", "similarity", "mirrored", "identical")


def _bodies(smpl, B, seed):
    """Targets: posed synthetic SMPL bodies up to 20 m from the origin; predictions: one of KINDS per body."""
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    transl = (torch.rand(B, 3, generator=g) - 0.5) * 40
    with torch.no_grad():
        out = smpl(betas=betas.to(DEV), body_pose=pose[:, 3:].to(DEV), global_orient=pose[:, :3].to(DEV),
                   transl=transl.to(DEV))
    tv, tj = out.vertices.double().cpu().numpy(), out.joints.double().cpu().numpy()
    rng = np.random.default_rng(seed)
    pv, pj = np.empty_like(tv), np.empty_like(tj)
    for b in range(B):
        kind = KINDS[b % len(KINDS)]
        both = _similar(np.concatenate([tv[b], tj[b]]), rng, kind)
        pv[b], pj[b] = both[:tv.shape[1]], both[tv.shape[1]:]
    f32 = lambda a: torch.from_numpy(a.astype(np.float32)).to(DEV)      # noqa: E731
    return f32(pv), f32(tv), f32(pj), f32(tj)


def _ref(pv=None, tv=None, pj=None, tj=None, jmap=None):
    c = lambda t: None if t is None else t.double().cpu().numpy()        # noqa: E731
    return M.reconstruction_errors(c(pv), c(tv), c(pj), c(tj), None if jmap is None else jmap.cpu().numpy())


def _close(got, want):
    got = got.double().cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    err = np.abs(got[ok] - want[ok])
    bound = 1e-5 * np.abs(want[ok]) + 1e-6
    assert (err <= bound).all(), (err.max(), np.argwhere(err > bound)[:5])


@pytest.mark.parametrize("B", [1, 37, 300])
def test_matches_oracle(smpl, B):
    pv, tv, pj, tj = _bodies(smpl, B, B)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    got = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    assert got.shape == (B, 6) and got.dtype == torch.float32
    want = _ref(pv, tv, pj, tj, jmap)
    _close(got, want)
    if B >= 5:                                            # the identical pair is exact; the others are not trivial
        assert (want[4::5, [0, 3]] == 0).all() and (want[4::5] < 1e-9).all() and (want[0::5] > 1e-4).all()
    # each pair alone: the other pair's columns are NaN
    _close(ops.reconstruction_errors(pv, tv), np.concatenate([want[:, :3], np.full((B, 3), np.nan)], 1))
    _close(ops.reconstruction_errors(pred_joints=pj, target_joints=tj, joint_map=jmap),
           np.concatenate([np.full((B, 3), np.nan), want[:, 3:]], 1))


@pytest.mark.parametrize("V", [3, 100, 6890, 20000])
def test_mesh_sizes_and_long_maps(V):
    g = torch.Generator().manual_seed(V)
    B, NJ = 9, 45
    tv = (torch.randn(B, V, 3, generator=g) * torch.tensor([0.2, 0.8, 0.1]) + torch.randn(B, 1, 3, generator=g) * 10)
    pv = tv + 0.03 * torch.randn(B, V, 3, generator=g)
    pv[1] = tv[1] * torch.tensor([-1.0, 1.0, 1.0])         # mirrored
    pv[2] = tv[2] * 1.2 + 5.0                               # similarity with R = I
    pv[3] = 7.0                                             # all predicted points coincide
    tj = torch.randn(B, NJ, 3, generator=g) + 20.0
    pj = tj + 0.05 * torch.randn(B, NJ, 3, generator=g)
    jmap = torch.randint(0, NJ, (70,), generator=g)         # longer than a warp, with repeated rows
    pv, tv, pj, tj, jmap = (t.to(DEV) for t in (pv, tv, pj, tj, jmap))
    got = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    want = _ref(pv, tv, pj, tj, jmap)
    _close(got, want)
    assert len(set(jmap.tolist())) < 70


def test_non_finite_points_poison_their_own_set_only(smpl):
    pv, tv, pj, tj = _bodies(smpl, 4, 3)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    pv[1, 100, 2] = float("nan")
    tv[2, 5, 0] = float("inf")
    pj[3, J14[4], 1] = float("-inf")
    got = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    _close(got, _ref(pv, tv, pj, tj, jmap))
    assert torch.isnan(got[1, :3]).all() and torch.isfinite(got[1, 3:]).all() and torch.isnan(got[3, 3:]).all()


def test_deterministic_and_batch_position_independent(smpl):
    pv, tv, pj, tj = _bodies(smpl, 37, 5)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    a = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    b = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    for i in (0, 17, 36):
        alone = ops.reconstruction_errors(pv[i:i + 1].clone(), tv[i:i + 1].clone(), pj[i:i + 1].clone(),
                                          tj[i:i + 1].clone(), jmap)
        assert torch.equal(alone.view(torch.int32), a[i:i + 1].view(torch.int32))


def _shifted(t, byte_offset):
    """A copy of t whose data starts `byte_offset` bytes past a 16-byte boundary."""
    n = t.numel()
    buf = torch.empty(n + 8, dtype=torch.float32, device=DEV)
    k = ((16 - buf.data_ptr() % 16) % 16 + byte_offset) // 4
    v = buf[k:k + n].view_as(t)
    v.copy_(t)
    assert v.data_ptr() % 16 == byte_offset
    return v


def _args(B, pv, tv, pj, tj, jmap, **kw):
    a = dict(batch=B, num_verts=0 if pv is None else pv.shape[1], num_joints=0 if pj is None else pj.shape[1],
             num_map=0 if jmap is None else jmap.numel(), reserved0=0, reserved1=0,
             pred_vertices=None if pv is None else pv.data_ptr(), target_vertices=None if tv is None else tv.data_ptr(),
             pred_joints=None if pj is None else pj.data_ptr(), target_joints=None if tj is None else tj.data_ptr(),
             joint_map=None if jmap is None else jmap.data_ptr())
    a.update(kw)
    return _lib.ReconErrorArgs(**a)


def _call(args, out_ptr):
    stream = ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    return _lib.load().b200smpl_reconstruction_errors(ctypes.byref(args), ctypes.c_void_p(out_ptr), stream)


@pytest.mark.parametrize("offset", [4, 8])
def test_unaligned_inputs_and_guard_bands(smpl, offset):
    B = 7
    pv, tv, pj, tj = _bodies(smpl, B, 9)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    want = ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    spv, stv, spj, stj = (_shifted(t, offset) for t in (pv, tv, pj, tj))
    sentinel = -12345.5
    guard = 37
    buf = torch.full((guard + B * 6 + guard + 1,), sentinel, dtype=torch.float32, device=DEV)
    k = guard + ((16 - buf.data_ptr() % 16) % 16 + offset) // 4
    out = buf[k:k + B * 6]
    assert _call(_args(B, spv, stv, spj, stj, jmap), out.data_ptr()) == 0
    torch.cuda.synchronize()
    assert torch.equal(out.view(B, 6), want)
    assert (buf[:k] == sentinel).all() and (buf[k + B * 6:] == sentinel).all()
    # an absent pair's columns are left as they were
    out.fill_(sentinel)
    assert _call(_args(B, spv, stv, None, None, None), out.data_ptr()) == 0
    assert torch.equal(out.view(B, 6)[:, :3], want[:, :3]) and (out.view(B, 6)[:, 3:] == sentinel).all()
    out.fill_(sentinel)
    assert _call(_args(B, None, None, spj, stj, jmap), out.data_ptr()) == 0
    assert torch.equal(out.view(B, 6)[:, 3:], want[:, 3:]) and (out.view(B, 6)[:, :3] == sentinel).all()
    assert (buf[:k] == sentinel).all() and (buf[k + B * 6:] == sentinel).all()


def test_graph_capture_and_one_launch_per_call(smpl):
    B = 16
    pv, tv, pj, tj = _bodies(smpl, B, 21)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    want = ops.reconstruction_errors(pv, tv, pj, tj, jmap)          # also checks the map once, outside the capture
    lib = _lib.load()
    before = lib.b200smpl_launch_count()
    ops.reconstruction_errors(pv, tv, pj, tj, jmap)
    assert lib.b200smpl_launch_count() - before == 1
    s_pv, s_tv, s_pj, s_tj = (torch.zeros_like(t) for t in (pv, tv, pj, tj))
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        ops.reconstruction_errors(s_pv, s_tv, s_pj, s_tj, jmap)
    torch.cuda.current_stream(DEV).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        got = ops.reconstruction_errors(s_pv, s_tv, s_pj, s_tj, jmap)
    for src, dst in zip((pv, tv, pj, tj), (s_pv, s_tv, s_pj, s_tj)):
        dst.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(got, want)


def test_argument_errors_launch_nothing_and_write_nothing(smpl):
    B = 3
    pv, tv, pj, tj = _bodies(smpl, B, 2)
    jmap = torch.tensor(J14, dtype=torch.int32, device=DEV)
    out = torch.full((B, 6), 7.0, device=DEV)
    lib = _lib.load()
    before = lib.b200smpl_launch_count()
    for kw in (dict(batch=0), dict(target_vertices=None), dict(pred_joints=None), dict(num_verts=0),
               dict(num_joints=0), dict(num_map=0), dict(joint_map=None),
               dict(pred_vertices=None, target_vertices=None, pred_joints=None, target_joints=None)):
        assert _call(_args(B, pv, tv, pj, tj, jmap, **kw), out.data_ptr()) == _lib.ERR_INVALID, kw
    assert _call(_args(B, pv, tv, pj, tj, jmap), 0) == _lib.ERR_INVALID
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == before and (out == 7.0).all()
    with pytest.raises(ValueError):
        ops.reconstruction_errors(pv, None)
    with pytest.raises(ValueError):
        ops.reconstruction_errors(pv, tv[:, :100])
    with pytest.raises(ValueError):
        ops.reconstruction_errors(pred_joints=pj, target_joints=tj)
    with pytest.raises(IndexError):
        ops.reconstruction_errors(pred_joints=pj, target_joints=tj, joint_map=torch.tensor([0, 90], device=DEV))
    with pytest.raises(TypeError):
        ops.reconstruction_errors(pv.double(), tv.double())
    assert lib.b200smpl_launch_count() == before


# ---- validation_step ------------------------------------------------------------------------------------------------
LOSSES = ("verts", "joints2D", "joints3D", "shape_params", "pose_params")


def _val_batch(model, B, seed):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, 64, generator=g)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
    cam = torch.tensor([0.9, 0.0, 0.0]).repeat(B, 1)
    out = O.SMPLOracle(model, dtype=torch.float64).forward(betas.double(), rot[:, 1:].double(), rot[:, :1].double(),
                                                           None, False)
    j2d = O.undo_keypoint_normalisation(O.orthographic_project(out.joints, cam.double()), 512)
    labels = {"joints2D": j2d[:, config.SMPL_TO_KPRCNN_MAP], "verts": out.vertices, "shape_params": betas,
              "pose_params_rot_matrices": rot, "joints3D": out.joints[:, config.ALL_JOINTS_TO_COCO_MAP]}
    return feats.to(DEV), {k: v.float().to(DEV) for k, v in labels.items()}


@pytest.mark.parametrize("fused", [False, True])
def test_validation_step_matches_oracle(smpl, synthetic_model, fused):
    B = 12
    torch.manual_seed(0)
    head = regressor.IEFModule((48, 48), in_features=64).to(DEV)
    crit = regressor.MultiTaskLoss(LOSSES, {"verts": 1.0, "joints2D": 0.1}).to(DEV)
    opt = torch.optim.Adam(list(head.parameters()) + list(crit.parameters()), lr=1e-3)
    feats, labels = _val_batch(synthetic_model, B, 3)
    g6, gproj = regressor.gpu_ops()
    regressor.train_step(head, crit, opt, smpl, feats, labels, g6, gproj, fused_loss=fused)   # Adam state exists
    params = {k: v.clone() for k, v in list(head.state_dict().items()) + list(crit.state_dict().items())}
    state = [{k: v.clone() if torch.is_tensor(v) else v for k, v in s.items()} for s in opt.state.values()]
    grads = [None if p.grad is None else p.grad.clone() for p in opt.param_groups[0]["params"]]

    loss, errors = regressor.validation_step(head, crit, smpl, feats, labels, g6, gproj, fused_loss=fused)
    assert errors.shape == (B, 7) and errors.device == DEV and not loss.requires_grad
    # the loss is the criterion's value on the same predictions
    with torch.no_grad():
        out = regressor.predict(head, smpl, feats, g6, None if fused else gproj)
        want_loss = (crit.forward_fused(labels, out) if fused else crit(labels, out))[0]
    assert torch.equal(loss, want_loss)
    # the errors are the oracle's on the same predictions and targets
    rot = labels["pose_params_rot_matrices"]
    with torch.no_grad():
        tgt = smpl(body_pose=rot[:, 1:], global_orient=rot[:, :1], betas=labels["shape_params"], pose2rot=False)
        eye = torch.eye(3, device=DEV).expand(B, 24, 3, 3)
        tp = smpl(body_pose=eye[:, 1:], global_orient=eye[:, :1], betas=out["shape_params"], pose2rot=False)
        tt = smpl(body_pose=eye[:, 1:], global_orient=eye[:, :1], betas=labels["shape_params"], pose2rot=False)
    jmap = torch.tensor(J14, device=DEV)
    want = _ref(out["verts"], tgt.vertices, out["joints"], tgt.joints, jmap)
    want = np.concatenate([want, _ref(tp.vertices, tt.vertices)[:, 1:2]], 1)
    _close(errors, want)
    assert (want > 1e-4).all()
    # no parameter, gradient or optimiser state changed
    now = dict(list(head.state_dict().items()) + list(crit.state_dict().items()))
    assert all(torch.equal(now[k], v) for k, v in params.items())
    for s0, s1 in zip(state, opt.state.values()):
        assert all(torch.equal(v, s1[k]) if torch.is_tensor(v) else v == s1[k] for k, v in s0.items())
    for g0, p in zip(grads, opt.param_groups[0]["params"]):
        assert (g0 is None and p.grad is None) or torch.equal(g0, p.grad)


def test_validation_step_does_not_synchronise(smpl, synthetic_model):
    B = 8
    torch.manual_seed(1)
    head = regressor.IEFModule((48, 48), in_features=64).to(DEV)
    crit = regressor.MultiTaskLoss(LOSSES).to(DEV)
    feats, labels = _val_batch(synthetic_model, B, 4)
    g6, gproj = regressor.gpu_ops()
    sums = torch.zeros(7, device=DEV)
    regressor.validation_step(head, crit, smpl, feats, labels, g6, None, fused_loss=True)   # checks the map once
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(2):
            loss, errors = regressor.validation_step(head, crit, smpl, feats, labels, g6, None, fused_loss=True)
            sums += errors.sum(0)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(sums).all()
