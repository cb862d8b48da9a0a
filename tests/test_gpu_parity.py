"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C-ABI
library, against the CPU oracle on the same seeded inputs, against the committed known answers,
and -- at BASELINE.json's batch sizes -- through size-independent properties.

Tolerances (BASELINE.json north_star): vertices / joints 1e-5 m absolute in fp32 modes, 1e-4 m in
bf16-GEMM mode; gradients 1e-4 relative in every mode the north_star names (the bf16-GEMM mode runs its gradient
GEMM in the bf16x3 split for that; measured 2e-5).  "Relative" = max |error| / max |reference| per gradient
tensor (`_rel`).  The extra `bf16_fast` mode (single-product bf16 gradient GEMM) is OUTSIDE that bound by design:
measured 2.2e-3 on grad_betas, tested at 5e-3.  Index / topology work bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib
from soccerplayershapepose_b200.engine import SMPLEngine
from soccerplayershapepose_b200.smpl import SMPL, SMPLLayer, SMPLOutput

pytestmark = pytest.mark.gpu

POS_TOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-4, "bf16_fast": 1e-4}
GRAD_TOL = {"fp32": 1e-4, "fp32_simt": 1e-4, "bf16": 1e-4, "bf16_fast": 5e-3}
MODES = ["fp32_simt", "fp32", "bf16", "bf16_fast"]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def engine(synthetic_model, dev):
    return SMPLEngine(synthetic_model, dev)


@pytest.fixture(scope="module")
def oracle64(synthetic_model):
    return O.SMPLOracle(synthetic_model, dtype=torch.float64)


def make_inputs(B, seed):
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    trans = torch.rand(B, 3, generator=g) * 2 - 1
    cam = torch.stack([torch.rand(B, generator=g) * 0.6 + 0.6, torch.rand(B, generator=g) * 0.4 - 0.2,
                       torch.rand(B, generator=g) * 0.4 - 0.2], 1)
    return betas, pose, trans, cam


def rotmats_of(pose):
    return O.batch_rodrigues(pose.double().reshape(-1, 3)).reshape(pose.shape[0], 24, 3, 3).float()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [1, 5, 37, 130])
def test_forward_rotmat_surface(engine, oracle64, dev, mode, B):
    betas, pose, trans, cam = make_inputs(B, 100 + B)
    rot = rotmats_of(pose)
    ref = oracle64.forward_flat(betas.double(), rot.double(), trans.double(), pose2rot=False)
    v, j, j2d = engine.forward(betas.to(dev), rot.to(dev), trans.to(dev), cam.to(dev), mode=_lib.MODES[mode])
    torch.cuda.synchronize()
    assert v.shape == (B, 6890, 3) and j.shape == (B, 90, 3) and j2d.shape == (B, 90, 2)
    assert (v.cpu().double() - ref.vertices).abs().max().item() < POS_TOL[mode]
    assert (j.cpu().double() - ref.joints).abs().max().item() < POS_TOL[mode]
    ref2d = O.orthographic_project(ref.joints, cam.double())
    assert (j2d.cpu().double() - ref2d).abs().max().item() < 2 * POS_TOL[mode]


@pytest.mark.parametrize("mode", MODES)
def test_forward_axis_angle_surface_no_transl(engine, oracle64, dev, mode):
    betas, pose, _, _ = make_inputs(9, 7)
    ref = oracle64.forward_flat(betas.double(), pose.double(), None, pose2rot=True)
    v, j, j2d = engine.forward(betas.to(dev), pose.to(dev), None, None, axis_angle=True, mode=_lib.MODES[mode])
    assert j2d is None
    assert (v.cpu().double() - ref.vertices).abs().max().item() < POS_TOL[mode]
    assert (j.cpu().double() - ref.joints).abs().max().item() < POS_TOL[mode]


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_known_answers(engine, smpl_kat, dev, mode):
    k = smpl_kat
    f = lambda a: torch.from_numpy(a).float().to(dev)  # noqa: E731
    v, j, _ = engine.forward(f(k["betas"]), f(k["rotmats"]), f(k["trans"]), None, mode=_lib.MODES[mode])
    sub = torch.from_numpy(k["vert_subset"]).to(dev)
    assert np.abs(v[:, sub].cpu().numpy() - k["verts_sub"]).max() < POS_TOL[mode]
    assert np.abs(j.cpu().numpy() - k["joints"]).max() < POS_TOL[mode]
    va, ja, _ = engine.forward(f(k["betas"][:5]), f(k["pose_aa"]), None, None, axis_angle=True,
                               mode=_lib.MODES[mode])
    assert np.abs(va[:, sub].cpu().numpy() - k["aa_verts_sub"]).max() < POS_TOL[mode]
    assert np.abs(ja.cpu().numpy() - k["aa_joints"]).max() < POS_TOL[mode]


def test_tpose_is_template(engine, synthetic_model, dev):
    v, j, _ = engine.forward(torch.zeros(3, 10, device=dev), torch.zeros(3, 72, device=dev), None, None,
                             axis_angle=True, mode=_lib.MODE_FP32)
    vt = torch.from_numpy(synthetic_model["v_template"]).to(dev)
    assert (v - vt).abs().max().item() < 1e-6


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _oracle_grads(oracle64, betas, pose, trans, cam, dV, dJ, dJ2, axis_angle):
    b = betas.double().requires_grad_(True)
    p = pose.double().requires_grad_(True)
    t = trans.double().requires_grad_(True) if trans is not None else None
    c = cam.double().requires_grad_(True) if cam is not None else None
    out = oracle64.forward_flat(b, p, t, pose2rot=axis_angle)
    loss = 0.0
    if dV is not None:
        loss = loss + (out.vertices * dV.double()).sum()
    if dJ is not None:
        loss = loss + (out.joints * dJ.double()).sum()
    if dJ2 is not None:
        loss = loss + (O.orthographic_project(out.joints, c) * dJ2.double()).sum()
    loss.backward()
    return b.grad, p.grad, (None if t is None else t.grad), (None if c is None or c.grad is None else c.grad)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("axis_angle", [False, True])
def test_backward_full(engine, oracle64, dev, mode, axis_angle):
    B = 37
    betas, pose_aa, trans, cam = make_inputs(B, 5)
    pose = pose_aa if axis_angle else rotmats_of(pose_aa)
    g = torch.Generator().manual_seed(9)
    dV = torch.randn(B, 6890, 3, generator=g)
    dJ = torch.randn(B, 90, 3, generator=g)
    dJ2 = torch.randn(B, 90, 2, generator=g)
    rb, rp, rt, rc = _oracle_grads(oracle64, betas, pose, trans, cam, dV, dJ, dJ2, axis_angle)
    m = _lib.MODES[mode]
    d = lambda x: x.to(dev)  # noqa: E731
    _, joints, _ = engine.forward(d(betas), d(pose), d(trans), d(cam), axis_angle=axis_angle, mode=m)
    gb, gp, gt, gc = engine.backward(d(betas), d(pose), d(trans), d(cam), joints, d(dV), d(dJ), d(dJ2),
                                     axis_angle=axis_angle, mode=m)
    tol = GRAD_TOL[mode]
    assert _rel(gb.cpu().double(), rb) < tol
    assert _rel(gp.cpu().double().reshape(rp.shape), rp) < tol
    assert _rel(gt.cpu().double(), rt) < tol
    assert _rel(gc.cpu().double(), rc) < tol
    # same gradients when forward keeps the blend output for backward instead of recomputing it
    out = engine.forward(d(betas), d(pose), d(trans), d(cam), axis_angle=axis_angle, mode=m, save=True)
    sb, sp, st_, sc = engine.backward(d(betas), d(pose), d(trans), d(cam), out[1], d(dV), d(dJ), d(dJ2),
                                      axis_angle=axis_angle, mode=m, saved=out[3])
    for a_, b_ in ((sb, gb), (sp, gp), (st_, gt), (sc, gc)):
        assert _rel(a_, b_) < 1e-5


@pytest.mark.parametrize("mode", ["fp32_simt", "fp32"])
@pytest.mark.parametrize("which", ["verts_only", "joints_only", "j2d_only"])
def test_backward_partial_gradients(engine, oracle64, dev, mode, which):
    B = 6
    betas, pose_aa, trans, cam = make_inputs(B, 11)
    pose = rotmats_of(pose_aa)
    g = torch.Generator().manual_seed(2)
    dV = torch.randn(B, 6890, 3, generator=g) if which == "verts_only" else None
    dJ = torch.randn(B, 90, 3, generator=g) if which == "joints_only" else None
    dJ2 = torch.randn(B, 90, 2, generator=g) if which == "j2d_only" else None
    rb, rp, rt, rc = _oracle_grads(oracle64, betas, pose, trans, cam, dV, dJ, dJ2, False)
    m = _lib.MODES[mode]
    d = lambda x: None if x is None else x.to(dev)  # noqa: E731
    _, joints, _ = engine.forward(d(betas), d(pose), d(trans), d(cam), mode=m, want_vertices=dV is not None)
    gb, gp, gt, gc = engine.backward(d(betas), d(pose), d(trans), d(cam), joints, d(dV), d(dJ), d(dJ2), mode=m)
    assert _rel(gb.cpu().double(), rb) < 1e-4
    assert _rel(gp.cpu().double().reshape(rp.shape), rp) < 1e-4
    assert _rel(gt.cpu().double(), rt) < 1e-4
    if which == "j2d_only":
        assert _rel(gc.cpu().double(), rc) < 1e-4
    else:
        assert gc.abs().max().item() == 0.0


def test_reference_module_surface(synthetic_model, oracle64, dev):
    """Call pattern of player_recon.py:1192-1210,1280: leaf rotmats / betas with requires_grad, keyword
    call with pose2rot=False, loss.backward()."""
    smpl = SMPL(synthetic_model, batch_size=1).to(dev)
    names = set(dict(smpl.named_buffers()).keys())
    assert {"v_template", "shapedirs", "posedirs", "J_regressor", "lbs_weights", "parents", "faces_tensor",
            "J_regressor_extra", "J_regressor_cocoplus", "J_regressor_h36m"} <= names
    assert smpl.faces.shape == (13776, 3) and np.array_equal(smpl.faces, synthetic_model["faces"])
    assert torch.equal(smpl.faces_tensor.cpu(), torch.from_numpy(synthetic_model["faces"]))
    assert torch.equal(smpl.parents.cpu(), torch.from_numpy(synthetic_model["parents"]))
    betas, pose_aa, _, cam = make_inputs(2, 3)
    rot = rotmats_of(pose_aa)
    go = rot[:, :1].clone().to(dev).requires_grad_(True)
    bp = rot[:, 1:].clone().to(dev).requires_grad_(True)
    be = betas.clone().to(dev).requires_grad_(True)
    out = smpl(body_pose=bp, global_orient=go, betas=be, pose2rot=False)
    assert isinstance(out, SMPLOutput) and out.vertices.shape == (2, 6890, 3) and out.joints.shape == (2, 90, 3)
    assert out["joints"] is out.joints and out.full_pose is None and out.betas is be
    ref = oracle64.forward_flat(betas.double(), rot.double(), None, pose2rot=False)
    assert (out.vertices.detach().cpu().double() - ref.vertices).abs().max().item() < 1e-5
    loss = (out.joints[:, :45] ** 2).sum() + out.vertices.sum()
    loss.backward()
    b64 = betas.double().requires_grad_(True)
    r64 = rot.double().requires_grad_(True)
    o = oracle64.forward_flat(b64, r64, None, pose2rot=False)
    ((o.joints[:, :45] ** 2).sum() + o.vertices.sum()).backward()
    assert _rel(be.grad.cpu().double(), b64.grad) < 1e-4
    assert _rel(torch.cat([go.grad, bp.grad], 1).cpu().double(), r64.grad) < 1e-4
    # default-pose call smpl(betas=pred_shape) (predict/predict_3D.py:148) with a batch of betas
    out0 = smpl(betas=be.detach())
    ref0 = oracle64.forward_flat(betas.double(), torch.zeros(2, 72, dtype=torch.float64), None, pose2rot=True)
    assert (out0.vertices.cpu().double() - ref0.vertices).abs().max().item() < 1e-5
    # north_star positional surface
    layer = SMPLLayer(synthetic_model).to(dev)
    v, j = layer(be.detach(), rot.to(dev), None)
    assert (j.cpu().double() - ref.joints).abs().max().item() < 1e-5
    # errors: CPU tensors are refused (no CPU path), wrong shapes raise
    with pytest.raises(RuntimeError):
        layer(betas, rot, None)
    with pytest.raises(ValueError):
        layer(be.detach()[:, :5], rot.to(dev), None)


def test_joints_only_autograd_skips_vertices(synthetic_model, oracle64, dev):
    smpl = SMPL(synthetic_model).to(dev)
    betas, pose_aa, trans, cam = make_inputs(4, 8)
    rot = rotmats_of(pose_aa).to(dev).requires_grad_(True)
    be = betas.to(dev).requires_grad_(True)
    camd = cam.to(dev).requires_grad_(True)
    out = smpl(body_pose=rot[:, 1:], global_orient=rot[:, :1], betas=be, transl=trans.to(dev), pose2rot=False,
               cam=camd, return_verts=False)
    assert out.vertices is None
    (out.joints2d ** 2).sum().backward()
    b64, r64 = betas.double().requires_grad_(True), rotmats_of(pose_aa).double().requires_grad_(True)
    c64 = cam.double().requires_grad_(True)
    o = oracle64.forward_flat(b64, r64, trans.double(), pose2rot=False)
    (O.orthographic_project(o.joints, c64) ** 2).sum().backward()
    assert _rel(be.grad.cpu().double(), b64.grad) < 1e-4
    assert _rel(rot.grad.cpu().double(), r64.grad) < 1e-4
    assert _rel(camd.grad.cpu().double(), c64.grad) < 1e-4


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_full_size_properties(engine, dev, mode):
    """BASELINE.json config 2 size (B=4096): slab invariance, determinism of the forward,
    translation equivariance, and linearity of the backward in the upstream gradient."""
    B = 4096
    m = _lib.MODES[mode]
    betas, pose_aa, trans, _ = make_inputs(B, 1)
    d = lambda x: x.to(dev)  # noqa: E731
    betas, pose_aa, trans = d(betas), d(pose_aa), d(trans)
    v1, j1, _ = engine.forward(betas, pose_aa, trans, None, axis_angle=True, mode=m, slab=1024)
    v1, j1 = v1.clone(), j1.clone()
    v2, j2, _ = engine.forward(betas, pose_aa, trans, None, axis_angle=True, mode=m, slab=512)
    assert torch.equal(v1, v2) and torch.equal(j1, j2)          # slab size never changes a body's result
    v3, j3, _ = engine.forward(betas, pose_aa, None, None, axis_angle=True, mode=m)
    assert (v3 + trans[:, None] - v1).abs().max().item() < 1e-6
    assert (j3 + trans[:, None] - j1).abs().max().item() < 1e-6
    # a body computed alone equals the same body inside the batch
    for i in (0, 1717, 4095):
        vi, ji, _ = engine.forward(betas[i:i + 1], pose_aa[i:i + 1], trans[i:i + 1], None, axis_angle=True, mode=m)
        assert torch.equal(vi[0], v1[i]) and torch.equal(ji[0], j1[i])
    # backward: linear in (dV, dJ)
    g = torch.Generator(device="cpu").manual_seed(4)
    dV = d(torch.randn(256, 6890, 3, generator=g))
    dJ = d(torch.randn(256, 90, 3, generator=g))
    sl = slice(100, 356)
    ga = engine.backward(betas[sl], pose_aa[sl], trans[sl], None, None, dV, dJ, None, axis_angle=True, mode=m)
    gb = engine.backward(betas[sl], pose_aa[sl], trans[sl], None, None, 2 * dV, 2 * dJ, None, axis_angle=True, mode=m)
    for a, b in zip(ga[:3], gb[:3]):
        assert _rel(b, 2 * a) < 1e-5


@pytest.mark.parametrize("nb,B", [(1, 37), (1, 256), (4, 130), (16, 256), (16, 300)])
def test_other_beta_counts_and_tile_counts(synthetic_model, dev, nb, B):
    """Models with another number of betas (other K layouts / gradient widths: the CTA-pair gradient GEMM with
    nf_pad 208 for 1 beta, 224 otherwise) at batch sizes with an odd (37 -> 1, 300 -> 3: the last cluster has a
    padding CTA), or even (130 -> 2, 256 -> 2) number of 128-body tiles: forward and backward against the oracle."""
    model = dict(synthetic_model)
    sd = synthetic_model["shapedirs"]
    if nb <= sd.shape[2]:
        model["shapedirs"] = np.ascontiguousarray(sd[:, :, :nb])
    else:
        rng = np.random.default_rng(7)
        model["shapedirs"] = np.concatenate([sd, (rng.standard_normal((sd.shape[0], 3, nb - sd.shape[2])) * 0.002).astype(np.float32)], 2)
    eng = SMPLEngine(model, dev)
    orc = O.SMPLOracle(model, dtype=torch.float64)
    g = torch.Generator().manual_seed(11 + nb)
    betas = torch.randn(B, nb, generator=g)
    pose = rotmats_of(torch.randn(B, 72, generator=g) * 0.3)
    trans = torch.rand(B, 3, generator=g)
    dV = torch.randn(B, 6890, 3, generator=g)
    dJ = torch.randn(B, 90, 3, generator=g)
    rb, rp, rt, _ = _oracle_grads(orc, betas, pose, trans, None, dV, dJ, None, False)
    ref = orc.forward_flat(betas.double(), pose.double(), trans.double(), pose2rot=False)
    d = lambda x: x.to(dev)  # noqa: E731
    v, j, _ = eng.forward(d(betas), d(pose), d(trans), None, mode=_lib.MODES["fp32"])
    assert (v.cpu().double() - ref.vertices).abs().max().item() < POS_TOL["fp32"]
    assert (j.cpu().double() - ref.joints).abs().max().item() < POS_TOL["fp32"]
    gb, gp, gt, _ = eng.backward(d(betas), d(pose), d(trans), None, None, d(dV), d(dJ), None, mode=_lib.MODES["fp32"])
    assert _rel(gb.cpu().double(), rb) < GRAD_TOL["fp32"]
    assert _rel(gp.cpu().double().reshape(rp.shape), rp) < GRAD_TOL["fp32"]
    assert _rel(gt.cpu().double(), rt) < GRAD_TOL["fp32"]


def test_silhouette_handoff_layout(synthetic_model, dev):
    """player_recon.py:288-289, 694-697: vertices (B,6890,3), faces (B,F,3) float, t (B,1,3)."""
    smpl = SMPL(model_data=synthetic_model).to(dev)
    betas, pose, trans, cam = make_inputs(3, 2)
    rot = rotmats_of(pose).to(dev)
    out = smpl(betas=betas.to(dev), body_pose=rot[:, 1:], global_orient=rot[:, :1], pose2rot=False)
    h = smpl.silhouette_inputs(out.vertices, cam.to(dev))
    assert h["vertices"].data_ptr() == out.vertices.data_ptr() and h["vertices"].shape == (3, 6890, 3)
    assert h["faces"].shape == (3, smpl.faces.shape[0], 3) and h["faces"].dtype == torch.float32
    assert np.array_equal(h["faces"][1].cpu().numpy().astype(np.int64), smpl.faces.astype(np.int64))
    t = O.weak_perspective_to_translation(cam.double(), 5000.0, 512)
    assert h["t"].shape == (3, 1, 3) and np.allclose(h["t"][:, 0].cpu().double().numpy(), t.numpy(), rtol=1e-5)


def test_batch_past_int32_element_index(engine, dev):
    """Maximum sizes: B * 6890 * 3 > 2^31 elements (B = 106 000, one 8.8 GB vertex tensor), BASELINE.json
    config 4's per-box batch and beyond.  64 distinct bodies repeated down the batch: every copy must equal the
    result of the 64-body batch bit for bit (forward), and the gradients of the copies at the far end -- past
    the 32-bit element index -- must equal those of the small batch (backward; fp32 RED order only)."""
    B, P = 106000, 64
    assert B * 6890 * 3 > 2 ** 31
    betas, pose_aa, trans, _ = make_inputs(P, 77)
    betas, pose_aa, trans = betas.to(dev), pose_aa.to(dev), trans.to(dev)
    rep = lambda x: x.repeat((B + P - 1) // P, 1)[:B].contiguous()  # noqa: E731
    v0, j0, _ = engine.forward(betas, pose_aa, trans, None, axis_angle=True)
    v0, j0 = v0.clone(), j0.clone()
    v, j, _ = engine.forward(rep(betas), rep(pose_aa), rep(trans), None, axis_angle=True)
    assert v.shape == (B, 6890, 3)
    nfull = B // P
    assert torch.equal(v[:nfull * P].view(nfull, P, 6890, 3), v0.expand(nfull, -1, -1, -1))
    assert torch.equal(j[:nfull * P].view(nfull, P, 90, 3), j0.expand(nfull, -1, -1, -1))
    assert torch.equal(v[nfull * P:], v0[:B - nfull * P])
    del v, j
    g = torch.Generator().manual_seed(5)
    dV0 = torch.randn(P, 6890, 3, generator=g).to(dev)
    dJ0 = torch.randn(P, 90, 3, generator=g).to(dev)
    g0 = engine.backward(betas, pose_aa, trans, None, None, dV0, dJ0, None, axis_angle=True)
    g0 = [x.clone() for x in g0[:3]]
    dV = dV0.repeat((B + P - 1) // P, 1, 1)[:B].contiguous()
    dJ = dJ0.repeat((B + P - 1) // P, 1, 1)[:B].contiguous()
    gB = engine.backward(rep(betas), rep(pose_aa), rep(trans), None, None, dV, dJ, None, axis_angle=True)
    # the 64-body batch and the 4096-body slabs split the K range of the gradient GEMM differently, so the two
    # differ by fp32 accumulation rounding (measured <= 3e-5 on grad_betas, 5e-7 on the others)
    for a, b in zip(g0, gB[:3]):
        last = b[(nfull - 1) * P:nfull * P]
        assert _rel(last, a) < 1e-4
        assert _rel(b[:P], a) < 1e-4
        assert torch.isfinite(b).all()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_forward_full_size_vs_oracle(engine, oracle64, dev, mode):
    """BASELINE.json config 2 size (B = 4096): vertices and joints of 64 random bodies of the batch against the
    fp64 oracle run on just those bodies, both pose surfaces."""
    B = 4096
    m = _lib.MODES[mode]
    betas, pose_aa, trans, _ = make_inputs(B, 31)
    pick = torch.randperm(B, generator=torch.Generator().manual_seed(32))[:64]
    pick[:4] = torch.tensor([0, 127, 128, 4095])
    d = lambda x: x.to(dev)  # noqa: E731
    for axis_angle in (True, False):
        pose = pose_aa if axis_angle else rotmats_of(pose_aa)
        v, j, _ = engine.forward(d(betas), d(pose), d(trans), None, axis_angle=axis_angle, mode=m)
        ref = oracle64.forward_flat(betas[pick].double(), pose[pick].double(), trans[pick].double(), pose2rot=axis_angle)
        ev = (v[pick.to(dev)].cpu().double() - ref.vertices).abs().max().item()
        ej = (j[pick.to(dev)].cpu().double() - ref.joints).abs().max().item()
        print("full-size forward errors vs fp64 oracle, 64 bodies (vertices, joints) [m]:", mode, axis_angle, ev, ej)
        assert ev < POS_TOL[mode] and ej < POS_TOL[mode]


@pytest.mark.parametrize("tree", ["chain", "bushy"])
@pytest.mark.parametrize("axis_angle", [False, True])
def test_other_kinematic_trees(synthetic_model, dev, tree, axis_angle):
    """The pose kernels walk the tree level by level (csrc/pose.cu P3, ChainTables::order / level_ptr): a 24-joint
    chain (24 levels of one joint) and a tree where joints have up to four children (4 levels), forward and backward
    against the fp64 oracle."""
    model = dict(synthetic_model)
    if tree == "chain":
        parents = np.arange(-1, 23)
    else:
        parents = np.array([-1, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 5, 5, 5, 5, 9, 9])
    model["parents"] = parents.astype(np.asarray(synthetic_model["parents"]).dtype)
    eng = SMPLEngine(model, dev)
    orc = O.SMPLOracle(model, dtype=torch.float64)
    B = 37
    betas, pose_aa, trans, cam = make_inputs(B, 77)
    pose_aa = pose_aa * 0.5                                   # a 24-deep chain compounds the rotations
    pose = pose_aa if axis_angle else rotmats_of(pose_aa)
    g = torch.Generator().manual_seed(78)
    dV, dJ, dJ2 = torch.randn(B, 6890, 3, generator=g), torch.randn(B, 90, 3, generator=g), torch.randn(B, 90, 2, generator=g)
    d = lambda x: x.to(dev)  # noqa: E731
    m = _lib.MODES["fp32"]
    out = eng.forward(d(betas), d(pose), d(trans), d(cam), axis_angle=axis_angle, mode=m, save=True)
    ref = orc.forward_flat(betas.double(), pose.double(), trans.double(), pose2rot=axis_angle)
    scale = max(1.0, ref.vertices.abs().max().item())
    assert (out[0].cpu().double() - ref.vertices).abs().max().item() < POS_TOL["fp32"] * scale
    assert (out[1].cpu().double() - ref.joints).abs().max().item() < POS_TOL["fp32"] * scale
    rb, rp, rt, rc = _oracle_grads(orc, betas, pose, trans, cam, dV, dJ, dJ2, axis_angle)
    for saved in (out[3], None):
        gb, gp, gt, gc = eng.backward(d(betas), d(pose), d(trans), d(cam), out[1], d(dV), d(dJ), d(dJ2),
                                      axis_angle=axis_angle, mode=m, saved=saved)
        errs = (_rel(gb.cpu().double(), rb), _rel(gp.cpu().double().reshape(rp.shape), rp), _rel(gt.cpu().double(), rt),
                _rel(gc.cpu().double(), rc))
        assert max(errs) < GRAD_TOL["fp32"], errs


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_wide_statistics_model_parity(wide_model, dev, mode):
    """The 'wide' synthetic model (H36M / COCO-plus regressor rows over 6-10 mesh parts -> twice the virtual joint
    rows; skinning rows with 1-3 influences): forward and backward against the fp64 oracle at a ragged batch, and
    a 4096-body batch against the same bodies computed in small batches."""
    eng = SMPLEngine(wide_model, dev)
    orc = O.SMPLOracle(wide_model, dtype=torch.float64)
    m = _lib.MODES[mode]
    B = 70
    betas, pose_aa, trans, cam = make_inputs(B, 41)
    rot = rotmats_of(pose_aa)
    g = torch.Generator().manual_seed(42)
    dV, dJ, dJ2 = torch.randn(B, 6890, 3, generator=g), torch.randn(B, 90, 3, generator=g), torch.randn(B, 90, 2, generator=g)
    d = lambda x: x.to(dev)  # noqa: E731
    out = eng.forward(d(betas), d(rot), d(trans), d(cam), mode=m, save=True)
    ref = orc.forward_flat(betas.double(), rot.double(), trans.double(), pose2rot=False)
    assert (out[0].cpu().double() - ref.vertices).abs().max().item() < POS_TOL[mode]
    assert (out[1].cpu().double() - ref.joints).abs().max().item() < POS_TOL[mode]
    rb, rp, rt, rc = _oracle_grads(orc, betas, rot, trans, cam, dV, dJ, dJ2, False)
    for saved in (out[3], None):
        gb, gp, gt, gc = eng.backward(d(betas), d(rot), d(trans), d(cam), out[1], d(dV), d(dJ), d(dJ2), mode=m, saved=saved)
        errs = (_rel(gb.cpu().double(), rb), _rel(gp.cpu().double().reshape(rp.shape), rp), _rel(gt.cpu().double(), rt),
                _rel(gc.cpu().double(), rc))
        assert max(errs) < GRAD_TOL[mode], errs
    # production size: the same body inside a 4096 batch and inside a small batch
    B2 = 4096
    betas2, pose2, trans2, _ = make_inputs(B2, 43)
    v, j, _ = eng.forward(d(betas2), d(pose2), d(trans2), None, axis_angle=True, mode=m)
    for i in (0, 2500, 4095):
        vi, ji, _ = eng.forward(d(betas2[i:i + 1]), d(pose2[i:i + 1]), d(trans2[i:i + 1]), None, axis_angle=True, mode=m)
        assert torch.equal(vi[0], v[i]) and torch.equal(ji[0], j[i])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_backward_full_size_vs_oracle(engine, oracle64, dev, mode):
    """BASELINE.json config 2 size (B = 4096, the CTA-pair GEMMs with their production split-K counts): the
    gradients of a handful of bodies spread over the batch against the fp64 oracle run on just those bodies
    (bodies are independent, so the oracle does not need the other 4090)."""
    B = 4096
    m = _lib.MODES[mode]
    betas, pose_aa, trans, cam = make_inputs(B, 21)
    pick = torch.tensor([0, 1, 127, 128, 2049, 4095])
    g = torch.Generator().manual_seed(22)
    dVs = torch.randn(len(pick), 6890, 3, generator=g)
    dJs = torch.randn(len(pick), 90, 3, generator=g)
    dV = torch.zeros(B, 6890, 3)
    dJ = torch.zeros(B, 90, 3)
    dV[pick], dJ[pick] = dVs, dJs
    d = lambda x: x.to(dev)  # noqa: E731
    gb, gp, gt, _ = engine.backward(d(betas), d(pose_aa), d(trans), None, None, d(dV), d(dJ), None,
                                    axis_angle=True, mode=m)
    rb, rp, rt, _ = _oracle_grads(oracle64, betas[pick], pose_aa[pick], trans[pick], None, dVs, dJs, None, True)
    tol = GRAD_TOL[mode]
    errs = (_rel(gb[pick.to(dev)].cpu().double(), rb), _rel(gp[pick.to(dev)].cpu().double(), rp),
            _rel(gt[pick.to(dev)].cpu().double(), rt))
    print("full-size gradient errors vs fp64 oracle (betas, pose, transl):", errs)
    assert max(errs) < tol
    # bodies whose upstream gradient is zero get exactly zero
    others = torch.ones(B, dtype=torch.bool)
    others[pick] = False
    assert gb[others.to(dev)].abs().max().item() == 0.0 and gp[others.to(dev)].abs().max().item() == 0.0


@pytest.mark.parametrize("B", [1, 37, 130, 300, 541])
def test_no_write_outside_caller_buffers(engine, dev, monkeypatch, B):
    """Every buffer the host side hands to the C-ABI (outputs, gradients, workspace, saved-for-backward) is
    allocated between two sentinel-filled guard bands; ragged batches (not multiples of the 32-body group or
    the 128-body GEMM tile) must leave every band untouched in all three modes."""
    GUARD = 4096                                   # bytes on each side; keeps the 512-byte alignment torch gives
    real_empty = torch.empty
    bands = []

    def guarded_empty(*size, dtype=torch.float32, device=None, **kw):
        shape = tuple(size[0]) if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)) else tuple(size)
        if device is None or torch.device(device).type != "cuda":
            return real_empty(shape, dtype=dtype, device=device, **kw)
        item = torch.empty((), dtype=dtype).element_size()
        n = 1
        for s in shape:
            n *= int(s)
        pad = (-(n * item)) % 512                  # round the payload up so the upper band starts 512-aligned
        raw = real_empty(GUARD + n * item + pad + GUARD, dtype=torch.uint8, device=device)
        raw.fill_(0xA5)
        bands.append((raw, GUARD, GUARD + n * item))
        return raw[GUARD:GUARD + n * item].view(dtype).view(shape)

    monkeypatch.setattr(torch, "empty", guarded_empty)
    engine._ws.clear()                             # force fresh (guarded) workspaces
    betas, pose_aa, trans, cam = (x.to(dev) for x in make_inputs(B, 300 + B))
    g = torch.Generator().manual_seed(B)
    dV = torch.randn(B, 6890, 3, generator=g).to(dev)
    dJ = torch.randn(B, 90, 3, generator=g).to(dev)
    dJ2 = torch.randn(B, 90, 2, generator=g).to(dev)
    for mode in MODES:
        m = _lib.MODES[mode]
        out = engine.forward(betas, pose_aa, trans, cam, axis_angle=True, mode=m, save=True)
        engine.backward(betas, pose_aa, trans, cam, out[1], dV, dJ, dJ2, axis_angle=True, mode=m, saved=out[3])
        engine.backward(betas, pose_aa, trans, cam, out[1], dV, dJ, dJ2, axis_angle=True, mode=m)
        engine.forward(betas, pose_aa, None, None, axis_angle=True, mode=m, want_vertices=False)
        engine.forward(betas, pose_aa, trans, cam, axis_angle=True, mode=m)      # forward-only: the fused kernel
    torch.cuda.synchronize(dev)
    monkeypatch.setattr(torch, "empty", real_empty)
    engine._ws.clear()
    assert len(bands) >= 10
    for raw, lo, hi in bands:
        assert bool((raw[:lo] == 0xA5).all()), "write below a caller buffer"
        assert bool((raw[hi:] == 0xA5).all()), "write above a caller buffer"


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B", [515, 700, 1300])
def test_fused_forward_equals_two_kernel_forward(engine, dev, mode, B):
    """Forward-only calls run the blend GEMM with the skinning in its epilogue (csrc/fused_fwd.cu); calls that keep the
    forward products run blend GEMM + skinning kernel.  Same MMAs in the same K order, same skinning arithmetic: the
    vertices and joints must agree bit for bit (ragged batches over several CTA pairs; calls below 512 bodies run the
    two kernels either way)."""
    betas, pose, trans, _ = make_inputs(B, 900 + B)
    rot = rotmats_of(pose)
    b, r, t = betas.to(dev), rot.to(dev), trans.to(dev)
    v0, j0, _ = engine.forward(b, r, t, None, mode=_lib.MODES[mode])[:3]                  # fused
    v1, j1, _, _ = engine.forward(b, r, t, None, mode=_lib.MODES[mode], save=True)         # two kernels
    torch.cuda.synchronize()
    assert torch.equal(v0, v1) and torch.equal(j0, j1)


def test_forward_only_wider_slab_than_worklist(engine, dev):
    """A forward-only call (the fused forward) asking for a slab wider than the forward GEMM's work list holds
    (40960 bodies) runs at the widest slab and matches the default slab bit for bit."""
    B = 41088
    betas, pose, trans, _ = make_inputs(B, 41)
    b, p, t = betas.to(dev), pose.to(dev), trans.to(dev)
    v0, j0, _ = engine.forward(b, p, t, None, axis_angle=True)[:3]
    v1, j1, _ = engine.forward(b, p, t, None, axis_angle=True, slab=65536)[:3]
    torch.cuda.synchronize()
    assert torch.equal(v0, v1) and torch.equal(j0, j1)
