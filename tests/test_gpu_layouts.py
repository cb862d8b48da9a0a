"""GPU tests (run on the B200 box with -m gpu) of the SMPL forward and backward where the kernels leave their vector
paths: caller buffers that are only 4- or 8-byte aligned, and meshes with other vertex counts and fewer output joints.

- The pose kernels stage the pose rows with 16-byte loads only when `pose` is 16-byte aligned; the skinning kernels
  and the fused forward move vertex and vertex-gradient rows in 8-byte pieces only when V is even and the buffer is
  8-byte aligned.  Otherwise they copy element by element.  The results must not depend on the path: forwards are
  bit-identical to the aligned call, backwards agree with it up to the order of the fp32 REDs that accumulate dL/dA.
- The public surfaces hand such pointers to the kernels: a (1, 85) parameter row sliced into betas / pose / transl is
  contiguous with its pose 8 bytes past a 16-byte boundary, and `torch.cat` hands its inputs' gradients back as
  slices at their element offset.
- Other meshes (tests/test_layouts_host.py::derive_model): vertex counts with a ragged or no vertex-tile tail, odd
  counts, odd and even GEMM row-tile counts, and models with 54, 45 or 24 output joints; a 24-joint model has no
  virtual joint rows, so a joints-only call blends an empty row range.
- The multi-task loss with an odd number of vertex elements and with vertices that are only 4-byte aligned.

Tolerances are those of tests/test_gpu_parity.py (on the derived meshes see `mesh_grad_tol`); the fp64 oracle runs
on a few bodies of each batch (bodies are independent)."""
import ctypes

import pytest
import torch

from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib, config, regressor
from soccerplayershapepose_b200.engine import SMPLEngine
from soccerplayershapepose_b200.smpl import SMPL, SMPLLayer
from test_layouts_host import REGRESSORS, derive_model

pytestmark = pytest.mark.gpu

POS_TOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-4, "bf16_fast": 1e-4}
GRAD_TOL = {"fp32": 1e-4, "fp32_simt": 1e-4, "bf16": 1e-4, "bf16_fast": 5e-3}
MODES = ["fp32_simt", "fp32", "bf16", "bf16_fast"]
OFFSETS = (4, 8, 12)
GUARD = 1024                  # bytes of sentinel on each side of an offset buffer (a multiple of 16)
SENTINEL = 0xA5
# same call, other load path: only the order of the fp32 REDs that accumulate dL/dA and dL/dtransl may differ (the
# gradient of one body's translation sums ~7000 vertex terms that way: 1.2e-6 measured at B = 1)
RED_TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def engine(synthetic_model, dev):
    return SMPLEngine(synthetic_model, dev)


@pytest.fixture(scope="module")
def oracle64(synthetic_model):
    return O.SMPLOracle(synthetic_model, dtype=torch.float64)


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def offset_tensor(values, byte_offset, guard=GUARD):
    """A contiguous CUDA copy of `values` that starts `byte_offset` bytes past a 512-byte boundary (so data_ptr() % 16
    == byte_offset % 16), carved out of a larger uint8 allocation between two sentinel-filled guard bands;
    `assert_guards_intact` checks the bands."""
    if values is None:
        return None
    assert guard % 16 == 0 and 0 <= byte_offset < guard
    values = values.contiguous()
    nbytes = values.numel() * values.element_size()
    raw = torch.full((guard + byte_offset + nbytes + guard,), SENTINEL, dtype=torch.uint8, device=values.device)
    lo = guard + byte_offset
    t = raw[lo:lo + nbytes].view(values.dtype).view(values.shape)
    t.copy_(values)
    assert raw.data_ptr() % 512 == 0 and t.is_contiguous() and t.data_ptr() == raw.data_ptr() + lo
    t._guard_band = (raw, lo, lo + nbytes)
    return t


def offset_buffer(nbytes, byte_offset, device):
    """Scratch bytes (workspace, saved-for-backward) of exactly `nbytes` at `byte_offset` between guard bands."""
    return offset_tensor(torch.empty(nbytes, dtype=torch.uint8, device=device), byte_offset)


def assert_guards_intact(*tensors):
    torch.cuda.synchronize()
    for t in tensors:
        if t is None:
            continue
        raw, lo, hi = t._guard_band
        assert bool((raw[:lo] == SENTINEL).all()), "write below a caller buffer"
        assert bool((raw[hi:] == SENTINEL).all()), "write above a caller buffer"


def make_inputs(B, seed, nb=10):
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, nb, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    trans = torch.rand(B, 3, generator=g) * 2 - 1
    cam = torch.stack([torch.rand(B, generator=g) * 0.6 + 0.6, torch.rand(B, generator=g) * 0.4 - 0.2,
                       torch.rand(B, generator=g) * 0.4 - 0.2], 1)
    return betas, pose, trans, cam


def make_grads(B, V, NJ, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, V, 3, generator=g), torch.randn(B, NJ, 3, generator=g), torch.randn(B, NJ, 2, generator=g)


def rotmats_of(pose):
    return O.batch_rodrigues(pose.double().reshape(-1, 3)).reshape(pose.shape[0], 216).float()


def picked(B):
    return sorted({0, B // 2, B - 1})


def _oracle_grads(orc, betas, pose, trans, cam, dV, dJ, dJ2, axis_angle):
    b = betas.double().requires_grad_(True)
    p = pose.double().requires_grad_(True)
    t = trans.double().requires_grad_(True)
    c = cam.double().requires_grad_(True)
    out = orc.forward_flat(b, p, t, pose2rot=axis_angle)
    loss = (out.joints * dJ.double()).sum() + (O.orthographic_project(out.joints, c) * dJ2.double()).sum()
    if dV is not None:
        loss = loss + (out.vertices * dV.double()).sum()
    loss.backward()
    return b.grad, p.grad, t.grad, c.grad


def _check_forward(orc, v, j, j2d, betas, pose, trans, cam, axis_angle, pick, tol):
    ref = orc.forward_flat(betas[pick].double(), pose[pick].double(), trans[pick].double(), pose2rot=axis_angle)
    idx = torch.tensor(pick, device=j.device)
    if v is not None:
        ev = (v[idx].cpu().double() - ref.vertices).abs().max().item()
        assert ev < tol, ev
    ej = (j[idx].cpu().double() - ref.joints).abs().max().item()
    assert ej < tol, ej
    if j2d is not None:
        ref2d = O.orthographic_project(ref.joints, cam[pick].double())
        assert (j2d[idx].cpu().double() - ref2d).abs().max().item() < 2 * tol


def _check_grads(got, ref, pick, tol):
    idx = torch.tensor(pick, device=got[0].device)
    errs = [_rel(g[idx].cpu().double().reshape(r.shape), r) for g, r in zip(got, ref)]
    assert max(errs) < tol, errs


# ---- 1. unaligned inputs ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("axis_angle", [False, True])
@pytest.mark.parametrize("B", [1, 37, 515])
@pytest.mark.parametrize("mode", MODES)
def test_unaligned_inputs(engine, oracle64, dev, mode, B, axis_angle):
    """betas / pose / transl / cam at 4, 8 and 12 bytes past a 16-byte boundary (all four, or pose alone): forwards
    (two-kernel with save=True, and forward-only, the fused kernel at B = 515) bit-identical to the aligned call;
    backwards with the upstream gradients and joints at the same offsets, with and without the saved products, equal
    to the aligned call up to the RED order and to the fp64 oracle."""
    m = _lib.MODES[mode]
    betas, pose_aa, trans, cam = make_inputs(B, 500 + B)
    pose = pose_aa if axis_angle else rotmats_of(pose_aa)
    dV, dJ, dJ2 = make_grads(B, 6890, 90, 600 + B)
    pick = picked(B)
    kw = dict(axis_angle=axis_angle, mode=m)
    A = [x.to(dev) for x in (betas, pose, trans, cam)]
    Gd = [x.to(dev) for x in (dV, dJ, dJ2)]
    v0, j0, p0, s0 = engine.forward(*A, save=True, **kw)
    f0 = engine.forward(*A, **kw)
    _check_forward(oracle64, v0, j0, p0, betas, pose, trans, cam, axis_angle, pick, POS_TOL[mode])
    ref = _oracle_grads(oracle64, betas[pick], pose[pick], trans[pick], cam[pick], dV[pick], dJ[pick], dJ2[pick],
                        axis_angle)
    g_saved = engine.backward(*A, j0, *Gd, saved=s0, **kw)
    g_plain = engine.backward(*A, j0, *Gd, **kw)
    _check_grads(g_saved, ref, pick, GRAD_TOL[mode])
    _check_grads(g_plain, ref, pick, GRAD_TOL[mode])
    for off in OFFSETS:
        for which in ("all", "pose"):
            U = [offset_tensor(x, off) if which == "all" or i == 1 else x for i, x in enumerate(A)]
            assert U[1].data_ptr() % 16 == off
            v, j, p, s = engine.forward(*U, save=True, **kw)
            assert torch.equal(v, v0) and torch.equal(j, j0) and torch.equal(p, p0)
            f = engine.forward(*U, **kw)
            assert all(torch.equal(a, b) for a, b in zip(f, f0))
            J = offset_tensor(j0, off)
            G = [offset_tensor(x, off) for x in Gd]
            for saved, want in ((s, g_saved), (None, g_plain)):
                got = engine.backward(*U, J, *G, saved=saved, **kw)
                for a, b in zip(got, want):
                    assert _rel(a, b) < RED_TOL
                _check_grads(got, ref, pick, GRAD_TOL[mode])
            assert_guards_intact(*[u for u, a in zip(U, A) if u is not a], J, *G)


# ---- 2. unaligned outputs and scratch through the C-ABI ------------------------------------------------------------------
def _cabi_forward(eng, B, mode, A, verts, joints, j2d, ws, saved):
    args = _lib.ForwardArgs(batch=B, mode=mode, pose_is_axis_angle=1, slab_bodies=0,
                            betas=A[0].data_ptr(), pose=A[1].data_ptr(), transl=A[2].data_ptr(), cam=A[3].data_ptr(),
                            vertices=verts.data_ptr(), joints=joints.data_ptr(), joints2d=j2d.data_ptr(),
                            workspace=ws.data_ptr(), workspace_bytes=ws.numel(),
                            saved=None if saved is None else saved.data_ptr(),
                            saved_bytes=0 if saved is None else saved.numel())
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    _lib.check(eng.lib.b200smpl_forward(eng.handle, ctypes.byref(args), ctypes.c_void_p(stream)), "b200smpl_forward")


def _cabi_backward(eng, B, mode, A, joints, G, outs, ws, saved):
    args = _lib.BackwardArgs(batch=B, mode=mode, pose_is_axis_angle=1, slab_bodies=0,
                             betas=A[0].data_ptr(), pose=A[1].data_ptr(), transl=A[2].data_ptr(), cam=A[3].data_ptr(),
                             joints=joints.data_ptr(), grad_vertices=G[0].data_ptr(), grad_joints=G[1].data_ptr(),
                             grad_joints2d=G[2].data_ptr(), grad_betas=outs[0].data_ptr(), grad_pose=outs[1].data_ptr(),
                             grad_transl=outs[2].data_ptr(), grad_cam=outs[3].data_ptr(),
                             workspace=ws.data_ptr(), workspace_bytes=ws.numel(),
                             saved=None if saved is None else saved.data_ptr(),
                             saved_bytes=0 if saved is None else saved.numel())
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    _lib.check(eng.lib.b200smpl_backward(eng.handle, ctypes.byref(args), ctypes.c_void_p(stream)), "b200smpl_backward")


@pytest.mark.parametrize("B", [37, 300, 515, 1300])
@pytest.mark.parametrize("mode", MODES)
def test_unaligned_outputs_and_scratch(engine, dev, mode, B):
    """vertices / joints / joints2d and the four gradient outputs at 4, 8 and 12 bytes past a 16-byte boundary,
    workspace and saved buffer at 4, 512 and 1020 bytes and exactly the size the library asks for.  B = 37 and 300 keep
    the forward products (two kernels); B = 515 and 1300 are forward-only (the fused blend + skinning kernel).  Results
    equal the aligned call; no byte outside a buffer changes."""
    m = _lib.MODES[mode]
    lib, h = engine.lib, engine.handle
    save = B < 512
    betas, pose, trans, cam = make_inputs(B, 700 + B)
    dV, dJ, dJ2 = make_grads(B, 6890, 90, 800 + B)
    A = [x.to(dev) for x in (betas, pose, trans, cam)]
    Gd = [x.to(dev) for x in (dV, dJ, dJ2)]
    ref = engine.forward(*A, axis_angle=True, mode=m, save=save)
    ref_g = engine.backward(*A, ref[1], *Gd, axis_angle=True, mode=m, saved=ref[3] if save else None)
    for off, soff in zip(OFFSETS, (4, 512, 1020)):
        verts = offset_tensor(torch.empty(B, 6890, 3, device=dev), off)
        joints = offset_tensor(torch.empty(B, 90, 3, device=dev), off)
        j2d = offset_tensor(torch.empty(B, 90, 2, device=dev), off)
        ws_f = offset_buffer(lib.b200smpl_forward_workspace_bytes(h, B, m, 0), soff, dev)
        saved = offset_buffer(lib.b200smpl_saved_bytes(h, B, 0), soff, dev) if save else None
        _cabi_forward(engine, B, m, A, verts, joints, j2d, ws_f, saved)
        assert torch.equal(verts, ref[0]) and torch.equal(joints, ref[1]) and torch.equal(j2d, ref[2])
        G = [offset_tensor(x, off) for x in Gd]
        outs = [offset_tensor(torch.empty(B, n, device=dev), off) for n in (10, 72, 3, 3)]
        ws_b = offset_buffer(lib.b200smpl_backward_workspace_bytes(h, B, m, 0), soff, dev)
        _cabi_backward(engine, B, m, A, joints, G, outs, ws_b, saved)
        for a, b in zip(outs, ref_g):
            assert _rel(a, b) < RED_TOL
        assert_guards_intact(verts, joints, j2d, ws_f, saved, *G, *outs, ws_b)


# ---- 3. the public surfaces that produce such pointers ---------------------------------------------------------------------
def test_public_surfaces_hand_over_unaligned_pointers(synthetic_model, oracle64, dev):
    """B = 1 with betas / pose / transl sliced from one (1, 85) parameter row (the pose starts 40 bytes in: 8 mod 16,
    so both pose kernels stage it element by element), through `SMPLLayer` and the keyword `SMPL` surface; and a loss
    that hands the vertex gradient back at storage offset 3 (a `torch.cat` of 3 values and the flattened vertices), so
    the skinning backward reads it element by element.  Against the fp64 oracle and against aligned copies."""
    layer = SMPLLayer(synthetic_model).to(dev)
    smpl = SMPL(synthetic_model).to(dev)
    betas, pose, trans, _ = make_inputs(1, 31)
    row = torch.cat([betas, pose, trans], 1)
    dV, dJ, _ = make_grads(1, 6890, 90, 32)
    dVd, dJd = dV.to(dev), dJ.to(dev)

    params = row.to(dev).requires_grad_(True)
    b, p, t = params[:, :10], params[:, 10:82], params[:, 82:85]
    assert p.is_contiguous() and p.contiguous().data_ptr() == p.data_ptr() and p.data_ptr() % 16 == 8
    v, j = layer(b, p, t)
    torch.autograd.backward([v, j], [dVd, dJd])

    al = [x.detach().clone().requires_grad_(True) for x in (b, p, t)]
    assert all(x.data_ptr() % 16 == 0 for x in al)
    va, ja = layer(*al)
    torch.autograd.backward([va, ja], [dVd, dJd])
    assert torch.equal(v, va) and torch.equal(j, ja)
    g_al = torch.cat([x.grad for x in al], 1)
    assert _rel(params.grad, g_al) < RED_TOL

    b64, p64, t64 = (x.double().requires_grad_(True) for x in (betas, pose, trans))
    ref = oracle64.forward_flat(b64, p64, t64, pose2rot=True)
    ((ref.vertices * dV.double()).sum() + (ref.joints * dJ.double()).sum()).backward()
    assert (v.detach().cpu().double() - ref.vertices).abs().max().item() < POS_TOL["fp32"]
    assert (j.detach().cpu().double() - ref.joints).abs().max().item() < POS_TOL["fp32"]
    g64 = torch.cat([b64.grad, p64.grad, t64.grad], 1)
    for sl in (slice(0, 10), slice(10, 82), slice(82, 85)):
        assert _rel(params.grad[:, sl].cpu().double(), g64[:, sl]) < GRAD_TOL["fp32"]

    # keyword surface: SMPL.forward concatenates global_orient and body_pose into a fresh (aligned) tensor
    params_k = row.to(dev).requires_grad_(True)
    out = smpl(betas=params_k[:, :10], global_orient=params_k[:, 10:13], body_pose=params_k[:, 13:82],
               transl=params_k[:, 82:85], pose2rot=True)
    assert torch.equal(out.vertices, v) and torch.equal(out.joints, j)
    torch.autograd.backward([out.vertices, out.joints], [dVd, dJd])
    assert _rel(params_k.grad, g_al) < RED_TOL

    # vertex gradient at storage offset 3 (12 bytes: 4 mod 8)
    params_c = row.to(dev).requires_grad_(True)
    vc, jc = layer(params_c[:, :10], params_c[:, 10:82], params_c[:, 82:85])
    seen = []
    vc.register_hook(lambda g: seen.append((g.storage_offset(), g.is_contiguous(), g.data_ptr() % 8)))
    x3 = torch.zeros(3, device=dev, requires_grad=True)
    w = torch.cat([torch.zeros(3), dV.reshape(-1)]).to(dev)
    ((torch.cat([x3, vc.reshape(-1)]) * w).sum() + (jc * dJd).sum()).backward()
    assert seen == [(3, True, 4)]
    assert _rel(params_c.grad, g_al) < RED_TOL
    for sl in (slice(0, 10), slice(10, 82), slice(82, 85)):
        assert _rel(params_c.grad[:, sl].cpu().double(), g64[:, sl]) < GRAD_TOL["fp32"]


# ---- 4. other mesh sizes -------------------------------------------------------------------------------------------------
MESHES = [(V, REGRESSORS, True) for V in (1, 33, 129, 1001, 6889, 6912, 10475)] + [
    (33, (), True), (33, (), False), (6889, (), True), (6889, (), False)]
CASES = [(spec, mode) for spec in MESHES for mode in (MODES if spec[0] in (33, 6889) else ["fp32", "bf16"])]
_ENGINES = {}
_ORACLES = {}


def mesh_grad_tol(mode, V):
    """GRAD_TOL, except where the precision of a bf16 mode shows through on a derived mesh.  The bf16 modes blend the
    pose correctives from single-bf16 model rows (vertex error up to POS_TOL = 1e-4 m); the pose gradient is built
    from those vertices, and with a few hundred vertices or fewer the rounding no longer averages out (grad_pose
    measured on a B200: up to 7.6e-4 at V = 1, 1.7e-4 at V = 33, 1.03e-4 at V = 129, below 1e-4 from V = 1001 on;
    the fp32 modes stay below 7e-6 on the same bodies).  bf16_fast (single-product gradient GEMM, 5e-3 on the SMPL mesh) measured
    5.1e-3 on grad_betas of the 45-joint model."""
    if mode == "bf16" and V < 1000:
        return 1e-3
    if mode == "bf16_fast":
        return 1e-2
    return GRAD_TOL[mode]


def _njout(spec):
    return 24 + 21 * spec[2] + sum({"extra": 9, "cocoplus": 19, "h36m": 17}[k] for k in spec[1])


def _mesh_id(case):
    spec = case[0] if isinstance(case[0], tuple) else case
    return "V{}-{}j".format(spec[0], _njout(spec)) + ("-" + case[1] if isinstance(case[0], tuple) else "")


def _derived(synthetic_model, dev, spec):
    if spec not in _ENGINES:
        model = derive_model(synthetic_model, *spec)
        _ENGINES[spec] = SMPLEngine(model, dev)
        _ORACLES[spec] = O.SMPLOracle(model, dtype=torch.float64)
    return _ENGINES[spec], _ORACLES[spec]


@pytest.mark.parametrize("case", CASES, ids=_mesh_id)
def test_other_mesh_sizes(synthetic_model, dev, case):
    """Forward and backward on derived meshes against the fp64 oracle at B = 1, 37 and 515: the two-kernel forward
    (save=True), the forward-only call (the fused kernel at B = 515, bit-equal to the two kernels), backwards with and
    without the saved products, and joints-only forwards (same joints as the full call) and backwards."""
    spec, mode = case
    eng, orc = _derived(synthetic_model, dev, spec)
    V, NJ = spec[0], _njout(spec)
    assert eng.num_verts == V and eng.num_joints_out == NJ
    m = _lib.MODES[mode]
    tol, gtol = POS_TOL[mode], mesh_grad_tol(mode, V)
    for B in (1, 37, 515):
        betas, pose, trans, cam = make_inputs(B, 40 + B + V)
        dV, dJ, dJ2 = make_grads(B, V, NJ, 50 + B + V)
        pick = picked(B)
        A = [x.to(dev) for x in (betas, pose, trans, cam)]
        Gd = [x.to(dev) for x in (dV, dJ, dJ2)]
        kw = dict(axis_angle=True, mode=m)
        v, j, p, s = eng.forward(*A, save=True, **kw)
        assert v.shape == (B, V, 3) and j.shape == (B, NJ, 3)
        _check_forward(orc, v, j, p, betas, pose, trans, cam, True, pick, tol)
        f = eng.forward(*A, **kw)
        assert all(torch.equal(a, b) for a, b in zip(f, (v, j, p)))
        ref = _oracle_grads(orc, betas[pick], pose[pick], trans[pick], cam[pick], dV[pick], dJ[pick], dJ2[pick], True)
        for saved in (s, None):
            _check_grads(eng.backward(*A, j, *Gd, saved=saved, **kw), ref, pick, gtol)
        # joints only: the blend GEMMs run over the virtual joint rows alone (none for a 24-joint model)
        for save in (False, True):
            o = eng.forward(*A, want_vertices=False, save=save, **kw)
            assert o[0] is None and torch.equal(o[1], j) and torch.equal(o[2], p)
        ref_j = _oracle_grads(orc, betas[pick], pose[pick], trans[pick], cam[pick], None, dJ[pick], dJ2[pick], True)
        for saved in (o[3], None):
            _check_grads(eng.backward(*A, j, None, Gd[1], Gd[2], saved=saved, **kw), ref_j, pick, gtol)


ODD_MESHES = [spec for spec in MESHES if spec[0] % 2]


@pytest.mark.parametrize("spec", ODD_MESHES, ids=_mesh_id)
@pytest.mark.parametrize("B", [37, 300])
def test_no_write_outside_caller_buffers_odd_meshes(synthetic_model, dev, monkeypatch, spec, B):
    """Odd vertex counts (element-wise row copies in the skinning kernels) at ragged batches: every buffer the host
    side hands to the C-ABI sits between two sentinel-filled guard bands, in all four modes."""
    eng, _ = _derived(synthetic_model, dev, spec)
    V, NJ = spec[0], _njout(spec)
    real_empty = torch.empty
    bands = []

    def guarded_empty(*size, dtype=torch.float32, device=None, **kw):
        shape = tuple(size[0]) if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)) else tuple(size)
        if device is None or torch.device(device).type != "cuda":
            return real_empty(shape, dtype=dtype, device=device, **kw)
        t = offset_tensor(real_empty(shape, dtype=dtype, device=device), 0, guard=4096)
        bands.append(t)
        return t

    A = [x.to(dev) for x in make_inputs(B, 900 + B)]
    Gd = [x.to(dev) for x in make_grads(B, V, NJ, 901 + B)]
    monkeypatch.setattr(torch, "empty", guarded_empty)
    eng._ws.clear()
    for mode in MODES:
        kw = dict(axis_angle=True, mode=_lib.MODES[mode])
        out = eng.forward(*A, save=True, **kw)
        eng.backward(*A, out[1], *Gd, saved=out[3], **kw)
        eng.backward(*A, out[1], *Gd, **kw)
        eng.backward(*A, out[1], None, Gd[1], Gd[2], **kw)
        eng.forward(*A[:2], None, None, want_vertices=False, **kw)
        eng.forward(*A, **kw)
    monkeypatch.setattr(torch, "empty", real_empty)
    eng._ws.clear()
    assert len(bands) >= 10
    assert_guards_intact(*bands)


# ---- 5. multi-task loss ---------------------------------------------------------------------------------------------
LOSSES = ("verts", "joints2D", "joints3D", "shape_params", "pose_params")
WEIGHTS = {"verts": 1.0, "joints2D": 0.1, "joints3D": 1.0, "shape_params": 0.1, "pose_params": 0.1}


@pytest.mark.parametrize("unaligned", ["none", "verts", "verts_label", "both"])
def test_multitask_loss_odd_vertex_count_and_unaligned_vertices(dev, unaligned):
    """B = 7, V = 49: B * V * 3 is odd, so the vertex term has a last element outside its 8-byte pieces; `verts` and
    `verts_label` also at 4 bytes past a 16-byte boundary (as a contiguous slice hands them over).  Loss, parts and
    every gradient against the eager criterion in float64 on the CPU (pinned to the reference class in
    tests/test_oracle.py) and fp64 autograd."""
    B, V = 7, 49
    assert B * V * 3 % 2 == 1
    g = torch.Generator().manual_seed(77)
    pred = {"verts": torch.randn(B, V, 3, generator=g), "joints": torch.randn(B, 90, 3, generator=g) * 0.5,
            "cam": torch.stack([torch.rand(B, generator=g) * 0.4 + 0.7, torch.rand(B, generator=g) * 0.2 - 0.1,
                                torch.rand(B, generator=g) * 0.2 - 0.1], 1),
            "shape_params": torch.randn(B, 10, generator=g),
            "pose_params_rot_matrices": torch.randn(B, 24, 3, 3, generator=g)}
    # labels near the prediction (1 cm), so that the vertex term's last element weighs in the mean
    lab = {"verts": pred["verts"] + 0.01 * torch.randn(B, V, 3, generator=g),
           "joints2D": torch.rand(B, 17, 2, generator=g) * config.REGRESSOR_IMG_WH,
           "vis": torch.rand(B, 17, generator=g) > 0.3,
           "joints3D": torch.randn(B, 17, 3, generator=g) * 0.5,
           "shape_params": torch.randn(B, 10, generator=g),
           "pose_params_rot_matrices": torch.randn(B, 24, 3, 3, generator=g)}
    off_v = 4 if unaligned in ("verts", "both") else 0
    off_l = 4 if unaligned in ("verts_label", "both") else 0
    leaves = {k: x.to(dev).requires_grad_(True) for k, x in pred.items() if k != "verts"}
    leaves["verts"] = offset_tensor(pred["verts"].to(dev), off_v).requires_grad_(True)
    lab_d = {k: x.to(dev) for k, x in lab.items() if k != "verts"}
    lab_d["verts"] = offset_tensor(lab["verts"].to(dev), off_l)
    assert leaves["verts"].data_ptr() % 8 == off_v and lab_d["verts"].data_ptr() % 8 == off_l
    torch.manual_seed(0)
    crit = regressor.MultiTaskLoss(LOSSES, WEIGHTS).to(dev)
    loss, parts = crit.forward_fused(lab_d, leaves)
    (2.5 * loss).backward()
    assert_guards_intact(leaves["verts"], lab_d["verts"])

    crit64 = regressor.MultiTaskLoss(LOSSES, WEIGHTS).double()
    l64 = {k: x.double().requires_grad_(True) for k, x in pred.items()}
    o64 = dict(l64)
    o64["joints2D"] = O.undo_keypoint_normalisation(O.orthographic_project(l64["joints"], l64["cam"]), 512)[
        :, config.SMPL_TO_KPRCNN_MAP, :]
    o64["joints3D"] = l64["joints"][:, config.ALL_JOINTS_TO_COCO_MAP, :]
    lab64 = {k: (x.double() if x.dtype.is_floating_point else x) for k, x in lab.items()}
    ref, parts64 = crit64(lab64, o64)
    (2.5 * ref).backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item()))
    for name in LOSSES:
        assert abs(parts[name].item() - parts64[name].item()) < 1e-5 * max(1e-3, abs(parts64[name].item())), name
        gl, gl64 = getattr(crit, name + "_log_var").grad, getattr(crit64, name + "_log_var").grad
        assert abs(gl.item() - gl64.item()) < 1e-5 * max(1.0, abs(gl64.item())), name
    for k in pred:
        g64 = l64[k].grad
        err = (leaves[k].grad.cpu().double() - g64).abs().max().item()
        assert err < 2e-5 * g64.abs().max().item() + 1e-12, (k, err)
