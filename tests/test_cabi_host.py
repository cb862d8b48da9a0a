"""CPU-side tests of the C-ABI library (no GPU, no compute calls): it loads, exports every symbol
the header declares, refuses to compute without a device, and its HOST packing logic (blend
operand split, skinning plan, joint terms) reproduces the oracle when emulated in numpy."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import smpl_oracle as O
from soccerplayershapepose_b200 import _lib
from soccerplayershapepose_b200.engine import SMPLEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "b200smpl.h")).read()
    declared = set(re.findall(r"B200SMPL_API [\w\* ]+?(b200smpl_\w+)\(", header))
    assert len(declared) >= 18
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    assert _lib.load().b200smpl_abi_version() == 1


@pytest.fixture(scope="module")
def host_engine(synthetic_model):
    return SMPLEngine(synthetic_model, device=None)


def test_host_only_handle_refuses_compute(host_engine):
    lib = _lib.load()
    args = _lib.ForwardArgs(batch=1, mode=0)
    rc = lib.b200smpl_forward(host_engine.handle, ctypes.byref(args), None)
    assert rc == _lib.ERR_WORKSPACE or rc == _lib.ERR_CUDA
    args.workspace = 1
    rc = lib.b200smpl_forward(host_engine.handle, ctypes.byref(args), None)
    assert rc == _lib.ERR_CUDA and "no CPU fallback" in _lib.last_error()
    with pytest.raises(RuntimeError):
        host_engine.forward(torch.zeros(1, 10), torch.zeros(1, 216))


def test_model_validation_errors(synthetic_model):
    bad = dict(synthetic_model)
    bad["parents"] = np.array([-1] + [5] * 23)
    with pytest.raises(ValueError):
        SMPLEngine(bad, device=None)
    bad = dict(synthetic_model)
    w = synthetic_model["lbs_weights"].copy()
    w[0, :] = 1.0 / 24
    bad["lbs_weights"] = w
    with pytest.raises(ValueError, match="more than 4"):
        SMPLEngine(bad, device=None)


def test_chain_level_tables(host_engine, synthetic_model):
    """The pose kernels walk the kinematic tree one level at a time (csrc/pose.cu, P3): `chain_order` must list every
    joint once, sorted by depth, every parent on an earlier level than its child; `chain_level_ptr` delimits the
    levels (smplx kintree: 24 joints, 9 levels)."""
    parents = np.asarray(synthetic_model["parents"]).astype(int)
    depth = np.zeros(24, int)
    for j in range(1, 24):
        depth[j] = depth[parents[j]] + 1
    order = host_engine.debug_array("chain_order", np.int8).astype(int)
    ptr = host_engine.debug_array("chain_level_ptr", np.int8).astype(int)
    assert sorted(order.tolist()) == list(range(24))
    assert ptr[0] == 0 and ptr[-1] == 24 and np.all(np.diff(ptr) >= 0)
    nlev = depth.max() + 1
    assert nlev == 9
    for d in range(nlev):
        level = order[ptr[d]:ptr[d + 1]]
        assert len(level) > 0 and np.all(depth[level] == d)
        assert np.all(np.diff(level) > 0)                        # stable: joints of a level in index order
    assert np.all(ptr[nlev:] == 24)
    level_of = {int(j): int(depth[j]) for j in order}
    assert all(level_of[int(parents[j])] == level_of[j] - 1 for j in range(1, 24))


def _bf16_to_f32(u16):
    return (u16.astype(np.uint32) << 16).view(np.float32)


def _f32_to_bf16_rn(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    return r


def test_packed_model_emulation_matches_oracle(host_engine, synthetic_model):
    """Emulate the GPU dataflow in numpy from the PACKED arrays only and compare with the oracle."""
    _check_packed_emulation(host_engine, synthetic_model)


def test_packed_model_emulation_wide_statistics(wide_model):
    """The same on the 'wide' synthetic model: regressor rows spread over 6-10 mesh parts (twice the virtual joint
    rows) and skinning rows with 1-3 influences (VERDICT r01: the compact model may flatter the virtual-row trick)."""
    assert set(np.unique((wide_model["lbs_weights"] > 0).sum(1))) == {1, 2, 3, 4}
    eng = SMPLEngine(wide_model, device=None)
    assert eng.info.num_virtual_groups > 1000
    _check_packed_emulation(eng, wide_model)


def _check_packed_emulation(eng, model):
    info = eng.info
    V, n_pad, nq = info.num_verts, info.num_blend_rows_padded, info.num_virtual_groups
    nb, nf = 10, 217
    W32 = eng.debug_array("W32", np.float32).reshape(1 + nf, n_pad).astype(np.float64)
    vmeta = eng.debug_array("vmeta", np.uint32)
    vwts = eng.debug_array("vwts", np.float32).reshape(-1, 4).astype(np.float64)
    term_ptr = eng.debug_array("term_ptr", np.int32)
    term_joint = eng.debug_array("term_joint", np.uint8)
    term_qrow = eng.debug_array("term_qrow", np.int32)
    term_c = eng.debug_array("term_c", np.float32).astype(np.float64)
    Jt = eng.debug_array("Jt", np.float32).reshape(24, 3).astype(np.float64)
    Jsd = eng.debug_array("Jsd", np.float32).reshape(24, 3, nb).astype(np.float64)
    ntiles = len(vmeta) // 32
    n_virt0 = ntiles * 96
    assert info.num_blend_rows == n_virt0 + 3 * nq and n_pad % 128 == 0 and n_virt0 % 128 == 0

    gen = torch.Generator().manual_seed(3)
    betas = torch.randn(2, 10, generator=gen, dtype=torch.float64)
    pose = torch.randn(2, 72, generator=gen, dtype=torch.float64) * 0.3
    trans = torch.rand(2, 3, generator=gen, dtype=torch.float64)
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(2, 24, 3, 3)
    ref = O.SMPLOracle(model, dtype=torch.float64).forward_flat(betas, rot, trans, pose2rot=False)
    parents = np.asarray(model["parents"])

    for b in range(2):
        R = rot[b].numpy()
        beta = betas[b].numpy()
        feat = np.concatenate([beta, (R[1:] - np.eye(3)).reshape(-1)])
        vp = W32[0] + feat @ W32[1:]                                  # blend rows (real + virtual)
        # pose stage: rest joints from the folded regressor, chain, A
        Jr = Jt + Jsd @ beta
        G = np.zeros((24, 4, 4))
        for j in range(24):
            L = np.eye(4)
            L[:3, :3] = R[j]
            L[:3, 3] = Jr[j] if j == 0 else Jr[j] - Jr[parents[j]]
            G[j] = L if j == 0 else G[parents[j]] @ L
        A = G[:, :3, :].copy()
        A[:, :, 3] -= np.einsum("jrc,jc->jr", G[:, :3, :3], Jr)
        # skinning from the plan
        verts = np.zeros((V, 3))
        seen = np.zeros(V, bool)
        slots = [0, 0, 0, 0]
        for t in range(ntiles):
            for i in range(32):
                m = int(vmeta[t * 32 + i])
                if i == 0:
                    m |= 0xF << 20
                if not (m >> 29) & 1:
                    continue
                for s in range(4):
                    if (m >> (20 + s)) & 1:
                        slots[s] = (m >> (5 * s)) & 31
                    else:
                        assert slots[s] == (m >> (5 * s)) & 31      # plan is consistent
                v = t * 32 + ((m >> 24) & 31)
                p = np.append(vp[3 * v:3 * v + 3], 1.0)
                verts[v] = sum(vwts[t * 32 + i, s] * (A[slots[s]] @ p) for s in range(4)) + trans[b].numpy()
                assert not seen[v]
                seen[v] = True
        assert seen.all()
        np.testing.assert_allclose(verts, ref.vertices[b].numpy(), atol=2e-7)
        # joints from the terms
        joints = np.zeros((info.num_joints_out, 3))
        joints[:24] = G[:, :3, 3] + trans[b].numpy()
        for J in range(24, info.num_joints_out):
            acc = trans[b].numpy().copy()
            for k in range(term_ptr[J - 24], term_ptr[J - 24 + 1]):
                q = np.append(vp[term_qrow[k]:term_qrow[k] + 3], term_c[k])
                acc = acc + A[term_joint[k]] @ q
            joints[J] = acc
        np.testing.assert_allclose(joints, ref.joints[b].numpy(), atol=2e-7)
        # ... and from the virtual-tile plan the GPU kernels walk (32 q-groups per tile)
        qmeta = eng.debug_array("qmeta", np.uint32)
        qcoef = eng.debug_array("qcoef", np.float32).astype(np.float64)
        vt_j0 = eng.debug_array("vt_j0", np.int32)
        vt_nj = eng.debug_array("vt_nj", np.int32)
        assert len(qmeta) == 32 * len(vt_j0) == nq
        joints2 = np.full((info.num_joints_out, 3), np.nan)
        joints2[:24] = joints[:24]
        for tv in range(len(vt_j0)):
            # groups of a tile are ordered by skinning joint; every output joint of the tile accumulates its terms
            accs = np.tile(trans[b].numpy(), (int(vt_nj[tv]), 1)).astype(np.float64)
            cur = -1
            for i in range(32):
                mw = int(qmeta[tv * 32 + i])
                if not (mw >> 14) & 1:
                    continue
                if (mw >> 5) & 1:
                    assert (mw & 31) > cur or cur == -1      # sorted by skinning joint: each one loaded once
                    cur = mw & 31
                assert cur == (mw & 31)
                jl = (mw >> 8) & 31
                assert jl < vt_nj[tv]
                row = n_virt0 + 3 * (tv * 32 + i)
                accs[jl] = accs[jl] + A[cur] @ np.append(vp[row:row + 3], qcoef[tv * 32 + i])
            joints2[24 + vt_j0[tv]:24 + vt_j0[tv] + vt_nj[tv]] = accs
        np.testing.assert_allclose(joints2, ref.joints[b].numpy(), atol=2e-7)


def test_bf16_split_operand(host_engine):
    """The K-concatenated bf16x3 operand reproduces the fp32 rows to ~2^-16 relative."""
    eng = host_engine
    info = eng.info
    n_pad, pitch, nf = info.num_blend_rows_padded, info.feature_pitch, 217
    W32 = eng.debug_array("W32", np.float32).reshape(1 + nf, n_pad)
    Wf = _bf16_to_f32(eng.debug_array("Wf", np.uint16)).reshape(n_pad, pitch).astype(np.float64)
    Wb_hi = _bf16_to_f32(eng.debug_array("Wb_hi", np.uint16)).reshape(-1, n_pad)
    Wb_lo = _bf16_to_f32(eng.debug_array("Wb_lo", np.uint16)).reshape(-1, n_pad)
    assert pitch == 576 and Wb_hi.shape[0] == 224
    # template: exact 3-way split
    np.testing.assert_array_equal((Wf[:, 0] + Wf[:, 1] + Wf[:, 2]).astype(np.float32), W32[0])
    rng = np.random.default_rng(0)
    beta = rng.standard_normal(10).astype(np.float32)
    pf = (rng.standard_normal(207) * 0.3).astype(np.float32)
    x = np.concatenate([beta, pf])
    hi = _bf16_to_f32(_f32_to_bf16_rn(x))
    lo = _bf16_to_f32(_f32_to_bf16_rn(x - hi))
    # feature row as pose.cu writes it: slab 0 = [1 1 1 | b_hi b_lo b_hi], then the pf_hi and pf_lo segments
    feat = np.zeros(pitch)
    feat[0:3] = 1.0
    feat[3:13], feat[13:23], feat[23:33] = hi[:10], lo[:10], hi[:10]
    feat[64:271], feat[320:527] = hi[10:], lo[10:]
    exact = W32[0].astype(np.float64) + x.astype(np.float64) @ W32[1:].astype(np.float64)
    # the kernel's K schedule: slab 0 position by position; pf_hi.P_hi + pf_lo.P_hi (+ pf_hi.P_lo in fp32 mode)
    P_hi, P_lo = Wf[:, 64:320], Wf[:, 320:576]
    bf16_mode = Wf[:, :64] @ feat[:64] + P_hi @ feat[64:320] + P_hi @ feat[320:576]
    split = bf16_mode + P_lo @ feat[64:320]
    assert np.abs(split - exact).max() < 1e-6           # "fp32 mode": bf16x3 split (~2^-16 rel)
    err = np.abs(bf16_mode - exact).max()
    assert 1e-7 < err < 1e-4                            # "bf16 mode": single-bf16 pose-corrective model operand
    # backward operands: hi + lo reproduces the fp32 rows to 2^-16 relative
    rec = (Wb_hi[:nf].astype(np.float64) + Wb_lo[:nf]).astype(np.float64)
    scale = np.abs(W32[1:]).max()
    assert np.abs(rec - W32[1:]).max() < scale * 2.0 ** -15
    assert not Wb_hi[nf:].any() and not Wb_lo[nf:].any()


def test_slab_request_is_capped(host_engine):
    """A slab wider than the forward GEMMs' work lists hold (40960 bodies) plans exactly like the widest slab."""
    lib, h, B = _lib.load(), host_engine.handle, 65536
    assert lib.b200smpl_saved_bytes(h, B, 65536) == lib.b200smpl_saved_bytes(h, B, 40960)
    for mode in _lib.MODES.values():
        assert lib.b200smpl_forward_workspace_bytes(h, B, mode, 65536) == lib.b200smpl_forward_workspace_bytes(h, B, mode, 40960)
        assert lib.b200smpl_backward_workspace_bytes(h, B, mode, 65536) == lib.b200smpl_backward_workspace_bytes(h, B, mode, 40960)


def test_forward_gemm_worklist_covers_every_tile_once():
    """Host arithmetic of the forward blend GEMM's cluster work list (no device): for every slab width and row
    range, every (body-tile pair, row-tile pair) is covered exactly once, no cluster is empty, the list fits one
    wave of CTA pairs whenever the tile count allows, and the longest cluster is within one tile of the ideal."""
    import ctypes
    lib = _lib.load()
    cap = 160
    buf = (ctypes.c_uint16 * (3 * cap))()
    for num_sms in (148, 132, 2):
        tpcs = max(1, num_sms // 2)
        for body_tiles in (1, 2, 3, 8, 15, 16, 29, 30, 31, 32, 64, 319, 320):   # 320 = the widest slab, 40960 bodies
            for row_tiles in (1, 2, 3, 17, 162, 177, 178):
                n = lib.b200smpl_debug_fwd_gemm_worklist(body_tiles, row_tiles, num_sms, ctypes.cast(buf, ctypes.c_void_p), cap)
                bp_total, wtp_total = (body_tiles + 1) // 2, (row_tiles + 1) // 2
                assert 0 < n <= cap, (num_sms, body_tiles, row_tiles, n)
                seen = np.zeros((bp_total, wtp_total), np.int32)
                longest = 0
                for c in range(n):
                    bp, w0, w1 = buf[3 * c], buf[3 * c + 1], buf[3 * c + 2]
                    assert bp < bp_total and w0 < w1 <= wtp_total
                    seen[bp, w0:w1] += 1
                    longest = max(longest, w1 - w0)
                assert (seen == 1).all(), (num_sms, body_tiles, row_tiles)
                total = bp_total * wtp_total
                if bp_total <= tpcs:
                    ideal = -(-total // min(total, tpcs))
                    # rectangular or flattened, whichever was chosen: never worse than the rectangular split
                    rect_chunks = max(1, min(wtp_total, tpcs // bp_total))
                    assert longest <= -(-wtp_total // rect_chunks)
                    assert longest >= min(ideal, wtp_total) - 0
