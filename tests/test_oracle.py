"""CPU tests of the oracle itself (runs in the build container, no GPU).

* in-tree functions of the oracle vs golden vectors produced by EXECUTING the reference files
  (tests/golden/make_golden_from_reference.py) -- this is the pinned part;
* the smplx restatement ("parity unpinned"): two independent restatements agree, invariance
  properties hold, committed known answers reproduce.
"""
import numpy as np
import pytest
import torch

from oracle import smpl_oracle as O
from oracle.smpl_numpy import rodrigues_one, smpl_one_body
from soccerplayershapepose_b200 import config as cfg
from soccerplayershapepose_b200.model_io import SMPL_PARENTS, SMPL_EXTRA_JOINT_VERTEX_IDS


# ----------------------------------------------------------------------------- pinned: in-tree
def test_config_tables_bit_exact(intree_golden):
    g = intree_golden
    for k in ("ALL_JOINTS_TO_COCO_MAP", "ALL_JOINTS_TO_H36M_MAP", "H36M_TO_J17", "H36M_TO_J14",
              "SMPL_TO_KPRCNN_MAP"):
        assert np.array_equal(np.asarray(getattr(cfg, k), np.int64), g["cfg_" + k]), k
    assert cfg.FOCAL_LENGTH == float(g["cfg_FOCAL_LENGTH"])
    assert cfg.REGRESSOR_IMG_WH == int(g["cfg_REGRESSOR_IMG_WH"])


def test_orthographic_and_pixels(intree_golden):
    g = intree_golden
    out = O.orthographic_project(torch.from_numpy(g["ortho_points"]), torch.from_numpy(g["ortho_cam"]))
    assert np.array_equal(out.numpy(), g["ortho_out"])                      # same fp32 op order
    px = O.undo_keypoint_normalisation(out, 512)
    assert np.array_equal(px.numpy(), g["undo_norm_out"])


def test_weak_perspective_conversions(intree_golden):
    g = intree_golden
    cam = torch.from_numpy(g["ortho_cam"])
    t = O.weak_perspective_to_translation(cam, 5000.0, 512)
    assert np.array_equal(t.numpy(), g["wp2t_out"])
    wp = O.translation_to_weak_perspective(t, 5000.0, 512)
    assert np.array_equal(wp.numpy(), g["t2wp_out"])
    assert np.array_equal(O.intrinsics_matrix(512, 512, 5000.0), g["intrinsics_512_5000"])


def test_perspective_projection(intree_golden):
    g = intree_golden
    out = O.perspective_project(torch.from_numpy(g["ortho_points"]), torch.from_numpy(g["persp_rot"]),
                                torch.from_numpy(g["persp_trans"]), focal_length=5000.0, img_wh=512)
    np.testing.assert_allclose(out.numpy(), g["persp_out"], rtol=0, atol=0)


def test_rot6d(intree_golden):
    g = intree_golden
    out = O.rot6d_to_rotmat(torch.from_numpy(g["rot6d_in"]))
    assert out.shape == (6 * 24, 3, 3)
    assert np.array_equal(out.numpy(), g["rot6d_out"])


def test_joints2d_loss(intree_golden):
    g = intree_golden
    pred, label = torch.from_numpy(g["loss_j2d_pred"]), torch.from_numpy(g["loss_j2d_label"])
    lv = torch.tensor(O.init_log_var(1.0), dtype=torch.float32)
    assert np.float32(lv) == g["loss_j2d_log_var"]
    out = O.joints2d_loss(pred, label, lv, img_wh=256.0)
    np.testing.assert_allclose(out.numpy(), g["loss_j2d_out"], rtol=1e-6)
    out_v = O.joints2d_loss(pred, label, lv, img_wh=256.0, vis=torch.from_numpy(g["loss_j2d_vis"]))
    np.testing.assert_allclose(out_v.numpy(), g["loss_j2d_vis_out"], rtol=1e-6)
    # two-term loss: joints2D (w=100) + shape_params (w=0.01)
    lv2 = [torch.tensor(O.init_log_var(w), dtype=torch.float32) for w in (100.0, 0.01)]
    np.testing.assert_allclose(np.array([float(v) for v in lv2], np.float32), g["loss2_log_vars"], rtol=1e-6)
    sp, sl = torch.from_numpy(g["loss2_shape_pred"]), torch.from_numpy(g["loss2_shape_label"])
    shape_term = torch.mean((sp - sl) ** 2) * torch.exp(-lv2[1]) + lv2[1]
    total = O.joints2d_loss(pred, label, lv2[0], img_wh=256.0) + shape_term
    np.testing.assert_allclose(total.numpy(), g["loss2_out"], rtol=1e-5)


# ------------------------------------------------------------------- unpinned: smplx restatement
def _inputs(B, seed, dtype=torch.float64):
    gen = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=gen, dtype=dtype)
    pose = torch.randn(B, 72, generator=gen, dtype=dtype) * 0.3
    trans = torch.rand(B, 3, generator=gen, dtype=dtype) * 2 - 1
    return betas, pose, trans


def test_bit_exact_tables():
    assert SMPL_PARENTS.tolist() == [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19,
                                     20, 21]
    assert SMPL_EXTRA_JOINT_VERTEX_IDS.tolist() == [332, 6260, 2800, 4071, 583, 3216, 3226, 3387, 6617, 6624,
                                                    6787, 2746, 2319, 2445, 2556, 2673, 6191, 5782, 5905,
                                                    6016, 6133]
    # consistency with the in-tree COCO map: nose 24, l-eye 26, r-eye 25, l-ear 28, r-ear 27
    assert cfg.ALL_JOINTS_TO_COCO_MAP[:5] == [24, 26, 25, 28, 27]


def test_rodrigues_identity_and_orthonormal():
    R0 = O.batch_rodrigues(torch.zeros(4, 3, dtype=torch.float64))
    assert torch.allclose(R0, torch.eye(3, dtype=torch.float64).expand(4, 3, 3), atol=1e-15)
    r = torch.randn(50, 3, dtype=torch.float64)
    R = O.batch_rodrigues(r)
    eye = torch.eye(3, dtype=torch.float64)
    assert torch.allclose(R @ R.transpose(1, 2), eye.expand(50, 3, 3), atol=1e-7)
    assert torch.allclose(torch.linalg.det(R), torch.ones(50, dtype=torch.float64), atol=1e-7)
    for i in range(5):
        np.testing.assert_allclose(R[i].numpy(), rodrigues_one(r[i].numpy()), atol=1e-14)


def test_two_restatements_agree(synthetic_model):
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    betas, pose, trans = _inputs(3, 11)
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(3, 24, 3, 3)
    out = orc.forward_flat(betas, rot, trans, pose2rot=False)
    for b in range(3):
        v, j = smpl_one_body(synthetic_model, betas[b].numpy(), rot[b].numpy(), trans[b].numpy())
        np.testing.assert_allclose(out.vertices[b].numpy(), v, atol=1e-12)
        np.testing.assert_allclose(out.joints[b].numpy(), j, atol=1e-12)


def test_tpose_zero_beta_is_template(synthetic_model):
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float32)
    out = orc.forward_flat(torch.zeros(2, 10), torch.zeros(2, 72), None, pose2rot=True)
    err = (out.vertices - orc.v_template).abs().max().item()
    assert err < 5e-7, err
    j24 = O.vertices2joints(orc.J_regressor, orc.v_template[None])
    assert (out.joints[:, :24] - j24).abs().max().item() < 5e-7


def test_pose2rot_paths_agree(synthetic_model):
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    betas, pose, trans = _inputs(2, 3)
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(2, 24, 3, 3)
    a = orc.forward_flat(betas, pose, trans, pose2rot=True)
    b = orc.forward_flat(betas, rot, trans, pose2rot=False)
    assert torch.allclose(a.vertices, b.vertices, atol=1e-13)
    assert torch.allclose(a.joints, b.joints, atol=1e-13)


def test_global_rotation_and_translation_equivariance(synthetic_model):
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    betas, pose, trans = _inputs(2, 5)
    rot = O.batch_rodrigues(pose.reshape(-1, 3)).reshape(2, 24, 3, 3)
    base = orc.forward_flat(betas, rot, None, pose2rot=False)
    Q = O.batch_rodrigues(torch.tensor([[0.3, -1.1, 0.7]], dtype=torch.float64))[0]
    rot2 = rot.clone()
    rot2[:, 0] = Q @ rot[:, 0]
    out = orc.forward_flat(betas, rot2, trans, pose2rot=False)
    # rotating the root rotates everything about the root joint's rest position
    J0 = base.joints[:, :1] - 0  # posed root == rest root (G_0 translation = J_0)
    exp_v = (base.vertices - J0) @ Q.T + J0 + trans[:, None]
    exp_j = (base.joints - J0) @ Q.T + J0 + trans[:, None]
    # exact up to (sum_j w_vj - 1): skinning-weight rows sum to 1 only to fp32 rounding
    assert torch.allclose(out.vertices, exp_v, atol=2e-7)
    assert torch.allclose(out.joints[:, :24], exp_j[:, :24], atol=1e-12)
    assert torch.allclose(out.joints[:, 24:45], exp_j[:, 24:45], atol=2e-7)
    # regressed joints are affine in the vertices only up to (row sum - 1): rows sum to 1 in fp32
    assert torch.allclose(out.joints[:, 45:], exp_j[:, 45:], atol=5e-7)


def test_joint_layout(synthetic_model):
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    betas, pose, trans = _inputs(2, 9)
    out = orc.forward_flat(betas, pose, trans, pose2rot=True)
    assert out.vertices.shape == (2, 6890, 3) and out.joints.shape == (2, 90, 3)
    v = out.vertices
    assert torch.equal(out.joints[:, 24:45], v[:, torch.as_tensor(SMPL_EXTRA_JOINT_VERTEX_IDS)])
    for lo, hi, reg in ((45, 54, orc.J_regressor_extra), (54, 73, orc.J_regressor_cocoplus),
                        (73, 90, orc.J_regressor_h36m)):
        assert torch.allclose(out.joints[:, lo:hi], torch.einsum("jv,bvk->bjk", reg, v), atol=1e-13)


def test_known_answers(synthetic_model, smpl_kat):
    k = smpl_kat
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    out = orc.forward_flat(torch.from_numpy(k["betas"]), torch.from_numpy(k["rotmats"]),
                           torch.from_numpy(k["trans"]), pose2rot=False)
    np.testing.assert_allclose(out.vertices[:, k["vert_subset"]].numpy(), k["verts_sub"], atol=1e-12)
    np.testing.assert_allclose(out.joints.numpy(), k["joints"], atol=1e-12)
    np.testing.assert_allclose(out.vertices.sum(1).numpy(), k["verts_sum"], atol=1e-9)
    out_aa = orc.forward_flat(torch.from_numpy(k["betas"][:5]), torch.from_numpy(k["pose_aa"]), None,
                              pose2rot=True)
    np.testing.assert_allclose(out_aa.joints.numpy(), k["aa_joints"], atol=1e-12)
    # fp32 oracle (the reference's arithmetic) sits within 1e-5 m of the fp64 answers
    orc32 = O.SMPLOracle(synthetic_model, dtype=torch.float32)
    o32 = orc32.forward_flat(torch.from_numpy(k["betas"]).float(), torch.from_numpy(k["rotmats"]).float(),
                             torch.from_numpy(k["trans"]).float(), pose2rot=False)
    assert np.abs(o32.joints.double().numpy() - k["joints"]).max() < 1e-5


def test_oracle_gradcheck_small(synthetic_model):
    """Autograd through the oracle is what the GPU backward is compared with: sanity-check it
    by finite differences on a reduced loss."""
    orc = O.SMPLOracle(synthetic_model, dtype=torch.float64)
    betas, pose, trans = _inputs(1, 21)
    gen = torch.Generator().manual_seed(1)
    dV = torch.randn(1, 6890, 3, generator=gen, dtype=torch.float64)
    dJ = torch.randn(1, 90, 3, generator=gen, dtype=torch.float64)

    def loss(b, p, t):
        o = orc.forward_flat(b, p, t, pose2rot=True)
        return (o.vertices * dV).sum() + (o.joints * dJ).sum()

    b, p, t = (x.clone().requires_grad_(True) for x in (betas, pose, trans))
    loss(b, p, t).backward()
    eps = 1e-6
    for x, gx, idxs in ((betas, b.grad, [0, 7]), (pose, p.grad, [0, 4, 40, 71]), (trans, t.grad, [1])):
        for i in idxs:
            xp, xm = x.clone(), x.clone()
            xp[0, i] += eps
            xm[0, i] -= eps
            args_p = [betas, pose, trans]
            args_m = [betas, pose, trans]
            k = [id(betas), id(pose), id(trans)].index(id(x))
            args_p[k], args_m[k] = xp, xm
            fd = (loss(*args_p) - loss(*args_m)) / (2 * eps)
            assert abs(fd.item() - gx[0, i].item()) <= 1e-5 * max(1.0, abs(fd.item())), (k, i)


def test_vertices2joints_helper_matches_oracle():
    from soccerplayershapepose_b200.lbs import vertices2joints
    g = torch.Generator().manual_seed(0)
    v = torch.randn(3, 50, 3, generator=g, dtype=torch.float64)
    J = torch.rand(7, 50, generator=g, dtype=torch.float64)
    assert torch.allclose(vertices2joints(J, v), O.vertices2joints(J, v), rtol=0, atol=1e-12)


def test_perspective_projection_with_explicit_intrinsics(intree_golden):
    """cam_K argument of utils/cam_utils.py:54-85: batched matrices with skew, unequal focal lengths, off-centre
    principal point and a non-trivial third row (which the reference computes and drops)."""
    g = intree_golden
    out = O.perspective_project(torch.from_numpy(g["ortho_points"]), torch.from_numpy(g["persp_rot"]),
                                torch.from_numpy(g["persp_trans"]), cam_K=torch.from_numpy(g["persp_camK"]))
    np.testing.assert_allclose(out.numpy(), g["persp_camK_out"], rtol=0, atol=0)


def test_five_term_multitask_loss_matches_the_reference_class(intree_golden):
    """regressor.MultiTaskLoss (the eager restatement the fused kernels are tested against) reproduces
    HomoscedasticUncertaintyWeightedMultiTaskLoss executed from the reference file: all five MSE terms, a vis mask,
    unequal initial weights."""
    from soccerplayershapepose_b200 import regressor
    g = intree_golden
    names = ["verts", "joints2D", "joints3D", "shape_params", "pose_params"]
    w5 = {"verts": 2.0, "joints2D": 0.3, "joints3D": 1.5, "shape_params": 0.05, "pose_params": 0.7}
    crit = regressor.MultiTaskLoss(names, w5)
    np.testing.assert_allclose([getattr(crit, k + "_log_var").item() for k in names], g["loss5_log_vars"], rtol=1e-6)
    keys = ("verts", "joints2D", "joints3D", "shape_params", "pose_params_rot_matrices")
    outputs = {k: torch.from_numpy(g["loss5_pred_" + k]) for k in keys}
    labels = {k: torch.from_numpy(g["loss5_label_" + k]) for k in keys}
    labels["vis"] = torch.from_numpy(g["loss5_label_vis"])
    total, parts = crit(labels, outputs)
    np.testing.assert_allclose(total.item(), g["loss5_out"], rtol=1e-6)
    np.testing.assert_allclose([parts[k].item() for k in names], g["loss5_parts"], rtol=1e-6)


def test_fit_loss_per_player_is_joints2d_loss_per_player_plus_shape_term():
    """The per-player fitting loss the fit_loss kernel is checked against: for each player, `joints2d_loss` on that
    player alone plus shape_weight * mean(beta^2), values and gradients; a player with no visible keypoint gets
    log_var + the shape term and no keypoint gradient (where `joints2d_loss` is NaN)."""
    g = torch.Generator().manual_seed(7)
    B, K, lv, sw, wh = 6, 45, -0.7, 0.3, 200.0
    pred = (torch.rand(B, K, 2, generator=g, dtype=torch.float64) * 512).requires_grad_(True)
    label = torch.rand(B, K, 2, generator=g, dtype=torch.float64) * 512
    betas = torch.randn(B, 10, generator=g, dtype=torch.float64).requires_grad_(True)
    vis = torch.rand(B, K, generator=g) > 0.4
    vis[2] = False
    vis[3] = False
    vis[3, 5] = True
    got = O.fit_loss_per_player(pred, label, lv, betas, sw, wh, vis)
    got.sum().backward()
    pred2 = pred.detach().clone().requires_grad_(True)
    betas2 = betas.detach().clone().requires_grad_(True)
    lv_t = torch.tensor(lv, dtype=torch.float64)
    for b in range(B):
        shape = sw * (betas2[b] ** 2).mean()
        if b == 2:
            assert torch.isnan(O.joints2d_loss(pred2[b:b + 1], label[b:b + 1], lv_t, wh, vis[b:b + 1]))
            want = lv_t + shape
        else:
            want = O.joints2d_loss(pred2[b:b + 1], label[b:b + 1], lv_t, wh, vis[b:b + 1]) + shape
        want.backward()
        assert abs(got[b].item() - want.item()) < 1e-12 * max(1.0, abs(want.item())), b
    torch.testing.assert_close(pred.grad, pred2.grad, rtol=1e-12, atol=1e-15)
    torch.testing.assert_close(betas.grad, betas2.grad, rtol=1e-12, atol=1e-15)
    assert pred.grad[2].abs().max().item() == 0.0
    # without a mask every keypoint counts
    full = O.fit_loss_per_player(pred.detach(), label, lv, betas.detach(), sw, wh)
    for b in range(B):
        want = O.joints2d_loss(pred.detach()[b:b + 1], label[b:b + 1], lv_t, wh) + sw * (betas.detach()[b] ** 2).mean()
        assert abs(full[b].item() - want.item()) < 1e-12 * max(1.0, abs(want.item())), b
