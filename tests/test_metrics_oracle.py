"""CPU tests of the reconstruction-error definition (DESIGN.md section 13): the fp64 oracle against the float64
transcription of the reference's eval functions and against an independent rotation solver, its exact cases and its
degenerate rule, and the C-ABI entry's argument checks (which run before any device work)."""
import ctypes

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle import metrics_oracle as M
from soccerplayershapepose_b200 import _lib, config


def _bodies(rng, B=6, N=200):
    P = rng.standard_normal((B, N, 3)) * np.array([0.2, 0.8, 0.15]) + rng.standard_normal((B, 1, 3)) * 5
    Q = P + 0.03 * rng.standard_normal((B, N, 3))
    Q = Q @ Rotation.random(B, random_state=1).as_matrix().transpose(0, 2, 1) * 1.1 + 2.0
    return P, Q


def test_oracle_matches_reference_transcription():
    P, Q = _bodies(np.random.default_rng(0))
    ref = M.reference_errors(P, Q)
    got = M.reconstruction_errors(P, Q)[:, :3]
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12)
    # joints: the mapped rows with their own transforms
    jm = np.array(config.ALL_JOINTS_TO_J14_MAP) - 60
    got_j = M.reconstruction_errors(pred_joints=P, target_joints=Q, joint_map=jm)
    np.testing.assert_allclose(got_j[:, 3:], M.reference_errors(P[:, jm], Q[:, jm]), rtol=1e-12, atol=1e-12)
    assert np.isnan(got_j[:, :3]).all()


def test_j14_map_is_the_h36m_then_j14_selection():
    j = np.arange(config.NUM_ALL_JOINTS)
    assert config.ALL_JOINTS_TO_J14_MAP == j[config.ALL_JOINTS_TO_H36M_MAP][config.H36M_TO_J14].tolist()


def test_rotation_matches_an_independent_solver():
    rng = np.random.default_rng(1)
    for _ in range(5):
        P, Q = _bodies(rng, B=1)
        s, R, t = M.procrustes(P[0], Q[0])
        X, Y = P[0] - P[0].mean(0), Q[0] - Q[0].mean(0)
        rot, _ = Rotation.align_vectors(Y, X)            # R minimising sum |y_i - R x_i|^2
        np.testing.assert_allclose(R, rot.as_matrix(), atol=1e-10)
        assert abs(np.linalg.det(R) - 1) < 1e-12


def test_exact_similarity_gives_zero_error():
    rng = np.random.default_rng(2)
    Q = rng.standard_normal((300, 3))
    R = Rotation.random(random_state=3).as_matrix()
    P = 0.7 * Q @ R.T + np.array([20.0, -3.0, 1.0])
    assert M.set_errors(P, Q)[2] < 1e-12
    P = 1.3 * Q + np.array([20.0, -3.0, 1.0])            # R = I: SC is exact as well
    e, e_sc, e_pa = M.set_errors(P, Q)
    assert e > 1 and e_sc < 1e-12 and e_pa < 1e-12


def test_mirrored_prediction_gets_a_proper_rotation():
    rng = np.random.default_rng(4)
    Q = rng.standard_normal((300, 3)) * np.array([0.3, 0.9, 0.1])
    P = Q * np.array([1.0, 1.0, -1.0])
    s, R, _ = M.procrustes(P, Q)
    assert abs(np.linalg.det(R) - 1) < 1e-12
    assert M.set_errors(P, Q)[2] > 1e-3
    np.testing.assert_allclose(M.set_errors(P, Q)[2], M.reference_errors(P[None], Q[None])[0, 2], rtol=1e-12)


def test_degenerate_and_non_finite_bodies():
    rng = np.random.default_rng(5)
    Q = rng.standard_normal((50, 3))
    P = np.tile(np.array([[3.0, 1.0, -2.0]]), (50, 1))
    want = np.linalg.norm(Q.mean(0) - Q, axis=1).mean()
    e, e_sc, e_pa = M.set_errors(P, Q)
    assert e_sc == pytest.approx(want, rel=1e-14) and e_pa == pytest.approx(want, rel=1e-14)
    for bad in (np.nan, np.inf):
        P2 = rng.standard_normal((50, 3))
        P2[7, 1] = bad
        assert np.isnan(M.set_errors(P2, Q)).all()
    # one non-finite vertex leaves the joint columns alone
    Pv, Qv = rng.standard_normal((2, 1, 30, 3))
    Pv[0, 3, 0] = np.nan
    out = M.reconstruction_errors(Pv, Qv, Qv[:, :10] + 0.01, Qv[:, :10], np.arange(10))
    assert np.isnan(out[0, :3]).all() and np.isfinite(out[0, 3:]).all()


def _args(**kw):
    base = dict(batch=2, num_verts=10, num_joints=5, num_map=3, reserved0=0, reserved1=0,
                pred_vertices=16, target_vertices=32, pred_joints=48, target_joints=64, joint_map=80)
    base.update(kw)
    return _lib.ReconErrorArgs(**base)


@pytest.mark.parametrize("bad", [
    dict(batch=0), dict(batch=-1),
    dict(target_vertices=None), dict(pred_vertices=None),
    dict(target_joints=None), dict(pred_joints=None),
    dict(num_verts=0), dict(num_joints=0), dict(num_map=0), dict(joint_map=None),
    dict(pred_vertices=None, target_vertices=None, pred_joints=None, target_joints=None),
])
def test_entry_refuses_invalid_arguments_without_a_device(bad):
    lib = _lib.load()
    before = lib.b200smpl_launch_count()
    args = _args(**bad)
    out = ctypes.c_void_p(96)                            # never dereferenced: the checks come first
    assert lib.b200smpl_reconstruction_errors(ctypes.byref(args), out, None) == _lib.ERR_INVALID
    assert "reconstruction_errors" in _lib.last_error()
    assert lib.b200smpl_reconstruction_errors(ctypes.byref(_args()), None, None) == _lib.ERR_INVALID
    assert lib.b200smpl_reconstruction_errors(None, out, None) == _lib.ERR_INVALID
    assert lib.b200smpl_launch_count() == before

