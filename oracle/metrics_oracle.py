"""fp64 numpy restatement of the reconstruction errors (DESIGN.md section 13): per body the mean Euclidean distance
between predicted and target points, plain, scale-corrected (SC) and Procrustes-aligned (PA).

`reference_procrustes_batch` and `reference_scale_and_translation_batch` transcribe, in float64 numpy, the two
functions of the reference's utils/eval_utils.py as they are understood (procrustes_analysis_batch with the numpy SVD
and the sign(det) fix, scale_and_translation_transform_batch); `reference_errors` is the tracker's use of them.  They
divide by zero on degenerate bodies, where the oracle applies the repository's rule instead."""
from __future__ import annotations

import numpy as np


def mean_distance(P: np.ndarray, Q: np.ndarray) -> float:
    """E(P, Q) = (1/N) sum_i |p_i - q_i|, the mean Euclidean distance (not the RMS)."""
    return float(np.linalg.norm(np.asarray(P, np.float64) - np.asarray(Q, np.float64), axis=-1).mean())


def scale_correct(P: np.ndarray, Q: np.ndarray) -> np.ndarray:
    """p_i' = (p_i - mu_P) r_Q / r_P + mu_Q with r = sqrt(sum |p_i - mu|^2 / N); p_i' = mu_Q when r_P = 0."""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    mp, mq = P.mean(0), Q.mean(0)
    rp = np.sqrt(((P - mp) ** 2).sum() / len(P))
    rq = np.sqrt(((Q - mq) ** 2).sum() / len(Q))
    s = rq / rp if rp > 0 else 0.0
    return (P - mp) * s + mq


def procrustes(P: np.ndarray, Q: np.ndarray):
    """The similarity (s, R, t) with R in SO(3) maximising tr(R K), K = sum x_i y_i^T of the centred points:
    K = U S V^T, R = V diag(1, 1, det(V U^T)) U^T, s = tr(R K) / sum |x_i|^2, t = mu_Q - s R mu_P.  s = 0 (so
    p_i' = mu_Q) when all predicted points coincide."""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    mp, mq = P.mean(0), Q.mean(0)
    X, Y = P - mp, Q - mq
    K = X.T @ Y
    U, _, Vt = np.linalg.svd(K)
    V = Vt.T
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(V @ U.T)) or 1.0])
    R = V @ D @ U.T
    sxx = (X ** 2).sum()
    s = np.trace(R @ K) / sxx if sxx > 0 else 0.0
    return s, R, mq - s * R @ mp


def procrustes_align(P: np.ndarray, Q: np.ndarray) -> np.ndarray:
    s, R, t = procrustes(P, Q)
    return s * np.asarray(P, np.float64) @ R.T + t


def set_errors(P: np.ndarray, Q: np.ndarray):
    """(E, E_SC, E_PA) of one point set; all NaN when an input is not finite."""
    if not (np.all(np.isfinite(P)) and np.all(np.isfinite(Q))):
        return np.nan, np.nan, np.nan
    return mean_distance(P, Q), mean_distance(scale_correct(P, Q), Q), mean_distance(procrustes_align(P, Q), Q)


def reconstruction_errors(pred_vertices=None, target_vertices=None, pred_joints=None, target_joints=None,
                          joint_map=None) -> np.ndarray:
    """(B, 6) float64: pve, pve_sc, pve_pa, mpjpe, mpjpe_sc, mpjpe_pa; the columns of an absent pair are NaN.  The
    joints are rows joint_map of the joints and get their own transforms."""
    B = len(pred_vertices if pred_vertices is not None else pred_joints)
    out = np.full((B, 6), np.nan)
    for b in range(B):
        if pred_vertices is not None:
            out[b, :3] = set_errors(pred_vertices[b], target_vertices[b])
        if pred_joints is not None:
            m = np.asarray(joint_map)
            out[b, 3:] = set_errors(np.asarray(pred_joints[b])[m], np.asarray(target_joints[b])[m])
    return out


# ---- float64 transcription of the reference (utils/eval_utils.py) ---------------------------------------------------
def reference_procrustes_batch(S1: np.ndarray, S2: np.ndarray) -> np.ndarray:
    """procrustes_analysis_batch(S1, S2): S1, S2 (B, N, 3) -> S1 aligned to S2 by a similarity transform."""
    S1, S2 = np.asarray(S1, np.float64), np.asarray(S2, np.float64)
    mu1 = S1.mean(axis=1, keepdims=True)
    mu2 = S2.mean(axis=1, keepdims=True)
    X1 = S1 - mu1
    X2 = S2 - mu2
    var1 = np.sum(X1 ** 2, axis=(1, 2))
    K = np.matmul(X1.transpose(0, 2, 1), X2)
    U, s, V = np.linalg.svd(K)
    V = V.transpose(0, 2, 1)
    Z = np.tile(np.eye(3)[None], (S1.shape[0], 1, 1))
    Z[:, -1, -1] *= np.sign(np.linalg.det(np.matmul(U, V.transpose(0, 2, 1))))
    R = np.matmul(np.matmul(V, Z), U.transpose(0, 2, 1))
    trace = np.trace(np.matmul(R, K), axis1=1, axis2=2)
    scale = trace / var1
    trans = mu2.squeeze(1) - scale[:, None] * np.matmul(R, mu1.transpose(0, 2, 1)).squeeze(2)
    return scale[:, None, None] * np.matmul(S1, R.transpose(0, 2, 1)) + trans[:, None, :]


def reference_scale_and_translation_batch(P: np.ndarray, T: np.ndarray) -> np.ndarray:
    """scale_and_translation_transform_batch(P, T): P (B, N, 3) scaled and translated onto T's mean and RMS radius."""
    P, T = np.asarray(P, np.float64), np.asarray(T, np.float64)
    P_mean = np.mean(P, axis=1, keepdims=True)
    P_trans = P - P_mean
    P_scale = np.sqrt(np.sum(P_trans ** 2, axis=(1, 2), keepdims=True) / P.shape[1])
    P_normalised = P_trans / P_scale
    T_mean = np.mean(T, axis=1, keepdims=True)
    T_scale = np.sqrt(np.sum((T - T_mean) ** 2, axis=(1, 2), keepdims=True) / T.shape[1])
    return P_normalised * T_scale + T_mean


def reference_errors(pred: np.ndarray, target: np.ndarray) -> np.ndarray:
    """The tracker's per-body (E, E_SC, E_PA) for (B, N, 3) arrays: np.linalg.norm(. - target, axis=-1) per point,
    averaged over the points."""
    pred, target = np.asarray(pred, np.float64), np.asarray(target, np.float64)
    err = lambda a: np.linalg.norm(a - target, axis=-1).mean(axis=1)   # noqa: E731
    return np.stack([err(pred), err(reference_scale_and_translation_batch(pred, target)),
                     err(reference_procrustes_batch(pred, target))], axis=1)
