"""fp64 numpy restatement of the proxy representation (DESIGN.md section 12), the regressor's 1 + K channel input:
channel 0 the nearest-neighbour resize of the binary mask, channels 1 + j Gaussian heatmaps of the keypoints.

`reference_float32` transcribes the reference's two functions for one crop as written (float32 numpy,
create_proxy_representation at predict/predict_3D.py:67-81 over convert_2Djoints_to_gaussian_heatmaps at
utils/label_conversions.py:58-87), with the mask resize written as the integer nearest rule cv2.INTER_NEAREST
applies for 512 -> 256 (cv2 is not a dependency)."""
from __future__ import annotations

import numpy as np

INT16_MIN, INT16_MAX = -32768, 32767


def binary_mask(mask: np.ndarray) -> np.ndarray:
    """The repository's mask rule: floating point `>= 0.5`, any other dtype non-zero."""
    mask = np.asarray(mask)
    return mask >= 0.5 if mask.dtype.kind == "f" else mask != 0


def nearest_index(out_wh: int, in_wh: int) -> np.ndarray:
    """Source row / column of each destination one: (dst * in_wh) // out_wh in exact integer arithmetic."""
    return (np.arange(out_wh, dtype=np.int64) * in_wh) // out_wh


def centres(keypoints: np.ndarray, in_wh: int, out_wh: int, vis=None):
    """Truncated keypoint centres (..., K, 2) int64 and a (..., K) validity mask: the keypoint scaled by out_wh / in_wh
    in double precision and truncated toward zero (astype(np.int16)); invalid when vis == 0, not finite, or the
    truncated centre leaves the int16 range (where numpy's cast would wrap)."""
    kp = np.asarray(keypoints, dtype=np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        scaled = kp * np.array([out_wh / float(in_wh), out_wh / float(in_wh)])
        t = np.trunc(scaled)
        ok = np.all(np.isfinite(t) & (t >= INT16_MIN) & (t <= INT16_MAX), axis=-1)
    if vis is not None:
        ok &= np.asarray(vis) != 0
    c = np.where(ok[..., None], t, 0.0).astype(np.int64)
    return c, ok


def proxy_representation(masks, keypoints, vis=None, out_wh: int = 256, std: float = 4.0) -> np.ndarray:
    """masks (B, in_wh, in_wh), keypoints (B, K, 2) pixels (x, y) of the in_wh image, vis (B, K) or None ->
    (B, 1 + K, out_wh, out_wh) float64."""
    m = binary_mask(masks)
    B, in_wh = m.shape[0], m.shape[1]
    src = nearest_index(out_wh, in_wh)
    c, ok = centres(keypoints, in_wh, out_wh, vis)
    K = c.shape[1]
    out = np.zeros((B, 1 + K, out_wh, out_wh))
    out[:, 0] = m[:, src][:, :, src]
    u = np.arange(out_wh, dtype=np.float64)
    for b in range(B):
        for j in range(K):
            if not ok[b, j]:
                continue
            gx = ((u - c[b, j, 0]) / std) ** 2 / 2
            gy = ((u - c[b, j, 1]) / std) ** 2 / 2
            out[b, 1 + j] = np.exp(-gx[None, :] - gy[:, None])
    return out


def convert_2Djoints_to_gaussian_heatmaps(joints2D: np.ndarray, img_wh: int, std: int = 4) -> np.ndarray:
    """The reference function as written: joints2D (K, 2) -> (img_wh, img_wh, K) float32."""
    xx, yy = np.meshgrid(np.arange(img_wh), np.arange(img_wh))
    xx = xx[None, :, :].astype(np.float32)
    yy = yy[None, :, :].astype(np.float32)
    j2d_u = joints2D[:, 0, None, None]
    j2d_v = joints2D[:, 1, None, None]
    heatmap = np.exp(-(((xx - j2d_u) / std) ** 2) / 2 - (((yy - j2d_v) / std) ** 2) / 2).transpose(1, 2, 0)
    return heatmap


def reference_float32(silhouette: np.ndarray, joints2D: np.ndarray, in_wh: int, out_wh: int, std: int = 4):
    """create_proxy_representation as written, for one crop: (in_wh, in_wh) mask, (K, 2) keypoints -> (1 + K,
    out_wh, out_wh) float32.  The resize is the integer nearest rule in place of cv2.resize(INTER_NEAREST)."""
    src = nearest_index(out_wh, in_wh)
    silhouette = silhouette[src][:, src]
    joints2D = joints2D[:, :2]
    joints2D = joints2D * np.array([out_wh / float(in_wh), out_wh / float(in_wh)])
    heatmaps = convert_2Djoints_to_gaussian_heatmaps(joints2D.astype(np.int16), out_wh, std)
    proxy_rep = np.concatenate([silhouette[:, :, None].astype(np.float32), heatmaps], axis=-1)
    return np.transpose(proxy_rep, [2, 0, 1])
