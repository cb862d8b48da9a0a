"""fp64 restatement of the silhouette definition (DESIGN.md section 11) -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Camera: R = I, t = cam_t (B,3), K = [[f,0,S/2],[0,f,S/2],[0,0,1]]:  u = f (x+tx)/(z+tz) + S/2, v likewise with y.
Image element [i, j] is the pixel centred at (u, v) = (j + 0.5, i + 0.5); no vertical flip.
Faces with a vertex at z+tz <= 1e-3 or with |projected signed area| < 1e-8 px^2 are dropped; winding is ignored.
Hard (sigma == 0): a pixel is 1 when its centre is inside or on the boundary of a kept face.
Soft (sigma > 0, px^2): D_f = sigmoid(+d^2/sigma) inside, sigmoid(-d^2/sigma) outside, d = distance from the pixel
centre to the face's nearest edge segment; an outside face with d^2 > sigma ln(1/eps - 1), eps = 1e-4, contributes
nothing; alpha = 1 - prod_f (1 - D_f).

Every (face, pixel) pair is evaluated whose pixel centre lies in the face's bounding box grown by the cut-off radius
sqrt(sigma ln(1/eps - 1)); by the definition no other pair contributes.  The product is taken as
exp(sum log(1 - D_f)) with log(1 - D_f) = -softplus(+-d^2/sigma), which never saturates in fp64 -- an independent
formulation of what the kernels keep as an unsaturated product and a saturated count.  Gradients come from autograd.
The arithmetic runs on the device and in the dtype of `vertices` (scripts/silhouette_bench.py times it in fp32 on
the GPU as the eager baseline).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

EPS = 1e-4
ZMIN = 1e-3
AREA_MIN = 1e-8


def cutoff_d2(sigma: float) -> float:
    return sigma * math.log(1.0 / EPS - 1.0)


def project(vertices: torch.Tensor, cam_t: torch.Tensor, focal_length: float, img_wh: int):
    """(B,V,3), (B,3) -> uv (B,V,2) in pixels, Z = z + tz (B,V)."""
    Xc = vertices + cam_t[:, None, :]
    Z = Xc[..., 2]
    uv = focal_length * Xc[..., :2] / Z[..., None] + img_wh / 2.0
    return uv, Z


def face_table(vertices, cam_t, faces, focal_length, img_wh):
    """Projected triangles (B,F,3,2), kept mask (B,F) and signed area (B,F) in px^2."""
    uv, Z = project(vertices, cam_t, focal_length, img_wh)
    fl = faces.long()
    tri = uv[:, fl]                                                  # (B,F,3,2)
    zf = Z[:, fl]
    e1, e2 = tri[:, :, 1] - tri[:, :, 0], tri[:, :, 2] - tri[:, :, 0]
    area = 0.5 * (e1[..., 0] * e2[..., 1] - e1[..., 1] * e2[..., 0])
    kept = (zf > ZMIN).all(-1) & (area.abs() >= AREA_MIN)
    return tri, kept, area


def _inside(tri, p):
    """tri (...,3,2), p (...,2) -> inside or on the boundary (winding ignored)."""
    w = []
    for k in range(3):
        a, b = tri[..., k, :], tri[..., (k + 1) % 3, :]
        e = b - a
        w.append(e[..., 0] * (p[..., 1] - a[..., 1]) - e[..., 1] * (p[..., 0] - a[..., 0]))
    w = torch.stack(w, -1)
    return (w >= 0).all(-1) | (w <= 0).all(-1)


def _edge_d2(tri, p):
    """Squared distance from p to the nearest edge segment of tri (differentiable)."""
    ds = []
    for k in range(3):
        a, b = tri[..., k, :], tri[..., (k + 1) % 3, :]
        e = b - a
        t = (((p - a) * e).sum(-1) / (e * e).sum(-1)).clamp(0.0, 1.0)
        q = p - a - t[..., None] * e
        ds.append((q * q).sum(-1))
    return torch.stack(ds, -1).min(-1).values


def _pairs(tri_b, kept_b, S, rad):
    """Integer (face, row, col) triples of every pixel centre inside the face's box grown by rad."""
    with torch.no_grad():
        lo = tri_b.min(1).values
        hi = tri_b.max(1).values
        c0 = torch.ceil(lo[:, 0] - rad - 0.5).clamp(0, S - 1).long()
        c1 = torch.floor(hi[:, 0] + rad - 0.5).clamp(-1, S - 1).long()
        r0 = torch.ceil(lo[:, 1] - rad - 0.5).clamp(0, S - 1).long()
        r1 = torch.floor(hi[:, 1] + rad - 0.5).clamp(-1, S - 1).long()
        w = (c1 - c0 + 1).clamp(min=0)
        h = (r1 - r0 + 1).clamp(min=0)
        n = torch.where(kept_b, w * h, torch.zeros_like(w))
        fid = torch.repeat_interleave(torch.arange(tri_b.shape[0], device=tri_b.device), n)
        start = torch.cumsum(n, 0) - n
        local = torch.arange(int(n.sum()), device=tri_b.device) - start[fid]
        col = c0[fid] + local % w[fid]
        row = r0[fid] + local // w[fid]
    return fid, row, col


def render(vertices, faces, cam_t, img_wh: int, focal_length: float, sigma: float = 0.0, chunk: int = 1 << 22):
    """alpha (B,S,S) in the dtype of `vertices`; differentiable w.r.t. vertices and cam_t when sigma > 0."""
    S = int(img_wh)
    tri, kept, _ = face_table(vertices, cam_t, faces, focal_length, S)
    B = vertices.shape[0]
    rad = math.sqrt(cutoff_d2(sigma)) if sigma > 0 else 0.0
    out = []
    for b in range(B):
        fid, row, col = _pairs(tri[b].detach(), kept[b], S, rad)
        pix = row * S + col
        if sigma == 0:
            cov = torch.zeros(S * S, dtype=torch.bool, device=vertices.device)
            for s in range(0, fid.numel(), chunk):
                sl = slice(s, s + chunk)
                p = torch.stack([col[sl], row[sl]], -1).to(vertices.dtype) + 0.5
                ins = _inside(tri[b].detach()[fid[sl]], p)
                cov[pix[sl][ins]] = True
            out.append(cov.to(vertices.dtype).reshape(S, S))
            continue
        logom = torch.zeros(S * S, dtype=vertices.dtype, device=vertices.device)
        for s in range(0, fid.numel(), chunk):
            sl = slice(s, s + chunk)
            p = torch.stack([col[sl], row[sl]], -1).to(vertices.dtype) + 0.5
            t = tri[b][fid[sl]]
            d2 = _edge_d2(t, p)
            ins = _inside(t.detach(), p)
            live = ins | (d2.detach() <= cutoff_d2(sigma))
            x = torch.where(ins, d2, -d2) / sigma
            logom = logom.index_add(0, pix[sl][live], -F.softplus(x[live]))
        out.append((1.0 - torch.exp(logom)).reshape(S, S))
    return torch.stack(out)


def loss(vertices, faces, cam_t, target, img_wh, focal_length, sigma, weight):
    """Per body: weight * mean over the S^2 pixels of (alpha - target)^2."""
    alpha = render(vertices, faces, cam_t, img_wh, focal_length, sigma)
    return weight * ((alpha - target.to(alpha.dtype)) ** 2).mean(dim=(1, 2))


def edge_distance(vertices, faces, cam_t, img_wh, focal_length, b, rows, cols):
    """Distance (px) from the given pixel centres of body b to the nearest edge of any kept face of b."""
    with torch.no_grad():
        tri, kept, _ = face_table(vertices[b:b + 1], cam_t[b:b + 1], faces, focal_length, img_wh)
        tri = tri[0][kept[0]]
        p = torch.stack([cols, rows], -1).to(tri.dtype) + 0.5
        best = torch.full((p.shape[0],), float("inf"), dtype=tri.dtype)
        for s in range(0, tri.shape[0], 4096):
            d2 = _edge_d2(tri[None, s:s + 4096], p[:, None, :])
            best = torch.minimum(best, d2.min(1).values)
        return best.sqrt()
