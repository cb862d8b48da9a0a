"""CPU tests of the fp64 silhouette oracle (oracle/silhouette_oracle.py), the checker of csrc/silhouette.cu:
analytic coverage counts, the soft-to-hard limit, autograd against finite differences and the product of two
overlapping faces deep inside both."""
import math

import torch

from oracle import silhouette_oracle as SO

D64 = torch.float64
# camera that maps (x, y, 0) to pixel (x + S/2, y + S/2): f = 1, t = (0, 0, 1)
CAM_T = torch.tensor([[0.0, 0.0, 1.0]], dtype=D64)


def _mesh(pix, S):
    """Vertices (1,N,3) whose projection is `pix` (N,2) under CAM_T with f = 1."""
    p = torch.as_tensor(pix, dtype=D64)
    return torch.cat([p - S / 2.0, torch.zeros(p.shape[0], 1, dtype=D64)], 1)[None]


def test_hard_coverage_single_triangle_and_square():
    S = 32
    # right triangle (2,3) (12,3) (2,13): centres (j+.5, i+.5) with j >= 2, i >= 3, (j-2) + (i-3) <= 9 -> 55 pixels,
    # the ten centres on the hypotenuse included
    v = _mesh([[2, 3], [12, 3], [2, 13]], S)
    a = SO.render(v, torch.tensor([[0, 1, 2]]), CAM_T, S, 1.0, 0.0)
    assert int(a.sum()) == 55
    assert a[0, 3, 2] == 1 and a[0, 12, 2] == 1 and a[0, 3, 11] == 1 and a[0, 2, 2] == 0 and a[0, 12, 3] == 0
    # square [4, 20]^2 as two triangles of opposite winding: 16 x 16 centres, the shared diagonal counted once
    v = _mesh([[4, 4], [20, 4], [20, 20], [4, 20]], S)
    a = SO.render(v, torch.tensor([[0, 1, 2], [0, 3, 2]]), CAM_T, S, 1.0, 0.0)
    assert int(a.sum()) == 256 and a[0, 4:20, 4:20].all()


def test_dropped_faces():
    S = 16
    v = _mesh([[2, 2], [10, 2], [2, 10], [4, 4], [8, 8], [12, 12]], S)
    v_behind = v.clone()
    v_behind[0, 2, 2] = -1.0 + 1e-4                  # z + tz <= 1e-3: the first face is dropped
    faces = torch.tensor([[0, 1, 2], [3, 4, 5]])        # the second face is collinear: zero area, dropped
    assert int(SO.render(v, faces, CAM_T, S, 1.0, 0.0).sum()) > 0
    assert int(SO.render(v_behind, faces, CAM_T, S, 1.0, 0.0).sum()) == 0
    assert float(SO.render(v_behind, faces, CAM_T, S, 1.0, 1.0).abs().max()) == 0.0


def test_soft_converges_to_hard_away_from_edges():
    g = torch.Generator().manual_seed(0)
    S = 24
    pix = torch.rand(12, 2, generator=g, dtype=D64) * 20 + 2
    faces = torch.tensor([[0, 1, 2], [3, 4, 5], [6, 7, 8], [9, 10, 11], [0, 4, 8]])
    v = _mesh(pix, S)
    hard = SO.render(v, faces, CAM_T, S, 1.0, 0.0)[0]
    ii, jj = torch.meshgrid(torch.arange(S), torch.arange(S), indexing="ij")
    dist = SO.edge_distance(v, faces, CAM_T, S, 1.0, 0, ii.flatten(), jj.flatten()).reshape(S, S)
    far = dist > 0.5
    assert int(far.sum()) > 200
    errs = [float((SO.render(v, faces, CAM_T, S, 1.0, s)[0] - hard)[far].abs().max()) for s in (0.5, 0.1, 0.02)]
    assert errs[0] > errs[1] > errs[2] and errs[2] < 1e-5


def test_gradient_matches_central_differences():
    g = torch.Generator().manual_seed(1)
    S, sigma = 16, 2.0
    pix = torch.rand(6, 2, generator=g, dtype=D64) * 10 + 3
    faces = torch.tensor([[0, 1, 2], [3, 4, 5], [1, 2, 4]])
    v = _mesh(pix, S)
    v[0, :, 2] = torch.rand(6, generator=g, dtype=D64) * 0.2      # depth varies: z enters the projection
    t = torch.tensor([[0.3, -0.2, 1.5]], dtype=D64)
    w = torch.randn(1, S, S, generator=g, dtype=D64)
    f = 3.0

    def obj(vv, tt):
        return (SO.render(vv, faces, tt, S, f, sigma) * w).sum()

    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    obj(vv, tt).backward()
    h = 1e-6
    for x, grad in ((v, vv.grad), (t, tt.grad)):
        num = torch.zeros_like(x)
        for idx in range(x.numel()):
            xp, xm = x.clone(), x.clone()
            xp.view(-1)[idx] += h
            xm.view(-1)[idx] -= h
            fp = obj(xp, t) if x is v else obj(v, xp)
            fm = obj(xm, t) if x is v else obj(v, xm)
            num.view(-1)[idx] = (fp - fm) / (2 * h)
        assert (num - grad).abs().max() <= 1e-6 * max(1.0, float(grad.abs().max())), (num, grad)


def test_product_exact_inside_two_overlapping_faces():
    """A pixel deep inside two overlapping faces: 1 - D_f is ~1e-200, far below where a product with a division by
    (1 - D_f) stays meaningful.  alpha and d alpha / d d_f^2 must equal the closed forms
    alpha = 1 - (1 - D_1)(1 - D_2),  d alpha / d D_1 = 1 - D_2."""
    S, sigma = 40, 0.05
    v = _mesh([[2, 2], [38, 2], [2, 38], [4, 3], [37, 6], [6, 36]], S)
    faces = torch.tensor([[0, 1, 2], [3, 4, 5]])
    vv = v.clone().requires_grad_(True)
    a = SO.render(vv, faces, CAM_T, S, 1.0, sigma)
    i, j = 10, 10
    assert float(a.detach()[0, i, j]) == 1.0
    a[0, i, j].backward()
    # every factor is saturated: the exact gradient underflows to zero, never NaN / inf
    assert torch.isfinite(vv.grad).all() and float(vv.grad.abs().max()) < 1e-100
    # a pixel near an edge of face 2 and deep inside face 1: d alpha / d d2_2 = (1 - D_1) dD_2/dd2 ~ 0
    vv.grad = None
    p = torch.tensor([5.5, 6.5], dtype=D64)
    tri = v[0, faces[1].long(), :2] + S / 2.0
    d2_2 = float(SO._edge_d2(tri[None], p[None])[0])
    a = SO.render(vv, faces, CAM_T, S, 1.0, sigma)
    x2 = d2_2 / sigma * (1 if bool(SO._inside(tri, p)) else -1)
    D2 = 1 / (1 + math.exp(-x2))
    tri1 = v[0, faces[0].long(), :2] + S / 2.0
    x1 = float(SO._edge_d2(tri1[None], p[None])[0]) / sigma
    om1 = 1 / (1 + math.exp(x1))
    assert abs(float(a.detach()[0, 6, 5]) - (1 - om1 * (1 - D2))) < 1e-15
