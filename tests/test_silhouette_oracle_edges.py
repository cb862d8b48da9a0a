"""CPU tests that pin the fp64 silhouette oracle (oracle/silhouette_oracle.py) on the scenes of
tests/test_gpu_silhouette_edges.py: faces across the image border, a vertex behind the near plane and a ragged image
size, by analytic pixel counts and closed forms."""
import math

import torch

from oracle import silhouette_oracle as SO

D64 = torch.float64
# camera that maps (x, y, 0) to pixel (x + S/2, y + S/2): f = 1, t = (0, 0, 1)
CAM_T = torch.tensor([[0.0, 0.0, 1.0]], dtype=D64)


def _mesh(pix, S, z=None):
    """Vertices (1,N,3) whose projection under CAM_T with f = 1 is `pix` (N,2) for the vertices at z = 0."""
    p = torch.as_tensor(pix, dtype=D64)
    zz = torch.zeros(p.shape[0], dtype=D64) if z is None else torch.as_tensor(z, dtype=D64)
    return torch.cat([p - S / 2.0, zz[:, None]], 1)[None]


def test_hard_coverage_across_the_image_border():
    """Only pixel centres inside the image count.  Right triangle (-6,2) (10,2) (-6,18): centres (j+.5, i+.5) with
    j >= 0, i >= 2 and i + j <= 11 -> 55.  Right triangle (10,10) (30,10) (10,30) on a 16-pixel image: every centre
    with i, j in [10, 15] -> 36, the hypotenuse lies outside."""
    S = 16
    v = _mesh([[-6, 2], [10, 2], [-6, 18]], S)
    a = SO.render(v, torch.tensor([[0, 1, 2]]), CAM_T, S, 1.0, 0.0)[0]
    ii, jj = torch.meshgrid(torch.arange(S), torch.arange(S), indexing="ij")
    assert int(a.sum()) == 55 and torch.equal(a.bool(), (ii >= 2) & (ii + jj <= 11))
    v = _mesh([[10, 10], [30, 10], [10, 30]], S)
    a = SO.render(v, torch.tensor([[0, 1, 2]]), CAM_T, S, 1.0, 0.0)[0]
    assert int(a.sum()) == 36 and bool(a[10:, 10:].all())


def test_blur_of_a_face_outside_the_image():
    """A face wholly outside the image whose blur reaches in: alpha = sigmoid(-d^2 / sigma) at the nearest pixel
    centres, 0 beyond the cut-off radius.  Triangle right of a 16-pixel image with its left edge on x = 17 (1.5 px
    from the last centres); sigma = 2, radius sqrt(2 ln 9999) = 4.29 px."""
    S, sigma = 16, 2.0
    v = _mesh([[17, 4], [17, 12], [30, 8]], S)
    a = SO.render(v, torch.tensor([[0, 1, 2]]), CAM_T, S, 1.0, sigma)[0]
    for j, d in ((15, 1.5), (14, 2.5), (13, 3.5)):
        assert float((a[4:12, j] - 1 / (1 + math.exp(d * d / sigma))).abs().max()) < 1e-15
    assert float(a[:, :12].abs().max()) == 0.0


def test_vertex_behind_the_near_plane_drops_its_face():
    """A face with one vertex at z + tz = -0.5 is dropped, hard and soft (projected through the negative depth, that
    vertex would land at pixel (16, 20)).  A kept face next to it renders exactly as alone."""
    S = 16
    v = _mesh([[2, 3], [12, 3], [2, 13], [14, 14], [15, 8], [4, 2]], S, z=[0, 0, 0, 0, 0, -1.5])
    kept = torch.tensor([[0, 1, 2]])
    both = torch.tensor([[0, 1, 2], [3, 4, 5]])
    _, keep, _ = SO.face_table(v, CAM_T, both, 1.0, S)
    assert keep.tolist() == [[True, False]]
    hard = SO.render(v, both, CAM_T, S, 1.0, 0.0)
    assert int(hard.sum()) == 55 and torch.equal(hard, SO.render(v, kept, CAM_T, S, 1.0, 0.0))
    for sigma in (0.5, 4.0):
        assert torch.equal(SO.render(v, both, CAM_T, S, 1.0, sigma), SO.render(v, kept, CAM_T, S, 1.0, sigma))
    # the same face with the vertex in front of the camera does cover pixels
    v_front = v.clone()
    v_front[0, 5, 2] = 0.0
    assert int(SO.render(v_front, both, CAM_T, S, 1.0, 0.0).sum()) > 55


def test_square_at_a_ragged_size():
    """S = 33 (one pixel past a 32-pixel tile): the square [3.5, 29.5]^2 covers centres j, i in [3, 29] with the
    ones on its boundary -> 27^2 = 729; the square [20, 40]^2 is clipped to the 13 x 13 centres j, i in [20, 32]."""
    S = 33
    faces = torch.tensor([[0, 1, 2], [0, 3, 2]])
    v = _mesh([[3.5, 3.5], [29.5, 3.5], [29.5, 29.5], [3.5, 29.5]], S)
    a = SO.render(v, faces, CAM_T, S, 1.0, 0.0)[0]
    assert int(a.sum()) == 729 and bool(a[3:30, 3:30].all())
    v = _mesh([[20, 20], [40, 20], [40, 40], [20, 40]], S)
    a = SO.render(v, faces, CAM_T, S, 1.0, 0.0)[0]
    assert int(a.sum()) == 169 and bool(a[20:, 20:].all())
    # soft, last row: centre (26.5, 32.5) is inside the second triangle, 18^0.5 px from its nearest edge (the
    # diagonal), and beyond the cut-off of the first: alpha = sigmoid(18 / sigma)
    a = SO.render(v, faces, CAM_T, S, 1.0, 1.0)[0]
    assert abs(float(a[S - 1, 26]) - 1 / (1 + math.exp(-18.0))) < 1e-15

