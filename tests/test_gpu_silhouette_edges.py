"""GPU tests of the silhouette kernels (csrc/silhouette.cu) where their tiling can break: forward CTAs that render
several bands, ragged image sizes, bodies across the image border or behind the near plane, sparse gradients, blur
radii that span several tiles and bands, other meshes, and the size and argument limits of the C-ABI.

The reference is the fp64 oracle (oracle/silhouette_oracle.py), run on the GPU.  The bounds are those of
tests/test_gpu_silhouette.py: hard mismatches only within 1e-3 px of a kept edge, soft |d alpha| < 1e-4 away from
faces of |area| < 1e-4 px^2, gradients < 1e-3 max-norm relative, the fused loss within 1e-5 of render + loss +
backward."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import silhouette_oracle as SO
from soccerplayershapepose_b200 import _lib, config, ops
from soccerplayershapepose_b200.cam_utils import convert_weak_perspective_to_camera_translation_torch
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
BAND = 32          # rows per band and columns per tile in csrc/silhouette.cu


@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


@pytest.fixture(scope="module")
def faces(smpl):
    return smpl.faces_int32(DEV)


def _sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def _split(B, S):
    """CTAs per body of b200smpl_silhouette_render: the bands of a body are spread over ceil(SMs / B) CTAs."""
    return max(1, min(-(-S // BAND), -(-_sms() // B)))


def _focal(S):
    return config.FOCAL_LENGTH * S / 512


def _posed(smpl, cams, seed):
    """Posed vertices (B,6890,3) of random bodies seen through the weak-perspective cameras `cams` (B,3), and the
    camera translation (B,3)."""
    cams = torch.as_tensor(cams, dtype=torch.float32)
    B = cams.shape[0]
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=g)
    pose = torch.randn(B, 72, generator=g) * 0.3
    out = smpl(betas=betas.to(DEV), body_pose=pose[:, 3:].to(DEV), global_orient=pose[:, :3].to(DEV))
    t = convert_weak_perspective_to_camera_translation_torch(cams.to(DEV), config.FOCAL_LENGTH, 512)
    return out.vertices.detach().contiguous(), t.contiguous()


def _random_cams(B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.rand(B, generator=g) * 0.6 + 0.6, torch.rand(B, generator=g) * 0.4 - 0.2,
                        torch.rand(B, generator=g) * 0.4 - 0.2], 1)


def _at_corner(v, t, S, f):
    """Move every body in the image plane (each vertex by the same pixel offset, depths unchanged) so that its vertex
    extreme in the +u+v direction projects to (S - 1.5, S - 1.5).  The centre of pixel (S-1, S-1) then lies outside
    the silhouette within sqrt(2) px of its outline, and the body covers the last band and the last tile column."""
    uv, Z = SO.project(v.double(), t.double(), f, S)
    k = uv.sum(-1).argmax(1)
    duv = (S - 1.5) - uv[torch.arange(v.shape[0], device=v.device), k]
    out = v.double().clone()
    out[..., :2] += duv[:, None, :] * Z[..., None] / f
    return out.float().contiguous()


def _mesh(pix, S, z=None):
    """Vertices (1,N,3) that project to the pixel positions `pix` (N,2) under `_cam_t()` with f = 1 (exact in fp32 for
    pixel positions on a 1/8-px grid)."""
    p = torch.as_tensor(pix, dtype=torch.float64)
    zz = torch.zeros(p.shape[0], 1, dtype=torch.float64) if z is None else torch.as_tensor(z, dtype=torch.float64)[:, None]
    return torch.cat([p - S / 2.0, zz], 1)[None].float().to(DEV)


def _cam_t():
    """The camera of `_mesh`: t = (0, 0, 1)."""
    return torch.tensor([[0.0, 0.0, 1.0]], device=DEV)


def _ambiguous(v, t, faces, S, f, sigma):
    """Pixels near a face whose kept / dropped status fp32 may decide differently from fp64 (|area| < 1e-4 px^2);
    excluded from the soft and gradient comparisons.  They must be rare."""
    tri, _, area = SO.face_table(v.double(), t.double(), faces, f, S)
    mask = torch.zeros(v.shape[0], S, S, dtype=torch.bool, device=v.device)
    rad = math.sqrt(SO.cutoff_d2(sigma)) + 1.0
    for b, k in torch.nonzero(area.abs() < 1e-4).tolist():
        lo, hi = tri[b, k].min(0).values.tolist(), tri[b, k].max(0).values.tolist()
        c0, c1 = (int(np.clip(x, 0, S)) for x in (np.floor(lo[0] - rad), np.ceil(hi[0] + rad)))
        r0, r1 = (int(np.clip(x, 0, S)) for x in (np.floor(lo[1] - rad), np.ceil(hi[1] + rad)))
        mask[b, r0:r1, c0:c1] = True
    assert float(mask.float().mean()) < 0.05
    return mask


def _check_hard(v, faces, t, S, f, a=None):
    """Hard render against the oracle: mismatches only at pixel centres within 1e-3 px of a kept edge.  Returns the
    oracle's image."""
    if a is None:
        a = ops.render_silhouettes(v, faces, t, S, f, 0.0)
    ref = SO.render(v.double(), faces, t.double(), S, f, 0.0)
    assert a.shape == ref.shape and bool(((a == 0) | (a == 1)).all())
    bad = torch.nonzero(a.double() != ref)
    for b in bad[:, 0].unique().tolist():
        sel = bad[bad[:, 0] == b]
        d = SO.edge_distance(v.double(), faces, t.double(), S, f, b, sel[:, 1], sel[:, 2])
        assert float(d.max()) < 1e-3, (b, len(sel), float(d.max()))
    return ref


def _check_soft(v, faces, t, S, f, sigma, a=None, exact=False):
    """Soft render against the oracle, away from the pixels of `_ambiguous` unless the mesh is `exact`: vertices on
    a grid that fp32 projects exactly, so that fp32 and fp64 find the same areas."""
    if a is None:
        a = ops.render_silhouettes(v, faces, t, S, f, sigma)
    ref = SO.render(v.double(), faces, t.double(), S, f, sigma)
    err = (a.double() - ref).abs()
    if not exact:
        err = err[~_ambiguous(v, t, faces, S, f, sigma)]
    assert float(err.max()) < 1e-4, float(err.max())
    return ref


def _kernel_grads(v, faces, t, S, f, sigma, gs):
    """(grad_vertices, grad_t) of sum(alpha * g) from the render backward, one per g in gs."""
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    a = ops.render_silhouettes(vv, faces, tt, S, f, sigma)
    return [torch.autograd.grad(a, (vv, tt), g.float(), retain_graph=True) for g in gs]


def _oracle_grads(v, faces, t, S, f, sigma, gs):
    v64, t64 = v.double().requires_grad_(True), t.double().requires_grad_(True)
    a = SO.render(v64, faces, t64, S, f, sigma)
    return [torch.autograd.grad(a, (v64, t64), g.double(), retain_graph=True) for g in gs]


def _check_grads(v, faces, t, S, f, sigma, gs):
    for got, want in zip(_kernel_grads(v, faces, t, S, f, sigma, gs), _oracle_grads(v, faces, t, S, f, sigma, gs)):
        for x, y in zip(got, want):
            assert float(y.abs().max()) > 0.0
            rel = float((x.double() - y).abs().max() / y.abs().max())
            assert rel < 1e-3, rel


def _check_fused_loss(v, faces, t, S, f, sigma, target, weight=3.0):
    """silhouette_loss against the render, the squared-error loss and the render backward."""
    base = torch.rand(v.shape[0], device=DEV)
    loss, gv, gt = ops.silhouette_loss(v, faces, t, target, S, f, sigma, weight, loss_per_body=base.clone())
    vv, tt = v.clone().requires_grad_(True), t.clone().requires_grad_(True)
    a = ops.render_silhouettes(vv, faces, tt, S, f, sigma)
    ref = weight * ((a - target.float()) ** 2).mean(dim=(1, 2))
    ref.sum().backward()
    assert torch.allclose(loss - base, ref.detach(), rtol=1e-5, atol=1e-7)
    for got, want in ((gv, vv.grad), (gt, tt.grad)):
        assert float(want.abs().max()) > 0.0
        assert float((got - want).abs().max() / want.abs().max()) < 1e-5
    return loss - base, gv, gt


# ---- 1. launch geometry -----------------------------------------------------------------------------------------
NDISTINCT = 5


def _geometry(case):
    """(B, S) of a batch whose forward CTAs each render several bands."""
    sms = _sms()
    if case == "split1":
        B, S = sms + 3, 128
        assert _split(B, S) == 1 and B % NDISTINCT != 0
    else:
        B, S = -(-sms // 3), 256
        nb = S // BAND
        assert 1 < _split(B, S) < nb and nb % _split(B, S) != 0
    assert _split(1, S) == S // BAND                     # a body rendered alone: one band per CTA
    return B, S


def _batch(smpl, S, seed, B):
    v5, t5 = _posed(smpl, _random_cams(NDISTINCT, seed), seed)
    idx = torch.arange(B, device=DEV) % NDISTINCT
    return v5, t5, idx, v5[idx].contiguous(), t5[idx].contiguous()


@pytest.mark.parametrize("case", ["split1", "split3"])
def test_forward_ctas_over_several_bands(smpl, faces, case):
    """sil_fwd's band loop (band += gridDim.y) when a CTA renders several bands: split 1 with a ragged batch
    (SMs + 3 bodies, 4 bands each) and split 3 over 8 bands.  Every copy equals the body rendered alone bit for bit,
    and the distinct bodies match the oracle, hard and soft."""
    B, S = _geometry(case)
    f = _focal(S)
    v5, t5, idx, v, t = _batch(smpl, S, 100 + S, B)
    for sigma in (0.0, 1.0):
        a = ops.render_silhouettes(v, faces, t, S, f, sigma)
        alone = torch.cat([ops.render_silhouettes(v5[k:k + 1], faces, t5[k:k + 1], S, f, sigma)
                           for k in range(NDISTINCT)])
        assert torch.equal(a, alone[idx])
        if sigma == 0.0:
            assert float(_check_hard(v5, faces, t5, S, f, alone).sum()) > 100
        else:
            _check_soft(v5, faces, t5, S, f, sigma, alone)


@pytest.mark.parametrize("case", ["split1", "split3"])
def test_backward_and_loss_at_large_batches(smpl, faces, case):
    """sil_bwd and sil_loss at the batches of the forward test (one CTA per body over all its bands): every copy is
    within 1e-6 x max of the body computed alone (shared-memory atomics reorder the sums); the distinct bodies match
    the oracle (backward) and render + loss + backward (fused loss)."""
    B, S = _geometry(case)
    f, sigma = _focal(S), 1.0
    v5, t5, idx, v, t = _batch(smpl, S, 200 + S, B)
    g5 = torch.randn(NDISTINCT, S, S, generator=torch.Generator().manual_seed(S)).to(DEV)
    g5[_ambiguous(v5, t5, faces, S, f, sigma)] = 0.0
    (gv, gt), = _kernel_grads(v, faces, t, S, f, sigma, [g5[idx]])
    alone = [_kernel_grads(v5[k:k + 1], faces, t5[k:k + 1], S, f, sigma, [g5[k:k + 1]])[0] for k in range(NDISTINCT)]
    for k in range(NDISTINCT):
        for x, y in ((gv, alone[k][0]), (gt, alone[k][1])):
            assert float((x[idx == k] - y).abs().max()) <= 1e-6 * float(y.abs().max())
    _check_grads(v5, faces, t5, S, f, sigma, [g5])

    target5 = ops.render_silhouettes(v5 * 1.02, faces, t5, S, f, 0.0) > 0.5
    lossB, gvB, gtB = ops.silhouette_loss(v, faces, t, target5[idx], S, f, sigma, 3.0)
    for k in range(NDISTINCT):
        l1, gv1, gt1 = ops.silhouette_loss(v5[k:k + 1], faces, t5[k:k + 1], target5[k:k + 1], S, f, sigma, 3.0)
        for x, y in ((lossB, l1), (gvB, gv1), (gtB, gt1)):
            assert float((x[idx == k] - y).abs().max()) <= 1e-6 * float(y.abs().max())
    _check_fused_loss(v5, faces, t5, S, f, sigma, target5)


# ---- 2. ragged and large image sizes -------------------------------------------------------------------------
@pytest.fixture(scope="module", params=[33, 100, 257, 512])
def corner_bodies(request, smpl, faces):
    """Two bodies over the bottom-right corner of an S x S image (partial last band and tile column when S % 32), and
    the SMPL faces without those that project to under 1e-3 px^2 on either body: at S = 33 a few faces fall under the
    1e-4 px^2 that fp32 and fp64 may keep or drop differently, and their blur would cover a large part of the image."""
    S = request.param
    f = _focal(S)
    v, t = _posed(smpl, _random_cams(2, 300 + S), 300 + S)
    v = _at_corner(v, t, S, f)
    _, _, area = SO.face_table(v.double(), t.double(), faces, f, S)
    return S, f, v, t, faces[(area.abs() >= 1e-3).all(0)].contiguous()


def test_ragged_render(corner_bodies):
    """tile_fwd's row < S / col < S masks and the partial last band: hard and soft render against the oracle."""
    S, f, v, t, faces = corner_bodies
    ref = _check_hard(v, faces, t, S, f)
    nb = (S - 1) // BAND * BAND                           # first row of the last band, first column of the last tile
    assert float(ref[:, nb:].sum()) > 0 and float(ref[:, :, nb:].sum()) > 0
    _check_soft(v, faces, t, S, f, 1.0)


def test_ragged_sparse_backward(corner_bodies):
    """sil_bwd's grad_alpha read (row < S, col < S), the partial last tile column and band, and the per-tile early exit
    (__any_sync(need)): grad_alpha nonzero only (a) on the last band and the last tile column, (b) at the single pixel
    (S-1, S-1), against the oracle; an all-zero grad_alpha gives exactly zero gradients."""
    S, f, v, t, faces = corner_bodies
    sigma = 1.0
    amb = _ambiguous(v, t, faces, S, f, sigma)
    nb = (S - 1) // BAND * BAND
    edge = torch.zeros(2, S, S, dtype=torch.bool, device=DEV)
    edge[:, nb:, :] = True
    edge[:, :, nb:] = True
    ga = torch.randn(2, S, S, generator=torch.Generator().manual_seed(S)).to(DEV) * (edge & ~amb)
    gb = torch.zeros(2, S, S, device=DEV)
    gb[:, S - 1, S - 1] = 1.0
    assert not bool(amb[:, S - 1, S - 1].any())
    _check_grads(v, faces, t, S, f, sigma, [ga, gb])
    (gv, gt), = _kernel_grads(v, faces, t, S, f, sigma, [torch.zeros(2, S, S, device=DEV)])
    assert bool((gv == 0).all()) and bool((gt == 0).all())


def test_ragged_fused_loss(corner_bodies):
    """sil_loss's loss and target reads on the partial band and tile column (tile_bwd<true>)."""
    S, f, v, t, faces = corner_bodies
    target = ops.render_silhouettes(v * 1.02, faces, t, S, f, 0.0) > 0.5
    _check_fused_loss(v, faces, t, S, f, 1.0, target)


def _tiny_mesh(S):
    """Two faces of a few pixels on an S x S image, one partly outside it."""
    pix = [[0.125, 0.25], [S + 0.375, 0.75], [0.5, S - 0.125],
           [S * 0.5, S * 0.25], [S + 2.0, S * 0.75], [S * 0.625, S + 1.5]]
    return _mesh(pix, S), torch.tensor([[0, 1, 2], [3, 4, 5]], dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("S", [1, 7, 8])
def test_tiny_images(S):
    """Images smaller than one tile (a single partial band and tile column) on a hand-built mesh: hard, soft and the
    backward against the oracle."""
    v, fc = _tiny_mesh(S)
    t = _cam_t()
    assert float(_check_hard(v, fc, t, S, 1.0).sum()) >= 1
    _check_soft(v, fc, t, S, 1.0, 0.5)
    g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(S)).to(DEV)
    _check_grads(v, fc, t, S, 1.0, 0.5, [g])


# ---- 3. scenes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene", ["across_border", "fills_frame"])
def test_scene_render_and_backward(smpl, faces, scene):
    """band_list / tile_hit culling against the pixel centres [0.5, S - 0.5] with boxes grown by the blur radius:
    a body crossing all four image borders (weak-perspective [2.5, 0.5, -0.3]) and a body filling the whole frame
    (scale 8, faces tens of pixels wide).  Hard, soft and the backward against the oracle."""
    S, sigma = 256, 1.0
    f = _focal(S)
    cam = [[2.5, 0.5, -0.3], [2.5, -0.4, 0.35]] if scene == "across_border" else [[8.0, 0.0, 0.0]]
    v, t = _posed(smpl, cam, 400)
    uv, _ = SO.project(v.double(), t.double(), f, S)
    if scene == "across_border":
        assert float(uv.min()) < -50 and float(uv.max()) > S + 50
    ref = _check_hard(v, faces, t, S, f)
    assert float(ref.mean()) > (0.9 if scene == "fills_frame" else 0.1)
    _check_soft(v, faces, t, S, f, sigma)
    g = torch.randn(v.shape[0], S, S, generator=torch.Generator().manual_seed(401)).to(DEV)
    g[_ambiguous(v, t, faces, S, f, sigma)] = 0.0
    if scene == "across_border":
        _check_grads(v, faces, t, S, f, sigma, [g])
    else:
        # every pixel lies deep inside two or more faces: the exact gradient underflows to 0 in fp64, and the
        # kernel's count of saturated factors (1 - D_f < 1e-30) leaves at most products of such factors
        (gv, gt), = _kernel_grads(v, faces, t, S, f, sigma, [g])
        (gv64, gt64), = _oracle_grads(v, faces, t, S, f, sigma, [g])
        assert float(gv64.abs().max()) == 0.0 and float(gt64.abs().max()) == 0.0
        assert float(gv.abs().max()) < 1e-20 and float(gt.abs().max()) < 1e-20


def test_body_off_the_image(smpl, faces):
    """No face reaches the image: empty band lists.  alpha, grad_vertices and grad_t are exactly 0 and the loss is
    weight * mean(target)."""
    S, sigma, weight = 100, 1.0, 2.5
    f = _focal(S)
    v, t = _posed(smpl, [[1.0, 10.0, 0.0], [1.0, -3.0, -12.0]], 500)
    uv, _ = SO.project(v.double(), t.double(), f, S)
    assert bool(((uv[..., 0].min(1).values > S + 20) | (uv[..., 1].max(1).values < -20)).all())
    for sg in (0.0, sigma):
        assert bool((ops.render_silhouettes(v, faces, t, S, f, sg) == 0).all())
    g = torch.randn(2, S, S, generator=torch.Generator().manual_seed(501)).to(DEV)
    (gv, gt), = _kernel_grads(v, faces, t, S, f, sigma, [g])
    assert bool((gv == 0).all()) and bool((gt == 0).all())
    target = torch.rand(2, S, S, generator=torch.Generator().manual_seed(502)).to(DEV) > 0.7
    loss, gv, gt = ops.silhouette_loss(v, faces, t, target, S, f, sigma, weight)
    assert bool((gv == 0).all()) and bool((gt == 0).all())
    assert torch.allclose(loss, weight * target.float().mean(dim=(1, 2)), rtol=1e-6, atol=0)


def test_limb_behind_the_near_plane(smpl, faces):
    """project_body's z + tz <= 1e-3 rule: one side of the body is moved to z + tz = -0.5.  band_list drops every face
    touching it (NaN area), the flush writes zero gradient rows for its vertices, and hard, soft, the backward and
    the fused loss match the oracle."""
    S, sigma = 256, 1.0
    f = _focal(S)
    v, t = _posed(smpl, [[1.0, 0.0, 0.0], [0.8, 0.1, -0.1]], 600)
    behind = v[..., 0] > torch.quantile(v[..., 0], 0.85, dim=1, keepdim=True)
    v = v.clone()
    v[..., 2] = torch.where(behind, -0.5 - t[:, 2:3], v[..., 2])
    _, kept, _ = SO.face_table(v.double(), t.double(), faces, f, S)
    assert 0.05 < float(1 - kept.double().mean()) < 0.5
    assert float(_check_hard(v, faces, t, S, f).sum()) > 1000
    _check_soft(v, faces, t, S, f, sigma)
    g = torch.randn(2, S, S, generator=torch.Generator().manual_seed(601)).to(DEV)
    g[_ambiguous(v, t, faces, S, f, sigma)] = 0.0
    _check_grads(v, faces, t, S, f, sigma, [g])
    (gv, _), = _kernel_grads(v, faces, t, S, f, sigma, [g])
    assert bool((gv[behind] == 0).all())
    target = ops.render_silhouettes(v * 1.02, faces, t, S, f, 0.0) > 0.5
    _, gv, _ = _check_fused_loss(v, faces, t, S, f, sigma, target)
    assert bool((gv[behind] == 0).all())


@pytest.mark.parametrize("S,sigma", [(128, 0.05), (256, 8.0), (256, 16.0)])
def test_sigma_sweep(smpl, faces, S, sigma):
    """soft_term at sigma = 0.05 (many factors saturate: the unsaturated product and the saturated count) and at
    sigma = 8 / 16 (blur radii 8.6 / 12.1 px: grown boxes span several tiles and bands).  Soft render and backward
    against the oracle."""
    f = _focal(S)
    v, t = _posed(smpl, _random_cams(2, 700 + S), 700 + S)
    _check_soft(v, faces, t, S, f, sigma)
    g = torch.randn(2, S, S, generator=torch.Generator().manual_seed(701)).to(DEV)
    g[_ambiguous(v, t, faces, S, f, sigma)] = 0.0
    _check_grads(v, faces, t, S, f, sigma, [g])


# hand-built triangles on a 257 x 257 image (pixel positions); each spans several bands and tile columns or lies
# just outside the image within the blur radius (4.29 px at sigma = 2)
BIG_TRIANGLES = [
    [(-40.0, 20.0), (150.0, -30.0), (60.0, 200.0)],      # off the top-left corner
    [(100.0, 100.0), (300.0, 140.0), (180.0, 290.0)],    # across the right and bottom borders
    [(257.0, 20.0), (275.0, 30.0), (257.0, 90.0)],       # 0.5 px right of the last pixel centre
    [(30.0, 257.5), (120.0, 257.5), (70.0, 300.0)],      # 1 px below the last pixel centre
    [(-1.0, 150.0), (-30.0, 170.0), (-1.0, 240.0)],      # 1.5 px left of the first pixel centre
    [(40.0, 40.0), (90.0, 45.0), (50.0, 230.0)],         # inside, overlapping the first
]


def test_large_hand_built_triangles():
    """Triangles spanning several bands and tile columns, some partly or wholly off the image: band_list / tile_hit
    keep a face outside the image whose blur reaches in.  Hard, soft, backward and fused loss against the oracle."""
    S, sigma = 257, 2.0
    v = _mesh([p for tri in BIG_TRIANGLES for p in tri], S)
    fc = torch.arange(3 * len(BIG_TRIANGLES), dtype=torch.int32, device=DEV).reshape(-1, 3)
    t = _cam_t()
    _check_hard(v, fc, t, S, 1.0)
    ref = _check_soft(v, fc, t, S, 1.0, sigma)
    # the faces outside the image reach the last column, the last row and the first column alone:
    # alpha = sigmoid(-d^2 / sigma) at d = 0.5, 1 and 1.5 px
    for a, d in ((ref[0, 22:88, S - 1], 0.5), (ref[0, S - 1, 35:115], 1.0), (ref[0, 152:238, 0], 1.5)):
        assert float((a - 1 / (1 + math.exp(d * d / sigma))).abs().max()) < 1e-12
    g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(800)).to(DEV)
    _check_grads(v, fc, t, S, 1.0, sigma, [g])
    target = torch.zeros(1, S, S, dtype=torch.bool, device=DEV)
    target[0, 50:200, 60:250] = True
    loss, gv, gt = _check_fused_loss(v, fc, t, S, 1.0, sigma, target)
    v64, t64 = v.double().requires_grad_(True), t.double().requires_grad_(True)
    ref_loss = SO.loss(v64, fc, t64, target, S, 1.0, sigma, 3.0)
    ref_loss.sum().backward()
    assert abs(float(loss) - float(ref_loss.detach())) < 1e-5 * float(ref_loss.detach())
    for got, want in ((gv, v64.grad), (gt, t64.grad)):
        assert float((got.double() - want).abs().max() / want.abs().max()) < 1e-3


# ---- 4. other meshes and size limits ------------------------------------------------------------------------------
def test_triangle_soup_with_degenerate_faces():
    """A random mesh (V = 37, F = 50, varying depth) with a face repeating an index and a collinear face: band_list's
    area test drops both, like the oracle.  The soup renders bit for bit as without them; hard, soft and the backward
    match the oracle."""
    S, sigma = 100, 1.0
    g = torch.Generator().manual_seed(900)
    pix = torch.rand(37, 2, generator=g, dtype=torch.float64) * (S + 20) - 10
    pix[:3] = torch.tensor([[10.0, 10.0], [20.0, 20.0], [40.0, 40.0]])         # collinear
    z = torch.rand(37, generator=g, dtype=torch.float64) * 0.2
    z[:3] = 0.0
    v = _mesh(pix, S, z)
    good = torch.randint(0, 37, (48, 3), generator=g)
    good = good[(good[:, 0] != good[:, 1]) & (good[:, 1] != good[:, 2]) & (good[:, 0] != good[:, 2])]
    degenerate = torch.tensor([[0, 1, 2], [5, 9, 5]])
    soup = torch.cat([good[:20], degenerate[:1], good[20:], degenerate[1:]]).int().to(DEV)
    clean = torch.cat([good[:20], good[20:]]).int().to(DEV)
    assert soup.shape[0] >= 40
    t = _cam_t()
    for sg in (0.0, sigma):
        a = ops.render_silhouettes(v, soup, t, S, 1.0, sg)
        assert torch.equal(a, ops.render_silhouettes(v, clean, t, S, 1.0, sg))
        assert bool((ops.render_silhouettes(v, degenerate.int().to(DEV), t, S, 1.0, sg) == 0).all())
        assert float(SO.render(v.double(), degenerate.to(DEV), t.double(), S, 1.0, sg).abs().max()) == 0.0
    _check_hard(v, soup, t, S, 1.0)
    _check_soft(v, soup, t, S, 1.0, sigma, exact=True)
    gr = torch.randn(1, S, S, generator=g).to(DEV)
    _check_grads(v, soup, t, S, 1.0, sigma, [gr])


def _wide_mesh(V, S):
    """V vertices, four faces over vertices at both ends of the index range; the unused vertices sit at the image
    centre."""
    g = torch.Generator().manual_seed(V)
    ids = [0, 1, 2, 3, V // 2, V - 3, V - 2, V - 1]
    pix = torch.full((V, 2), S / 2.0, dtype=torch.float64)
    pix[ids] = torch.rand(len(ids), 2, generator=g, dtype=torch.float64) * S
    fc = torch.tensor([[0, 1, 2], [V - 3, V - 2, V - 1], [2, V // 2, V - 1], [3, V // 2, 1]], dtype=torch.int32)
    return _mesh(pix, S), fc.to(DEV), ids


def test_shared_memory_limits():
    """sil_prepare's shared-memory check (smem + 1024 <= opt-in per block): the largest mesh the backward accepts (16 B
    per vertex) renders and back-propagates correctly; one more vertex is refused by the backward and the fused loss
    but still renders; the largest mesh the forward accepts (8 B per vertex) renders correctly and one more vertex is
    refused.  A 3-vertex mesh renders first, so every kernel's dynamic shared-memory attribute has to grow."""
    S, sigma, F = 64, 1.0, 4
    optin = torch.cuda.get_device_properties(DEV).shared_memory_per_block_optin
    v_bwd = (optin - 1024 - 6 * F) // 16          # sil_smem(bwd) = 16 V + 6 F
    v_fwd = (optin - 1024 - 6 * F) // 8           # sil_smem(fwd) = 8 V + 6 F
    assert 6890 < v_bwd < v_fwd <= 65535
    t = _cam_t()

    v3 = _mesh([[5.0, 6.0], [50.0, 10.0], [20.0, 60.0]], S)
    f3 = torch.tensor([[0, 1, 2]], dtype=torch.int32, device=DEV)
    _check_soft(v3, f3, t, S, 1.0, sigma)

    v, fc, ids = _wide_mesh(v_bwd, S)
    _check_hard(v, fc, t, S, 1.0)
    a = _check_soft(v, fc, t, S, 1.0, sigma)
    g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(1000)).to(DEV)
    _check_grads(v, fc, t, S, 1.0, sigma, [g])
    (gv, _), = _kernel_grads(v, fc, t, S, 1.0, sigma, [g])
    unused = torch.ones(v_bwd, dtype=torch.bool, device=DEV)
    unused[ids] = False
    assert bool((gv[0, unused] == 0).all())
    _check_fused_loss(v, fc, t, S, 1.0, sigma, a > 0.5)

    # one more vertex (unused): too large for the backward, the same image from the forward
    v1 = torch.cat([v, v[:, :1]], 1).contiguous()
    assert torch.equal(ops.render_silhouettes(v1, fc, t, S, 1.0, sigma), ops.render_silhouettes(v, fc, t, S, 1.0, sigma))
    with pytest.raises(ValueError, match="shared-memory"):
        _kernel_grads(v1, fc, t, S, 1.0, sigma, [g])
    with pytest.raises(ValueError, match="shared-memory"):
        ops.silhouette_loss(v1, fc, t, a > 0.5, S, 1.0, sigma)

    v, fc, _ = _wide_mesh(v_fwd, S)
    _check_hard(v, fc, t, S, 1.0)
    _check_soft(v, fc, t, S, 1.0, sigma)
    v1 = torch.cat([v, v[:, :1]], 1).contiguous()
    with pytest.raises(ValueError, match="shared-memory"):
        ops.render_silhouettes(v1, fc, t, S, 1.0, 0.0)


def test_c_abi_argument_checks():
    """sil_prepare and the entry points' pointer checks: each bad argument gives B200SMPL_ERR_INVALID (ValueError
    through _lib.check) without launching a kernel or writing an output."""
    lib = _lib.load()
    S, B, V = 16, 2, 3
    v = _mesh([[2.0, 2.0], [14.0, 3.0], [5.0, 13.0]], S).expand(B, V, 3).contiguous()
    t = _cam_t().expand(B, 3).contiguous()
    fc = torch.tensor([[0, 1, 2]], dtype=torch.int32, device=DEV)
    alpha = torch.full((B, S, S), 7.0, device=DEV)
    ga = torch.ones(B, S, S, device=DEV)
    gv, gt = torch.full_like(v, 7.0), torch.full_like(t, 7.0)
    target = torch.ones(B, S, S, dtype=torch.uint8, device=DEV)
    loss = torch.full((B,), 7.0, device=DEV)

    def args(**kw):
        a = dict(batch=B, num_verts=V, num_faces=1, img_wh=S, focal_length=1.0, sigma=1.0, vertices=v.data_ptr(),
                 cam_t=t.data_ptr(), faces=fc.data_ptr(), workspace=None, workspace_bytes=0)
        a.update(kw)
        return ctypes.byref(_lib.SilhouetteArgs(**a))

    def calls(p, alpha_p=alpha.data_ptr(), ga_p=ga.data_ptr(), gv_p=gv.data_ptr(), gt_p=gt.data_ptr(),
              target_p=target.data_ptr(), loss_p=loss.data_ptr(), weight=1.0):
        return [lambda: lib.b200smpl_silhouette_render(p, alpha_p, None),
                lambda: lib.b200smpl_silhouette_render_backward(p, ga_p, gv_p, gt_p, None),
                lambda: lib.b200smpl_silhouette_loss(p, target_p, weight, loss_p, gv_p, gt_p, None)]

    bad = [args(batch=0), args(num_verts=2), args(num_verts=65536), args(num_faces=0), args(img_wh=0),
           args(img_wh=16385), args(sigma=float("nan")), args(sigma=-1.0), args(sigma=float("inf")),
           args(focal_length=0.0), args(focal_length=float("inf")), args(focal_length=float("nan")),
           args(vertices=None), args(cam_t=None), args(faces=None), None]
    cases = [c for p in bad for c in calls(p)]
    cases += [calls(args(), alpha_p=None)[0], calls(args(), ga_p=None)[1], calls(args(), gv_p=None)[1],
              calls(args(), gt_p=None)[1], calls(args(), target_p=None)[2], calls(args(), loss_p=None)[2],
              calls(args(), gv_p=None)[2], calls(args(), gt_p=None)[2], calls(args(), weight=float("nan"))[2],
              calls(args(sigma=0.0))[1], calls(args(sigma=0.0))[2]]
    torch.cuda.synchronize()
    n0 = lib.b200smpl_launch_count()
    for i, call in enumerate(cases):
        rc = call()
        assert rc == _lib.ERR_INVALID, (i, rc)
        with pytest.raises(ValueError):
            _lib.check(rc, "case {}".format(i))
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0
    for x in (alpha, gv, gt, loss):
        assert bool((x == 7.0).all())
    # the valid arguments do launch
    _lib.check(calls(args())[0](), "render")
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 + 1 and float(alpha.max()) > 0.5
