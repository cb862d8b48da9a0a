"""GPU tests of the proxy-representation kernel (csrc/proxy.cu, b200smpl_proxy_representation, ops.proxy_representation)
against the fp64 oracle (oracle/proxy_oracle.py), and of the regressor's graphed training step fed by detections
(regressor.ProxyInputs)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import proxy_oracle as PO
from soccerplayershapepose_b200 import _lib, config, ops, regressor
from soccerplayershapepose_b200.smpl import SMPL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
K = 17
HEAT_TOL = 2e-6


def _inputs(B, in_wh, seed, K=K, vis=True, mask_dtype=torch.uint8):
    """Masks (blobs plus noise), keypoints spread over and past the image with the border and the special values
    mixed in, and vis with some zeros."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(in_wh), torch.arange(in_wh), indexing="ij")
    cx, cy = torch.rand(B, 1, 1, generator=g) * in_wh, torch.rand(B, 1, 1, generator=g) * in_wh
    r = torch.rand(B, 1, 1, generator=g) * in_wh * 0.4 + 1
    masks = ((xx - cx) ** 2 + (yy - cy) ** 2 < r ** 2) ^ (torch.rand(B, in_wh, in_wh, generator=g) < 0.05)
    kp = torch.rand(B, K, 2, generator=g) * 1.4 * in_wh - 0.2 * in_wh
    special = torch.tensor([0.0, in_wh - 1.0, float(in_wh), -0.75, -1.0, in_wh - 0.5, float("nan"), float("inf"),
                            -1e9, 0.999])
    pick = torch.rand(B, K, 2, generator=g) < 0.25
    kp = torch.where(pick, special[torch.randint(0, len(special), (B, K, 2), generator=g)], kp).float()
    v = (torch.rand(B, K, generator=g) > 0.2) if vis else None
    if mask_dtype == torch.float32:
        masks = torch.where(masks, 0.5 + 0.5 * torch.rand(masks.shape, generator=g),
                            0.4999 * torch.rand(masks.shape, generator=g))
    else:
        masks = masks.to(mask_dtype)
    return masks.to(DEV), kp.to(DEV), None if v is None else v.to(DEV)


def _check(got, masks, kp, vis, out_wh, bodies):
    """got (B, 1 + K, S, S) against the fp64 oracle on the given bodies: channel 0 exact, heatmaps within HEAT_TOL."""
    idx = torch.tensor(bodies, device=DEV)
    ref = PO.proxy_representation(masks[idx].cpu().numpy(), kp[idx].cpu().numpy(),
                                  None if vis is None else vis[idx].cpu().numpy(), out_wh)
    g = got[idx].cpu().double().numpy()
    np.testing.assert_array_equal(g[:, 0], ref[:, 0])
    err = np.abs(g[:, 1:] - ref[:, 1:])
    assert err.max() <= HEAT_TOL, float(err.max())
    return ref


CASES = [(1, 512, 256), (37, 512, 255), (300, 512, 256), (1, 256, 1), (37, 100, 37), (37, 256, 300), (1, 100, 300),
         (300, 256, 37), (37, 512, 256), (300, 100, 1)]


@pytest.mark.parametrize("B,in_wh,out_wh", CASES)
def test_matches_oracle_in_both_layouts(B, in_wh, out_wh):
    masks, kp, vis = _inputs(B, in_wh, 10 * B + in_wh + out_wh)
    a = ops.proxy_representation(masks, kp, vis, out_wh)
    b = ops.proxy_representation(masks, kp, vis, out_wh, channels_last=True)
    assert a.is_contiguous() and b.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(a, b)                               # the same values, bit for bit
    bodies = sorted({0, B // 2, B - 1} | set(range(min(B, 4))))
    ref = _check(a, masks, kp, vis, out_wh, bodies)
    # the cases hold visible centres inside the image and zero channels from vis and from the special values
    assert (ref[:, 1:].reshape(len(bodies), K, -1).max(-1) == 1.0).any()
    assert (ref[:, 1:].reshape(len(bodies), K, -1).max(-1) == 0.0).any()


@pytest.mark.parametrize("mask_dtype", [torch.bool, torch.float32])
def test_mask_dtypes_and_no_vis(mask_dtype):
    masks, kp, _ = _inputs(5, 512, 3, vis=False, mask_dtype=mask_dtype)
    got = ops.proxy_representation(masks, kp, None, 256, std=2.5)
    ref = PO.proxy_representation(masks.cpu().numpy(), kp.cpu().numpy(), None, 256, std=2.5)
    np.testing.assert_array_equal(got[:, 0].cpu().numpy(), ref[:, 0])
    assert np.abs(got[:, 1:].cpu().double().numpy() - ref[:, 1:]).max() <= HEAT_TOL
    m7 = torch.from_numpy(PO.binary_mask(masks.cpu().numpy()).astype(np.uint8) * 7).to(DEV)   # non-zero = inside
    assert torch.equal(ops.proxy_representation(m7, kp, None, 256, std=2.5), got)


def test_peak_truncation_and_vis_at_512_to_256():
    """The three places a wrong rule shows at the reference's sizes: the centre is truncated, not rounded; the mask
    is sampled at 2 dst; vis zeroes its channel."""
    masks = torch.zeros(2, 512, 512, dtype=torch.uint8, device=DEV)
    masks[:, 1::2, 1::2] = 1                               # only odd source pixels are inside
    masks[1, 10, 20] = 1
    kp = torch.tensor([[[101.9, 57.3], [-1.5, -1.5]], [[3.0, 3.0], [7.0, 9.0]]], device=DEV)
    vis = torch.tensor([[1, 1], [1, 0]], device=DEV)
    out = ops.proxy_representation(masks, kp, vis, 256)
    assert not bool(out[0, 0].any()) and float(out[1, 0, 5, 10]) == 1.0 and float(out[1, 0].sum()) == 1.0
    assert float(out[0, 1, 28, 50]) == 1.0 and float(out[0, 1].max()) == 1.0
    assert float(out[0, 2, 0, 0]) == 1.0
    assert float(out[1, 1, 1, 1]) == 1.0
    assert not bool(out[1, 2].any())


def test_deterministic_and_batch_position_independent():
    B = 64
    masks, kp, vis = _inputs(B, 512, 5)
    for cl in (False, True):
        a = ops.proxy_representation(masks, kp, vis, 256, channels_last=cl)
        for _ in range(3):
            assert torch.equal(ops.proxy_representation(masks, kp, vis, 256, channels_last=cl), a)
        perm = torch.randperm(B, generator=torch.Generator().manual_seed(2)).to(DEV)
        p = ops.proxy_representation(masks[perm].contiguous(), kp[perm].contiguous(), vis[perm].contiguous(), 256,
                                     channels_last=cl)
        assert torch.equal(p, a[perm])


def _call(m, k, v, out_ptr, S, cl, **kw):
    """The C-ABI entry on masks m, keypoints k, vis v (uint8 or None); kw overrides fields of the argument struct."""
    a = dict(batch=m.shape[0], in_wh=m.shape[1], out_wh=S, num_keypoints=k.shape[1], channels_last=int(cl),
             reserved0=0, std=4.0, masks=m.data_ptr(), keypoints=k.data_ptr(), vis=None if v is None else v.data_ptr())
    a.update(kw)
    return _lib.load().b200smpl_proxy_representation(ctypes.byref(_lib.ProxyArgs(**a)), out_ptr,
                                                     ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream))


@pytest.mark.parametrize("out_wh", [37, 256, 300])
@pytest.mark.parametrize("cl", [False, True])
def test_unaligned_output_keeps_guard_bands(out_wh, cl):
    """The output at 4, 8 and 12 bytes past a 16-byte boundary: the same values, and the sentinel bands on both
    sides untouched (the kernel's scalar head and tail around its 16-byte stores)."""
    B, GUARD = 3, 1024
    masks, kp, vis = _inputs(B, 512, out_wh, mask_dtype=torch.uint8)
    vis8 = vis.to(torch.uint8)
    want = ops.proxy_representation(masks, kp, vis, out_wh, channels_last=cl)
    flat = want.permute(0, 2, 3, 1).reshape(-1) if cl else want.reshape(-1)
    n = flat.numel()
    for off in (1, 2, 3):
        raw = torch.full((GUARD + off + n + GUARD,), -7.25, device=DEV)
        assert raw.data_ptr() % 16 == 0
        view = raw[GUARD + off:GUARD + off + n]
        _lib.check(_call(masks, kp, vis8, view.data_ptr(), out_wh, cl), "proxy_representation")
        torch.cuda.synchronize()
        assert torch.equal(view, flat), off
        assert bool((raw[:GUARD + off] == -7.25).all()) and bool((raw[GUARD + off + n:] == -7.25).all())


def test_out_argument_and_graph_capture():
    B, S = 8, 256
    masks, kp, vis = _inputs(B, 512, 11)
    for cl in (False, True):
        fmt = torch.channels_last if cl else torch.contiguous_format
        out = torch.empty(B, 1 + K, S, S, device=DEV, memory_format=fmt)
        sm, sk, sv = masks.clone(), kp.clone(), vis.clone()
        ops.proxy_representation(sm, sk, sv, S, channels_last=cl, out=out)   # warm
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            r = ops.proxy_representation(sm, sk, sv, S, channels_last=cl, out=out)
        assert r is out
        m2, k2, v2 = _inputs(B, 512, 12)
        sm.copy_(m2); sk.copy_(k2); sv.copy_(v2)
        out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, ops.proxy_representation(m2, k2, v2, S, channels_last=cl))
        wrong = torch.empty(B, 1 + K, S, S, device=DEV,
                            memory_format=torch.contiguous_format if cl else torch.channels_last)
        with pytest.raises(ValueError):
            ops.proxy_representation(masks, kp, vis, S, channels_last=cl, out=wrong)
    with pytest.raises(ValueError):
        ops.proxy_representation(masks, kp, vis, S, out=torch.empty(B, K, S, S, device=DEV))
    with pytest.raises(TypeError):
        ops.proxy_representation(masks.to(torch.int32), kp, vis, S)
    with pytest.raises(ValueError):
        ops.proxy_representation(masks, kp[:, :3], vis, S)


def test_one_launch_per_call():
    lib = _lib.load()
    masks, kp, vis = _inputs(4, 512, 13)
    ops.proxy_representation(masks, kp, vis)
    torch.cuda.synchronize()
    n0 = lib.b200smpl_launch_count()
    ops.proxy_representation(masks, kp, vis, channels_last=True)
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 + 1


def test_cabi_argument_checks():
    """Each bad argument gives B200SMPL_ERR_INVALID without launching a kernel or writing the output; the limits
    themselves are accepted."""
    lib = _lib.load()
    masks, kp, vis = _inputs(2, 64, 14)
    vis8 = vis.to(torch.uint8)
    out = torch.full((2 * 18 * 16 * 16,), 3.0, device=DEV)
    p = out.data_ptr()
    bad = [dict(batch=0), dict(batch=-1), dict(in_wh=0), dict(in_wh=16385), dict(out_wh=0), dict(out_wh=16385),
           dict(num_keypoints=0), dict(num_keypoints=_lib.PROXY_MAX_KEYPOINTS + 1), dict(std=0.0), dict(std=-1.0),
           dict(std=float("nan")), dict(std=float("inf")), dict(channels_last=2), dict(masks=None),
           dict(keypoints=None)]
    torch.cuda.synchronize()
    n0 = lib.b200smpl_launch_count()
    for i, kw in enumerate(bad):
        rc = _call(masks, kp, vis8, p, 16, False, **kw)
        assert rc == _lib.ERR_INVALID, (i, kw, rc)
        with pytest.raises(ValueError):
            _lib.check(rc, "case {}".format(i))
    assert _call(masks, kp, vis8, None, 16, False) == _lib.ERR_INVALID
    assert lib.b200smpl_proxy_representation(None, p, None) == _lib.ERR_INVALID
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 and bool((out == 3.0).all())
    _lib.check(_call(masks, kp, vis8, p, 16, False), "valid")
    _lib.check(_call(masks, kp, None, p, 16, True, std=1e-3), "valid, no vis")
    kp32 = torch.zeros(2, _lib.PROXY_MAX_KEYPOINTS, 2, device=DEV)
    big = torch.empty(2, 1 + _lib.PROXY_MAX_KEYPOINTS, 16, 16, device=DEV)
    _lib.check(_call(masks, kp32, None, big.data_ptr(), 16, False), "K at the limit")
    torch.cuda.synchronize()
    assert lib.b200smpl_launch_count() == n0 + 3
    assert float(big[:, 1:, 0, 0].min()) == 1.0


# ---- the graphed training step fed by detections -------------------------------------------------------------------
@pytest.fixture(scope="module")
def smpl(synthetic_model):
    return SMPL(model_data=synthetic_model, mode="fp32").to(DEV)


def _labels(smpl, B, seed):
    g = torch.Generator().manual_seed(seed)
    betas = torch.randn(B, 10, generator=g).to(DEV)
    pose = (torch.randn(B, 72, generator=g) * 0.3).to(DEV)
    cam = torch.tensor([0.9, 0.0, 0.0], device=DEV).repeat(B, 1)
    with torch.no_grad():
        t = smpl(betas=betas, body_pose=pose[:, 3:], global_orient=pose[:, :3])
        rot = ops.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
        j2d = ops.orthographic_project(t.joints, cam, 512.0)[:, config.SMPL_TO_KPRCNN_MAP, :].contiguous()
        masks = smpl.render_silhouettes(t.vertices, cam, img_wh=512, sigma=0.0, proj_wh=512) > 0.5
    labels = {"verts": t.vertices, "joints3D": t.joints[:, config.ALL_JOINTS_TO_COCO_MAP, :].contiguous(),
              "shape_params": betas, "pose_params_rot_matrices": rot, "joints2D": j2d}
    return labels, masks, j2d


class _SmallEncoder(torch.nn.Module):
    """Non-overlapping convolution -> ReLU -> mean pool -> IEF head: every kernel of its step is deterministic under
    cudnn.deterministic."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(1 + K, 16, 8, 8)
        self.ief = regressor.IEFModule((32, 32), in_features=16)
        with torch.no_grad():
            self.ief.fc3.weight.mul_(0.05)

    def forward(self, x):
        return self.ief(torch.relu(self.conv(x)).mean(dim=(2, 3)))


def test_graphed_step_from_detections_is_bitwise_the_step_from_prebuilt_proxies(smpl):
    """GraphedTrainStep(ProxyInputs(...)) against GraphedTrainStep fed ops.proxy_representation(...) of the same
    inputs, from the same initial parameters: bitwise the same losses over three steps, with new inputs each step."""
    B = 6
    labels, masks, j2d = _labels(smpl, B, 1)
    crit_w = {"shape_params": 0.1, "pose_params": 0.1}
    was = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        torch.manual_seed(0)
        net_a = _SmallEncoder().to(DEV)
        net_b = _SmallEncoder().to(DEV)
        net_b.load_state_dict(net_a.state_dict())
        crit_a = regressor.MultiTaskLoss(tuple(crit_w), crit_w).to(DEV)
        crit_b = regressor.MultiTaskLoss(tuple(crit_w), crit_w).to(DEV)
        g6, gproj = regressor.gpu_ops()
        vis = torch.ones(B, K, dtype=torch.bool, device=DEV)
        feats = ops.proxy_representation(masks, j2d, vis)
        ga = regressor.GraphedTrainStep(net_a, crit_a, smpl, regressor.ProxyInputs(masks, j2d, vis), labels, g6, gproj,
                                        lr=1e-3, warmup=2)
        gb = regressor.GraphedTrainStep(net_b, crit_b, smpl, feats, labels, g6, gproj, lr=1e-3, warmup=2)
        assert ga.features.shape == (B, 1 + K, 256, 256) and ga.features.is_contiguous()
        gen = torch.Generator().manual_seed(3)
        la, lb = [], []
        for step in range(3):
            kp = (j2d + torch.randn(j2d.shape, generator=gen).to(DEV) * 4).contiguous()
            v = (torch.rand(B, K, generator=gen) > 0.2).to(DEV)
            m = masks.roll(step, dims=2).contiguous()
            la.append(ga(regressor.ProxyInputs(m, kp, v), labels).item())
            lb.append(gb(ops.proxy_representation(m, kp, v), labels).item())
            assert torch.equal(ga.features, gb.features)
        assert la == lb, (la, lb)
        assert la[0] != la[2]
        with pytest.raises(TypeError):
            ga(feats, labels)
    finally:
        torch.backends.cudnn.deterministic = was


def test_graphed_step_from_detections_with_the_encoder_and_fused_loss(smpl):
    """ResNet-18 in channels_last with the fused five-term loss: the step builds its proxy in the encoder's memory
    format and follows the step fed prebuilt proxies."""
    B = 4
    labels, masks, j2d = _labels(smpl, B, 2)
    w = {"verts": 1.0, "joints2D": 0.1, "joints3D": 1.0, "shape_params": 0.1, "pose_params": 0.1}
    torch.manual_seed(0)
    nets = [regressor.SingleInputRegressor(1 + K).to(DEV).to(memory_format=torch.channels_last) for _ in range(2)]
    nets[1].load_state_dict(nets[0].state_dict())
    crits = [regressor.MultiTaskLoss(tuple(w), w).to(DEV) for _ in range(2)]
    g6, _ = regressor.gpu_ops()
    u8 = masks.to(torch.uint8)
    feats = ops.proxy_representation(u8, j2d, channels_last=True)
    ga = regressor.GraphedTrainStep(nets[0], crits[0], smpl, regressor.ProxyInputs(u8, j2d), labels, g6, None,
                                    warmup=2, fused_loss=True)
    gb = regressor.GraphedTrainStep(nets[1], crits[1], smpl, feats, labels, g6, None, warmup=2, fused_loss=True)
    assert ga.features.is_contiguous(memory_format=torch.channels_last) and not ga.features.is_contiguous()
    la = [ga(regressor.ProxyInputs(u8, j2d), labels).item() for _ in range(3)]
    lb = [gb(feats, labels).item() for _ in range(3)]
    assert torch.equal(ga.features, feats)
    np.testing.assert_allclose(la, lb, rtol=1e-4)
