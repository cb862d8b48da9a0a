"""CPU tests of the fp64 proxy-representation oracle (oracle/proxy_oracle.py, DESIGN.md section 12): the pieces of
the definition one by one, and agreement with the reference's two functions transcribed literally in float32."""
import numpy as np
import pytest

from oracle import proxy_oracle as PO


def _one(kp, in_wh=512, out_wh=256, vis=None, std=4.0):
    masks = np.zeros((1, in_wh, in_wh), np.uint8)
    v = None if vis is None else np.asarray([vis])
    return PO.proxy_representation(masks, np.asarray([kp], np.float32), v, out_wh, std)[0]


def test_peak_is_one_at_the_truncated_centre():
    out = _one([[101.9, 57.3], [3.0, 500.0]])
    # 101.9 / 2 = 50.95 -> 50, 57.3 / 2 = 28.65 -> 28; (x, y) is (column, row)
    assert out[1].max() == 1.0 and np.unravel_index(out[1].argmax(), out[1].shape) == (28, 50)
    assert out[2][250, 1] == 1.0
    np.testing.assert_allclose(out[1][28, 54], np.exp(-0.5), rtol=1e-15)       # one std to the right
    np.testing.assert_allclose(out[1][32, 54], np.exp(-1.0), rtol=1e-15)


def test_negative_coordinates_truncate_toward_zero():
    out = _one([[-1.5, -1.5], [-2.5, 9.0]])               # -0.75 -> 0, -1.25 -> -1 (not floor: -2)
    assert out[1][0, 0] == 1.0
    np.testing.assert_allclose(out[2][4, 0], np.exp(-1.0 / 32), rtol=1e-15)   # centre (-1, 4): column 0 is 1 px off
    c, ok = PO.centres(np.array([[[-1.5, -1.5], [-2.5, 9.0]]], np.float32), 512, 256)
    assert ok.all() and c[0].tolist() == [[0, 0], [-1, 4]]


def test_downscale_samples_source_pixel_two_dst():
    rng = np.random.default_rng(0)
    m = rng.integers(0, 2, (2, 512, 512)).astype(np.uint8)
    out = PO.proxy_representation(m, np.zeros((2, 1, 2), np.float32), None, 256)
    np.testing.assert_array_equal(out[:, 0], m[:, ::2, ::2])
    assert not np.array_equal(out[:, 0], m[:, 1::2, 1::2])


@pytest.mark.parametrize("in_wh,out_wh", [(100, 256), (37, 300), (256, 256), (300, 37), (512, 1)])
def test_resize_rule_and_identity(in_wh, out_wh):
    rng = np.random.default_rng(in_wh + out_wh)
    m = rng.random((1, in_wh, in_wh)).astype(np.float32)
    out = PO.proxy_representation(m, np.zeros((1, 1, 2), np.float32), None, out_wh)
    src = [(d * in_wh) // out_wh for d in range(out_wh)]
    assert src[0] == 0 and src[-1] <= in_wh - 1
    want = (m[0] >= 0.5)[np.ix_(src, src)]
    np.testing.assert_array_equal(out[0, 0], want)
    if in_wh == out_wh:
        np.testing.assert_array_equal(out[0, 0], m[0] >= 0.5)
    if out_wh > in_wh:                                   # upscaling repeats source pixels
        assert len(set(src)) == in_wh


def test_upscale_and_same_size_scale_the_keypoints():
    out = _one([[10.0, 20.0]], in_wh=100, out_wh=256)     # 25.6, 51.2 -> 25, 51
    assert np.unravel_index(out[1].argmax(), out[1].shape) == (51, 25)
    out = _one([[10.7, 20.2]], in_wh=256, out_wh=256)
    assert np.unravel_index(out[1].argmax(), out[1].shape) == (20, 10)


def test_vis_zeroes_its_channel():
    out = _one([[100.0, 100.0], [200.0, 200.0]], vis=[1, 0])
    assert out[1].max() == 1.0 and not out[2].any()


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf, 65536.0 * 2, -65540.0 * 2, 1e30])
def test_non_finite_or_huge_coordinates_give_zero_channels(bad):
    out = _one([[bad, 10.0], [10.0, bad], [10.0, 10.0]])
    assert not out[1].any() and not out[2].any() and out[3].max() == 1.0


def test_int16_range_edges():
    # scaled 32767.5 truncates to 32767 (kept); -32768.5 -> -32768 (kept); 32768 and -32769 would wrap (zeroed)
    c, ok = PO.centres(np.array([[[65535.0, 0.0], [-65537.0, 0.0], [65536.0, 0.0], [-65538.0, 0.0]]], np.float32),
                       512, 256)
    assert ok[0].tolist() == [True, True, False, False]
    assert c[0, :2, 0].tolist() == [32767, -32768]


@pytest.mark.parametrize("in_wh,out_wh", [(512, 256), (256, 256), (100, 64)])
def test_oracle_agrees_with_float32_reference_transcription(in_wh, out_wh):
    rng = np.random.default_rng(7)
    K = 17
    mask = (rng.random((in_wh, in_wh)) > 0.4).astype(np.uint8)
    kp = (rng.random((K, 2)) * 1.2 * in_wh - 0.1 * in_wh).astype(np.float32)
    ref = PO.reference_float32(mask, kp, in_wh, out_wh)
    got = PO.proxy_representation(mask[None], kp[None], None, out_wh)[0]
    assert ref.dtype == np.float32 and ref.shape == got.shape == (1 + K, out_wh, out_wh)
    np.testing.assert_array_equal(got[0], ref[0])
    assert np.abs(got[1:] - ref[1:]).max() < 1e-6
    assert (ref[1:].reshape(K, -1).max(1) == 1.0).sum() >= 8        # most centres fall inside the image


def test_cabi_entry_is_exported_and_checks_arguments_before_the_device():
    import ctypes
    from soccerplayershapepose_b200 import _lib
    lib = _lib.load()
    assert ctypes.sizeof(_lib.ProxyArgs) == 56
    assert lib.b200smpl_proxy_representation(None, None, None) == _lib.ERR_INVALID
    args = _lib.ProxyArgs(batch=1, in_wh=8, out_wh=8, num_keypoints=_lib.PROXY_MAX_KEYPOINTS + 1, channels_last=0,
                          reserved0=0, std=4.0, masks=16, keypoints=16, vis=None)
    assert lib.b200smpl_proxy_representation(ctypes.byref(args), 16, None) == _lib.ERR_INVALID
    assert "num_keypoints" in _lib.last_error()
