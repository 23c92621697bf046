"""The YUV 4:2:0 -> BGR reference (yuv_ops.yuv420_to_bgr) against cv2.cvtColor, byte for byte: NV12, NV21 and I420,
random frames and the sample photos, packed and padded row strides.  CPU only."""
import cv2
import numpy as np
import pytest

import yuv_ops as yo

FORMATS = {yo.YUV_NV12: cv2.COLOR_YUV2BGR_NV12, yo.YUV_NV21: cv2.COLOR_YUV2BGR_NV21, yo.YUV_I420: cv2.COLOR_YUV2BGR_I420}


def i420_to(fmt, yuv, w, h):
    """Repacks a cv2 I420 frame ((3H/2) x W) into `fmt`."""
    if fmt == yo.YUV_I420:
        return yuv
    flat = yuv[h:].reshape(-1)
    u, v = flat[:w * h // 4], flat[w * h // 4:]
    uv = np.stack([u, v] if fmt == yo.YUV_NV12 else [v, u], -1).reshape(h // 2, w)
    return np.concatenate([yuv[:h], uv])


def pad_stride(yuv, w, h, fmt, stride):
    """The same frame with `stride` bytes per Y row (chroma rows: stride for NV12 / NV21, stride / 2 for I420)."""
    out = np.full(h * stride * 3 // 2, 77, np.uint8)
    out[:h * stride].reshape(h, stride)[:, :w] = yuv[:h]
    if fmt == yo.YUV_I420:
        cs = stride // 2
        flat = yuv[h:].reshape(-1)
        out[h * stride:].reshape(h, cs)[:, :w // 2] = flat.reshape(h, w // 2)
    else:
        out[h * stride:].reshape(h // 2, stride)[:, :w] = yuv[h:]
    return out


@pytest.mark.parametrize("fmt", list(FORMATS))
@pytest.mark.parametrize("w,h", [(2, 2), (6, 4), (130, 98), (1280, 720), (1920, 1080)])
def test_random_frames_equal_cv2(fmt, w, h):
    rng = np.random.default_rng(w * 31 + h + fmt)
    yuv = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    want = cv2.cvtColor(yuv, FORMATS[fmt])
    assert np.array_equal(yo.yuv420_to_bgr(yuv, w, h, fmt), want)
    for extra in (2, 64):
        assert np.array_equal(yo.yuv420_to_bgr(pad_stride(yuv, w, h, fmt, w + extra), w, h, fmt, w + extra), want)


@pytest.mark.parametrize("fmt", list(FORMATS))
def test_sample_photos_equal_cv2(fmt, sample_images):
    for name, img in sample_images.items():
        h, w = (img.shape[0] // 2) * 2, (img.shape[1] // 2) * 2
        bgr = np.ascontiguousarray(img[:h, :w])
        yuv = i420_to(fmt, cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420), w, h)
        want = cv2.cvtColor(yuv, FORMATS[fmt])
        assert np.array_equal(yo.yuv420_to_bgr(yuv, w, h, fmt), want), name
        assert np.array_equal(yo.yuv420_to_bgr(pad_stride(yuv, w, h, fmt, w + 64), w, h, fmt, w + 64), want), name
        # the round trip through YUV is lossy, but stays close to the photo
        assert np.abs(want.astype(int) - bgr.astype(int)).mean() < 4.0


def test_rejects_wrong_length_and_format():
    yuv = np.zeros((6, 4), np.uint8)
    with pytest.raises(ValueError):
        yo.yuv420_to_bgr(yuv[:5], 4, 4, yo.YUV_NV12)
    with pytest.raises(ValueError):
        yo.yuv420_to_bgr(yuv, 4, 4, 16)
