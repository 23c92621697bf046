"""YUV 4:2:0 -> BGR reference for the tests (test infrastructure, not product code): an integer restatement of
cv2.cvtColor(COLOR_YUV2BGR_NV12 / _NV21 / _I420), pinned byte for byte against cv2 in tests/test_oracle_yuv.py."""
from __future__ import annotations

import numpy as np

YUV_NV12, YUV_NV21, YUV_I420 = 0x1000, 0x1001, 0x1002


def yuv420_to_bgr(frame, width: int, height: int, fmt: int, row_stride: int = None) -> np.ndarray:
    """Integer restatement of OpenCV's 8-bit YUV420sp / YUV420p -> BGR conversion (imgproc/color_yuv.simd.hpp,
    BT.601 limited range, 20-bit fixed point).  `frame` holds height * row_stride * 3 / 2 bytes: the Y plane
    (row_stride bytes per row), then at height * row_stride either the interleaved chroma plane (NV12: U,V;
    NV21: V,U; same row stride) or, for I420, the U plane then the V plane (row_stride / 2 bytes per row).
    The chroma sample of pixel (x, y) is the one at (x / 2, y / 2).  Returns u8 [height, width, 3] BGR."""
    W, H = int(width), int(height)
    rs = W if row_stride is None else int(row_stride)
    buf = np.frombuffer(np.ascontiguousarray(frame).tobytes(), np.uint8)
    if buf.size != H * rs * 3 // 2:
        raise ValueError("frame length does not equal height * row_stride * 3 / 2")
    Y = buf[:H * rs].reshape(H, rs)[:, :W]
    if fmt in (YUV_NV12, YUV_NV21):
        uv = buf[H * rs:].reshape(H // 2, rs)[:, :W].reshape(H // 2, W // 2, 2)
        U, V = (uv[..., 0], uv[..., 1]) if fmt == YUV_NV12 else (uv[..., 1], uv[..., 0])
    elif fmt == YUV_I420:
        cs = rs // 2
        c = buf[H * rs:].reshape(H, cs)
        U, V = c[:H // 2, :W // 2], c[H // 2:, :W // 2]
    else:
        raise ValueError("unknown YUV format %#x" % fmt)
    up = lambda p: np.repeat(np.repeat(p.astype(np.int64), 2, 0), 2, 1)
    yy = np.maximum(Y.astype(np.int64) - 16, 0) * 1220542 + (1 << 19)
    u, v = up(U) - 128, up(V) - 128
    r = (yy + 1673527 * v) >> 20
    g = (yy - 852492 * v - 409993 * u) >> 20
    b = (yy + 2116026 * u) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)
