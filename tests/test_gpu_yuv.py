"""YUV 4:2:0 input (FDT_FMT_YUV_NV12 / _NV21 / _I420) through the C ABI.  The reference for every YUV frame is the library
itself run on cv2.cvtColor(frame) as a BGR frame (that path is pinned against the oracle elsewhere), so every comparison
here is exact equality: letterboxed bytes, face records, mesh / iris arrays and crops."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle import cv_ops as co
from test_oracle_yuv import FORMATS, i420_to, pad_stride
from yuv_ops import YUV_I420, YUV_NV12, YUV_NV21

pytestmark = pytest.mark.gpu

NV12, NV21, I420 = YUV_NV12, YUV_NV21, YUV_I420
S_OF = {"shortRange": 128, "full": 192, "backCamera": 256}


@pytest.fixture(scope="module")
def fdt(lib):
    import face_detection_tflite_b200 as pkg
    return pkg


_dets = {}


def detector(fdt, model, **kw):
    key = (model, tuple(sorted(kw.items())))
    if key not in _dets:
        _dets[key] = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], **kw)
    return _dets[key]


def even(img):
    h, w = img.shape[:2]
    return np.ascontiguousarray(img[:h - h % 2, :w - w % 2])


def to_yuv(bgr, fmt):
    """BGR photo -> YUV frame of `fmt` ((3H/2) x W u8) and the BGR frame it stands for (cvtColor of it)."""
    h, w = bgr.shape[:2]
    yuv = i420_to(fmt, cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420), w, h)
    return yuv, cv2.cvtColor(yuv, FORMATS[fmt])


def to_yuv_batch(frames, fmt):
    ys, bs = zip(*(to_yuv(f, fmt) for f in frames))
    return np.stack(ys), np.stack(bs)


def records(faces, counts, max_faces=100):
    """Raw bytes of every filled fdt_face slot, frame by frame."""
    sz = C.sizeof(faces._type_)
    base = C.addressof(faces)
    return [[C.string_at(base + (b * max_faces + j) * sz, sz) for j in range(int(counts[b]))] for b in range(len(counts))]


def h2d(d):
    return int(d._lib.fdt_last_h2d_bytes(d._h))


def run_device(d, frames, fmt, w, h, stride=None, **kw):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(frames).reshape(-1)).cuda()
    out = d.detectBatchRaw(int(t.data_ptr()), count=len(frames), width=w, height=h, matType=fmt, memKind=1, rowStride=stride, **kw)
    torch.cuda.synchronize()
    return out


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["shortRange", "full", "backCamera"])
@pytest.mark.parametrize("w,h", [(1280, 720), (1920, 1080), (130, 98), (6, 4), (128, 128)])
def test_letterbox_bytes_equal_bgr_path(fdt, model, w, h):
    d = detector(fdt, model)
    S = S_OF[model]
    rng = np.random.default_rng(w + 7 * h)
    for fmt in FORMATS:
        yuv = rng.integers(0, 256, (2, h * 3 // 2, w), dtype=np.uint8)
        want = [co.letterbox_u8(cv2.cvtColor(f, FORMATS[fmt]), S, S)[0] for f in yuv]
        d.detectBatchRaw(yuv, count=2, width=w, height=h, matType=fmt)
        got = d.debugLetterboxed(2)
        for b in range(2):
            assert np.array_equal(got[b], want[b]), (fmt, "host", b)
        run_device(d, yuv, fmt, w, h)
        got = d.debugLetterboxed(2)
        for b in range(2):
            assert np.array_equal(got[b], want[b]), (fmt, "device", b)


def _fast_frames(sample_images, w, h):
    from face_detection_tflite_b200 import synth
    return np.concatenate([synth.face_frames(5, w, h, start=1), synth.noise_frames(2, w, h, seed=9)])


def test_fast_mode_records_equal_bgr_path(fdt, sample_images):
    d = detector(fdt, "shortRange")
    photos = [even(img) for img in sample_images.values()]
    total = 0
    for fmt in FORMATS:
        for img in photos:
            h, w = img.shape[:2]
            yuv, bgr = to_yuv(img, fmt)
            f0, c0, _ = d.detectBatchRaw(bgr, count=1, width=w, height=h)
            f1, c1, _ = d.detectBatchRaw(yuv, count=1, width=w, height=h, matType=fmt)
            assert records(f1, c1) == records(f0, c0)
            faces = d.detectFacesFromMatBytes(yuv.tobytes(), width=w, height=h, matType=fmt, mode=fdt.FaceDetectionMode.fast)
            assert [f.detectionData for f in faces] == [f.detectionData for f in d.detectFacesFromMat(bgr, mode=fdt.FaceDetectionMode.fast)]
            total += int(c1.sum())
        yuv, bgr = to_yuv_batch(_fast_frames(sample_images, 1280, 720), fmt)
        f0, c0, _ = d.detectBatchRaw(bgr, count=len(bgr), width=1280, height=720)
        f1, c1, _ = d.detectBatchRaw(yuv, count=len(yuv), width=1280, height=720, matType=fmt)
        assert records(f1, c1) == records(f0, c0)
        total += int(c1.sum())
    assert total >= 3 * 5                                            # every format saw faces


def test_host_batch_crosses_chunks_and_slots(fdt):
    """600 frames with maxBatch 256: three chunks over both pipeline slots; 640x360 -> 128x72 uploads the Y plane sparse
    (rows 5k+2, 5k+3) and the chroma plane whole (rows {1, 3, 4} of every 5)."""
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange", maxBatch=256)
    base = np.concatenate([synth.face_frames(20, 640, 360, start=2, max_side=300), synth.noise_frames(4, 640, 360, seed=3)])
    for fmt in FORMATS:
        yuv, bgr = to_yuv_batch(base, fmt)
        yuv, bgr = np.tile(yuv, (25, 1, 1)), np.tile(bgr, (25, 1, 1, 1))
        f0, c0, _ = d.detectBatchRaw(bgr, count=600, width=640, height=360)
        f1, c1, _ = d.detectBatchRaw(yuv, count=600, width=640, height=360, matType=fmt)
        assert records(f1, c1) == records(f0, c0) and c1.sum() >= 100
        fb = 640 * 360 * 3 // 2
        assert h2d(d) == 600 * (360 // 5 * 2 * 640 + 640 * 360 // 2) < 600 * fb


@pytest.mark.parametrize("fmt", list(FORMATS))
def test_sparse_upload_bytes(fdt, fmt):
    from face_detection_tflite_b200 import synth
    n = 6
    for model, (w, h), per_frame in (("shortRange", (1280, 720), 276480), ("full", (1920, 1080), 622080), ("backCamera", (1280, 720), None)):
        d = detector(fdt, model)
        yuv, bgr = to_yuv_batch(synth.face_frames(n, w, h, start=1), fmt)
        f0, c0, _ = d.detectBatchRaw(bgr, count=n, width=w, height=h)
        f1, c1, _ = d.detectBatchRaw(yuv, count=n, width=w, height=h, matType=fmt)
        assert records(f1, c1) == records(f0, c0), model
        assert np.array_equal(d.debugLetterboxed(n), np.stack([co.letterbox_u8(b, S_OF[model], S_OF[model])[0] for b in bgr]))
        if per_frame is not None:
            assert h2d(d) == n * per_frame, model
        else:
            # back camera, 720 -> 144: Y rows 5k+2, 5k+3 go up sparse, the chroma plane (rows {1, 3, 4} of every 5) whole
            assert h2d(d) == n * (720 // 5 * 2 * 1280 + 1280 * 360) < n * w * h * 3 // 2


def _out_of_frame(img_hw, cx, cy, size, theta_arg, out):
    """True when the crop extractAlignedSquare(cx, cy, size, theta_arg, out) takes taps from outside the frame."""
    mask = np.full(img_hw + (3,), 255, np.uint8)
    m = co.extract_aligned_square(mask, cx, cy, size, theta_arg, out)
    return m is not None and bool((m < 255).any())


def test_standard_and_full_mode_equal_bgr_path(fdt, sample_images, lib):
    d = detector(fdt, "shortRange")
    photos = [even(img) for img in sample_images.values()]
    lm = sample_images["landmark-ex1.jpg"]
    photos.append(np.ascontiguousarray(lm[:640, 380:1020]))          # the face reaches the left and bottom borders
    border_crops = faces_seen = 0
    for fmt in FORMATS:
        for img in photos:
            h, w = img.shape[:2]
            yuv, bgr = to_yuv(img, fmt)
            for mode in (fdt.FaceDetectionMode.standard, fdt.FaceDetectionMode.full):
                taps = []
                for frame, mt in ((bgr, 16), (yuv, fmt)):
                    f, c, mesh, iris = d.detectBatchRaw(frame, count=1, width=w, height=h, matType=mt, mode=mode, withIris=True)
                    n = int(c[0])
                    mcrops, raw, flag = d.debugMeshStage(max(n, 1))
                    t = [records(f, c), mesh[:, :n].copy(), mcrops.copy(), raw.copy(), flag.copy()]
                    if mode == fdt.FaceDetectionMode.full:
                        icrops, rois, cont, ir = d.debugIrisStage(max(n, 1))
                        t += [iris[:, :n].copy(), icrops.copy(), rois.copy(), cont.copy(), ir.copy()]
                    taps.append(t)
                faces_seen += len(taps[0][0][0])
                for a, b in zip(taps[0], taps[1]):
                    if isinstance(a, list):
                        assert a == b
                    else:
                        assert a.shape == b.shape and np.array_equal(a, b, equal_nan=a.dtype.kind == "f")
                if mode == fdt.FaceDetectionMode.full:
                    for r in taps[1][7]:
                        border_crops += _out_of_frame((h, w), r[0], r[1], r[2], r[3], 64)
            # face crops: the ROI of the detector's keypoints (fast mode)
            ff, fc, _ = d.detectBatchRaw(bgr, count=1, width=w, height=h)
            for j in range(int(fc[0])):
                out10 = (C.c_double * 10)()
                lib.fdt_host_face_roi((C.c_double * 12)(*ff[j].keypoints), float(w), float(h), 192, out10)
                border_crops += _out_of_frame((h, w), out10[1], out10[2], out10[3], -out10[0], 192)
    assert faces_seen >= 3 * 2 * 3
    assert border_crops >= 1                                         # the BGR-zero rule for out-of-frame taps was exercised


def test_padded_row_stride(fdt, sample_images):
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange")
    frames = np.concatenate([synth.face_frames(3, 1280, 720, start=1), synth.noise_frames(1, 1280, 720, seed=4)])
    w, h = 1280, 720
    for fmt in FORMATS:
        yuv, _ = to_yuv_batch(frames, fmt)
        padded = np.stack([pad_stride(f, w, h, fmt, w + 64) for f in yuv])
        f0, c0, _ = d.detectBatchRaw(yuv, count=4, width=w, height=h, matType=fmt)
        lb0 = d.debugLetterboxed(4)
        f1, c1, _ = d.detectBatchRaw(padded, count=4, width=w, height=h, matType=fmt, rowStride=w + 64)
        assert records(f1, c1) == records(f0, c0) and np.array_equal(d.debugLetterboxed(4), lb0)
        f2, c2, _ = run_device(d, padded, fmt, w, h, stride=w + 64)
        assert records(f2, c2) == records(f0, c0) and np.array_equal(d.debugLetterboxed(4), lb0)
        # the crop warps read the padded planes too
        img = even(sample_images["landmark-ex1.jpg"])
        ph, pw = img.shape[:2]
        y, _ = to_yuv(img, fmt)
        full = fdt.FaceDetectionMode.full
        a = d.detectBatchRaw(y, count=1, width=pw, height=ph, matType=fmt, mode=full, withIris=True)
        b = d.detectBatchRaw(pad_stride(y, pw, ph, fmt, pw + 64), count=1, width=pw, height=ph, matType=fmt, mode=full,
                             rowStride=pw + 64, withIris=True)
        c = run_device(d, pad_stride(y, pw, ph, fmt, pw + 64)[None], fmt, pw, ph, stride=pw + 64, mode=full, withIris=True)
        assert int(a[1][0]) == 1
        for other in (b, c):
            assert records(other[0], other[1]) == records(a[0], a[1])
            assert np.array_equal(other[2], a[2]) and np.array_equal(other[3], a[3])


def test_multi_device_nv12(fdt):
    import torch
    from face_detection_tflite_b200 import synth
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    frames, _ = to_yuv_batch(np.concatenate([synth.face_frames(21, 640, 360, max_side=300), synth.noise_frames(2, 640, 360)]), NV12)
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=8)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=8)
    for mode in (fdt.FaceDetectionMode.fast, fdt.FaceDetectionMode.full):
        a = multi.detectBatchRaw(frames, count=23, width=640, height=360, matType=NV12, mode=mode, withIris=True)
        b = one.detectBatchRaw(frames, count=23, width=640, height=360, matType=NV12, mode=mode, withIris=True)
        assert records(a[0], a[1]) == records(b[0], b[1]) and int(b[1].sum()) >= 10
        if mode == fdt.FaceDetectionMode.full:
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    one.dispose(); multi.dispose()


def test_status_codes(fdt, lib):
    from face_detection_tflite_b200 import _ffi
    d = detector(fdt, "shortRange")
    h = d._h
    faces = (_ffi.FdtFace * 100)()
    cnt = C.c_int32()
    buf = np.zeros(4096, np.uint8)
    p = buf.ctypes.data
    for fmt in FORMATS:
        assert lib.fdt_detect_batch(h, p, 1, 7, 4, 8, fmt, 0, 0, faces, C.byref(cnt), None, None) == _ffi.FDT_ERR_BAD_ARG     # odd width
        assert lib.fdt_detect_batch(h, p, 1, 8, 5, 8, fmt, 0, 0, faces, C.byref(cnt), None, None) == _ffi.FDT_ERR_BAD_ARG     # odd height
        assert lib.fdt_detect_batch(h, p, 1, 8, 4, 6, fmt, 0, 0, faces, C.byref(cnt), None, None) == _ffi.FDT_ERR_SIZE_MISMATCH
        assert lib.fdt_detect_one(h, p, 47, 8, 4, fmt, 0, faces, C.byref(cnt), None, None) == _ffi.FDT_ERR_SIZE_MISMATCH
        assert lib.fdt_detect_one(h, p, 48, 8, 4, fmt, 0, faces, C.byref(cnt), None, None) == _ffi.FDT_OK and cnt.value == 0
        rc_odd = lib.fdt_detect_batch(h, p, 1, 8, 4, 9, fmt, 0, 0, faces, C.byref(cnt), None, None)
        assert rc_odd == (_ffi.FDT_ERR_BAD_ARG if fmt == I420 else _ffi.FDT_OK)                                   # odd stride: I420 only
        rois = np.array([[4.0, 2.0, 4.0, 0.0]])
        crops = np.zeros((1, 8, 8, 3), np.uint8)
        assert lib.fdt_extract_aligned_squares(h, p, 8, 4, 8, fmt, rois.ctypes.data, 1, 8, crops.ctypes.data, None) == _ffi.FDT_ERR_BAD_ARG
        with pytest.raises(ValueError):
            d.detectBatchRaw(buf[:47], count=1, width=8, height=4, matType=fmt)
        with pytest.raises(ValueError):
            d.detectFacesFromMatBytes(buf[:47], width=8, height=4, matType=fmt)
        assert d.detectBatchRaw(buf[:48], count=1, width=8, height=4, matType=fmt)[1][0] == 0
