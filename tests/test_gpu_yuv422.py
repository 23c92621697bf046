"""Packed YUV 4:2:2 frames (FDT_FMT_YUYV / _UYVY / _YVYU) through every detect entry point.

The library converts each tap as cv2.cvtColor(frame, COLOR_YUV2BGR_YUYV / _UYVY / _YVYU) converts the pixel (the rule is pinned
against cv2 in test_yuv422_host.py), before it is weighted.  So the bar throughout is bitwise equality with the library's own
BGR call on cv2.cvtColor(frame): face records, counts, mesh and iris arrays, letterboxed bytes, mesh / iris crops and the
caller's face crops, in all eight orientations, from host and device memory, uniform and mixed calls."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle.jpeg_ops import exif_transform
from test_gpu_orientation import INVERSE, Frame, assert_same, even, records, run, to_device
from test_gpu_rgb import as_format, border_crop, photos

pytestmark = pytest.mark.gpu

GRAY, BGR = 0, 16
NV12 = 0x1000
RGB, PLANAR = 0x1010, 0x1012
YUYV, UYVY, YVYU = 0x1020, 0x1021, 0x1022
NEW = [YUYV, UYVY, YVYU]
TO = {YUYV: cv2.COLOR_BGR2YUV_YUYV, UYVY: cv2.COLOR_BGR2YUV_UYVY, YVYU: cv2.COLOR_BGR2YUV_YVYU}
FROM = {YUYV: cv2.COLOR_YUV2BGR_YUYV, UYVY: cv2.COLOR_YUV2BGR_UYVY, YVYU: cv2.COLOR_YUV2BGR_YVYU}
S_OF = {"shortRange": 128, "full": 192, "backCamera": 256}


@pytest.fixture(scope="module")
def fdt(lib):
    import face_detection_tflite_b200 as pkg
    return pkg


_dets = {}


@pytest.fixture(scope="module", autouse=True)
def _release():
    """The handles of this module and torch's cached blocks go back before the next module runs."""
    yield
    import torch
    for d in _dets.values():
        d.dispose()
    _dets.clear()
    torch.cuda.empty_cache()


def detector(fdt, model, **kw):
    key = (model, tuple(sorted(kw.items())))
    if key not in _dets:
        _dets[key] = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], **kw)
    return _dets[key]


def as_422(s, mt, pad=0):
    """The BGR image s (even width) as a packed YUV 4:2:2 frame of format mt with `pad` bytes of row padding: (data [h, stride],
    row stride, the reference BGR image cv2.cvtColor(frame, COLOR_YUV2BGR_*))."""
    h, w = s.shape[:2]
    img = cv2.cvtColor(s, TO[mt])                                       # h x w x 2
    buf = np.full((h, 2 * w + pad), 77, np.uint8)
    buf[:, :2 * w] = img.reshape(h, 2 * w)
    return buf, 2 * w + pad, cv2.cvtColor(img, FROM[mt])


def stored(upright_bgr, o, mt, pad=0, seed=0):
    """The frame of format mt stored in orientation o whose upright image is upright_bgr; its reference (for the new formats)
    is the same oriented call on the stored frame converted to BGR."""
    s = exif_transform(upright_bgr, INVERSE[o])
    h, w = s.shape[:2]
    if mt in NEW:
        data, stride, ref = as_422(s, mt, pad)
    else:
        data, stride, ref = as_format(s, mt, pad, seed)
    return Frame(data, w, h, mt, stride, o, None if ref is None else Frame(ref, w, h, BGR, w * 3, o))


def ref_or_self(fr):
    return fr.ref if fr.mt in NEW else fr


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["shortRange", "full", "backCamera"])
def test_letterbox_bytes(fdt, sample_images, model):
    """Letterboxed bytes and records at camera sizes, an odd height, a tiny frame and the identity letterbox (S x S), with row
    strides of 2w and 2w + 3, uniform and mixed calls."""
    d = detector(fdt, model)
    S = S_OF[model]
    lm = sample_images["landmark-ex1.jpg"]
    for w, h in ((1280, 720), (1920, 1080), (130, 97), (6, 4), (S, S)):
        img = cv2.resize(lm, (w, h), interpolation=cv2.INTER_AREA)
        for mt in NEW:
            for pad in (0, 3):
                fr = stored(img, 1, mt, pad)
                want, _ = run(d, fr.ref)
                assert_same(run(d, fr)[0], want, (model, w, h, mt, pad))
                f = d.detectFramesRaw([fr.desc()])
                assert records(*f[:2]) == want[0] and np.array_equal(d.debugLetterboxed(1), want[1]), (model, w, h, mt, pad, "frames")


@pytest.mark.parametrize("mt", NEW)
def test_all_orientations_fast_host_and_device(fdt, sample_images, mt):
    d = detector(fdt, "shortRange")
    frames = []
    for k, img in enumerate(photos(sample_images)):
        for o in range(1, 9):
            frames.append(stored(even(img), o, mt, pad=(0, 6, 3)[(k + o) % 3]))
    faces = 0
    for fr in frames:
        want, n = run(d, fr.ref)
        faces += n
        assert_same(run(d, fr)[0], want, ("host", fr.o, fr.w, fr.h))
        t = to_device([fr.data])
        assert_same(run(d, fr, ptr=int(t[0].data_ptr()))[0], want, ("device", fr.o, fr.w, fr.h))
    assert faces >= 8 * 2
    # the same frames as one mixed call, host and device
    orients = [fr.o for fr in frames]
    got = d.detectFramesRaw([fr.desc() for fr in frames], orientations=orients)
    lb = d.debugLetterboxed(len(frames))
    ts = to_device([fr.data for fr in frames])
    got_dev = d.detectFramesRaw([fr.desc(int(t.data_ptr())) for fr, t in zip(frames, ts)], memKind=1, orientations=orients)
    assert records(*got_dev[:2]) == records(*got[:2])
    assert np.array_equal(d.debugLetterboxed(len(frames)), lb)
    for b, fr in enumerate(frames):
        want, _ = run(d, fr.ref)
        assert records(*got[:2])[b] == want[0][0], b
        assert np.array_equal(lb[b], want[1][0]), b


def test_standard_and_full_mode(fdt, sample_images):
    """Records, mesh and iris arrays and the mesh / iris crops (including taps past the frame border) in every orientation;
    uniform and mixed calls."""
    d = detector(fdt, "shortRange")
    imgs = [even(sample_images["landmark-ex1.jpg"]), border_crop(sample_images), even(sample_images["iris-detection-ex1.jpg"])]
    faces = 0
    for o in range(1, 9):
        for k, img in enumerate(imgs):
            mt = NEW[(o + k) % 3]
            fr = stored(img, o, mt, pad=(0, 8, 3)[k])
            for mode in (1, 2):
                want, n = run(d, fr.ref, mode)
                assert_same(run(d, fr, mode)[0], want, (o, mt, mode, img.shape))
                faces += n
                f = d.detectFramesRaw([fr.desc()], mode=mode, orientations=[o])
                w = d.detectBatchRaw(fr.ref.data, count=1, width=fr.w, height=fr.h, matType=BGR, mode=mode, withIris=True,
                                     orientation=o)
                assert records(*f[:2]) == records(*w[:2]), (o, mt, mode)
                assert np.array_equal(f[2], w[2]) and (mode == 1 or np.array_equal(f[3], w[3])), (o, mt, mode)
    assert faces >= 24
    # the border crop's mesh crop has out-of-frame taps, which stay BGR 0
    want, n = run(d, stored(imgs[1], 1, UYVY).ref, 1)
    assert n >= 1 and (want[3].reshape(-1, 3) == 0).all(axis=1).any()


def test_detect_one_and_batch_device(fdt, sample_images, lib):
    """fdt_detect_one (full mode, exactly 2 * width * height bytes) and fdt_detect_batch_device (fast mode)."""
    d = detector(fdt, "shortRange")
    mf = d._max_faces
    imgs = [even(sample_images["landmark-ex1.jpg"]), cv2.resize(sample_images["iris-detection-ex1.jpg"], (642, 359))]

    def one(data, w, h, mt):
        faces = (fdt._ffi.FdtFace * mf)()
        n = C.c_int32(0)
        mesh = np.zeros((mf, 468, 3), np.float32)
        iris = np.zeros((mf, 152, 3), np.float32)
        rc = lib.fdt_detect_one(d._h, data.ctypes.data, data.size, w, h, mt, 2, faces, C.byref(n), mesh.ctypes.data_as(fdt._ffi.f32p),
                                iris.ctypes.data_as(fdt._ffi.f32p))
        assert rc == 0, lib.fdt_last_error(d._h)
        return records(faces, [n.value]), mesh[:n.value].copy(), iris[:n.value].copy(), d.debugMeshStage(max(n.value, 1))[0].copy()

    def on_device(data, w, h, stride, mt, count):
        t = to_device([np.tile(data.reshape(-1), count)])[0]
        pf, pc = C.c_void_p(), C.c_void_p()
        assert lib.fdt_detect_batch_device(d._h, t.data_ptr(), count, w, h, stride, mt, 0, C.byref(pf), C.byref(pc)) == 0
        counts = np.zeros(count, np.int32)
        faces = (fdt._ffi.FdtFace * (count * mf))()
        assert lib.fdt_copy_to_host(d._h, counts.ctypes.data, pc, counts.nbytes) == 0
        assert lib.fdt_copy_to_host(d._h, C.addressof(faces), pf, C.sizeof(faces)) == 0
        return records(faces, counts), d.debugLetterboxed(count).copy()

    found = 0
    for img in imgs:
        h, w = img.shape[:2]
        for mt in NEW:
            data, stride, ref = as_422(img, mt)
            assert data.size == 2 * w * h
            want = one(ref, w, h, BGR)
            got = one(data, w, h, mt)
            assert got[0] == want[0], (mt, w, h)
            assert_same(got[1:], want[1:], (mt, w, h))
            found += len(want[0][0])
            a, b = on_device(data, w, h, stride, mt, 5), on_device(ref, w, h, w * 3, BGR, 5)
            assert a[0] == b[0] and np.array_equal(a[1], b[1]), (mt, w, h)
    assert found >= 2


def test_upload_bytes_and_launch_counts(fdt, sample_images):
    """Fast mode, host frames: a 1280x720 frame uploads rows 10k+4 and 10k+5 at 2 bytes per pixel (368,640 B, also stored
    sideways); launch counts equal BGR's for uniform and mixed calls, fast and full mode."""
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange")
    n = 6
    nbytes = lambda: int(d._lib.fdt_last_h2d_bytes(d._h))
    for (w, h), o in (((1280, 720), 1), ((1280, 720), 6), ((642, 359), 1)):
        src = synth.face_frames(n, w, h, start=1)
        for mt in NEW:
            frs = [stored(s, o, mt) for s in src]
            data = np.stack([f.data for f in frs])
            f, c, _ = d.detectBatchRaw(data, count=n, width=frs[0].w, height=frs[0].h, matType=mt, rowStride=frs[0].stride,
                                       orientation=o)
            got_bytes = nbytes()
            lb = d.debugLetterboxed(n)
            ref = np.stack([fr.ref.data for fr in frs])
            rf, rc, _ = d.detectBatchRaw(ref, count=n, width=frs[0].w, height=frs[0].h, matType=BGR, orientation=o)
            assert records(f, c) == records(rf, rc), (w, h, o, mt)
            assert np.array_equal(lb, d.debugLetterboxed(n)), (w, h, o, mt)
            if h == 720:
                assert got_bytes == n * 368640, (o, mt, got_bytes)
            else:
                assert got_bytes == n * 2 * w * h, (o, mt, got_bytes)     # 359 rows: no period, whole frames
    lm = even(sample_images["landmark-ex1.jpg"])
    for o in (1, 6):
        for mode in (0, 2):
            base = stored(lm, o, BGR)
            run(d, base, mode)
            want = d.lastLaunchCount()
            d.detectFramesRaw([base.desc()], mode=mode, orientations=[o])
            want_frames = d.lastLaunchCount()
            for mt in NEW:
                fr = stored(lm, o, mt)
                run(d, fr, mode)
                assert d.lastLaunchCount() == want, (o, mode, mt)
                d.detectFramesRaw([fr.desc()], mode=mode, orientations=[o])
                assert d.lastLaunchCount() == want_frames, (o, mode, mt, "frames")


def mixed(sample_images):
    """YUYV, UYVY, BGR, GRAY, NV12, RGB and planar RGB frames of different sizes and orientations, with padded rows."""
    lm, iris, group = (sample_images[k] for k in ("landmark-ex1.jpg", "iris-detection-ex1.jpg", "group-shot-bounding-box-ex1.jpeg"))
    imgs = [even(lm), even(iris), even(cv2.resize(group, (1920, 1080), interpolation=cv2.INTER_AREA)), cv2.resize(lm, (202, 134)),
            border_crop(sample_images)]
    kinds = [YUYV, UYVY, BGR, GRAY, NV12, RGB, PLANAR, YVYU]
    out = []
    k = 0
    for o in range(1, 9):
        for i, img in enumerate(imgs):
            mt = kinds[(k + i) % len(kinds)]
            out.append(stored(img, o, mt, pad=(0, 4, 16)[k % 3] if mt != NV12 else (0, 2, 16)[k % 3], seed=k))
            k += 1
    return out


@pytest.mark.parametrize("mode", [0, 2])
def test_mixed_call(fdt, sample_images, mode):
    """One mixed call over 4:2:2 and five other formats equals the same call with every 4:2:2 frame replaced by its BGR
    image, from host and device memory, over chunks of 4 (the call crosses max_batch)."""
    d = detector(fdt, "shortRange", maxBatch=4)
    frames = mixed(sample_images)
    assert {f.mt for f in frames} == {YUYV, UYVY, YVYU, BGR, GRAY, NV12, RGB, PLANAR}
    orients = [f.o for f in frames]
    got = d.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=orients)
    want = d.detectFramesRaw([ref_or_self(f).desc() for f in frames], mode=mode, orientations=orients)
    rec = records(*got[:2])
    assert rec == records(*want[:2])
    assert sum(map(len, rec)) >= 20
    if mode:
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    ts = to_device([f.data for f in frames])
    dev = d.detectFramesRaw([f.desc(int(t.data_ptr())) for f, t in zip(frames, ts)], mode=mode, memKind=1, orientations=orients)
    assert records(*dev[:2]) == rec
    if mode:
        assert np.array_equal(dev[2], got[2]) and np.array_equal(dev[3], got[3])
    # a 4-frame chunk's letterboxes against the same chunk with BGR references
    d.detectFramesRaw([f.desc() for f in frames[:4]], orientations=orients[:4])
    lb = d.debugLetterboxed(4).copy()
    d.detectFramesRaw([ref_or_self(f).desc() for f in frames[:4]], orientations=orients[:4])
    assert np.array_equal(lb, d.debugLetterboxed(4))


def test_uniform_call_crosses_max_batch(fdt, sample_images):
    """10 frames through chunks of 4, full mode, upright and sideways."""
    d4 = detector(fdt, "shortRange", maxBatch=4)
    lm = even(sample_images["landmark-ex1.jpg"])
    for mt in NEW:
        for o in (1, 6):
            frs = [stored(np.roll(lm, 16 * k, axis=1), o, mt, pad=3) for k in range(10)]
            got = d4.detectBatchRaw(np.stack([f.data for f in frs]), count=10, width=frs[0].w, height=frs[0].h, matType=mt,
                                    rowStride=frs[0].stride, mode=2, withIris=True, orientation=o)
            want = d4.detectBatchRaw(np.stack([f.ref.data for f in frs]), count=10, width=frs[0].w, height=frs[0].h, matType=BGR,
                                     mode=2, withIris=True, orientation=o)
            assert records(*got[:2]) == records(*want[:2]) and np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), (mt, o)
            assert sum(map(len, records(*got[:2]))) >= 10


@pytest.mark.parametrize("spec", [dict(kind="embedding", size=112, order="rgb", chw=True, dtype=np.float32,
                                       scale=(1 / 127.5,) * 3, bias=(-1.0,) * 3),
                                  dict(kind="face", size=96)])
def test_face_crops(fdt, sample_images, spec):
    """The caller's face crops (both kinds; float CHW RGB and u8 BGR) equal the BGR call's: uniform host and device calls in
    several orientations, fast and full mode, and a mixed call."""
    d = detector(fdt, "shortRange", maxBatch=4)
    d.setFaceCrops(fdt.FaceCropSpec(**spec))
    try:
        lm = even(sample_images["landmark-ex1.jpg"])
        total = 0
        for o in (1, 3, 6, 7):
            for k, mt in enumerate(NEW):
                fr = stored(lm, o, mt, pad=3 * k)
                for mode in (0, 2):
                    want, n = run(d, fr.ref, mode)
                    wc, wok = d.faceCrops()
                    got, _ = run(d, fr, mode)
                    gc, gok = d.faceCrops()
                    assert_same(got, want, (o, mt, mode))
                    assert len(wc) == n >= 1 and np.array_equal(gc, wc) and np.array_equal(gok, wok), (o, mt, mode)
                    total += n
                t = to_device([fr.data])
                got, _ = run(d, fr, 0, ptr=int(t[0].data_ptr()))
                gc, _ = d.faceCrops()
                run(d, fr.ref)
                assert np.array_equal(gc, d.faceCrops()[0]), (o, mt, "device")
        assert total >= 24
        frames = mixed(sample_images)[:12]
        orients = [f.o for f in frames]
        for mode in (0, 2):
            got = d.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=orients)
            gc, gok = d.faceCrops()
            want = d.detectFramesRaw([ref_or_self(f).desc() for f in frames], mode=mode, orientations=orients)
            wc, wok = d.faceCrops()
            assert records(*got[:2]) == records(*want[:2])
            assert len(wc) >= 6 and np.array_equal(gc, wc) and np.array_equal(gok, wok), mode
    finally:
        d.setFaceCrops(None)


def test_status_codes(fdt, lib):
    d = detector(fdt, "shortRange")
    ffi = fdt._ffi
    faces = (ffi.FdtFace * 300)()
    counts = (C.c_int32 * 3)()
    buf = np.zeros(4 * 64 * 64 * 2, np.uint8)
    for mt in NEW:
        for fn in (lambda w, s: lib.fdt_detect_batch(d._h, buf.ctypes.data, 1, w, 48, s, mt, 0, 0, faces, counts, None, None),
                   lambda w, s: lib.fdt_detect_batch_oriented(d._h, buf.ctypes.data, 1, w, 48, s, mt, 6, 0, 0, faces, counts, None, None)):
            assert fn(64, 127) == ffi.FDT_ERR_SIZE_MISMATCH, mt
            assert fn(63, 128) == ffi.FDT_ERR_BAD_ARG, mt                  # odd (stored) width
            assert fn(64, 128) == ffi.FDT_OK, mt
            assert fn(64, 131) == ffi.FDT_OK, mt                           # odd strides are fine
        good = ffi.FdtFrame(buf.ctypes.data, 64, 48, 128, mt)
        short = ffi.FdtFrame(buf.ctypes.data, 64, 48, 127, mt)
        odd = ffi.FdtFrame(buf.ctypes.data, 63, 48, 128, mt)
        assert lib.fdt_detect_frames(d._h, (ffi.FdtFrame * 3)(good, short, good), 3, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_SIZE_MISMATCH
        assert b"frame 1" in lib.fdt_last_error(d._h)
        assert lib.fdt_detect_frames_oriented(d._h, (ffi.FdtFrame * 3)(good, good, odd), (C.c_int32 * 3)(1, 6, 8), 3, 0, 0, faces, counts,
                                              None, None) == ffi.FDT_ERR_BAD_ARG
        assert b"frame 2" in lib.fdt_last_error(d._h)
        # fdt_detect_one: nbytes must be 2 * width * height
        n = C.c_int32(0)
        size = 64 * 48 * 2
        for wrong in (size - 1, size + 1, 64 * 48 * 3 // 2, 64 * 48 * 3):
            assert lib.fdt_detect_one(d._h, buf.ctypes.data, wrong, 64, 48, mt, 0, faces, C.byref(n), None, None) == ffi.FDT_ERR_SIZE_MISMATCH
        assert lib.fdt_detect_one(d._h, buf.ctypes.data, size, 63, 48, mt, 0, faces, C.byref(n), None, None) == ffi.FDT_ERR_BAD_ARG
        assert lib.fdt_detect_one(d._h, buf.ctypes.data, size, 64, 48, mt, 0, faces, C.byref(n), None, None) == ffi.FDT_OK
        # the aligned-square crop keeps to the formats it always took
        rois = (C.c_double * 4)(32, 24, 20, 0)
        out = np.zeros(16 * 16 * 3, np.uint8)
        ok = (C.c_int32 * 1)()
        assert lib.fdt_extract_aligned_squares(d._h, buf.ctypes.data, 64, 48, 128, mt, rois, 1, 16, out.ctypes.data, ok) == ffi.FDT_ERR_BAD_ARG


def test_python_api(fdt, sample_images):
    d = detector(fdt, "shortRange")
    lm = even(sample_images["landmark-ex1.jpg"])
    h, w = lm.shape[:2]
    for name, mt in (("yuyv", YUYV), ("uyvy", UYVY), ("yvyu", YVYU)):
        m = cv2.cvtColor(lm, TO[mt])                                    # cv2's CV_8UC2 form, h x w x 2
        ref = cv2.cvtColor(m, FROM[mt])
        want = d.detectFacesFromMat(ref)
        assert len(want) == 1

        def same(got, what):
            assert len(got) == len(want) and got[0].originalSize.width == w and got[0].originalSize.height == h, what
            assert np.array_equal(got[0].mesh.packed, want[0].mesh.packed) and np.array_equal(got[0].irisPacked, want[0].irisPacked), what
            assert got[0].detectionData.boundingBox.xmin == want[0].detectionData.boundingBox.xmin, what

        same(d.detectFacesFromMat(m, layout=name), name)
        same(d.detectFacesFromMatBytes(m.tobytes(), width=w, height=h, matType=mt), (name, "bytes"))
        same(d.detectFacesBatch(m, count=1, width=w, height=h, matType=mt, mode=2)[0], (name, "batch"))
        # a row-padded view goes in uncopied with its row stride
        wide = np.zeros((h, w + 8, 2), np.uint8)
        wide[:, 3:3 + w] = m
        for got in d.detectFacesFromMats([wide[:, 3:3 + w], m], layout=name):
            same(got, (name, "mats"))
        # sideways: the faces of the upright image
        s = cv2.rotate(lm, cv2.ROTATE_90_COUNTERCLOCKWISE)               # stored so that a 90 degree clockwise turn is upright
        sm = cv2.cvtColor(s, TO[mt])
        got = d.detectFacesFromMat(sm, layout=name, orientation=6)
        wref = d.detectFacesFromMat(cv2.cvtColor(sm, FROM[mt]), orientation=6)
        assert [f.anchorIndex for f in got] == [f.anchorIndex for f in wref] and len(got) == 1
        assert np.array_equal(got[0].mesh.packed, wref[0].mesh.packed)


def test_multi_device(fdt, sample_images):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=8)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=8)
    frames = mixed(sample_images)
    for mode in (0, 2):
        a = multi.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=[f.o for f in frames])
        b = one.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=[f.o for f in frames])
        assert records(*a[:2]) == records(*b[:2])
        if mode:
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    fr = stored(even(sample_images["landmark-ex1.jpg"]), 6, UYVY, pad=8)
    data = np.stack([fr.data] * 20)
    a = multi.detectBatchRaw(data, count=20, width=fr.w, height=fr.h, matType=UYVY, rowStride=fr.stride, orientation=6, mode=2,
                             withIris=True)
    b = one.detectBatchRaw(np.stack([fr.ref.data] * 20), count=20, width=fr.w, height=fr.h, matType=BGR, orientation=6, mode=2,
                           withIris=True)
    assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    one.dispose(); multi.dispose()
