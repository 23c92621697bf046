"""Aligned face crops of the detect calls (fdt_set_face_crops / fdt_get_face_crops / fdt_copy_face_crops).

Each crop is extractAlignedSquare on the upright BGR image with the ROI of the face the call returned, so the bar throughout is
exact equality with oracle.cv_ops.extract_aligned_square on that image, the ROI from oracle.geometry.compute_embedding_alignment
(kind "embedding") or fdt_host_face_roi (kind "face") on the returned records, put into the requested layout in numpy (channel
order, CHW, float32 v * scale + bias).  The crops come packed in output order, one per returned face."""
import ctypes as C

import cv2
import numpy as np
import pytest

from face_detection_tflite_b200 import _ffi
from face_detection_tflite_b200.synth import face_frame
from oracle import cv_ops as co
from oracle import geometry as geo
from oracle.jpeg_ops import exif_transform
from test_gpu_orientation import BGR, BGRA, GRAY, I420, INVERSE, NV12, NV21, assert_same, even, records, stored
from test_gpu_yuv_planes import layout as plane_layout, split, to_device as planes_to_device, yuv_planes
from yuv_ops import yuv420_to_bgr

pytestmark = pytest.mark.gpu

RGB, RGBA, RGB_PLANAR = _ffi.FDT_FMT_RGB, _ffi.FDT_FMT_RGBA, _ffi.FDT_FMT_RGB_PLANAR
SCALE, BIAS = (1 / 127.5, 1 / 58.0, 0.75), (-1.0, -0.25, 3.5)


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


def detector(fdt, model="shortRange", **kw):
    key = (model, tuple(sorted(kw.items())))
    if key not in _dets:
        _dets[key] = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], **kw)
    return _dets[key]


def spec_of(fdt, kind="embedding", size=112, layout=0):
    return fdt.FaceCropSpec(kind, size, "rgb" if layout & 1 else "bgr", bool(layout & 2),
                            np.float32 if layout & 4 else np.uint8, SCALE, BIAS)


def to_layout(crop, spec):
    """A u8 HWC BGR crop in the spec's layout, as numpy computes it."""
    c = crop[..., ::-1] if spec.order == "rgb" else crop
    if spec.dtype == np.float32:
        c = c.astype(np.float32) * np.array(spec.scale, np.float32) + np.array(spec.bias, np.float32)
    return np.ascontiguousarray(c.transpose(2, 0, 1) if spec.chw else c)


def roi(lib, kind, kp, w, h):
    """(cx, cy, size, theta) of a returned face's crop ROI in the upright image of w x h."""
    if kind == "embedding":
        theta, cx, cy, size = geo.compute_embedding_alignment((kp[0] * w, kp[1] * h), (kp[2] * w, kp[3] * h))
    else:
        out = (C.c_double * 10)()
        lib.fdt_host_face_roi((C.c_double * 12)(*kp), float(w), float(h), 1, out)
        theta, cx, cy, size = out[:4]
    return cx, cy, size, theta


def expected(d, spec, faces, counts, uprights):
    """(crops, ok) for the records of one call: frame b's faces against uprights[b] (u8 BGR, or GRAY HxW)."""
    mf, out, ok = d._max_faces, [], []
    for b, img in enumerate(uprights):
        img = cv2.cvtColor(img, cv2.COLOR_GRAY2BGR) if img.ndim == 2 else img
        for j in range(int(counts[b])):
            kp = list(faces[b * mf + j].keypoints)
            cx, cy, size, theta = roi(d._lib, spec.kind, kp, img.shape[1], img.shape[0])
            c = co.extract_aligned_square(img, cx, cy, size, -theta, spec.size)
            ok.append(c is not None)
            out.append(to_layout(c, spec) if c is not None else np.zeros(spec.shape(1)[1:], spec.dtype))
    return (np.stack(out) if out else np.zeros(spec.shape(0), spec.dtype)), np.array(ok, bool)


def check(d, spec, faces, counts, uprights):
    got, ok = d.faceCrops()
    want, wok = expected(d, spec, faces, counts, uprights)
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, want.shape)
    assert np.array_equal(ok, wok) and ok.all()
    assert np.array_equal(got, want), int(np.argmax([not np.array_equal(a, b) for a, b in zip(got, want)]))
    return got


def photos(sample_images):
    """The sample photos (even sizes; the group shot at 1920x1080, where the short-range detector finds no face) and a synthetic
    1280x720 frame of four faces."""
    return [even(img if img.shape[1] <= 1920 else cv2.resize(img, (1920, 1080), interpolation=cv2.INTER_AREA))
            for img in sample_images.values()] + [face_frame(4, 1280, 720)]


def frames_of(imgs):
    return [(np.ascontiguousarray(m), m.shape[1], m.shape[0], BGR) for m in imgs]


def as_format(bgr, mt):
    """(stored bytes, row stride) of an upright BGR image in format mt (o = 1)."""
    h, w = bgr.shape[:2]
    if mt == RGB:
        return cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB), 3 * w
    if mt == RGBA:
        return cv2.cvtColor(bgr, cv2.COLOR_BGR2RGBA), 4 * w
    if mt == RGB_PLANAR:
        return np.ascontiguousarray(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB).transpose(2, 0, 1)), w
    raise ValueError(mt)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["embedding", "face"])
@pytest.mark.parametrize("layout", range(8))
def test_kinds_and_layouts(fdt, sample_images, kind, layout):
    d = detector(fdt)
    spec = spec_of(fdt, kind, 112 if kind == "embedding" else 160, layout)
    d.setFaceCrops(spec)
    imgs = photos(sample_images)
    faces, counts, _, _ = d.detectFramesRaw(frames_of(imgs), mode=1)
    assert counts.sum() >= 3
    check(d, spec, faces, counts, imgs)
    d.setFaceCrops(None)


def test_layout_zero_equals_embedding_crop(fdt, sample_images):
    d = detector(fdt)
    d.setFaceCrops(fdt.FaceCropSpec())
    imgs = photos(sample_images)
    per_frame = d.detectFacesFromMats(imgs, mode=fdt.FaceDetectionMode.full)
    got, ok = d.faceCrops()
    want = [d.embeddingCrop(f, m) for m, fs in zip(imgs, per_frame) for f in fs]
    assert ok.all() and len(want) == len(got) >= 3
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    d.setFaceCrops(None)


def test_face_kind_equals_mesh_crops(fdt, sample_images):
    """FDT_CROP_FACE at 192 is the standard-mode mesh crop (every face passes a presence gate of 0)."""
    d = detector(fdt, minFacePresenceConfidence=0.0)
    d.setFaceCrops(fdt.FaceCropSpec("face", 192))
    img = photos(sample_images)[3]
    faces, counts, _ = d.detectBatchRaw(img, count=1, width=img.shape[1], height=img.shape[0], mode=1)
    got, _ = d.faceCrops()
    mesh_crops = d.debugMeshStage(int(counts[0]))[0]
    assert int(counts[0]) >= 2 and np.array_equal(got, mesh_crops)
    d.setFaceCrops(None)


@pytest.mark.parametrize("mt", [GRAY, BGR, BGRA, NV12, NV21, I420, RGB, RGBA, RGB_PLANAR])
def test_formats_orientations_host_and_device(fdt, sample_images, mt):
    import torch
    d = detector(fdt)
    spec = spec_of(fdt, "embedding", 112, 7)
    d.setFaceCrops(spec)
    up = photos(sample_images)[0]
    for o in range(1, 9):
        if mt in (GRAY, BGR, BGRA, NV12, NV21, I420):
            fr = stored(up, o, mt)
            data, w, h, stride = fr.data, fr.w, fr.h, fr.stride
            ref = fr.ref.data.reshape(fr.ref.h, fr.ref.w, -1) if fr.ref.mt != GRAY else fr.ref.data.reshape(fr.ref.h, fr.ref.w)
        else:
            s = exif_transform(up, INVERSE[o])
            data, stride = as_format(s, mt)
            h, w = s.shape[:2]
            ref = up
        if ref.ndim == 3 and ref.shape[2] == 4:
            ref = cv2.cvtColor(ref, cv2.COLOR_BGRA2BGR)
        for mem in (0, 1):
            src = data if mem == 0 else torch.from_numpy(np.ascontiguousarray(data).reshape(-1)).cuda()
            faces, counts, _ = d.detectBatchRaw(src if mem == 0 else src.data_ptr(), count=1, width=w, height=h, matType=mt,
                                                rowStride=stride, mode=0, memKind=mem, orientation=o)
            assert int(counts[0]) == 1, (o, mem)
            check(d, spec, faces, counts, [ref])
    d.setFaceCrops(None)


@pytest.mark.parametrize("kind", ["nvdec", "ffmpeg", "android2", "split"])
def test_separate_planes(fdt, sample_images, kind):
    """fdt_detect_yuv_planes from host memory, and from device memory through FrameD (nvdec, android2) and through the
    plane table (ffmpeg, split: U and V with different strides)."""
    d = detector(fdt)
    spec = spec_of(fdt, "face", 128, 6)
    d.setFaceCrops(spec)
    imgs = photos(sample_images)
    lays = [split(*yuv_planes(m), 2) if kind == "split" else plane_layout(kind, *yuv_planes(m), seed=i) for i, m in enumerate(imgs)]
    refs = [yuv420_to_bgr(l.ref, l.w, l.h, I420) for l in lays]
    for mode in (0, 2):
        faces, counts, _, _ = d.detectYuvPlanesRaw([l.host() for l in lays], mode=mode, orientations=[1] * len(lays))
        check(d, spec, faces, counts, refs)
        ts = planes_to_device(lays)
        faces, counts, _, _ = d.detectYuvPlanesRaw([l.device(t) for l, t in zip(lays, ts)], mode=mode, memKind=1)
        check(d, spec, faces, counts, refs)
    d.setFaceCrops(None)


def test_entry_points(fdt, sample_images):
    d = detector(fdt)
    spec = spec_of(fdt, "embedding", 96, 5)
    d.setFaceCrops(spec)
    imgs = photos(sample_images)
    lm = imgs[0]
    h, w = lm.shape[:2]
    # fdt_detect_batch, fdt_detect_batch_oriented
    faces, counts, _ = d.detectBatchRaw(np.stack([lm, lm]), count=2, width=w, height=h, mode=1)
    check(d, spec, faces, counts, [lm, lm])
    s = exif_transform(lm, INVERSE[6])
    faces, counts, _ = d.detectBatchRaw(s, count=1, width=s.shape[1], height=s.shape[0], mode=0, orientation=6)
    check(d, spec, faces, counts, [lm])
    # fdt_detect_one
    got_faces = d.detectFacesFromMatBytes(lm.tobytes(), width=w, height=h, mode=fdt.FaceDetectionMode.standard)
    got, _ = d.faceCrops()
    want = [to_layout(d.embeddingCrop(f, lm, 96), spec) for f in got_faces]
    assert len(got) == len(want) == 1 and np.array_equal(got[0], want[0])
    # fdt_detect_frames, fdt_detect_frames_oriented
    faces, counts, _, _ = d.detectFramesRaw(frames_of(imgs), mode=2)
    check(d, spec, faces, counts, imgs)
    st = [exif_transform(m, INVERSE[o]) for m, o in zip(imgs, (3, 5, 8, 2))]
    faces, counts, _, _ = d.detectFramesRaw(frames_of(st), mode=0, orientations=[3, 5, 8, 2])
    check(d, spec, faces, counts, imgs)
    # fdt_detect_jpeg, fdt_detect_jpeg_batch with a failed image
    from conftest import ASSETS
    jpgs = [(ASSETS / "samples" / n).read_bytes() for n in ("landmark-ex1.jpg", "iris-detection-ex1.jpg")]
    decoded = [d.decodeImage(b) for b in jpgs]
    got_faces = d.detectFacesFromBytes(jpgs[0], mode=fdt.FaceDetectionMode.full)
    got, _ = d.faceCrops()
    assert len(got) == len(got_faces) == 1
    assert np.array_equal(got[0], to_layout(d.embeddingCrop(got_faces[0], decoded[0], 96), spec))
    faces, counts, _, _, wh, status = d.detectBytesBatchRaw([jpgs[0], b"not a jpeg", jpgs[1]], mode=1)
    assert list(status) == [0, _ffi.FDT_ERR_FORMAT, 0] and counts[1] == 0
    check(d, spec, faces, counts, [decoded[0], np.zeros((2, 2, 3), np.uint8), decoded[1]])
    d.setFaceCrops(None)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_modes_and_bitwise_unchanged(fdt, sample_images, mode):
    """Records, mesh, iris and the debug taps are bitwise those of crops off; full mode crops use the iris-refined eyes."""
    d = detector(fdt)
    imgs = photos(sample_images)
    spec = spec_of(fdt, "embedding", 112, 4)

    def run():
        out = list(d.detectFramesRaw(frames_of(imgs), mode=mode))
        taps = [d.debugLetterboxed(len(imgs))]
        if mode:
            taps += [np.copy(x) for x in d.debugMeshStage(100)]
        if mode == 2:
            taps += [np.copy(x) for x in d.debugIrisStage(100)]
        return out, taps

    d.setFaceCrops(None)
    (f0, c0, m0, i0), t0 = run()
    assert d.faceCrops()[0].shape[0] == 0
    d.setFaceCrops(spec)
    (f1, c1, m1, i1), t1 = run()
    assert records(f0, c0) == records(f1, c1)
    assert (m0 is None and m1 is None) or np.array_equal(m0, m1)
    assert (i0 is None and i1 is None) or np.array_equal(i0, i1)
    assert_same(t0, t1, "taps")
    check(d, spec, f1, c1, imgs)
    if mode == 2:
        assert all(f1[b * 100 + j].has_iris for b in range(len(imgs)) for j in range(int(c1[b])))
    d.setFaceCrops(None)


def c4_frames(n, distinct):
    """n 1280x720 synthetic frames cycling over the given (F)-distribution frames."""
    base = [face_frame(k, 1280, 720) for k in distinct]
    return np.stack([base[i % len(base)] for i in range(n)]), base


@pytest.mark.parametrize("max_batch,n,mode", [(2, 11, 1), (4, 19, 0), (4, 13, 2), (32, 1024, 1), (32, 1024, 0)])
def test_chunks_and_passes(fdt, max_batch, n, mode):
    """More than two chunks, and (maxBatch 32: mesh passes and crop passes of 64 faces) a C4-shaped 1024-frame device batch of
    up to 4 faces per frame whose chunks hold more faces than one pass: the packed index must follow the output order."""
    import torch
    d = detector(fdt, maxBatch=max_batch, maxFaces=4)
    spec = spec_of(fdt, "embedding", 112, 6)
    d.setFaceCrops(spec)
    frames, base = c4_frames(n, [4, 9, 14, 19, 24, 29] if n >= 64 else [4, 3, 9, 0, 8, 2])
    dev = torch.from_numpy(frames.reshape(-1)).cuda()
    faces, counts, _ = d.detectBatchRaw(dev.data_ptr(), count=n, width=1280, height=720, mode=mode, memKind=1)
    got, ok = d.faceCrops()
    assert ok.all() and got.shape[0] == counts.sum()
    assert max(counts[k * max_batch:(k + 1) * max_batch].sum() for k in range((n + max_batch - 1) // max_batch)) > 2 * max_batch or n < 64
    # identical frames give identical records: the expected crops of each distinct frame once, then in output order
    rec = records(faces, counts, d._max_faces)
    per = {}
    for b in range(n):
        k = b % len(base)
        if k not in per:
            per[k] = expected(d, spec, faces[b * d._max_faces:], counts[b:b + 1], [base[k]])[0]
        assert rec[b] == rec[b % len(base)]
    want = np.concatenate([per[b % len(base)] for b in range(n)])
    assert np.array_equal(got, want)
    d.setFaceCrops(None)


def test_zero_faces_and_off(fdt):
    d = detector(fdt)
    noise = np.random.default_rng(3).integers(0, 256, (4, 240, 320, 3), dtype=np.uint8)
    d.setFaceCrops(fdt.FaceCropSpec())
    _, counts, _ = d.detectBatchRaw(noise, count=4, width=320, height=240, mode=1)
    got, ok = d.faceCrops()
    assert counts.sum() == 0 and got.shape == (0, 112, 112, 3) and ok.shape == (0,)
    n = C.c_int64(-1)
    assert d._lib.fdt_get_face_crops(d._h, C.byref(n), None) == 0 and n.value == 0
    d.setFaceCrops(None)
    assert d._lib.fdt_get_face_crops(d._h, C.byref(n), None) == 0 and n.value == 0


def test_fast_mode_uploads_whole_frames(fdt):
    d = detector(fdt)
    frames, _ = c4_frames(6, [4, 3])
    nbytes = lambda: int(d._lib.fdt_last_h2d_bytes(d._h))
    d.setFaceCrops(None)
    a = d.detectBatchRaw(frames, count=6, width=1280, height=720, mode=0)
    sparse = nbytes()
    d.setFaceCrops(fdt.FaceCropSpec())
    b = d.detectBatchRaw(frames, count=6, width=1280, height=720, mode=0)
    assert sparse < frames.nbytes and nbytes() == frames.nbytes
    assert records(a[0], a[1]) == records(b[0], b[1])
    d.setFaceCrops(None)


def test_copies_launches_and_status_codes(fdt, sample_images):
    import torch
    d = detector(fdt)
    lib, h = d._lib, d._h
    imgs = photos(sample_images)
    spec = spec_of(fdt, "face", 112, 7)
    d.setFaceCrops(None)
    d.detectFramesRaw(frames_of(imgs), mode=1)
    base_launches = d.lastLaunchCount()
    d.setFaceCrops(spec)
    lib.fdt_set_stage_timing(h, 1)
    faces, counts, _, _ = d.detectFramesRaw(frames_of(imgs), mode=1)
    lib.fdt_set_stage_timing(h, 0)
    ms, launches = C.c_float(), C.c_int32()
    assert lib.fdt_get_stage_ms(h, 9, C.byref(ms), C.byref(launches)) == 0 and launches.value >= 1 and ms.value > 0
    assert d.lastLaunchCount() == base_launches + launches.value
    got = check(d, spec, faces, counts, imgs)
    # device copies: the arena pointer and a torch tensor
    t = torch.zeros(got.size, dtype=torch.float32, device="cuda")
    assert d.copyFaceCropsRaw(t.data_ptr(), t.numel() * 4) == got.shape[0]
    assert np.array_equal(t.cpu().numpy().reshape(got.shape), got)
    n, p = C.c_int64(), C.c_void_p()
    assert lib.fdt_get_face_crops(h, C.byref(n), C.byref(p)) == 0 and n.value == got.shape[0] and p.value
    host = np.empty_like(got)
    assert lib.fdt_copy_to_host(h, host.ctypes.data, p, host.nbytes) == 0 and np.array_equal(host, got)
    # capacity, mem_kind, fdt_detect_batch_device
    assert lib.fdt_copy_face_crops(h, host.ctypes.data, host.nbytes - 1, 0, None) == _ffi.FDT_ERR_SIZE_MISMATCH
    assert lib.fdt_copy_face_crops(h, host.ctypes.data, host.nbytes, 7, None) == _ffi.FDT_ERR_BAD_ARG
    lm = imgs[0]
    dev = torch.from_numpy(lm.reshape(-1)).cuda()
    pf, pc = C.c_void_p(), C.c_void_p()
    assert lib.fdt_detect_batch_device(h, dev.data_ptr(), 1, lm.shape[1], lm.shape[0], lm.shape[1] * 3, BGR, 0, C.byref(pf),
                                       C.byref(pc)) == _ffi.FDT_ERR_UNSUPPORTED
    # bad specs leave the setting as it was
    def bad(**kw):
        c = spec._struct()
        for k, v in kw.items():
            if k in ("scale", "bias"):
                getattr(c, k)[1] = v
            else:
                setattr(c, k, v)
        return lib.fdt_set_face_crops(h, C.byref(c))
    for kw in ({"struct_size": 36}, {"kind": 2}, {"kind": -1}, {"layout": 8}, {"out_size": 0}, {"out_size": 4097},
               {"scale": float("nan")}, {"bias": float("inf")}):
        assert bad(**kw) == _ffi.FDT_ERR_BAD_ARG, kw
    faces, counts, _, _ = d.detectFramesRaw(frames_of(imgs), mode=1)
    check(d, spec, faces, counts, imgs)
    d.setFaceCrops(None)
    pf, pc = C.c_void_p(), C.c_void_p()
    assert lib.fdt_detect_batch_device(h, dev.data_ptr(), 1, lm.shape[1], lm.shape[0], lm.shape[1] * 3, BGR, 0, C.byref(pf),
                                       C.byref(pc)) == 0


def test_python_spec_errors(fdt):
    d = detector(fdt)
    with pytest.raises(ValueError):
        d.setFaceCrops("embedding")
    with pytest.raises(ValueError):
        d.copyFaceCropsRaw(0, -1)


def test_multi_device(fdt, sample_images):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    imgs = photos(sample_images)
    spec = spec_of(fdt, "embedding", 112, 5)
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=2)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=2)
    for d in (one, multi):
        d.setFaceCrops(spec)
    frames = frames_of(imgs * 3)
    for mode in (0, 2):
        a = multi.detectFramesRaw(frames, mode=mode)
        b = one.detectFramesRaw(frames, mode=mode)
        assert records(*a[:2]) == records(*b[:2])
        ga, gb = multi.faceCrops()[0], one.faceCrops()[0]
        assert ga.shape[0] == a[1].sum() and np.array_equal(ga, gb)
    n, p = C.c_int64(), C.c_void_p()
    assert multi._lib.fdt_get_face_crops(multi._h, C.byref(n), C.byref(p)) == _ffi.FDT_ERR_UNSUPPORTED
    t = torch.zeros(ga.size, dtype=torch.float32, device="cuda")
    assert multi._lib.fdt_copy_face_crops(multi._h, t.data_ptr(), ga.nbytes, 1, None) == _ffi.FDT_ERR_UNSUPPORTED
    one.dispose(); multi.dispose()
