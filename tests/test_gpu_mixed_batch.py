"""Mixed batches through the C ABI: fdt_detect_frames (frames of different sizes and formats in one call) and
fdt_detect_jpeg_batch (many encoded images in one call).  Every stage is exact or independent of an image's position in its
chunk, so the bar throughout is bitwise equality with fdt_detect_batch / fdt_detect_jpeg run on each frame alone: face
records, meshes, iris arrays and letterboxed bytes."""
import ctypes as C

import cv2
import numpy as np
import pytest

from test_oracle_jpeg import CASES, SAMPLES, SAMPLING, synth_image, with_exif_orientation
from test_oracle_yuv import FORMATS, i420_to, pad_stride

pytestmark = pytest.mark.gpu

S_OF = {"shortRange": 128, "full": 192, "backCamera": 256}
GRAY, BGR, BGRA = 0, 16, 24
NV12, NV21, I420 = list(FORMATS)


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


def records(faces, counts, max_faces=100):
    """Raw bytes of every filled fdt_face slot, frame by frame (as in test_gpu_yuv.py)."""
    sz = C.sizeof(faces._type_)
    base = C.addressof(faces)
    return [[C.string_at(base + (b * max_faces + j) * sz, sz) for j in range(int(counts[b]))] for b in range(len(counts))]


class Frame:
    """One frame's bytes (exactly height * stride, or * 3 / 2 for YUV) and its descriptor."""

    def __init__(self, data, w, h, mt, stride=None):
        self.data = np.ascontiguousarray(data).reshape(-1)
        self.w, self.h, self.mt = w, h, mt
        self.stride = stride if stride is not None else (w if mt in FORMATS else w * {GRAY: 1, BGR: 3, BGRA: 4}[mt])

    def desc(self, data=None):
        return (self.data if data is None else data, self.w, self.h, self.mt, self.stride)


def packed(img, mt, pad=0):
    h, w = img.shape[:2]
    img = {GRAY: lambda: cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), BGR: lambda: img, BGRA: lambda: cv2.cvtColor(img, cv2.COLOR_BGR2BGRA)}[mt]()
    ch = 1 if img.ndim == 2 else img.shape[2]
    rows = np.zeros((h, w * ch + pad), np.uint8)
    rows[:, :w * ch] = img.reshape(h, w * ch)
    rows[:, w * ch:] = 77                                             # padding bytes must not matter
    return Frame(rows, w, h, mt, w * ch + pad)


def yuv(img, fmt, pad=0):
    h, w = img.shape[:2]
    img = np.ascontiguousarray(img[:h - h % 2, :w - w % 2])
    h, w = img.shape[:2]
    f = i420_to(fmt, cv2.cvtColor(img, cv2.COLOR_BGR2YUV_I420), w, h)
    return Frame(pad_stride(f, w, h, fmt, w + pad) if pad else f, w, h, fmt, w + pad)


def mixed_frames(sample_images, S=128):
    """About 30 frames: the sample photos at native size, rotated to portrait and downscaled below the model input; a frame
    of exactly S x S; odd sizes; every format; padded row strides."""
    photos = list(sample_images.values())
    out = []
    for i, img in enumerate(photos):
        out.append(packed(img, BGR))
        out.append(packed(cv2.rotate(img, cv2.ROTATE_90_CLOCKWISE), BGR))
        out.append(packed(cv2.resize(img, (S * 3 // 4 + i, S // 2 + 3 * i), interpolation=cv2.INTER_AREA), BGR))
        oh, ow = img.shape[0] - 1 - img.shape[0] % 2 - 2 * i, img.shape[1] - 1 - img.shape[1] % 2 - 2 * i
        out.append(packed(np.ascontiguousarray(img[:oh, 1:ow + 1]), [GRAY, BGRA, BGR][i]))                     # odd sizes
        for fmt in FORMATS:
            out.append(yuv(img, fmt))
    lm = sample_images["landmark-ex1.jpg"]
    out.append(packed(cv2.resize(lm, (S, S), interpolation=cv2.INTER_AREA), BGR))            # identity letterbox
    out.append(yuv(cv2.resize(lm, (S, S), interpolation=cv2.INTER_AREA), NV12))
    out.append(packed(np.ascontiguousarray(lm[:640, 380:1020]), BGR))                       # the face reaches two borders
    out.append(packed(lm, GRAY))
    out.append(packed(lm, BGRA, pad=40))
    out.append(packed(cv2.rotate(lm, cv2.ROTATE_90_COUNTERCLOCKWISE), BGR, pad=7))
    out.append(yuv(lm, NV21, pad=64))
    out.append(yuv(lm, I420, pad=32))
    out.append(packed(cv2.resize(lm, (1001, 667), interpolation=cv2.INTER_AREA), BGRA))
    return out


def per_frame(d, fr, mode=None, **kw):
    mode = mode if mode is not None else 0
    return d.detectBatchRaw(fr.data, count=1, width=fr.w, height=fr.h, matType=fr.mt, rowStride=fr.stride, mode=mode, withIris=True, **kw)


def to_device(frames):
    import torch
    ts = [torch.from_numpy(f.data).cuda() for f in frames]
    torch.cuda.synchronize()
    return ts, [f.desc(int(t.data_ptr())) for f, t in zip(frames, ts)]


def assert_equal_to_per_frame(d, frames, got, mode):
    f, c, mesh, iris = got
    rec = records(f, c)
    for b, fr in enumerate(frames):
        wf, wc, wm, wi = per_frame(d, fr, mode)
        assert rec[b] == records(wf, wc)[0], b
        n = int(wc[0])
        if mesh is not None:
            assert np.array_equal(mesh[b, :n], wm[0, :n]), b
        if iris is not None:
            assert np.array_equal(iris[b, :n], wi[0, :n]), b
    return int(np.sum(c))


# ---------------------------------------------------------------------------------------------------------------------
def test_fast_mode_host_and_device(fdt, sample_images):
    d = detector(fdt, "shortRange")
    frames = mixed_frames(sample_images)
    assert len(frames) >= 30 and len({(f.w, f.h) for f in frames}) >= 15
    got = d.detectFramesRaw([f.desc() for f in frames])
    assert int(d._lib.fdt_last_h2d_bytes(d._h)) == sum(f.data.size for f in frames)          # whole frames, frame bytes only
    lb = d.debugLetterboxed(len(frames))
    launches = d.lastLaunchCount()
    ts, ddesc = to_device(frames)
    got_dev = d.detectFramesRaw(ddesc, memKind=1)
    lb_dev = d.debugLetterboxed(len(frames))
    assert records(*got_dev[:2]) == records(*got[:2])
    assert np.array_equal(lb_dev, lb)
    faces = assert_equal_to_per_frame(d, frames, got, 0)
    assert faces >= 20
    for b, fr in enumerate(frames):
        per_frame(d, fr)
        assert np.array_equal(lb[b], d.debugLetterboxed(1)[0]), b
    # one batched call: as many launches as fdt_detect_batch over that many equal frames
    f0 = frames[0]
    d.detectBatchRaw(np.tile(f0.data, len(frames)), count=len(frames), width=f0.w, height=f0.h, matType=f0.mt, rowStride=f0.stride)
    assert launches == d.lastLaunchCount()


@pytest.mark.parametrize("model", ["shortRange", "full", "backCamera"])
def test_standard_and_full_mode(fdt, sample_images, model):
    d = detector(fdt, model)
    frames = mixed_frames(sample_images, S_OF[model])
    for mode in (fdt.FaceDetectionMode.standard, fdt.FaceDetectionMode.full):
        got = d.detectFramesRaw([f.desc() for f in frames], mode=mode)
        assert assert_equal_to_per_frame(d, frames, got, mode) >= 10


def test_chunks_cross_slots_and_staging_budget(fdt, sample_images):
    d = detector(fdt, "shortRange", maxBatch=4)
    base = mixed_frames(sample_images)
    frames = [base[(7 * i) % len(base)] for i in range(37)]
    got = d.detectFramesRaw([f.desc() for f in frames], mode=fdt.FaceDetectionMode.full)
    with pytest.raises(ValueError):
        d.debugLetterboxed(1)               # ten chunks: slot 0 no longer holds the first (checked before other calls replace it)
    assert assert_equal_to_per_frame(d, frames, got, fdt.FaceDetectionMode.full) >= 20
    # maxBatch 2 stages at most 16 MiB of host frames per chunk: a 3840x2160 BGRA frame (33 MB) is a chunk of its own
    d2 = detector(fdt, "shortRange", maxBatch=2)
    lm = sample_images["landmark-ex1.jpg"]
    big = packed(cv2.resize(lm, (3840, 2160)), BGRA)
    small = base[0]
    d2.detectFramesRaw([small.desc(), big.desc()])
    lb = d2.debugLetterboxed(1)                                        # the first chunk is [small]
    with pytest.raises(ValueError):
        d2.debugLetterboxed(2)
    per_frame(d2, small)
    assert np.array_equal(lb, d2.debugLetterboxed(1))
    frames = [small, big, base[5], big, big, base[9], base[13]]
    for mode in (fdt.FaceDetectionMode.fast, fdt.FaceDetectionMode.full):
        got = d2.detectFramesRaw([f.desc() for f in frames], mode=mode)
        assert assert_equal_to_per_frame(d2, frames, got, mode) >= 4


def test_shuffled_list_permutes_results(fdt, sample_images):
    d = detector(fdt, "shortRange")
    frames = mixed_frames(sample_images)
    a = records(*d.detectFramesRaw([f.desc() for f in frames])[:2])
    perm = np.random.default_rng(5).permutation(len(frames))
    b = records(*d.detectFramesRaw([frames[i].desc() for i in perm])[:2])
    assert b == [a[i] for i in perm]


def test_uniform_batch_is_a_special_case(fdt):
    import torch
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange")
    base = np.concatenate([synth.face_frames(12, 1280, 720, start=1), synth.noise_frames(4, 1280, 720, seed=2)])
    t = torch.from_numpy(base).cuda().repeat(64, 1, 1, 1).contiguous()
    fb = 1280 * 720 * 3
    want = d.detectBatchRaw(int(t.data_ptr()), count=1024, width=1280, height=720, memKind=1)
    got = d.detectFramesRaw([(int(t.data_ptr()) + i * fb, 1280, 720, BGR) for i in range(1024)], memKind=1)
    assert records(*got[:2]) == records(*want[:2]) and int(want[1].sum()) >= 500
    del t


def test_status_codes(fdt, lib):
    from face_detection_tflite_b200 import _ffi
    d = detector(fdt, "shortRange")
    faces = (_ffi.FdtFace * (100 * 4))()
    counts = np.zeros(4, np.int32)
    buf = np.zeros(4096, np.uint8)
    good = (buf.ctypes.data, 8, 4, 24, BGR)

    def call(descs, h=d._h, mode=0, mem=0):
        arr = (_ffi.FdtFrame * len(descs))(*[_ffi.FdtFrame(*x) for x in descs])
        return lib.fdt_detect_frames(h, arr, len(descs), mode, mem, faces, counts.ctypes.data_as(_ffi.i32p), None, None)

    bad = [((None, 8, 4, 24, BGR), _ffi.FDT_ERR_BAD_ARG), ((buf.ctypes.data, 7, 4, 8, NV12), _ffi.FDT_ERR_BAD_ARG),
           ((buf.ctypes.data, 8, 4, 20, BGR), _ffi.FDT_ERR_SIZE_MISMATCH), ((buf.ctypes.data, 8, 4, 24, 5), _ffi.FDT_ERR_BAD_ARG),
           ((buf.ctypes.data, 0, 4, 24, BGR), _ffi.FDT_ERR_BAD_ARG)]
    for k, (desc, code) in enumerate(bad):
        descs = [good] * 3
        descs.insert(k % 3, desc)
        assert call(descs) == code, k
        assert ("frame %d" % (k % 3)).encode() in lib.fdt_last_error(d._h)
    assert lib.fdt_detect_frames(d._h, None, -1, 0, 0, faces, counts.ctypes.data_as(_ffi.i32p), None, None) == _ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_frames(d._h, None, 0, 0, 0, faces, counts.ctypes.data_as(_ffi.i32p), None, None) == _ffi.FDT_OK
    assert call([good], mode=7) == _ffi.FDT_ERR_BAD_ARG
    assert call([good], mem=1) == _ffi.FDT_ERR_BAD_ARG                                        # host memory as device frames
    fast_only = detector(fdt, "shortRange", withMesh=False)
    assert call([good], h=fast_only._h, mode=1) == _ffi.FDT_ERR_NOT_READY
    with pytest.raises(ValueError):
        d.detectFramesRaw([(buf[:31], 8, 4, BGR)])
    # the handle stays usable
    assert call([good, good]) == _ffi.FDT_OK and counts[:2].tolist() == [0, 0]
    ptrs = (C.c_void_p * 1)(buf.ctypes.data)
    sizes = (C.c_size_t * 1)(10)
    st = np.zeros(1, np.int32)
    assert lib.fdt_detect_jpeg_batch(d._h, ptrs, sizes, -1, 0, faces, counts.ctypes.data_as(_ffi.i32p), None, None, None,
                                     st.ctypes.data_as(_ffi.i32p)) == _ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_jpeg_batch(fast_only._h, ptrs, sizes, 1, 2, faces, counts.ctypes.data_as(_ffi.i32p), None, None, None,
                                     st.ctypes.data_as(_ffi.i32p)) == _ffi.FDT_ERR_NOT_READY


# ---------------------------------------------------------------------------------------------------------------------
def jpeg_list():
    """Sample photos, the oracle's encodings, greyscale, the eight EXIF orientations, and undecodable entries in between."""
    good = [p.read_bytes() for p in SAMPLES]
    for w, h, samp, q, prog, rst in CASES:
        good.append(cv2.imencode(".jpg", synth_image(w, h, w * 1000 + h), [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                 SAMPLING[samp], cv2.IMWRITE_JPEG_PROGRESSIVE, int(prog), cv2.IMWRITE_JPEG_RST_INTERVAL, rst])[1].tobytes())
    good.append(cv2.imencode(".jpg", synth_image(75, 49, 5)[:, :, 0], [cv2.IMWRITE_JPEG_QUALITY, 80])[1].tobytes())
    lm = cv2.imencode(".jpg", cv2.imread(str(SAMPLES[0])), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    good += [with_exif_orientation(lm, o) for o in range(1, 9)]
    bad = [b"", b"not a jpeg", SAMPLES[0].read_bytes()[:300], b"\xff\xd8\xff\xd9"]
    out = []
    for i, g in enumerate(good):
        out.append(g)
        if i % 6 == 2:
            out.append(bad[(i // 6) % len(bad)])
    return out + bad


def jpeg_one(d, data, mode):
    from face_detection_tflite_b200 import _ffi
    buf = np.frombuffer(data + b"\x00", np.uint8)
    faces, counts, mesh, iris = d._outputs(1, mode)
    wh = (C.c_int32 * 2)()
    rc = d._lib.fdt_detect_jpeg(d._h, buf.ctypes.data, len(data), int(mode), faces, counts.ctypes.data_as(_ffi.i32p),
                                mesh.ctypes.data_as(_ffi.f32p) if mesh is not None else None,
                                iris.ctypes.data_as(_ffi.f32p) if iris is not None else None, wh)
    return rc, (faces, counts, mesh, iris)


@pytest.mark.parametrize("max_batch", [0, 4])
def test_jpeg_batch_equals_per_image(fdt, max_batch):
    from face_detection_tflite_b200 import _ffi
    d = detector(fdt, "shortRange", maxBatch=max_batch)
    images = jpeg_list()
    for mode in (fdt.FaceDetectionMode.fast, fdt.FaceDetectionMode.full):
        faces, counts, mesh, iris, wh, status = d.detectBytesBatchRaw(images, mode=mode)
        rec = records(faces, counts)
        nbad = 0
        for i, data in enumerate(images):
            want = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR) if data else None
            rc, (wf, wc, wm, wi) = jpeg_one(d, data, mode)
            assert status[i] == rc, i
            if want is None:
                nbad += 1
                assert rc == _ffi.FDT_ERR_FORMAT and counts[i] == 0 and tuple(wh[i]) == (0, 0), i
                continue
            assert tuple(wh[i]) == (want.shape[1], want.shape[0]), i
            assert rec[i] == records(wf, wc)[0], i
            n = int(wc[0])
            if mesh is not None:
                assert np.array_equal(mesh[i, :n], wm[0, :n]) and np.array_equal(iris[i, :n], wi[0, :n]), i
        assert nbad >= 6 and int(counts.sum()) >= 3
    out = d.detectFacesFromBytesBatch(images[:6], mode=fdt.FaceDetectionMode.fast)
    assert [o is None for o in out] == [s != 0 for s in status[:6]]


# ---------------------------------------------------------------------------------------------------------------------
def test_mats_api(fdt, sample_images):
    d = detector(fdt, "shortRange")
    lm = sample_images["landmark-ex1.jpg"]
    mats = [lm, lm[100:700, 200:900], cv2.cvtColor(lm, cv2.COLOR_BGR2GRAY)[::1, 5:], cv2.cvtColor(lm, cv2.COLOR_BGR2BGRA)]
    got = d.detectFacesFromMats(mats)
    for m, faces in zip(mats, got):
        want = d.detectFacesFromMat(np.ascontiguousarray(m))
        assert len(faces) == len(want) >= 1
        for a, b in zip(faces, want):
            assert a.detectionData == b.detectionData and np.array_equal(a.mesh.packed, b.mesh.packed)
            assert np.array_equal(a.irisPacked, b.irisPacked)


def test_multi_device(fdt, sample_images):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=8)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=8)
    frames = mixed_frames(sample_images)
    for mode in (fdt.FaceDetectionMode.fast, fdt.FaceDetectionMode.full):
        a = multi.detectFramesRaw([f.desc() for f in frames], mode=mode)
        b = one.detectFramesRaw([f.desc() for f in frames], mode=mode)
        assert records(*a[:2]) == records(*b[:2])
        if mode == fdt.FaceDetectionMode.full:
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    images = jpeg_list()
    a, b = multi.detectBytesBatchRaw(images), one.detectBytesBatchRaw(images)
    assert records(*a[:2]) == records(*b[:2]) and all(np.array_equal(x, y) for x, y in zip(a[2:], b[2:]))
    ts, ddesc = to_device(frames[:2])
    with pytest.raises(NotImplementedError):
        multi.detectFramesRaw(ddesc, memKind=1)
    assert records(*multi.detectFramesRaw([f.desc() for f in frames[:3]])[:2]) == records(*one.detectFramesRaw([f.desc() for f in frames[:3]])[:2])
    one.dispose(); multi.dispose()
