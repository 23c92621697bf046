"""Rotated and mirrored frames (EXIF orientations 1-8) through fdt_detect_batch_oriented and fdt_detect_frames_oriented.

A 90-degree rotation or a flip is an exact pixel permutation, and the letterbox and crop kernels only change the address each
tap reads.  So the bar throughout is bitwise equality with the plain entry point run on the upright image
U = exif_transform(stored, orientation): face records, mesh and iris arrays, letterboxed bytes and mesh / iris crops.  For YUV
frames the reference is exif_transform(yuv420_to_bgr(stored), orientation) passed as BGR."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle.jpeg_ops import exif_transform
from test_oracle_yuv import i420_to, pad_stride
from yuv_ops import YUV_I420, YUV_NV12, YUV_NV21, yuv420_to_bgr

pytestmark = pytest.mark.gpu

GRAY, BGR, BGRA = 0, 16, 24
NV12, NV21, I420 = YUV_NV12, YUV_NV21, YUV_I420
FORMATS = [GRAY, BGR, BGRA, NV12, NV21, I420]
YUV = (NV12, NV21, I420)
CH = {GRAY: 1, BGR: 3, BGRA: 4}
S_OF = {"shortRange": 128, "full": 192, "backCamera": 256}
INVERSE = {1: 1, 2: 2, 3: 3, 4: 4, 5: 5, 6: 8, 7: 7, 8: 6}      # exif_transform(exif_transform(x, INVERSE[o]), o) == x


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
    sz = C.sizeof(faces._type_)
    base = C.addressof(faces)
    return [[C.string_at(base + (b * max_faces + j) * sz, sz) for j in range(int(counts[b]))] for b in range(len(counts))]


class Frame:
    """A stored frame (data holds height * stride bytes, * 3 / 2 for YUV) in orientation o, and its upright reference `ref`."""

    def __init__(self, data, w, h, mt, stride, o, ref=None):
        self.data, self.w, self.h, self.mt, self.stride, self.o, self.ref = np.ascontiguousarray(data).reshape(-1), w, h, mt, stride, o, ref

    def desc(self, ptr=None):
        return (self.data if ptr is None else ptr, self.w, self.h, self.mt, self.stride)


def stored(upright_bgr, o, mt, pad=0):
    """The frame of format mt stored in orientation o whose upright image is upright_bgr (even sizes for YUV), with `pad`
    bytes of row padding, and its reference: the upright image in the format the plain call takes for it."""
    s = exif_transform(upright_bgr, INVERSE[o])
    h, w = s.shape[:2]
    if mt in YUV:
        f = i420_to(mt, cv2.cvtColor(s, cv2.COLOR_BGR2YUV_I420), w, h)
        data = pad_stride(f, w, h, mt, w + pad) if pad else f
        ref = exif_transform(yuv420_to_bgr(data, w, h, mt, w + pad), o)
        return Frame(data, w, h, mt, w + pad, o, Frame(ref, ref.shape[1], ref.shape[0], BGR, ref.shape[1] * 3, 1))
    img = {GRAY: cv2.cvtColor(s, cv2.COLOR_BGR2GRAY), BGR: s, BGRA: cv2.cvtColor(s, cv2.COLOR_BGR2BGRA)}[mt]
    rb = w * CH[mt]
    buf = np.full((h, rb + pad), 77, np.uint8)
    buf[:, :rb] = img.reshape(h, rb)
    u = exif_transform(img.reshape(h, w, CH[mt]), o)
    return Frame(buf, w, h, mt, rb + pad, o, Frame(u, u.shape[1], u.shape[0], mt, u.shape[1] * CH[mt], 1))


def even(img):
    h, w = img.shape[:2]
    return np.ascontiguousarray(img[:h - h % 2, :w - w % 2])


def run(d, fr, mode=0, ptr=None):
    """One uniform call on fr (device memory when ptr is given): records, mesh, iris, letterbox, mesh crops, iris crops."""
    f, c, mesh, iris = d.detectBatchRaw(fr.data if ptr is None else ptr, count=1, width=fr.w, height=fr.h, matType=fr.mt,
                                        rowStride=fr.stride, mode=mode, memKind=0 if ptr is None else 1, withIris=True,
                                        orientation=fr.o)
    n = int(c[0])
    out = [records(f, c), d.debugLetterboxed(1)]
    if mode:
        out += [mesh[:, :n].copy(), d.debugMeshStage(max(n, 1))[0].copy()]
    if mode == 2:
        out += [iris[:, :n].copy(), d.debugIrisStage(max(n, 1))[0].copy()]
    return out, n


def assert_same(a, b, what):
    assert len(a) == len(b), what
    for i, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, np.ndarray):
            assert x.shape == y.shape and np.array_equal(x, y), (what, i)
        else:
            assert x == y, (what, i)


def to_device(arrays):
    import torch
    ts = [torch.from_numpy(np.ascontiguousarray(a).reshape(-1)).cuda() for a in arrays]
    torch.cuda.synchronize()
    return ts


def photos(sample_images):
    """The sample photos (even sizes; the 3840x2160 group shot at 1920x1080, so one detector's staging stays small) and one
    odd-sized crop of the first."""
    ps = [even(img if img.shape[1] <= 1920 else cv2.resize(img, (1920, 1080), interpolation=cv2.INTER_AREA))
          for img in sample_images.values()]
    lm = sample_images["landmark-ex1.jpg"]
    return ps, np.ascontiguousarray(lm[1:852, 3:1276])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mt", FORMATS)
def test_all_orientations_fast_host_and_device(fdt, sample_images, mt):
    d = detector(fdt, "shortRange")
    ps, odd = photos(sample_images)
    frames = []
    for k, img in enumerate(ps + ([odd] if mt not in YUV else [])):
        for o in range(1, 9):
            frames.append(stored(img, o, mt, pad=(0, 6, 32)[(k + o) % 3]))
    faces = 0
    for fr in frames:
        want, n = run(d, fr.ref)
        faces += n
        assert_same(run(d, fr)[0], want, ("host", fr.o, fr.w, fr.h))
        t = to_device([fr.data])
        assert_same(run(d, fr, ptr=int(t[0].data_ptr()))[0], want, ("device", fr.o, fr.w, fr.h))
    assert faces >= 8 * 2           # at least two photos with a face found in every orientation
    # the same frames as one mixed call, host and device
    descs = [fr.desc() for fr in frames]
    orients = [fr.o for fr in frames]
    got = d.detectFramesRaw(descs, orientations=orients)
    lb = d.debugLetterboxed(len(frames))
    ts = to_device([fr.data for fr in frames])
    got_dev = d.detectFramesRaw([fr.desc(int(t.data_ptr())) for fr, t in zip(frames, ts)], memKind=1, orientations=orients)
    assert records(*got_dev[:2]) == records(*got[:2])
    assert np.array_equal(d.debugLetterboxed(len(frames)), lb)
    for b, fr in enumerate(frames):
        want, _ = run(d, fr.ref)
        assert records(*got[:2])[b] == want[0][0], b
        assert np.array_equal(lb[b], want[1][0]), b


@pytest.mark.parametrize("model", ["shortRange", "backCamera"])
def test_identity_letterbox(fdt, sample_images, model):
    """A stored (and so upright) size of exactly S x S: the tap path at equal sizes must return the pixels."""
    d = detector(fdt, model)
    S = S_OF[model]
    lm = sample_images["landmark-ex1.jpg"]
    img = cv2.resize(lm[:, 200:1053], (S, S), interpolation=cv2.INTER_AREA)
    for o in (1, 3, 6, 7):
        for mt in (BGR, GRAY, NV12, I420):
            fr = stored(img, o, mt)
            want, _ = run(d, fr.ref)
            got, _ = run(d, fr)
            assert_same(got, want, (o, mt))
            f = d.detectFramesRaw([fr.desc()], orientations=[o])
            assert records(*f[:2]) == want[0] and np.array_equal(d.debugLetterboxed(1), want[1]), (o, mt, "frames")
    # an upright image of S x S / 2 (no resize, only padding) stored transposed, as S / 2 x S
    wide = cv2.resize(lm, (S, S // 2), interpolation=cv2.INTER_AREA)
    for o in (5, 6, 8):
        fr = stored(wide, o, BGR)
        assert_same(run(d, fr)[0], run(d, fr.ref)[0], o)


@pytest.mark.parametrize("model", ["shortRange", "full", "backCamera"])
def test_standard_and_full_mode(fdt, sample_images, model):
    d = detector(fdt, model)
    lm = sample_images["landmark-ex1.jpg"]
    imgs = [even(lm), np.ascontiguousarray(lm[:640, 380:1020]), even(sample_images["iris-detection-ex1.jpg"])]   # [1]: face at two borders
    faces = 0
    for o in (3, 6, 7):
        for img in imgs:
            for mt in ((BGR, NV12, BGRA) if model == "shortRange" else (BGR, NV21)):
                fr = stored(img, o, mt, pad=8 if mt == BGRA else 0)
                for mode in (1, 2):
                    want, n = run(d, fr.ref, mode)
                    assert_same(run(d, fr, mode)[0], want, (o, mt, mode, img.shape))
                    faces += n
                    f = d.detectFramesRaw([fr.desc()], mode=mode, orientations=[o])
                    w = d.detectBatchRaw(fr.ref.data, count=1, width=fr.ref.w, height=fr.ref.h, matType=fr.ref.mt, mode=mode, withIris=True)
                    assert records(*f[:2]) == records(*w[:2])
                    assert np.array_equal(f[2], w[2]) and (mode == 1 or np.array_equal(f[3], w[3]))
    assert faces >= 12


def test_border_crop_taps_stay_zero(fdt, sample_images):
    """The face of this crop reaches the frame border: its mesh crop has taps outside U, which must be BGR 0 in every
    orientation (bitwise the upright crop), also for YUV frames."""
    d = detector(fdt, "shortRange")
    img = np.ascontiguousarray(sample_images["landmark-ex1.jpg"][:640, 380:1020])
    want, n = run(d, stored(img, 1, BGR), 1)
    assert n >= 1
    crops = want[3]
    assert (crops.reshape(-1, 3) == 0).all(axis=1).any()          # some crop pixels come from outside the frame
    for o in range(2, 9):
        for mt in (BGR, NV12):
            fr = stored(img, o, mt)
            ref, _ = run(d, fr.ref, 1)
            got, _ = run(d, fr, 1)
            assert_same(got, ref, (o, mt))


@pytest.mark.parametrize("mt", [BGR, NV12, NV21, I420])
def test_sparse_upload_bytes(fdt, mt):
    """Fast mode, host frames: the rows the upright image's taps read go up (x taps for orientations 5-8).  At these sizes that
    is the same number of bytes as orientation 1 on the same stored frames."""
    from face_detection_tflite_b200 import synth
    n = 6
    for model, (w, h), per_frame in (("shortRange", (1280, 720), {BGR: 552960, NV12: 276480, NV21: 276480, I420: 276480}),
                                     ("full", (1920, 1080), None), ("backCamera", (1280, 720), None)):
        d = detector(fdt, model)
        src = synth.face_frames(n, w, h, start=1)
        base = None
        for o in range(1, 9):
            frs = [stored(exif_transform(s, o), o, mt) for s in src]          # stored frames = src, whatever o
            data = np.stack([f.data for f in frs])
            f, c, _ = d.detectBatchRaw(data, count=n, width=w, height=h, matType=mt, orientation=o)
            nb = int(d._lib.fdt_last_h2d_bytes(d._h))
            lb = d.debugLetterboxed(n)
            ref = np.stack([fr.ref.data for fr in frs])
            rf, rc, _ = d.detectBatchRaw(ref, count=n, width=frs[0].ref.w, height=frs[0].ref.h, matType=frs[0].ref.mt)
            assert records(f, c) == records(rf, rc), (model, o)
            assert np.array_equal(lb, d.debugLetterboxed(n)), (model, o)
            if base is None:
                base = nb
                if per_frame is not None:
                    assert nb == n * per_frame[mt], model
                assert nb < data.size, model
            assert nb == base, (model, o, nb, base)


def test_uniform_batch_crosses_chunks(fdt):
    """600 frames stored sideways with maxBatch 256: three chunks over both pipeline slots, equal to per-frame calls."""
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange", maxBatch=256)
    src = synth.face_frames(600, 320, 240)
    data = np.ascontiguousarray(np.stack([exif_transform(s, INVERSE[6]) for s in src]))     # 240 x 320 stored, upright 320 x 240
    f, c, _ = d.detectBatchRaw(data, count=600, width=240, height=320, orientation=6)
    got = records(f, c)
    assert sum(len(r) for r in got) >= 400
    for b in range(600):
        wf, wc, _ = d.detectBatchRaw(src[b], count=1, width=320, height=240)
        assert got[b] == records(wf, wc)[0], b
    fo, co, _ = d.detectBatchRaw(data[:5], count=5, width=240, height=320, orientation=6, mode=0)
    assert records(fo, co) == got[:5]


def mixed(sample_images):
    """All 8 orientations interleaved over different sizes and formats."""
    lm, iris, group = (sample_images[k] for k in ("landmark-ex1.jpg", "iris-detection-ex1.jpg", "group-shot-bounding-box-ex1.jpeg"))
    imgs = [even(lm), even(iris), even(cv2.resize(group, (1920, 1080), interpolation=cv2.INTER_AREA)), cv2.resize(lm, (200, 134)),
            np.ascontiguousarray(lm[:640, 380:1020])]
    out = []
    k = 0
    for o in range(1, 9):
        for i, img in enumerate(imgs):
            mt = FORMATS[(k + i) % len(FORMATS)]
            if mt in YUV and (img.shape[0] % 2 or img.shape[1] % 2):
                mt = BGR
            out.append(stored(img, o, mt, pad=(0, 4, 16)[k % 3] if mt not in YUV else (0, 2, 16)[k % 3]))
            k += 1
    return out


@pytest.mark.parametrize("mode", [0, 2])
def test_mixed_call_all_orientations(fdt, sample_images, mode):
    d = detector(fdt, "shortRange", maxBatch=4)
    frames = mixed(sample_images)
    got = d.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=[f.o for f in frames])
    rec = records(*got[:2])
    total = 0
    for b, fr in enumerate(frames):
        wf, wc, wm, wi = d.detectBatchRaw(fr.data, count=1, width=fr.w, height=fr.h, matType=fr.mt, rowStride=fr.stride,
                                          mode=mode, withIris=True, orientation=fr.o)
        assert rec[b] == records(wf, wc)[0], b
        n = int(wc[0])
        total += n
        if mode:
            assert np.array_equal(got[2][b, :n], wm[0, :n]) and np.array_equal(got[3][b, :n], wi[0, :n]), b
    assert total >= 20
    # shuffling the list together with its orientations permutes the results
    perm = np.random.default_rng(5).permutation(len(frames))
    sh = d.detectFramesRaw([frames[i].desc() for i in perm], mode=mode, orientations=[frames[i].o for i in perm])
    assert records(*sh[:2]) == [rec[i] for i in perm]


def test_launch_count_and_status_codes(fdt, sample_images, lib):
    d = detector(fdt, "shortRange")
    lm = even(sample_images["landmark-ex1.jpg"])
    for o in (2, 6):
        for mode in (0, 2):
            fr = stored(lm, o, NV12)
            run(d, fr.ref, mode)
            want = d.lastLaunchCount()
            run(d, fr, mode)
            assert d.lastLaunchCount() == want, (o, mode)
            d.detectFramesRaw([fr.ref.desc()], mode=mode)
            want = d.lastLaunchCount()
            d.detectFramesRaw([fr.desc()], mode=mode, orientations=[o])
            assert d.lastLaunchCount() == want, (o, mode, "frames")
    # status codes, straight through the C ABI (the Python checks would raise first)
    fr = stored(lm, 1, BGR)
    faces = (fdt._ffi.FdtFace * 300)()
    counts = (C.c_int32 * 3)()
    for bad in (0, 9, -1):
        assert lib.fdt_detect_batch_oriented(d._h, fr.data.ctypes.data, 1, fr.w, fr.h, fr.stride, BGR, bad, 0, 0, faces, counts,
                                             None, None) == fdt._ffi.FDT_ERR_BAD_ARG
        arr = (fdt._ffi.FdtFrame * 3)(*[fdt._ffi.FdtFrame(fr.data.ctypes.data, fr.w, fr.h, fr.stride, BGR)] * 3)
        ors = (C.c_int32 * 3)(1, 1, bad)
        assert lib.fdt_detect_frames_oriented(d._h, arr, ors, 3, 0, 0, faces, counts, None, None) == fdt._ffi.FDT_ERR_BAD_ARG
        assert b"frame 2" in lib.fdt_last_error(d._h)
    # NULL orientations equal all ones
    arr = (fdt._ffi.FdtFrame * 3)(*[fdt._ffi.FdtFrame(fr.data.ctypes.data, fr.w, fr.h, fr.stride, BGR)] * 3)
    assert lib.fdt_detect_frames_oriented(d._h, arr, None, 3, 0, 0, faces, counts, None, None) == fdt._ffi.FDT_OK
    a = records(faces, counts)
    assert lib.fdt_detect_frames_oriented(d._h, arr, (C.c_int32 * 3)(1, 1, 1), 3, 0, 0, faces, counts, None, None) == fdt._ffi.FDT_OK
    assert records(faces, counts) == a and sum(map(len, a)) == 3


def test_python_api(fdt, sample_images):
    d = detector(fdt, "shortRange")
    lm = even(sample_images["landmark-ex1.jpg"])
    fr = stored(lm, 6, BGR)
    s = fr.data.reshape(fr.h, fr.w, 3)
    up = d.detectFacesFromMat(lm)
    for got in (d.detectFacesFromMat(s, orientation=6), d.detectFacesFromMatBytes(s.tobytes(), width=fr.w, height=fr.h, orientation=6),
                d.detectFacesFromMats([s], orientations=[6])[0]):
        assert len(got) == len(up) == 1
        assert got[0].originalSize.width == lm.shape[1] and got[0].originalSize.height == lm.shape[0]
        assert np.array_equal(got[0].mesh.packed, up[0].mesh.packed) and np.array_equal(got[0].irisPacked, up[0].irisPacked)
    b = d.detectFacesBatch(s, count=1, width=fr.w, height=fr.h, orientation=6)[0]
    assert b[0].originalSize.width == lm.shape[1]


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
    lm = even(sample_images["landmark-ex1.jpg"])
    fr = stored(lm, 8, NV12)
    data = np.stack([fr.data] * 20)
    a = multi.detectBatchRaw(data, count=20, width=fr.w, height=fr.h, matType=NV12, orientation=8, mode=2, withIris=True)
    b = one.detectBatchRaw(data, count=20, width=fr.w, height=fr.h, matType=NV12, orientation=8, mode=2, withIris=True)
    assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    one.dispose(); multi.dispose()
