"""RGB, RGBA and planar RGB frames (FDT_FMT_RGB / _RGBA / _RGB_PLANAR) through every detect entry point.

Swapping channels or reading three planes only changes which bytes each letterbox and crop tap loads, so the bar throughout is
bitwise equality with the same call on the BGR image: cv2.cvtColor(frame, COLOR_RGB2BGR) / COLOR_RGBA2BGR, or
chw[::-1].transpose(1, 2, 0) for a planar frame.  Face records, mesh and iris arrays, letterboxed bytes and mesh / iris crops
are compared, in all eight orientations, from host and device memory."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle.jpeg_ops import exif_transform
from test_gpu_orientation import INVERSE, Frame, assert_same, even, records, run, to_device
from test_oracle_yuv import i420_to, pad_stride

pytestmark = pytest.mark.gpu

GRAY, BGR, BGRA = 0, 16, 24
NV12, NV21, I420 = 0x1000, 0x1001, 0x1002
RGB, RGBA, PLANAR = 0x1010, 0x1011, 0x1012
NEW = [RGB, RGBA, PLANAR]
ALL = [GRAY, BGR, BGRA, NV12, NV21, I420, RGB, RGBA, PLANAR]
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


def as_format(s, mt, pad=0, seed=0):
    """The stored BGR image s in format mt with `pad` bytes of row padding: (data, row stride, the BGR image the contract names
    for that data).  RGBA alpha is random (it must be ignored)."""
    h, w = s.shape[:2]
    if mt == PLANAR:
        chw = np.ascontiguousarray(cv2.cvtColor(s, cv2.COLOR_BGR2RGB).transpose(2, 0, 1))
        buf = np.full((3, h, w + pad), 91, np.uint8)
        buf[:, :, :w] = chw
        return buf, w + pad, np.ascontiguousarray(buf[:, :, :w][::-1].transpose(1, 2, 0))
    if mt in (NV12, NV21, I420):
        f = i420_to(mt, cv2.cvtColor(s, cv2.COLOR_BGR2YUV_I420), w, h)
        return (pad_stride(f, w, h, mt, w + pad) if pad else f), w + pad, None
    if mt == RGBA:
        img = cv2.cvtColor(s, cv2.COLOR_BGR2RGBA)
        img[..., 3] = np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)
        ref = cv2.cvtColor(img, cv2.COLOR_RGBA2BGR)
    elif mt == RGB:
        img = cv2.cvtColor(s, cv2.COLOR_BGR2RGB)
        ref = cv2.cvtColor(img, cv2.COLOR_RGB2BGR)
    else:
        img = {GRAY: cv2.cvtColor(s, cv2.COLOR_BGR2GRAY), BGR: s, BGRA: cv2.cvtColor(s, cv2.COLOR_BGR2BGRA)}[mt]
        ref = None
    ch = 1 if img.ndim == 2 else img.shape[2]
    buf = np.full((h, w * ch + pad), 77, np.uint8)
    buf[:, :w * ch] = img.reshape(h, w * ch)
    return buf, w * ch + pad, ref


def stored(upright_bgr, o, mt, pad=0, seed=0):
    """The frame of format mt stored in orientation o whose upright image is upright_bgr; its reference is the same oriented call
    on the stored frame converted to BGR."""
    s = exif_transform(upright_bgr, INVERSE[o])
    h, w = s.shape[:2]
    data, stride, ref = as_format(s, mt, pad, seed)
    return Frame(data, w, h, mt, stride, o, None if ref is None else Frame(ref, w, h, BGR, w * 3, o))


def photos(sample_images):
    """The sample photos (the 3840x2160 group shot at 1920x1080), and an odd-sized crop of the first."""
    ps = [img if img.shape[1] <= 1920 else cv2.resize(img, (1920, 1080), interpolation=cv2.INTER_AREA)
          for img in sample_images.values()]
    lm = sample_images["landmark-ex1.jpg"]
    return ps + [np.ascontiguousarray(lm[1:852, 3:1276])]


def border_crop(sample_images):
    """A crop whose face reaches two borders: its mesh and iris crops have taps outside the frame."""
    return np.ascontiguousarray(sample_images["landmark-ex1.jpg"][:640, 380:1020])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mt", NEW)
def test_all_orientations_fast_host_and_device(fdt, sample_images, mt):
    d = detector(fdt, "shortRange")
    frames = []
    for k, img in enumerate(photos(sample_images)):
        for o in range(1, 9):
            frames.append(stored(img, o, mt, pad=(0, 6, 32)[(k + o) % 3], seed=k * 8 + o))
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


def test_standard_and_full_mode_short_range(fdt, sample_images):
    """Mesh and iris crops (including taps past the frame border) in every orientation; uniform and mixed calls."""
    d = detector(fdt, "shortRange")
    lm = sample_images["landmark-ex1.jpg"]
    imgs = [lm, border_crop(sample_images), sample_images["iris-detection-ex1.jpg"]]
    faces = 0
    for o in range(1, 9):
        for k, img in enumerate(imgs):
            mt = NEW[(o + k) % 3]
            fr = stored(img, o, mt, pad=(0, 8, 3)[k], seed=o)
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
    want, n = run(d, stored(imgs[1], 1, PLANAR).ref, 1)
    assert n >= 1 and (want[3].reshape(-1, 3) == 0).all(axis=1).any()


@pytest.mark.parametrize("model", ["full", "backCamera"])
def test_fast_mode_other_letterboxes(fdt, sample_images, model):
    """The 192 and 256 letterboxes (the 128 one runs everywhere above)."""
    d = detector(fdt, model)
    for k, img in enumerate(photos(sample_images)):
        for o in (1, 4, 6):
            for mt in NEW:
                fr = stored(img, o, mt, pad=4 * k, seed=k)
                want, _ = run(d, fr.ref)
                assert_same(run(d, fr)[0], want, (model, k, o, mt))


@pytest.mark.parametrize("model", ["shortRange", "backCamera"])
def test_identity_letterbox(fdt, sample_images, model):
    """A stored size of exactly S x S: the identity read (orientation 1) and the tap path at equal sizes (the others)."""
    d = detector(fdt, model)
    S = S_OF[model]
    img = cv2.resize(sample_images["landmark-ex1.jpg"][:, 200:1053], (S, S), interpolation=cv2.INTER_AREA)
    for o in (1, 3, 6, 7):
        for mt in NEW:
            for pad in (0, 5):
                fr = stored(img, o, mt, pad=pad)
                want, _ = run(d, fr.ref)
                assert_same(run(d, fr)[0], want, (o, mt, pad))
                f = d.detectFramesRaw([fr.desc()], orientations=[o])
                assert records(*f[:2]) == want[0] and np.array_equal(d.debugLetterboxed(1), want[1]), (o, mt, "frames")


def test_detect_one_and_batch_device(fdt, sample_images, lib):
    """fdt_detect_one (full mode) and fdt_detect_batch_device (fast mode, results left on the device)."""
    d = detector(fdt, "shortRange")
    mf = d._max_faces
    imgs = [sample_images["landmark-ex1.jpg"], cv2.resize(sample_images["iris-detection-ex1.jpg"], (641, 359))]

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
        return records(faces, counts)

    found = 0
    for img in imgs:
        h, w = img.shape[:2]
        for mt in NEW:
            data, stride, ref = as_format(img, mt)
            want = one(ref, w, h, BGR)
            got = one(data, w, h, mt)
            assert got[0] == want[0], (mt, w, h)
            assert_same(got[1:], want[1:], (mt, w, h))
            found += len(want[0][0])
            assert on_device(data, w, h, stride, mt, 5) == on_device(ref, w, h, w * 3, BGR, 5), (mt, w, h)
    assert found >= 2


def test_sparse_upload_bytes_and_launch_counts(fdt, sample_images):
    """Fast mode, host frames: RGB / RGBA upload what BGR / BGRA do; planar frames the same rows of each plane (552,960 B for
    1280x720, also stored sideways), or whole frames when the tap rows are not periodic.  Launch counts equal BGR's."""
    from face_detection_tflite_b200 import synth
    d = detector(fdt, "shortRange")
    n = 6
    nbytes = lambda: int(d._lib.fdt_last_h2d_bytes(d._h))
    for (w, h), o in (((1280, 720), 1), ((1280, 720), 6), ((641, 359), 1), ((641, 359), 8)):
        src = synth.face_frames(n, w, h, start=1)
        per = {}
        for mt in (BGR, BGRA) + tuple(NEW):
            frs = [stored(s, o, mt) for s in src]
            data = np.stack([f.data for f in frs])
            f, c, _ = d.detectBatchRaw(data, count=n, width=frs[0].w, height=frs[0].h, matType=mt, rowStride=frs[0].stride,
                                       orientation=o)
            per[mt] = nbytes()
            lb = d.debugLetterboxed(n)
            if mt in NEW:
                ref = np.stack([fr.ref.data for fr in frs])
                rf, rc, _ = d.detectBatchRaw(ref, count=n, width=frs[0].w, height=frs[0].h, matType=BGR, orientation=o)
                assert records(f, c) == records(rf, rc), (w, h, o, mt)
                assert np.array_equal(lb, d.debugLetterboxed(n)), (w, h, o, mt)
        assert per[RGB] == per[BGR] and per[RGBA] == per[BGRA], (w, h, o, per)
        if h == 720:
            assert per[PLANAR] == per[BGR] == n * 552960, (o, per)
        else:
            assert per[PLANAR] == n * 3 * h * w, (o, per)                 # 359 rows: no period, whole frames
    # launch counts: uniform and mixed calls, fast and full mode
    lm = sample_images["landmark-ex1.jpg"]
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


def test_chunking(fdt, sample_images):
    """maxBatch 4 with 10 frames (uniform and mixed, full mode), and 600 uniform fast-mode frames over three chunks of 256."""
    from face_detection_tflite_b200 import synth
    d4 = detector(fdt, "shortRange", maxBatch=4)
    lm = even(sample_images["landmark-ex1.jpg"])
    for mt in NEW:
        frs = [stored(np.roll(lm, 16 * k, axis=1), 1 if k % 2 else 6, mt, pad=2, seed=k) for k in range(10)]
        same = [f for f in frs if f.o == 6]
        data = np.stack([f.data for f in same])
        got = d4.detectBatchRaw(data, count=len(same), width=same[0].w, height=same[0].h, matType=mt, rowStride=same[0].stride,
                                mode=2, withIris=True, orientation=6)
        ref = np.stack([f.ref.data for f in same])
        want = d4.detectBatchRaw(ref, count=len(same), width=same[0].w, height=same[0].h, matType=BGR, mode=2, withIris=True,
                                 orientation=6)
        assert records(*got[:2]) == records(*want[:2]) and np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), mt
        got = d4.detectFramesRaw([f.desc() for f in frs], mode=2, orientations=[f.o for f in frs])
        want = d4.detectFramesRaw([f.ref.desc() for f in frs], mode=2, orientations=[f.o for f in frs])
        assert records(*got[:2]) == records(*want[:2]) and np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), mt
        assert sum(map(len, records(*got[:2]))) >= 10
    d = detector(fdt, "shortRange", maxBatch=256)
    src = synth.face_frames(600, 320, 240)
    for mt in NEW:
        frs = [stored(s, 1, mt) for s in src]
        f, c, _ = d.detectBatchRaw(np.stack([x.data for x in frs]), count=600, width=320, height=240, matType=mt)
        rf, rc, _ = d.detectBatchRaw(np.stack([x.ref.data for x in frs]), count=600, width=320, height=240, matType=BGR)
        got = records(f, c)
        assert got == records(rf, rc), mt
        assert sum(len(r) for r in got) >= 400


def mixed(sample_images):
    """All nine formats over different sizes and orientations, with padded rows."""
    lm, iris, group = (sample_images[k] for k in ("landmark-ex1.jpg", "iris-detection-ex1.jpg", "group-shot-bounding-box-ex1.jpeg"))
    imgs = [even(lm), even(iris), even(cv2.resize(group, (1920, 1080), interpolation=cv2.INTER_AREA)), cv2.resize(lm, (201, 134)),
            border_crop(sample_images)]
    out = []
    k = 0
    for o in range(1, 9):
        for i, img in enumerate(imgs):
            mt = ALL[(k + i) % len(ALL)]
            if mt in (NV12, NV21, I420) and (img.shape[0] % 2 or img.shape[1] % 2):
                mt = PLANAR
            out.append(stored(img, o, mt, pad=(0, 4, 16)[k % 3] if mt not in (NV12, NV21, I420) else (0, 2, 16)[k % 3], seed=k))
            k += 1
    return out


@pytest.mark.parametrize("mode", [0, 2])
def test_mixed_call_all_formats(fdt, sample_images, mode):
    """Every frame of a mixed call over the nine formats equals its one-frame call, from host and device memory."""
    d = detector(fdt, "shortRange", maxBatch=4)
    frames = mixed(sample_images)
    assert {f.mt for f in frames} == set(ALL)
    orients = [f.o for f in frames]
    got = d.detectFramesRaw([f.desc() for f in frames], mode=mode, orientations=orients)
    rec = records(*got[:2])
    ts = to_device([f.data for f in frames])
    dev = d.detectFramesRaw([f.desc(int(t.data_ptr())) for f, t in zip(frames, ts)], mode=mode, memKind=1, orientations=orients)
    assert records(*dev[:2]) == rec
    if mode:
        assert np.array_equal(dev[2], got[2]) and np.array_equal(dev[3], got[3])
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
    # a 4-frame chunk's letterboxes against the one-frame calls
    d.detectFramesRaw([f.desc() for f in frames[:4]], orientations=orients[:4])
    lb = d.debugLetterboxed(4)
    for b, fr in enumerate(frames[:4]):
        assert np.array_equal(lb[b], run(d, fr)[0][1][0]), b


def test_status_codes(fdt, sample_images, lib):
    d = detector(fdt, "shortRange")
    ffi = fdt._ffi
    faces = (ffi.FdtFace * 300)()
    counts = (C.c_int32 * 3)()
    img = cv2.resize(sample_images["landmark-ex1.jpg"], (64, 48))
    buf = np.zeros(4 * 64 * 64 * 3, np.uint8)
    for mt, minimum in ((RGB, 3 * 64), (RGBA, 4 * 64), (PLANAR, 64)):
        for fn in (lambda s: lib.fdt_detect_batch(d._h, buf.ctypes.data, 1, 64, 48, s, mt, 0, 0, faces, counts, None, None),
                   lambda s: lib.fdt_detect_batch_oriented(d._h, buf.ctypes.data, 1, 64, 48, s, mt, 6, 0, 0, faces, counts, None, None)):
            assert fn(minimum - 1) == ffi.FDT_ERR_SIZE_MISMATCH, mt
            assert fn(minimum) == ffi.FDT_OK, mt
        good = ffi.FdtFrame(buf.ctypes.data, 64, 48, minimum, mt)
        bad = ffi.FdtFrame(buf.ctypes.data, 64, 48, minimum - 1, mt)
        assert lib.fdt_detect_frames(d._h, (ffi.FdtFrame * 3)(good, bad, bad), 3, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_SIZE_MISMATCH
        assert b"frame 1" in lib.fdt_last_error(d._h)
        assert lib.fdt_detect_frames_oriented(d._h, (ffi.FdtFrame * 3)(good, good, bad), (C.c_int32 * 3)(1, 6, 8), 3, 0, 0, faces, counts,
                                              None, None) == ffi.FDT_ERR_SIZE_MISMATCH
        assert b"frame 2" in lib.fdt_last_error(d._h)
        # fdt_detect_one: nbytes must be the frame's size
        data, _, _ = as_format(img, mt)
        n = C.c_int32(0)
        size = data.size
        assert size == {RGB: 64 * 48 * 3, RGBA: 64 * 48 * 4, PLANAR: 3 * 64 * 48}[mt]
        for wrong in (size - 1, size + 1, 64 * 48 * 3 // 2):
            if wrong != size:
                assert lib.fdt_detect_one(d._h, data.ctypes.data, wrong, 64, 48, mt, 0, faces, C.byref(n), None, None) == ffi.FDT_ERR_SIZE_MISMATCH
        assert lib.fdt_detect_one(d._h, data.ctypes.data, size, 64, 48, mt, 0, faces, C.byref(n), None, None) == ffi.FDT_OK
        # the aligned-square crop keeps to the formats it always took
        rois = (C.c_double * 4)(32, 24, 20, 0)
        out = np.zeros(16 * 16 * 3, np.uint8)
        ok = (C.c_int32 * 1)()
        assert lib.fdt_extract_aligned_squares(d._h, data.ctypes.data, 64, 48, minimum, mt, rois, 1, 16, out.ctypes.data, ok) == ffi.FDT_ERR_BAD_ARG
    # the profile entry takes the new formats
    t = to_device([np.zeros(3 * 48 * 64 * 4, np.uint8)])[0]
    ms = (C.c_float * 512)()
    nl = C.c_int32()
    for mt, stride in ((RGB, 192), (RGBA, 256), (PLANAR, 64)):
        assert lib.fdt_profile_chunk(d._h, t.data_ptr(), 2, 64, 48, stride, mt, 1, ms, 512, C.byref(nl)) == ffi.FDT_OK, mt


def test_python_api(fdt, sample_images):
    import torch
    d = detector(fdt, "shortRange")
    lm = sample_images["landmark-ex1.jpg"]
    rgb = cv2.cvtColor(lm, cv2.COLOR_BGR2RGB)
    rgba = cv2.cvtColor(lm, cv2.COLOR_BGR2RGBA)
    chw = np.ascontiguousarray(rgb.transpose(2, 0, 1))
    up = d.detectFacesFromMat(lm)
    assert len(up) == 1

    def same(got, what):
        assert len(got) == 1 and got[0].originalSize.width == lm.shape[1] and got[0].originalSize.height == lm.shape[0], what
        assert np.array_equal(got[0].mesh.packed, up[0].mesh.packed) and np.array_equal(got[0].irisPacked, up[0].irisPacked), what

    same(d.detectFacesFromMat(rgb, layout="rgb"), "rgb")
    same(d.detectFacesFromMat(rgba, layout="rgb"), "rgba")
    same(d.detectFacesFromMat(chw, layout="rgb_planar"), "planar")
    gray = cv2.cvtColor(lm, cv2.COLOR_BGR2GRAY)
    assert [f.anchorIndex for f in d.detectFacesFromMat(gray, layout="rgb")] == [f.anchorIndex for f in d.detectFacesFromMat(gray)]
    # a planar view with padded rows and evenly spaced planes (a column crop of a wider CHW array), and a view that must be copied
    wide = np.zeros((3, lm.shape[0], lm.shape[1] + 40), np.uint8)
    wide[:, :, 17:17 + lm.shape[1]] = chw
    view = wide[:, :, 17:17 + lm.shape[1]]
    assert view.strides == (lm.shape[0] * wide.shape[2], wide.shape[2], 1)
    tall = np.zeros((3, lm.shape[0] + 5, lm.shape[1]), np.uint8)
    tall[:, :lm.shape[0]] = chw
    uneven = tall[:, :lm.shape[0]]                                     # planes height + 5 rows apart: copied
    assert uneven.strides[0] != lm.shape[0] * uneven.strides[1]
    for got in d.detectFacesFromMats([view, uneven, chw], layout="rgb_planar"):
        same(got, "mats planar")
    same(d.detectFacesFromMats([rgb, rgba], layout="rgb")[1], "mats rgba")
    # a CUDA CHW tensor straight from torch: its data_ptr with FDT_MEM_DEVICE
    t = torch.from_numpy(np.stack([chw, chw])).cuda()
    torch.cuda.synchronize()
    f, c, _ = d.detectBatchRaw(t.data_ptr(), count=2, width=lm.shape[1], height=lm.shape[0], matType=fdt._ffi.FDT_FMT_RGB_PLANAR,
                               memKind=fdt._ffi.FDT_MEM_DEVICE)
    wf, wc, _ = d.detectBatchRaw(np.stack([lm, lm]), count=2, width=lm.shape[1], height=lm.shape[0])
    assert records(f, c) == records(wf, wc) and list(c) == [1, 1]
    b = d.detectFacesBatch(chw, count=1, width=lm.shape[1], height=lm.shape[0], matType=fdt._ffi.FDT_FMT_RGB_PLANAR, mode=2)[0]
    same(b, "batch")


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
    fr = stored(even(sample_images["landmark-ex1.jpg"]), 6, PLANAR, pad=8)
    data = np.stack([fr.data] * 20)
    a = multi.detectBatchRaw(data, count=20, width=fr.w, height=fr.h, matType=PLANAR, rowStride=fr.stride, orientation=6, mode=2,
                             withIris=True)
    b = one.detectBatchRaw(data, count=20, width=fr.w, height=fr.h, matType=PLANAR, rowStride=fr.stride, orientation=6, mode=2,
                           withIris=True)
    assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    one.dispose(); multi.dispose()
