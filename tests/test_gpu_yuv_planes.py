"""Separate-plane YUV 4:2:0 frames (fdt_detect_yuv_planes): decoder surfaces, FFmpeg frames and Android YUV_420_888 images.

A frame is a Y, a U and a V plane, each with its own base and row stride, U and V sharing a pixel stride of 1 or 2.  Only the
addresses of the samples differ from a contiguous I420 frame, so the bar throughout is bitwise equality with the library's own
FDT_FMT_YUV_I420 call on the same samples packed contiguously: face records, counts, mesh and iris arrays, letterboxed bytes and
the mesh and iris crops.  Every byte outside a plane's sampled extent (stride padding, the other plane's samples between ps-2
samples) is random noise, and buffers that end at their last sample are passed as they are."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle.jpeg_ops import exif_transform
from test_gpu_orientation import INVERSE, assert_same, even, records

pytestmark = pytest.mark.gpu

I420 = 0x1002
KINDS = ["nvdec", "nv21", "ffmpeg", "yv12", "android2", "android2_split", "android1"]


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


def yuv_planes(bgr):
    """The Y, U and V samples of an even-sized BGR image (cv2 BGR2YUV_I420)."""
    h, w = bgr.shape[:2]
    f = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420).reshape(-1)
    n, c = h * w, h * w // 4
    return f[:n].reshape(h, w), f[n:n + c].reshape(h // 2, w // 2), f[n + c:].reshape(h // 2, w // 2)


def put(buf, off, stride, step, arr):
    rows, cols = arr.shape
    buf[off + np.arange(rows)[:, None] * stride + np.arange(cols)[None, :] * step] = arr


class Layout:
    """Buffers of random noise holding the three planes: planes[k] = (buffer index, offset, row stride)."""

    def __init__(self, Y, U, V, ps, bufs, planes):
        self.w, self.h, self.ps, self.bufs, self.planes = Y.shape[1], Y.shape[0], ps, bufs, planes
        for arr, (b, off, stride), step in zip((Y, U, V), planes, (1, ps, ps)):
            put(bufs[b], off, stride, step, arr)
        self.ref = np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)])   # the contiguous I420 frame

    def strides(self):
        return tuple(p[2] for p in self.planes)

    def host(self):
        return (tuple(self.bufs[b][off:] for b, off, _ in self.planes), self.strides(), self.w, self.h, self.ps)

    def device(self, tensors):
        return (tuple(int(tensors[b].data_ptr()) + off for b, off, _ in self.planes), self.strides(), self.w, self.h, self.ps)

    def h2d(self):
        """fdt_last_h2d_bytes of the frame from host memory: the Y plane's sampled columns, then one interleaved chroma area of
        width bytes per row (pixel stride 2, V one byte from U, one stride of at least width), else U's and V's sampled columns."""
        (_, _, _), (bu, ou, su), (bv, ov, sv) = self.planes
        if self.ps == 2 and bu == bv and abs(ou - ov) == 1 and su == sv >= self.w:
            return self.w * self.h + (self.h // 2) * self.w
        return self.w * self.h + 2 * (self.h // 2) * ((self.w // 2 - 1) * self.ps + 1)


def extent(rows, cols, stride, step):
    return (rows - 1) * stride + (cols - 1) * step + 1


def layout(kind, Y, U, V, seed=0):
    rng = np.random.default_rng(seed)
    noise = lambda n: rng.integers(0, 256, n, dtype=np.uint8)
    h, w = Y.shape
    ch, cw = h // 2, w // 2
    if kind == "nvdec":           # pitched NV12 surface, chroma at pitch * surface height (1920x1080: 2048, 1088 rows)
        pitch = (w + 255) // 256 * 256
        sh = (h + 15) // 16 * 16 + (16 if h % 16 == 0 else 0)
        return Layout(Y, U, V, 2, [noise(pitch * sh * 3 // 2)], [(0, 0, pitch), (0, pitch * sh, pitch), (0, pitch * sh + 1, pitch)])
    if kind == "nv21":
        s = w + 6
        return Layout(Y, U, V, 2, [noise(s * h + s * ch)], [(0, 0, s), (0, s * h + 1, s), (0, s * h, s)])
    if kind == "ffmpeg":          # three planes with three different linesizes (1920: 1984 / 1024 / 1056)
        ly, lu = (w + 63) // 64 * 64 + 64, (cw + 63) // 64 * 64
        lv = lu + 32
        return Layout(Y, U, V, 1, [noise(ly * h), noise(lu * ch), noise(lv * ch)], [(0, 0, ly), (1, 0, lu), (2, 0, lv)])
    if kind == "yv12":            # the V plane stored before the U plane
        sy = w + 32
        sc = sy // 2
        return Layout(Y, U, V, 1, [noise(sy * h + 2 * sc * ch)], [(0, 0, sy), (0, sy * h + sc * ch, sc), (0, sy * h, sc)])
    sy = w + 16
    yb = noise(extent(h, w, sy, 1))
    if kind == "android2":        # YUV_420_888, pixelStride 2, U and V views of one interleaved buffer ending at V's last sample
        sc = w + 16
        return Layout(Y, U, V, 2, [yb, noise(extent(ch, cw, sc, 2) + 1)], [(0, 0, sy), (1, 0, sc), (1, 1, sc)])
    if kind == "android2_split":  # pixelStride 2, U and V buffers each truncated to its sampled extent
        sc = w + 16
        n = extent(ch, cw, sc, 2)
        return Layout(Y, U, V, 2, [yb, noise(n), noise(n)], [(0, 0, sy), (1, 0, sc), (2, 0, sc)])
    if kind == "android1":        # pixelStride 1, three truncated buffers
        sc = cw + 8
        n = extent(ch, cw, sc, 1)
        return Layout(Y, U, V, 1, [yb, noise(n), noise(n)], [(0, 0, sy), (1, 0, sc), (2, 0, sc)])
    raise ValueError(kind)


def split(Y, U, V, ps, seed=0):
    """U and V in allocations of their own with different row strides: device frames of this layout need the plane table."""
    rng = np.random.default_rng(seed)
    h, w = Y.shape
    su = (w // 2 - 1) * ps + 1 + 3
    sv = su + 40
    bufs = [rng.integers(0, 256, n, dtype=np.uint8) for n in (w * h, extent(h // 2, w // 2, su, ps), extent(h // 2, w // 2, sv, ps))]
    return Layout(Y, U, V, ps, bufs, [(0, 0, w), (1, 0, su), (2, 0, sv)])


def to_device(lays):
    import torch
    ts = [[torch.from_numpy(b).cuda() for b in lay.bufs] for lay in lays]
    torch.cuda.synchronize()
    return ts


def photos(sample_images):
    """The sample photos at even sizes, the group shot at 1920x1080 (the NVDEC surface of 1080-line video)."""
    return [even(img if img.shape[1] <= 1920 else cv2.resize(img, (1920, 1080), interpolation=cv2.INTER_AREA))
            for img in sample_images.values()]


def stored(img, o):
    """The Y, U, V samples of the frame stored in orientation o whose upright image is img."""
    return yuv_planes(np.ascontiguousarray(exif_transform(img, INVERSE[o])))


def call(d, descs, mode, mem, orients, ref):
    """(records, mesh, iris, letterboxed bytes of the first chunk) of one call: the planes call, or (ref) the I420 call."""
    if ref:
        got = d.detectFramesRaw(descs, mode=mode, orientations=orients)
    else:
        got = d.detectYuvPlanesRaw(descs, mode=mode, memKind=mem, orientations=orients)
    return records(*got[:2]), got[2], got[3], d.debugLetterboxed(min(len(descs), 4))


def ref_desc(lay):
    return (lay.ref, lay.w, lay.h, I420, lay.w)


def same(a, b, what):
    assert a[0] == b[0], what
    for x, y in zip(a[1:], b[1:]):
        assert (x is None and y is None) or np.array_equal(x, y), what


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_layouts_all_orientations_host_and_device(fdt, sample_images, kind):
    """Every layout, every orientation, from host memory (exact upload bytes), device memory as laid out, and device memory
    with U and V split into allocations of different strides (the plane-table kernels)."""
    d = detector(fdt, "shortRange")
    lays = []
    for k, img in enumerate(photos(sample_images)):
        for o in range(1, 9):
            lays.append(layout(kind, *stored(img, o), seed=8 * k + o))
    orients = [o for _ in photos(sample_images) for o in range(1, 9)]
    want = call(d, [ref_desc(l) for l in lays], 0, 0, orients, True)
    assert sum(map(len, want[0])) >= 2 * 8          # faces found in every orientation
    got = call(d, [l.host() for l in lays], 0, 0, orients, False)
    same(got, want, (kind, "host"))
    assert int(d._lib.fdt_last_h2d_bytes(d._h)) == sum(l.h2d() for l in lays), kind
    ts = to_device(lays)
    same(call(d, [l.device(t) for l, t in zip(lays, ts)], 0, 1, orients, False), want, (kind, "device"))
    sp = [split(*stored(img, o), lays[0].ps, seed=o) for img in photos(sample_images) for o in range(1, 9)]
    same(call(d, [l.device(t) for l, t in zip(sp, to_device(sp))], 0, 1, orients, False), want, (kind, "device, plane table"))
    # other noise outside the extents: the same results
    again = [layout(kind, *stored(img, o), seed=1000 + o) for img in photos(sample_images)[:1] for o in range(1, 9)]
    same(call(d, [l.host() for l in again], 0, 0, orients[:8], False), call(d, [ref_desc(l) for l in again], 0, 0, orients[:8], True),
         (kind, "noise"))


def single(d, desc, mode, mem, o, ref):
    """One frame: records, mesh, iris, letterbox, mesh crops, iris crops."""
    rec, mesh, iris, lb = call(d, [desc], mode, mem, [o], ref)
    n = len(rec[0])
    out = [rec, lb[:1]]
    if mode:
        out += [mesh[:, :n].copy(), d.debugMeshStage(max(n, 1))[0].copy()]
    if mode == 2:
        out += [iris[:, :n].copy(), d.debugIrisStage(max(n, 1))[0].copy()]
    return out, n


@pytest.mark.parametrize("mode", [1, 2])
def test_standard_and_full_mode_crops(fdt, sample_images, mode):
    """Mesh and iris crops through the FrameD route (host frames, NVDEC / NV21 device frames) and the plane-table route
    (FFmpeg linesizes, split planes), with the right eye's mirrored crop and taps past the frame border."""
    d = detector(fdt, "shortRange")
    lm = sample_images["landmark-ex1.jpg"]
    imgs = [even(lm), even(lm[:640, 380:1020]), even(sample_images["iris-detection-ex1.jpg"])]
    faces = 0
    for o in (1, 3, 6, 7):
        for k, img in enumerate(imgs):
            planes = stored(img, o)
            lay = layout(KINDS[(o + k) % len(KINDS)], *planes, seed=o)
            want, n = single(d, ref_desc(lay), mode, 0, o, True)
            faces += n
            assert_same(single(d, lay.host(), mode, 0, o, False)[0], want, (o, k, "host"))
            t = to_device([lay])[0]
            assert_same(single(d, lay.device(t), mode, 1, o, False)[0], want, (o, k, "device"))
            sp = split(*planes, 2 if k % 2 else 1, seed=k)
            t = to_device([sp])[0]
            assert_same(single(d, sp.device(t), mode, 1, o, False)[0], want, (o, k, "plane table"))
    assert faces >= 12


@pytest.mark.parametrize("model", ["full", "backCamera"])
def test_other_letterboxes(fdt, sample_images, model):
    d = detector(fdt, model)
    for k, img in enumerate(photos(sample_images)):
        for o in (1, 6):
            planes = stored(img, o)
            lays = [layout(kind, *planes, seed=k) for kind in ("nvdec", "ffmpeg", "android2_split")] + [split(*planes, 2)]
            want = call(d, [ref_desc(lays[0])], 0, 0, [o], True)
            same(call(d, [lays[0].host()], 0, 0, [o], False), want, (model, k, o, "host"))
            ts = to_device(lays)
            for lay, t in zip(lays, ts):
                same(call(d, [lay.device(t)], 0, 1, [o], False), want, (model, k, o, "device"))


def test_u_and_v_more_than_2gib_apart(fdt, sample_images):
    """One 3 GiB device allocation with U 16 MiB and V 2.5 GiB in: the offsets do not fit an int, so the plane table runs."""
    import torch
    d = detector(fdt, "shortRange")
    img = photos(sample_images)[0]
    Y, U, V = stored(img, 6)
    h, w = Y.shape
    big = torch.empty(3 << 30, dtype=torch.uint8, device="cuda")
    big[: 32 << 20].random_(0, 256)
    uo, vo, s = 16 << 20, (5 << 29), w + 64
    for off, arr, ps in ((0, Y, 1), (uo, U, 2), (vo, V, 2)):
        view = big[off: off + extent(*arr.shape, s, ps)]
        flat = np.random.default_rng(off).integers(0, 256, view.numel(), dtype=np.uint8)
        put(flat, 0, s, ps, arr)
        view.copy_(torch.from_numpy(flat))
    torch.cuda.synchronize()
    assert vo - uo > 2 ** 31
    ref = np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)])
    base = int(big.data_ptr())
    for mode in (0, 2):
        want = call(d, [(ref, w, h, I420, w)], mode, 0, [6], True)
        got = call(d, [((base, base + uo, base + vo), (s, s, s), w, h, 2)], mode, 1, [6], False)
        same(got, want, mode)
        assert len(want[0][0]) >= 1
    del big
    torch.cuda.empty_cache()


def test_chunks_and_slots(fdt, sample_images):
    """2 * maxBatch + 3 frames of different sizes and layouts, full mode: chunk boundaries and both pipeline slots."""
    d = detector(fdt, "shortRange", maxBatch=4)
    ps = photos(sample_images)
    lays, orients = [], []
    for k in range(11):
        img = ps[k % len(ps)]
        if k % 3 == 1:
            img = even(cv2.resize(img, (img.shape[1] // 2 + 2 * k, img.shape[0] // 2 + 2 * k)))
        o = 1 + (k * 3) % 8
        planes = stored(img, o)
        lays.append(layout(KINDS[k % len(KINDS)], *planes, seed=k) if k % 4 else split(*planes, 1 + k % 2, seed=k))
        orients.append(o)
    want = d.detectFramesRaw([ref_desc(l) for l in lays], mode=2, orientations=orients)
    host = d.detectYuvPlanesRaw([l.host() for l in lays], mode=2, orientations=orients)
    ts = to_device(lays)
    dev = d.detectYuvPlanesRaw([l.device(t) for l, t in zip(lays, ts)], mode=2, memKind=1, orientations=orients)
    for got, what in ((host, "host"), (dev, "device")):
        assert records(*got[:2]) == records(*want[:2]), what
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), what
    assert sum(map(len, records(*want[:2]))) >= 8
    # fast mode, one chunk's letterboxes
    d.detectFramesRaw([ref_desc(l) for l in lays[:4]], orientations=orients[:4])
    lb = d.debugLetterboxed(4)
    d.detectYuvPlanesRaw([l.host() for l in lays[:4]], orientations=orients[:4])
    assert np.array_equal(d.debugLetterboxed(4), lb)


def test_status_codes(fdt, lib):
    d = detector(fdt, "shortRange")
    ffi = fdt._ffi
    faces = (ffi.FdtFace * 300)()
    counts = (C.c_int32 * 3)()
    buf = np.zeros(64 * 48 * 4, np.uint8)
    p = buf.ctypes.data

    def desc(**kw):
        f = dict(plane=(p, p + 64 * 48, p + 64 * 48 + 1), row_stride=(64, 64, 64), width=64, height=48, pixel_stride=2)
        f.update(kw)
        r = ffi.FdtYuvPlanes()
        r.plane = (C.c_void_p * 3)(*f["plane"])
        r.row_stride = (C.c_int32 * 3)(*f["row_stride"])
        r.width, r.height, r.pixel_stride = f["width"], f["height"], f["pixel_stride"]
        return r

    good = desc()
    cases = [(dict(width=63), ffi.FDT_ERR_BAD_ARG, b""), (dict(height=47), ffi.FDT_ERR_BAD_ARG, b""),
             (dict(width=0), ffi.FDT_ERR_BAD_ARG, b""),
             (dict(plane=(p, None, p)), ffi.FDT_ERR_BAD_ARG, b"plane U"), (dict(plane=(None, p, p)), ffi.FDT_ERR_BAD_ARG, b"plane Y"),
             (dict(plane=(p, p, None)), ffi.FDT_ERR_BAD_ARG, b"plane V"),
             (dict(pixel_stride=0), ffi.FDT_ERR_BAD_ARG, b""), (dict(pixel_stride=3), ffi.FDT_ERR_BAD_ARG, b""),
             (dict(row_stride=(-64, 64, 64)), ffi.FDT_ERR_BAD_ARG, b"plane Y"), (dict(row_stride=(64, 0, 64)), ffi.FDT_ERR_BAD_ARG, b"plane U"),
             (dict(row_stride=(64, 64, -1)), ffi.FDT_ERR_BAD_ARG, b"plane V"),
             (dict(row_stride=(63, 64, 64)), ffi.FDT_ERR_SIZE_MISMATCH, b"plane Y"),
             (dict(row_stride=(64, 62, 64)), ffi.FDT_ERR_SIZE_MISMATCH, b"plane U"),
             (dict(row_stride=(64, 64, 62)), ffi.FDT_ERR_SIZE_MISMATCH, b"plane V"),
             (dict(row_stride=(64, 31, 32), pixel_stride=1), ffi.FDT_ERR_SIZE_MISMATCH, b"plane U")]
    for kw, code, plane in cases:
        for mem in (0, 1):
            arr = (ffi.FdtYuvPlanes * 3)(good, good, desc(**kw))
            assert lib.fdt_detect_yuv_planes(d._h, arr, None, 3, 0, mem, faces, counts, None, None) == code, kw
            assert b"frame 2" in lib.fdt_last_error(d._h) and plane in lib.fdt_last_error(d._h), kw
    # the minimum strides are accepted: 63 bytes of a ps-2 chroma row, 32 of a ps-1 one
    for kw in (dict(row_stride=(64, 63, 63)), dict(row_stride=(64, 32, 32), pixel_stride=1, plane=(p, p + 4000, p + 6000))):
        assert lib.fdt_detect_yuv_planes(d._h, (ffi.FdtYuvPlanes * 1)(desc(**kw)), None, 1, 0, 0, faces, counts, None, None) == 0, kw
    arr = (ffi.FdtYuvPlanes * 2)(good, good)
    assert lib.fdt_detect_yuv_planes(d._h, arr, (C.c_int32 * 2)(1, 9), 2, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    assert b"frame 1" in lib.fdt_last_error(d._h)
    assert lib.fdt_detect_yuv_planes(d._h, arr, None, 2, 7, 0, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_yuv_planes(d._h, arr, None, 2, 0, 5, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_yuv_planes(d._h, arr, None, 2, 0, 0, None, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    # host memory passed as device memory, also for one plane after planes of an allocation the call has already checked
    assert lib.fdt_detect_yuv_planes(d._h, arr, None, 2, 0, 1, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    import torch
    t = torch.zeros(64 * 48 * 2, dtype=torch.uint8, device="cuda")
    q = int(t.data_ptr())
    dev = desc(plane=(q, q + 64 * 48, q + 64 * 48 + 1))
    assert lib.fdt_detect_yuv_planes(d._h, (ffi.FdtYuvPlanes * 2)(dev, dev), None, 2, 0, 1, faces, counts, None, None) == ffi.FDT_OK
    mixed = desc(plane=(q, q + 64 * 48, p))
    assert lib.fdt_detect_yuv_planes(d._h, (ffi.FdtYuvPlanes * 2)(dev, mixed), None, 2, 0, 1, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    assert b"frame 1: plane V" in lib.fdt_last_error(d._h)
    assert lib.fdt_detect_yuv_planes(d._h, None, None, 0, 0, 0, faces, counts, None, None) == ffi.FDT_OK
    assert lib.fdt_detect_yuv_planes(None, arr, None, 2, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_NOT_READY


def test_python_api(fdt, sample_images):
    """detectFacesFromYuvPlanes on numpy views: an NV12 chroma plane as uv[:, 0::2], uv[:, 1::2], an I420 frame's planes and
    rotated frames."""
    d = detector(fdt, "shortRange")
    lm = even(sample_images["landmark-ex1.jpg"])
    h, w = lm.shape[:2]
    Y, U, V = yuv_planes(lm)
    ref = np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)])
    f, c, mesh, iris = d.detectFramesRaw([(ref, w, h, I420, w)], mode=2)
    uv = np.stack([U, V], -1).reshape(h // 2, w)
    pitched = np.zeros((h, w + 64), np.uint8)
    pitched[:, :w] = Y
    for frame in ((Y, U, V), (pitched[:, :w], uv[:, 0::2], uv[:, 1::2])):
        got = d.detectFacesFromYuvPlanes([frame, frame])
        assert [len(g) for g in got] == [1, 1]
        for g in got:
            assert g[0].originalSize.width == w and g[0].originalSize.height == h
            assert np.array_equal(g[0].mesh.packed, mesh[0, 0]) and np.array_equal(g[0].irisPacked, iris[0, 0])
            assert g[0].anchorIndex == f[0].anchor_index
    s = stored(lm, 8)
    got = d.detectFacesFromYuvPlanes([s], orientations=[8], mode=0)
    assert len(got[0]) == 1 and got[0][0].originalSize.width == w and got[0][0].originalSize.height == h


def test_multi_device(fdt, sample_images):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=8)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=8)
    lays, orients = [], []
    for k, img in enumerate(photos(sample_images) * 3):
        o = 1 + k % 8
        lays.append(layout(KINDS[k % len(KINDS)], *stored(img, o), seed=k))
        orients.append(o)
    for mode in (0, 2):
        a = multi.detectYuvPlanesRaw([l.host() for l in lays], mode=mode, orientations=orients)
        b = one.detectFramesRaw([ref_desc(l) for l in lays], mode=mode, orientations=orients)
        assert records(*a[:2]) == records(*b[:2])
        if mode:
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    one.dispose(); multi.dispose()
