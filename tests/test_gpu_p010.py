"""16-bit YUV 4:2:0 frames: FDT_FMT_P010 (P010 / P012 / P016 contiguous frames) and fdt_detect_yuv_planes16 (NVDEC P016
surfaces, FFmpeg yuv420p10le / p12le planes).

The library reduces every 16-bit sample s with `bits` significant bits to (s >> (bits - 8)) & 0xFF before anything else, so the
bar throughout is bitwise equality with the 8-bit call on the frame made by that rule: FDT_FMT_YUV_NV12 for the contiguous
format, fdt_detect_yuv_planes for the planes.  Compared are face records and counts, mesh and iris arrays, the letterboxed bytes,
the mesh and iris stage crops and the face crops.  Inputs are built as word = (v8 << (bits - 8)) | random low bits, with random
bits above `bits` as well for 10 and 12, so any use of the discarded bits shows."""
import ctypes as C

import cv2
import numpy as np
import pytest

from oracle.jpeg_ops import exif_transform
from test_gpu_orientation import INVERSE, Frame, assert_same, even, records, run, to_device
from test_gpu_yuv422 import as_422

pytestmark = pytest.mark.gpu

BGR, NV12, P010, YUYV = 16, 0x1000, 0x1003, 0x1020


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


def widen(v8, bits, rng):
    """16-bit words whose 8-bit sample under the rule is v8: v8 << (bits - 8), random bits below, and random bits above `bits`."""
    v = v8.astype(np.uint16) << (bits - 8)
    v |= rng.integers(0, 1 << (bits - 8), v8.shape, dtype=np.uint16)
    if bits < 16:
        v |= rng.integers(0, 1 << (16 - bits), v8.shape, dtype=np.uint16) << bits
    return v


def nv12_of(bgr):
    """The NV12 frame ((3H/2) x W uint8) of an even-sized BGR image."""
    h, w = bgr.shape[:2]
    f = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420).reshape(-1)
    n, c = h * w, h * w // 4
    uv = np.empty((h // 2, w), np.uint8)
    uv[:, 0::2] = f[n:n + c].reshape(h // 2, w // 2)
    uv[:, 1::2] = f[n + c:].reshape(h // 2, w // 2)
    return np.concatenate([f[:n].reshape(h, w), uv])


def p010_pair(upright_bgr, o, pad=0, seed=0):
    """The P010 frame stored in orientation o whose upright image is upright_bgr, with `pad` words of row padding (noise), and
    its reference: the NV12 frame of the words' high bytes, in the same orientation."""
    rng = np.random.default_rng(seed)
    s = exif_transform(upright_bgr, INVERSE[o])
    h, w = s.shape[:2]
    f8 = nv12_of(s)
    words = rng.integers(0, 1 << 16, (h * 3 // 2, w + pad), dtype=np.uint16)
    words[:, :w] = widen(f8, 16, rng)
    return Frame(words.view(np.uint8), w, h, P010, 2 * (w + pad), o), Frame(f8, w, h, NV12, w, o)


def lm(sample_images):
    return even(sample_images["landmark-ex1.jpg"])


# ---------------------------------------------------------------------------------------------------------------------
def test_all_orientations_fast_host_and_device(fdt, sample_images):
    d = detector(fdt, "shortRange")
    faces = 0
    for k, img in enumerate([even(im if im.shape[1] <= 1920 else cv2.resize(im, (1920, 1080), interpolation=cv2.INTER_AREA))
                             for im in sample_images.values()]):
        for o in range(1, 9):
            fr, ref = p010_pair(img, o, pad=(0, 6, 32)[(k + o) % 3], seed=k * 8 + o)
            want, n = run(d, ref)
            faces += n
            assert_same(run(d, fr)[0], want, ("host", k, o))
            t = to_device([fr.data])
            assert_same(run(d, fr, ptr=int(t[0].data_ptr()))[0], want, ("device", k, o))
    assert faces >= 8


@pytest.mark.parametrize("model", ["shortRange", "full", "backCamera"])
def test_standard_and_full_mode(fdt, sample_images, model):
    d = detector(fdt, model)
    for o in (1, 3, 6, 8):
        fr, ref = p010_pair(lm(sample_images), o, pad=4, seed=o)
        for mode in (1, 2):
            want, n = run(d, ref, mode)
            assert n >= 1, (model, o)
            assert_same(run(d, fr, mode)[0], want, (model, o, mode))
            t = to_device([fr.data])
            assert_same(run(d, fr, mode, ptr=int(t[0].data_ptr()))[0], want, (model, o, mode, "device"))


def test_detect_one_and_batch_device(fdt, sample_images, lib):
    d = detector(fdt, "shortRange")
    ffi = fdt._ffi
    img = lm(sample_images)
    fr, ref = p010_pair(img, 1, seed=3)
    h, w = img.shape[:2]

    def one(data, mt):
        faces = (ffi.FdtFace * 100)()
        n = C.c_int32(0)
        mesh = np.zeros((100, 468, 3), np.float32)
        iris = np.zeros((100, 152, 3), np.float32)
        buf = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
        assert lib.fdt_detect_one(d._h, buf.ctypes.data, buf.size, w, h, mt, 2, faces, C.byref(n),
                                  mesh.ctypes.data_as(ffi.f32p), iris.ctypes.data_as(ffi.f32p)) == ffi.FDT_OK
        return records(faces, [n.value]), mesh[:n.value].copy(), iris[:n.value].copy(), d.debugMeshStage(max(n.value, 1))[0].copy()

    want = one(ref.data, NV12)
    assert len(want[0][0]) >= 1
    assert_same(one(fr.data, P010), want, "fdt_detect_one")

    def on_device(data, stride, mt, count=3):
        t = to_device([np.tile(data.reshape(-1), count)])[0]
        pf, pc = C.c_void_p(), C.c_void_p()
        assert lib.fdt_detect_batch_device(d._h, t.data_ptr(), count, w, h, stride, mt, 0, C.byref(pf), C.byref(pc)) == 0
        counts = np.zeros(count, np.int32)
        faces = (ffi.FdtFace * (count * d._max_faces))()
        assert lib.fdt_copy_to_host(d._h, counts.ctypes.data, pc, counts.nbytes) == 0
        assert lib.fdt_copy_to_host(d._h, C.addressof(faces), pf, C.sizeof(faces)) == 0
        return records(faces, counts, d._max_faces), d.debugLetterboxed(count).copy(), counts

    a, b = on_device(fr.data, fr.stride, P010), on_device(ref.data, ref.stride, NV12)
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and b[2].min() >= 1


def test_upload_bytes_and_launch_counts(fdt, sample_images):
    d = detector(fdt, "shortRange")
    nbytes = lambda: int(d._lib.fdt_last_h2d_bytes(d._h))
    launches = lambda: int(d._lib.fdt_last_launch_count(d._h))
    rng = np.random.default_rng(5)
    img = cv2.resize(lm(sample_images), (1280, 720), interpolation=cv2.INTER_AREA)
    fr, ref = p010_pair(img, 1, seed=9)
    for n in (1, 4):
        for mode in (0, 2):
            d.detectBatchRaw(np.stack([ref.data] * n), count=n, width=1280, height=720, matType=NV12, mode=mode)
            nv12_bytes, nv12_launches = nbytes(), launches()
            d.detectBatchRaw(np.stack([fr.data] * n), count=n, width=1280, height=720, matType=P010, mode=mode)
            assert launches() == nv12_launches, (n, mode)
            # fast mode: Y rows 10k+4, 10k+5 and chroma row 5k+2 of 2560 bytes each; otherwise whole frames
            assert nbytes() == (552960 * n if mode == 0 else 1280 * 720 * 3 * n) == 2 * nv12_bytes, (n, mode)
    # mixed calls upload whole frames
    fr2, _ = p010_pair(img[:480, :640], 6, pad=8, seed=1)
    d.detectFramesRaw([fr.desc(), fr2.desc(), ref.desc()])
    assert nbytes() == 1280 * 720 * 3 + fr2.stride * 640 * 3 // 2 + 1280 * 720 * 3 // 2
    # planes16: each plane's sampled columns, twice the 8-bit rule's bytes
    f8 = ref.data.reshape(1080, 1280)
    y16 = widen(f8[:720], 16, rng)
    uv16 = widen(f8[720:], 16, rng)
    d.detectYuvPlanesRaw([((y16, uv16, uv16.reshape(-1)[1:]), (2560, 2560, 2560), 1280, 720, 2)], sampleBits=16)
    assert nbytes() == 2 * 1280 * 720 + 360 * 2 * 1280
    p10 = [widen(p, 10, rng) for p in (f8[:720], f8[720:, 0::2].copy(), f8[720:, 1::2].copy())]
    d.detectYuvPlanesRaw([(tuple(p10), (2560, 1280, 1280), 1280, 720, 1)], sampleBits=10)
    assert nbytes() == 2 * 1280 * 720 + 4 * 360 * 640


def mixed(sample_images, seed=0):
    """A mixed list: P010 frames (several sizes and orientations) next to BGR, NV12 and YUYV frames; with the reference list
    in which each P010 frame is its NV12 frame."""
    imgs = [even(im if im.shape[1] <= 1920 else cv2.resize(im, (1920, 1080), interpolation=cv2.INTER_AREA))
            for im in sample_images.values()]
    got, want = [], []
    for k, img in enumerate(imgs):
        for o in (1, 3, 6, 8):
            fr, ref = p010_pair(img, o, pad=2 * k, seed=seed + 10 * k + o)
            got.append(fr); want.append(ref)
        s = exif_transform(img, INVERSE[5])
        bgr = Frame(s, s.shape[1], s.shape[0], BGR, s.shape[1] * 3, 5)
        data, stride, _ = as_422(img, YUYV, pad=4)
        yuyv = Frame(data, img.shape[1], img.shape[0], YUYV, stride, 1)
        nv = Frame(nv12_of(img), img.shape[1], img.shape[0], NV12, img.shape[1], 1)
        for f in (bgr, yuyv, nv):
            got.append(f); want.append(f)
    return got, want


@pytest.mark.parametrize("mode", [0, 2])
def test_mixed_call(fdt, sample_images, mode):
    d = detector(fdt, "shortRange")
    got, want = mixed(sample_images)
    orients = [f.o for f in got]
    a = d.detectFramesRaw([f.desc() for f in got], mode=mode, orientations=orients)
    ga = d.debugLetterboxed(len(got))
    b = d.detectFramesRaw([f.desc() for f in want], mode=mode, orientations=orients)
    assert np.array_equal(ga, d.debugLetterboxed(len(got)))
    assert records(*a[:2]) == records(*b[:2]) and sum(map(len, records(*b[:2]))) >= 12
    if mode:
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    ts = to_device([f.data for f in got])
    c = d.detectFramesRaw([f.desc(int(t.data_ptr())) for f, t in zip(got, ts)], mode=mode, memKind=1, orientations=orients)
    assert records(*c[:2]) == records(*b[:2])
    if mode:
        assert np.array_equal(c[2], b[2]) and np.array_equal(c[3], b[3])


def test_more_than_two_chunks(fdt, sample_images):
    """maxBatch 4: a uniform call of 11 frames and a planes16 call of 11 frames each run 3 chunks through both slots."""
    d = detector(fdt, "shortRange", maxBatch=4)
    fr, ref = p010_pair(lm(sample_images), 6, pad=2, seed=2)
    for mode in (0, 2):
        a = d.detectBatchRaw(np.stack([fr.data] * 11), count=11, width=fr.w, height=fr.h, matType=P010, rowStride=fr.stride,
                             orientation=6, mode=mode, withIris=True)
        b = d.detectBatchRaw(np.stack([ref.data] * 11), count=11, width=ref.w, height=ref.h, matType=NV12, orientation=6,
                             mode=mode, withIris=True)
        assert records(*a[:2]) == records(*b[:2]) and min(a[1]) >= 1
        if mode:
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
        surfaces = [p016_surface(ref, 16, np.random.default_rng(i)) for i in range(11)]
        g = d.detectYuvPlanesRaw([s[0] for s in surfaces], mode=mode, orientations=[6] * 11, sampleBits=16)
        w8 = d.detectYuvPlanesRaw([s[1] for s in surfaces], mode=mode, orientations=[6] * 11)
        assert records(*g[:2]) == records(*w8[:2]) == records(*b[:2])
        if mode:
            assert np.array_equal(g[2], w8[2]) and np.array_equal(g[3], w8[3])


def p016_surface(nv, bits, rng, pitch_pad=64, extra_rows=8):
    """NVDEC-shaped pitched surfaces of the NV12 frame nv (a Frame): Y rows of `pitch` bytes, the chroma at pitch * surface
    height, U = chroma, V = chroma + 1 sample.  Returns the planes16 descriptor of the 16-bit surface (word = the rule's inverse
    with random low bits) and the planes descriptor of the 8-bit surface, both as detectYuvPlanesRaw tuples on host buffers."""
    w, h = nv.w, nv.h
    sh = h + extra_rows
    f8 = nv.data.reshape(h * 3 // 2, w)
    s8 = rng.integers(0, 256, (sh * 3 // 2, w + pitch_pad), dtype=np.uint8)
    s8[:h, :w] = f8[:h]
    s8[sh:sh + h // 2, :w] = f8[h:]
    s16 = rng.integers(0, 1 << 16, s8.shape, dtype=np.uint16)
    s16[:h, :w] = widen(f8[:h], bits, rng)
    s16[sh:sh + h // 2, :w] = widen(f8[h:], bits, rng)
    b8, b16 = s8.reshape(-1), s16.reshape(-1).view(np.uint8)
    p8, p16 = w + pitch_pad, 2 * (w + pitch_pad)
    c8, c16 = sh * p8, sh * p16
    return (((b16, b16[c16:], b16[c16 + 2:]), (p16, p16, p16), w, h, 2),
            ((b8, b8[c8:], b8[c8 + 1:]), (p8, p8, p8), w, h, 2))


def device_desc(desc, keep):
    """A detectYuvPlanesRaw tuple on host buffers (views of one buffer) as the same tuple on one device copy of that buffer."""
    import torch
    planes, strides, w, h, ps = desc
    base = planes[0].base if planes[0].base is not None else planes[0]
    while base.base is not None and isinstance(base.base, np.ndarray):
        base = base.base
    raw = base.reshape(-1).view(np.uint8)
    t = torch.from_numpy(raw.copy()).cuda()
    keep.append(t)
    off = [p.ctypes.data - raw.ctypes.data for p in planes]
    return (tuple(int(t.data_ptr()) + o for o in off), strides, w, h, ps)


@pytest.mark.parametrize("mode", [0, 2])
def test_nvdec_p016_surfaces(fdt, sample_images, mode):
    """Pitched P016 surfaces (chroma at pitch * surface height) in every orientation, host and device, against the 8-bit
    surfaces through fdt_detect_yuv_planes."""
    import torch
    d = detector(fdt, "shortRange")
    rng = np.random.default_rng(11)
    pairs = []
    for o in range(1, 9):
        _, ref = p010_pair(lm(sample_images), o, seed=o)
        pairs.append(p016_surface(ref, 16, rng, pitch_pad=(0, 64, 256)[o % 3], extra_rows=(0, 8)[o % 2]))
    orients = list(range(1, 9))
    a = d.detectYuvPlanesRaw([p[0] for p in pairs], mode=mode, orientations=orients, sampleBits=16)
    la = d.debugLetterboxed(8)
    b = d.detectYuvPlanesRaw([p[1] for p in pairs], mode=mode, orientations=orients)
    assert np.array_equal(la, d.debugLetterboxed(8))
    assert records(*a[:2]) == records(*b[:2]) and min(b[1]) >= 1
    if mode:
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    keep = []
    dev16 = [device_desc(p[0], keep) for p in pairs]
    dev8 = [device_desc(p[1], keep) for p in pairs]
    torch.cuda.synchronize()
    c = d.detectYuvPlanesRaw(dev16, mode=mode, memKind=1, orientations=orients, sampleBits=16)
    lc = d.debugLetterboxed(8)
    e = d.detectYuvPlanesRaw(dev8, mode=mode, memKind=1, orientations=orients)
    assert np.array_equal(lc, d.debugLetterboxed(8)) and np.array_equal(lc, la)
    assert records(*c[:2]) == records(*e[:2]) == records(*b[:2])
    if mode:
        assert np.array_equal(c[2], e[2]) and np.array_equal(c[3], b[3])


def ffmpeg_planes(nv, bits, rng, linesizes):
    """yuv420p10le / p12le-shaped planes of the NV12 frame nv: three uint16 planes with their own linesizes (bytes; noise in the
    padding), as a detectFacesFromYuvPlanes (y, u, v) triple of views, and the 8-bit (y, u, v) triple of the same samples."""
    w, h = nv.w, nv.h
    f8 = nv.data.reshape(h * 3 // 2, w)
    p8 = (f8[:h], f8[h:, 0::2], f8[h:, 1::2])
    out = []
    for p, ls in zip(p8, linesizes):
        buf = rng.integers(0, 1 << 16, (p.shape[0], ls // 2), dtype=np.uint16)
        buf[:, :p.shape[1]] = widen(p, bits, rng)
        out.append(buf[:, :p.shape[1]])
    return tuple(out), p8


@pytest.mark.parametrize("bits", [10, 12])
def test_ffmpeg_three_planes(fdt, sample_images, bits):
    import torch
    d = detector(fdt, "shortRange")
    rng = np.random.default_rng(bits)
    frames16, frames8, orients = [], [], []
    for k, o in enumerate((1, 2, 6, 7)):
        _, ref = p010_pair(lm(sample_images), o, seed=o)
        ls = [2 * ref.w + 64 * k, ref.w + 32 + 2 * k, ref.w + 96]
        p16, p8 = ffmpeg_planes(ref, bits, rng, ls)
        frames16.append(p16); frames8.append(p8); orients.append(o)
    for mode in (0, 2):
        got = d.detectFacesFromYuvPlanes(frames16, mode=mode, orientations=orients, sampleBits=bits)
        lg = d.debugLetterboxed(4)
        want = d.detectFacesFromYuvPlanes(frames8, mode=mode, orientations=orients)
        assert np.array_equal(lg, d.debugLetterboxed(4))
        assert [len(f) for f in got] == [len(f) for f in want] and min(len(f) for f in want) >= 1
        for gf, wf in zip(got, want):
            for g, w in zip(gf, wf):
                assert g.detectionData.boundingBox == w.detectionData.boundingBox
                if mode:
                    assert np.array_equal(g.mesh.packed, w.mesh.packed) and np.array_equal(g.irisPacked, w.irisPacked)
    # the same planes from device memory (each plane copied to an allocation of its own)
    keep = []
    descs16, descs8 = [], []
    for p16, p8 in zip(frames16, frames8):
        for planes, out in ((p16, descs16), (p8, descs8)):
            cs = [np.ascontiguousarray(p) for p in planes]
            ts = [torch.from_numpy(c.reshape(-1).view(np.uint8)).cuda() for c in cs]
            keep += ts
            out.append((tuple(int(t.data_ptr()) for t in ts), tuple(c.strides[0] for c in cs), cs[0].shape[1], cs[0].shape[0], 1))
    torch.cuda.synchronize()
    a = d.detectYuvPlanesRaw(descs16, memKind=1, orientations=orients, sampleBits=bits)
    b = d.detectYuvPlanesRaw(descs8, memKind=1, orientations=orients)
    assert records(*a[:2]) == records(*b[:2]) and min(b[1]) >= 1


@pytest.mark.parametrize("spec", [dict(kind="embedding", size=112, order="rgb", chw=True, dtype=np.float32,
                                       scale=(1 / 127.5,) * 3, bias=(-1.0,) * 3),
                                  dict(kind="face", size=96)])
def test_face_crops(fdt, sample_images, spec):
    """Face crops of P010 frames (uniform host and device, mixed) and of planes16 frames equal the 8-bit calls' crops."""
    d = detector(fdt, "shortRange", maxBatch=4)
    d.setFaceCrops(fdt.FaceCropSpec(**spec))
    try:
        total = 0
        for o in (1, 3, 6, 7):
            fr, ref = p010_pair(lm(sample_images), o, pad=2, seed=o)
            for mode in (0, 2):
                want, n = run(d, ref, mode)
                wc, wok = d.faceCrops()
                got, _ = run(d, fr, mode)
                gc, gok = d.faceCrops()
                assert_same(got, want, (o, mode))
                assert len(wc) == n >= 1 and np.array_equal(gc, wc) and np.array_equal(gok, wok), (o, mode)
                total += n
            t = to_device([fr.data])
            run(d, fr, 0, ptr=int(t[0].data_ptr()))
            gc, _ = d.faceCrops()
            run(d, ref)
            assert np.array_equal(gc, d.faceCrops()[0]), (o, "device")
        assert total >= 8
        got, want = mixed(sample_images)
        got, want = got[:9], want[:9]
        orients = [f.o for f in got]
        for mode in (0, 2):
            a = d.detectFramesRaw([f.desc() for f in got], mode=mode, orientations=orients)
            gc, gok = d.faceCrops()
            b = d.detectFramesRaw([f.desc() for f in want], mode=mode, orientations=orients)
            wc, wok = d.faceCrops()
            assert records(*a[:2]) == records(*b[:2])
            assert len(wc) >= 4 and np.array_equal(gc, wc) and np.array_equal(gok, wok), mode
        rng = np.random.default_rng(1)
        surf = [p016_surface(p010_pair(lm(sample_images), o, seed=o)[1], 16, rng) for o in (1, 6)]
        for mode in (0, 2):
            d.detectYuvPlanesRaw([s[0] for s in surf], mode=mode, orientations=[1, 6], sampleBits=16)
            gc, gok = d.faceCrops()
            d.detectYuvPlanesRaw([s[1] for s in surf], mode=mode, orientations=[1, 6])
            wc, wok = d.faceCrops()
            assert len(wc) >= 2 and np.array_equal(gc, wc) and np.array_equal(gok, wok), mode
    finally:
        d.setFaceCrops(None)


def test_status_codes(fdt, lib):
    d = detector(fdt, "shortRange")
    ffi = fdt._ffi
    faces = (ffi.FdtFace * 300)()
    counts = (C.c_int32 * 3)()
    buf = np.zeros(4 * 64 * 64 * 3, np.uint8)
    for fn in (lambda w, h, s: lib.fdt_detect_batch(d._h, buf.ctypes.data, 1, w, h, s, P010, 0, 0, faces, counts, None, None),
               lambda w, h, s: lib.fdt_detect_batch_oriented(d._h, buf.ctypes.data, 1, w, h, s, P010, 6, 0, 0, faces, counts, None, None)):
        assert fn(64, 48, 126) == ffi.FDT_ERR_SIZE_MISMATCH
        assert fn(63, 48, 128) == ffi.FDT_ERR_BAD_ARG                      # odd (stored) width
        assert fn(64, 47, 128) == ffi.FDT_ERR_BAD_ARG                      # odd (stored) height
        assert fn(64, 48, 131) == ffi.FDT_ERR_BAD_ARG                      # odd row stride
        assert fn(64, 48, 128) == ffi.FDT_OK
        assert fn(64, 48, 136) == ffi.FDT_OK
    good = ffi.FdtFrame(buf.ctypes.data, 64, 48, 128, P010)
    short = ffi.FdtFrame(buf.ctypes.data, 64, 48, 126, P010)
    odd = ffi.FdtFrame(buf.ctypes.data, 64, 48, 129, P010)
    assert lib.fdt_detect_frames(d._h, (ffi.FdtFrame * 3)(good, short, good), 3, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_SIZE_MISMATCH
    assert b"frame 1" in lib.fdt_last_error(d._h)
    assert lib.fdt_detect_frames_oriented(d._h, (ffi.FdtFrame * 3)(good, good, odd), (C.c_int32 * 3)(1, 6, 8), 3, 0, 0, faces, counts,
                                          None, None) == ffi.FDT_ERR_BAD_ARG
    assert b"frame 2" in lib.fdt_last_error(d._h)
    n = C.c_int32(0)
    size = 64 * 48 * 3
    for wrong in (size - 1, size + 1, 64 * 48 * 3 // 2, 64 * 48 * 2):
        assert lib.fdt_detect_one(d._h, buf.ctypes.data, wrong, 64, 48, P010, 0, faces, C.byref(n), None, None) == ffi.FDT_ERR_SIZE_MISMATCH
    assert lib.fdt_detect_one(d._h, buf.ctypes.data, size, 63, 48, P010, 0, faces, C.byref(n), None, None) == ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_one(d._h, buf.ctypes.data, size, 64, 48, P010, 0, faces, C.byref(n), None, None) == ffi.FDT_OK
    rois = (C.c_double * 4)(32, 24, 20, 0)
    out = np.zeros(16 * 16 * 3, np.uint8)
    ok = (C.c_int32 * 1)()
    assert lib.fdt_extract_aligned_squares(d._h, buf.ctypes.data, 64, 48, 128, P010, rois, 1, 16, out.ctypes.data, ok) == ffi.FDT_ERR_BAD_ARG
    # fdt_detect_yuv_planes16
    base = buf.ctypes.data

    def planes(y=0, u=64 * 48 * 2, v=64 * 48 * 2 + 64, ys=128, us=128, vs=128, ps=1, w=64, h=48):
        return ffi.FdtYuvPlanes((C.c_void_p * 3)(base + y, base + u, base + v), (C.c_int32 * 3)(ys, us, vs), w, h, ps, 0)

    def call(descs, bits=10):
        arr = (ffi.FdtYuvPlanes * len(descs))(*descs)
        return lib.fdt_detect_yuv_planes16(d._h, arr, None, len(descs), bits, 0, 0, faces, counts, None, None)

    assert call([planes()]) == ffi.FDT_OK
    assert call([planes(), planes(ps=2, us=128, vs=128, v=64 * 48 * 2 + 2)], 16) == ffi.FDT_OK
    for bits in (0, 8, 9, 11, 14, 15, 17, 32, -10):
        assert call([planes()], bits) == ffi.FDT_ERR_BAD_ARG, bits
    assert call([planes(), planes(u=64 * 48 * 2 + 1)]) == ffi.FDT_ERR_BAD_ARG
    assert b"frame 1" in lib.fdt_last_error(d._h) and b"plane U" in lib.fdt_last_error(d._h)
    assert call([planes(vs=129)]) == ffi.FDT_ERR_BAD_ARG and b"plane V" in lib.fdt_last_error(d._h)
    assert call([planes(y=1)]) == ffi.FDT_ERR_BAD_ARG and b"plane Y" in lib.fdt_last_error(d._h)
    assert call([planes(ys=126)]) == ffi.FDT_ERR_SIZE_MISMATCH
    assert call([planes(us=62)]) == ffi.FDT_ERR_SIZE_MISMATCH                  # 2 * ((64 / 2 - 1) * 1 + 1) = 64
    assert call([planes(us=64, vs=64)]) == ffi.FDT_OK
    assert call([planes(ps=2, us=124, vs=124)]) == ffi.FDT_ERR_SIZE_MISMATCH   # 2 * ((64 / 2 - 1) * 2 + 1) = 126
    assert call([planes(ps=2, us=126, vs=126)]) == ffi.FDT_OK
    assert call([planes(w=63)]) == ffi.FDT_ERR_BAD_ARG
    assert call([planes(ps=3)]) == ffi.FDT_ERR_BAD_ARG
    arr = (ffi.FdtYuvPlanes * 1)(planes())
    assert lib.fdt_detect_yuv_planes16(d._h, arr, (C.c_int32 * 1)(9), 1, 10, 0, 0, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG
    assert lib.fdt_detect_yuv_planes16(d._h, arr, None, 1, 10, 0, 1, faces, counts, None, None) == ffi.FDT_ERR_BAD_ARG   # host pointers


def test_python_api(fdt, sample_images):
    d = detector(fdt, "shortRange")
    img = lm(sample_images)
    fr, ref = p010_pair(img, 1, seed=4)
    mat16 = fr.data.view(np.uint16).reshape(img.shape[0] * 3 // 2, -1)
    got = d.detectFacesFromMat(mat16, layout="p010")
    want = d.detectFacesFromMatBytes(ref.data, width=ref.w, height=ref.h, matType=NV12)
    assert len(got) == len(want) >= 1
    for g, w in zip(got, want):
        assert g.detectionData.boundingBox == w.detectionData.boundingBox and np.array_equal(g.mesh.packed, w.mesh.packed)
    for o in (3, 6):
        fr, ref = p010_pair(img, o, pad=3, seed=o)
        m = fr.data.view(np.uint16).reshape(fr.h * 3 // 2, -1)
        got = d.detectFacesFromMats([np.ascontiguousarray(m[:, :fr.w]), m[:, :fr.w]], layout="p010", orientations=[o, o])
        want = d.detectFacesFromMatBytes(ref.data, width=ref.w, height=ref.h, matType=NV12, orientation=o)
        assert [len(f) for f in got] == [len(want)] * 2 and len(want) >= 1
        for g in got:
            assert [f.detectionData.boundingBox for f in g] == [f.detectionData.boundingBox for f in want]


@pytest.mark.parametrize("size", [(1680, 1050), (432, 286), (1278, 850)])
def test_heights_two_mod_four(fdt, sample_images, size):
    """Frames whose even height is 2 mod 4 (a 1680x1050 screen capture): the (3H/2) x W array goes in through both Python
    layouts and the raw calls, host and device, and every result equals the NV12 call's."""
    d = detector(fdt, "shortRange")
    w, h = size
    assert h % 4 == 2
    img = cv2.resize(lm(sample_images), (w, h), interpolation=cv2.INTER_AREA)
    for o in (1, 6):
        fr, ref = p010_pair(img, o, seed=w + o)
        want, n = run(d, ref, 2)
        assert n >= 1, (size, o)
        assert_same(run(d, fr, 2)[0], want, (size, o, "host"))
        t = to_device([fr.data])
        assert_same(run(d, fr, ptr=int(t[0].data_ptr()))[0], run(d, ref)[0], (size, o, "device"))
        m = fr.data.view(np.uint16).reshape(fr.h * 3 // 2, fr.w)
        got = d.detectFacesFromMat(m, layout="p010", orientation=o)
        wref = d.detectFacesFromMatBytes(ref.data, width=ref.w, height=ref.h, matType=NV12, orientation=o)
        assert len(got) == len(wref) >= 1
        for g, r in zip(got, wref):
            assert g.detectionData.boundingBox == r.detectionData.boundingBox and np.array_equal(g.mesh.packed, r.mesh.packed)
        per = d.detectFacesFromMats([m], layout="p010", orientations=[o])
        assert [f.detectionData.boundingBox for f in per[0]] == [f.detectionData.boundingBox for f in wref]


def test_multi_device(fdt, sample_images):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    one = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=[0], maxBatch=8)
    multi = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, devices=list(range(ndev)), maxBatch=8)
    try:
        fr, ref = p010_pair(lm(sample_images), 6, pad=4, seed=1)
        a = multi.detectBatchRaw(np.stack([fr.data] * 20), count=20, width=fr.w, height=fr.h, matType=P010, rowStride=fr.stride,
                                 orientation=6, mode=2, withIris=True)
        b = one.detectBatchRaw(np.stack([ref.data] * 20), count=20, width=ref.w, height=ref.h, matType=NV12, orientation=6, mode=2,
                               withIris=True)
        assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
        rng = np.random.default_rng(2)
        surf = [p016_surface(ref, 16, rng) for _ in range(12)]
        a = multi.detectYuvPlanesRaw([s[0] for s in surf], mode=2, orientations=[6] * 12, sampleBits=16)
        b = one.detectYuvPlanesRaw([s[1] for s in surf], mode=2, orientations=[6] * 12)
        assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
        got, want = mixed(sample_images)
        orients = [f.o for f in got]
        a = multi.detectFramesRaw([f.desc() for f in got], mode=2, orientations=orients)
        b = one.detectFramesRaw([f.desc() for f in want], mode=2, orientations=orients)
        assert records(*a[:2]) == records(*b[:2]) and np.array_equal(a[2], b[2])
    finally:
        one.dispose(); multi.dispose()
