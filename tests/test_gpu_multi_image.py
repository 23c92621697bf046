"""GPU parity where one CTA of an image-resident kernel runs several images.

k_tail_ws and k_chain_wide launch min(B, SMs) CTAs and walk images img = blockIdx.x, + gridDim.x, ...; k_fc_tc tiles the
faces of a mesh pass in M-tiles of 128.  A CTA's second and later images take paths of their own: the next input is
prefetched into buffer 0 after the planner's last_a_layer, the barrier phases follow the image count, the weight and tap
rings keep counting across images, and the channel pads of every buffer are zeroed only once.  These tests run chunks
larger than the SM count and check every image:
  * against the fp64 oracle, on a reference run whose chunks (64 frames, or mesh passes of <= 64 faces) are smaller than
    the SM count, so every image runs first in its CTA: raw heads <= 1e-4 of the SAME image's max|ref| per head, candidate
    index sets bit-exact except anchors whose oracle logit lies within 10x that image's largest score error of 0;
  * bitwise against that reference run, at positions beyond the SM count (second and third image of a CTA, second and
    third M-tile), where results must not depend on the position of an image in its chunk.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import cv_ops as co, detect_post as dp
from oracle.pipeline import OraclePipeline

pytestmark = pytest.mark.gpu

HEAD_REL_TOL = 1e-4       # of the same image's (crop's) max|ref|, per output tensor
CAND_MARGIN = 10.0        # candidate anchors closer to the threshold than this many times the image's score error may flip
REF_CHUNK = 64            # reference handle: one image per CTA (64 < SM count)
MESH_REF_CHUNK = 16       # reference handle for the mesh / iris passes: mesh_cap = 64 faces, one crop per CTA
ORACLE_BATCH = 16


@pytest.fixture(scope="module")
def fdt(lib):
    import face_detection_tflite_b200 as pkg
    return pkg


_cache = {}


def cached(key, make):
    if key not in _cache:
        _cache[key] = make()
    return _cache[key]


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def oracle(model_bytes, model):
    def make():
        from conftest import ASSETS
        iris = (ASSETS / "models" / "iris_landmark.tflite").read_bytes()
        return OraclePipeline(model_bytes[model], model, model_bytes["mesh"], "f64", iris_bytes=iris)
    return cached(("oracle", model), make)


def records(faces, counts):
    """Per frame: the raw bytes of its valid face records (FdtFace, no padding)."""
    n, sz = len(counts), C.sizeof(type(faces[0]))
    a = np.frombuffer(faces, np.uint8).reshape(n, -1)
    return [a[b, :int(counts[b]) * sz].tobytes() for b in range(n)]


# ---- detectors -------------------------------------------------------------------------------------------------------
def det_frames():
    """P = 2 * SMs + 3 distinct 640x360 frames: CTAs 0-2 of a P-frame chunk run three images each."""
    def make():
        from face_detection_tflite_b200 import synth
        P = 2 * sm_count() + 3
        n_noise = 6
        fr = [synth.face_frame(k, 640, 360) for k in range(P - n_noise)]
        fr += [synth.noise_frames(1, 640, 360, seed=100 + s)[0] for s in range(n_noise)]
        return np.ascontiguousarray(np.stack(fr))
    return cached("det_frames", make)


def reference_run(fdt, model):
    """Run R: maxBatch 64, single-chunk calls of 64 frames, so every image is the first (only) image of its CTA."""
    def make():
        frames = det_frames()
        P = len(frames)
        d = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], withMesh=False, maxBatch=REF_CHUNK)
        boxes, scores, cands, recs = [], [], [], []
        for off in range(0, P, REF_CHUNK):
            n = min(REF_CHUNK, P - off)
            faces, counts, _ = d.detectBatchRaw(frames[off:off + n], count=n, width=640, height=360)
            b, s = d.debugRawHeads(n)
            boxes.append(b)
            scores.append(s)
            cands += [d.debugCandidates(i) for i in range(n)]
            recs += records(faces, counts)
        d.dispose()
        return {"boxes": np.concatenate(boxes), "scores": np.concatenate(scores), "cands": cands, "recs": recs}
    return cached(("R", model), make)


def oracle_heads(model_bytes, model):
    def make():
        o = oracle(model_bytes, model)
        frames = det_frames()
        boxes, scores = [], []
        for off in range(0, len(frames), ORACLE_BATCH):
            r = o.det.run(np.stack([o.preprocess(fr)[0] for fr in frames[off:off + ORACLE_BATCH]]))
            boxes.append(np.asarray(r[0]).reshape(r[0].shape[0], -1, 16))
            scores.append(np.asarray(r[1]).reshape(r[1].shape[0], -1))
        return np.concatenate(boxes), np.concatenate(scores)
    return cached(("oracle_heads", model), make)


DET_MODELS = ["shortRange", "full", "backCamera"]


@pytest.mark.parametrize("model", DET_MODELS)
def test_every_image_of_reference_run_matches_f64_oracle(fdt, model_bytes, model):
    """Every image of R against the fp64 oracle, each with its own scale: a small-range image cannot hide behind the batch."""
    R = reference_run(fdt, model)
    want_b, want_s = oracle_heads(model_bytes, model)
    P = len(det_frames())
    assert R["boxes"].shape == want_b.shape and R["scores"].shape == want_s.shape
    worst = {"boxes": 0.0, "scores": 0.0}
    flips = 0
    for i in range(P):
        for name, got, want in (("boxes", R["boxes"][i], want_b[i]), ("scores", R["scores"][i], want_s[i])):
            err = float(np.abs(got - want).max() / np.abs(want).max())
            worst[name] = max(worst[name], err)
            assert err <= HEAD_REL_TOL, (model, i, name, err)
        idx, _ = dp.collect_candidates(want_s[i])
        got = set(R["cands"][i].tolist())
        assert list(R["cands"][i]) == sorted(got)                                  # ascending anchor order
        near = set(np.flatnonzero(np.abs(want_s[i]) <= CAND_MARGIN * np.abs(R["scores"][i] - want_s[i]).max()).tolist())
        if near:
            print("%s image %d: anchors within the score-error margin of the threshold: %s" % (model, i, sorted(near)))
        diff = got ^ set(idx)
        assert diff <= near, (model, i, sorted(diff - near))
        flips += len(diff)
    print("%s: %d images, worst rel err boxes %.2e scores %.2e (bar %.0e), candidate flips %d"
          % (model, P, worst["boxes"], worst["scores"], HEAD_REL_TOL, flips))


@pytest.mark.parametrize("model", DET_MODELS)
def test_chunk_beyond_sm_count_equals_reference_bitwise(fdt, model):
    """All P frames in one chunk (CTAs 0-2 run three images, the others two): heads and candidates of every image equal R."""
    R = reference_run(fdt, model)
    frames = det_frames()
    P, sms = len(frames), sm_count()
    d = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], withMesh=False, maxBatch=P)
    sizes = [P, sms + 1] if model == "shortRange" else [P]                          # sms + 1: only CTA 0 takes a second image
    for n in sizes:
        faces, counts, _ = d.detectBatchRaw(frames[:n], count=n, width=640, height=360)
        boxes, scores = d.debugRawHeads(n)
        for i in range(n):
            assert np.array_equal(boxes[i], R["boxes"][i]) and np.array_equal(scores[i], R["scores"][i]), (model, n, i)
            assert np.array_equal(d.debugCandidates(i), R["cands"][i]), (model, n, i)
        assert records(faces, counts) == R["recs"][:n]
        assert int(counts.sum()) > 0
        for b in range(n):                                                           # fast mode: no mesh, no iris, reserved zero
            for j in range(int(counts[b])):
                f = faces[b * d._max_faces + j]
                assert (f.has_mesh, f.has_iris, f.reserved) == (0, 0, 0), (model, n, b, j)
    d.dispose()


def test_short_range_chunk_1024_position_invariance(fdt):
    """bench.py C2's chunk of 1024 device-resident frames, frame i = frame i % P: P is not a multiple of the SM count, so
    one frame lands on different CTAs and at different positions within a CTA.  Its heads equal R's bitwise."""
    import torch
    R = reference_run(fdt, "shortRange")
    frames = det_frames()
    P, n = len(frames), 1024
    dev = torch.from_numpy(frames).cuda()[torch.arange(n) % P].contiguous()
    d = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=n)
    faces, counts, _ = d.detectBatchRaw(dev.data_ptr(), count=n, width=640, height=360, memKind=1)
    boxes, scores = d.debugRawHeads(n)
    recs = records(faces, counts)
    for i in range(n):
        assert np.array_equal(boxes[i], R["boxes"][i % P]) and np.array_equal(scores[i], R["scores"][i % P]), i
        assert recs[i] == R["recs"][i % P], i
    d.dispose()


def readable_tensor(d, t):
    try:
        return d.debugTensor(0, t, 1).shape[0] == 1
    except (ValueError, NotImplementedError):                  # not materialised, or its buffer is reused in this plan
        return False


@pytest.mark.parametrize("model", DET_MODELS)
def test_three_chunks_over_both_slots_and_tap_validity(fdt, model_bytes, model):
    """3 * P device-resident frames on a maxBatch = P handle: three chunks over both pipeline slots, each chunk a rotation
    of the P frames.  Every frame's face records equal R's.  The third chunk reuses slot 0, so the taps that read slot 0
    refuse; the candidate tap still holds chunk 0."""
    import torch
    R = reference_run(fdt, model)
    frames = det_frames()
    P = len(frames)
    n_tensors = len(oracle(model_bytes, model).det.model.tensors)
    dev_base = torch.from_numpy(frames).cuda()
    d = fdt.FaceDetector.create(fdt.FaceDetectionModel[model], withMesh=False, maxBatch=P)
    for chunks in (2, 3):
        order = np.concatenate([np.roll(np.arange(P), -c) for c in range(chunks)])
        dev = dev_base[torch.from_numpy(order)].contiguous()
        faces, counts, _ = d.detectBatchRaw(dev.data_ptr(), count=len(order), width=640, height=360, memKind=1)
        recs = records(faces, counts)
        for i, j in enumerate(order):
            assert recs[i] == R["recs"][j], (model, chunks, i)
        for i in range(P):                                                            # chunk 0 is the identity order
            assert np.array_equal(d.debugCandidates(i), R["cands"][i]), (model, chunks, i)
        if chunks == 2:                                                               # slot 0 still holds chunk 0
            boxes, scores = d.debugRawHeads(P)
            assert np.array_equal(boxes, R["boxes"]) and np.array_equal(scores, R["scores"])
            tensor = next(t for t in range(n_tensors) if readable_tensor(d, t))
            d.debugLetterboxed(1)
            d.debugInputTensor(1)
        else:
            for tap in (lambda: d.debugRawHeads(1), lambda: d.debugLetterboxed(1), lambda: d.debugInputTensor(1),
                        lambda: d.debugTensor(0, tensor, 1)):
                with pytest.raises(ValueError, match="more than two chunks"):
                    tap()
    d.dispose()


# ---- mesh and iris passes ----------------------------------------------------------------------------------------------
def mesh_frames(fdt):
    """1280x720 frames of four (5k + 4) and one (5k + 1) face tiles, and their detector face counts."""
    def make():
        from face_detection_tflite_b200 import synth
        four = np.stack([synth.face_frame(5 * k + 4, 1280, 720) for k in range(160)])
        one = np.stack([synth.face_frame(5 * k + 1, 1280, 720) for k in range(24)])
        d = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False)
        c4 = d.detectBatchRaw(four, count=len(four), width=1280, height=720)[1].copy()
        c1 = d.detectBatchRaw(one, count=len(one), width=1280, height=720)[1].copy()
        d.dispose()
        return four, c4, one, c1
    return cached("mesh_frames", make)


def select_frames(four, c4, one, c1, total=None, at_least=None):
    """Distinct frames whose detections add up to exactly `total` faces, or to at least `at_least`."""
    picked, s = [], 0
    for k in range(len(four)):
        if at_least is not None and s >= at_least:
            break
        if c4[k] > 0 and (total is None or s + c4[k] <= total):
            picked.append(four[k])
            s += int(c4[k])
    if total is not None:
        for k in np.flatnonzero(c1 == 1):
            if s == total:
                break
            picked.append(one[k])
            s += 1
        assert s == total, "the frame pool cannot make %d faces" % total
    else:
        assert s >= at_least, "the frame pool holds only %d faces" % s
    return np.ascontiguousarray(np.stack(picked)), s


def mesh_case(fdt, case):
    """One chunk's single mesh pass on the default handle (maxBatch 256, mesh_cap 512) and the same frames on a maxBatch
    16 handle (mesh passes of <= 64 faces).  "257": exactly 257 faces in standard mode (three k_fc_tc M-tiles, the last
    with one row; some tail CTAs take two faces).  "2sms": at least 2 * SMs + 1 faces in full mode (CTA 0 takes three)."""
    def make():
        four, c4, one, c1 = mesh_frames(fdt)
        if case == "257":
            frames, nf = select_frames(four, c4, one, c1, total=257)
            mode = fdt.FaceDetectionMode.standard
        else:
            frames, nf = select_frames(four, c4, one, c1, at_least=2 * sm_count() + 1)
            mode = fdt.FaceDetectionMode.full
        n = len(frames)
        out = {"frames": frames, "nf": nf, "mode": mode}
        d = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange)
        assert d.maxBatch == 256 and n <= 256
        faces, counts, mesh, iris = d.detectBatchRaw(frames, count=n, width=1280, height=720, mode=mode, withIris=True)
        out["got"] = (records(faces, counts), counts.copy(), mesh, iris)
        out["mesh_stage"] = d.debugMeshStage(nf + 1)
        if mode == fdt.FaceDetectionMode.full:
            out["iris_stage"] = d.debugIrisStage(nf + 1)
        d.dispose()
        r = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, maxBatch=MESH_REF_CHUNK)
        faces, counts, mesh, iris = r.detectBatchRaw(frames, count=n, width=1280, height=720, mode=mode, withIris=True)
        out["ref"] = (records(faces, counts), counts.copy(), mesh, iris)
        r.dispose()
        return out
    return cached(("mesh_case", case), make)


@pytest.mark.parametrize("case", ["257", "2sms"])
def test_mesh_pass_every_crop_matches_f64_oracle(fdt, model_bytes, case):
    """Raw 1404 outputs and face flag of every crop of the pass vs the fp64 mesh net on that same crop."""
    mc = mesh_case(fdt, case)
    crops, raw, flag = mc["mesh_stage"]
    assert len(crops) == mc["nf"]                                                     # one pass holds every face of the chunk
    if case == "257":
        assert mc["nf"] == 257
    else:
        assert mc["nf"] >= 2 * sm_count() + 1
    o = oracle(model_bytes, "shortRange")
    worst_raw = worst_flag = 0.0
    for off in range(0, len(crops), ORACLE_BATCH):
        ref = o.mesh.run(np.stack([co.normalize_bgr_u8(c) for c in crops[off:off + ORACLE_BATCH]]))
        li = int(np.argmax([x.shape[1] for x in ref]))
        for k in range(ref[li].shape[0]):
            f = off + k
            e = float(np.abs(raw[f] - ref[li][k]).max() / np.abs(ref[li][k]).max())
            ef = float(abs(flag[f] - ref[1 - li][k][0]) / max(1.0, abs(ref[1 - li][k][0])))
            worst_raw, worst_flag = max(worst_raw, e), max(worst_flag, ef)
            assert e <= HEAD_REL_TOL, (case, f, e)
            assert ef <= HEAD_REL_TOL, (case, f, ef)
    print("mesh pass %s: %d crops, worst rel err raw %.2e flag %.2e (bar %.0e)" % (case, len(crops), worst_raw, worst_flag, HEAD_REL_TOL))


@pytest.mark.parametrize("case", ["257", "2sms"])
def test_mesh_pass_equals_small_passes_bitwise(fdt, case):
    """Face records (detection data, mesh score, iris-refined eye keypoints), meshes and, in full mode, iris points of every
    face equal those of passes of <= 64 faces, where each crop runs alone in its CTA."""
    mc = mesh_case(fdt, case)
    recs, counts, mesh, iris = mc["got"]
    rrecs, rcounts, rmesh, riris = mc["ref"]
    assert np.array_equal(counts, rcounts)
    assert 2 * int(counts.sum()) >= mc["nf"]                                          # the presence gate keeps most faces
    for b in range(len(counts)):
        assert recs[b] == rrecs[b], (case, b)
        c = int(counts[b])
        assert np.array_equal(mesh[b, :c], rmesh[b, :c]), (case, b)
        if iris is not None:
            assert np.array_equal(iris[b, :c], riris[b, :c]), (case, b)


def test_iris_pass_beyond_sm_count_matches_f64_oracle(fdt, model_bytes):
    """Full mode: one iris pass of more than 2 * SMs eye crops; every crop's contours and iris outputs vs the fp64 iris
    net on that same crop."""
    mc = mesh_case(fdt, "2sms")
    crops, rois, cont, ir = mc["iris_stage"]
    assert len(crops) > 2 * sm_count()
    o = oracle(model_bytes, "shortRange")
    worst = 0.0
    for off in range(0, len(crops), 4 * ORACLE_BATCH):
        ref = o.iris.run(np.stack([co.normalize_bgr_u8(c) for c in crops[off:off + 4 * ORACLE_BATCH]]))
        for k in range(ref[0].shape[0]):
            e = off + k
            for got, want in ((cont[e], ref[0][k]), (ir[e], ref[1][k])):
                err = float(np.abs(got - want).max() / np.abs(want).max())
                worst = max(worst, err)
                assert err <= HEAD_REL_TOL, (e, err)
    print("iris pass: %d eye crops, worst rel err %.2e (bar %.0e)" % (len(crops), worst, HEAD_REL_TOL))
