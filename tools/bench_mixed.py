"""Mixed batches against what a caller could do before them, one process, one GPU.

Photo workload: 1024 frames over 12 sizes from 640x480 to 4032x3024, landscape and portrait (the sample photos resized,
6 unique frames per size, tiled), short-range detector, maxBatch 256.  For fast and standard mode, host (pageable) and device
frames, the variants alternate for --rounds rounds:
  (a) per_frame: one fdt_detect_batch call per frame;
  (b) per_size:  one fdt_detect_batch call per group of equal-sized frames (the best a caller could do without mixed batches);
  (c) mixed:     one fdt_detect_frames call over the whole list.
JPEG workload: --jpegs photos re-encoded at quality 90 over the same 12 sizes; fdt_detect_jpeg per image against one
fdt_detect_jpeg_batch call, fast and standard mode, next to the single-thread host Huffman decode time of the same images
(fdt_host_jpeg_info runs the whole entropy decoder).
Letterbox cost: stage 0 of fdt_set_stage_timing for a uniform C2 chunk (1024 device frames of 1280x720, maxBatch 1024):
k_letterbox (fdt_detect_batch) against k_letterbox_multi (fdt_detect_frames on the same frames).

Every time is a host clock around calls that end in a device synchronise (the library returns results on the host).

    python tools/bench_mixed.py [--rounds 3] [--out profiles/r04a_bench_mixed.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_yuv import card  # noqa: E402

SIZES = [(640, 480), (480, 640), (1024, 768), (1280, 720), (720, 1280), (1280, 960), (1920, 1080), (1080, 1920),
         (2048, 1536), (2592, 1944), (3024, 4032), (4032, 3024)]
UNIQUE = 6
BGR = 16


def photo_frames(n):
    """{size: [count, h, w, 3] contiguous frames} and the list order: frame i has size SIZES[i % 12], index i // 12 in its group."""
    import cv2
    samples = [cv2.imread(str(p)) for p in sorted((ROOT / "assets" / "samples").glob("*.jp*g"))]
    groups = {}
    for k, (w, h) in enumerate(SIZES):
        count = len(range(k, n, len(SIZES)))
        uniq = []
        for u in range(UNIQUE):
            img = samples[u % len(samples)]
            img = cv2.flip(img, 1) if u >= len(samples) else img
            uniq.append(cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA))
        groups[(w, h)] = np.ascontiguousarray(np.stack([uniq[i % UNIQUE] for i in range(count)]))
    order = [(SIZES[i % len(SIZES)], i // len(SIZES)) for i in range(n)]
    return groups, order


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--jpegs", type=int, default=300)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import cv2
    import torch
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi, build

    build.build()
    lib = _ffi.load()
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withIris=False, maxBatch=256)
    h, mf = det._h, det._max_faces

    def check(rc):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(h).decode())

    n = args.frames
    groups, order = photo_frames(n)
    dgroups = {k: torch.from_numpy(v).cuda() for k, v in groups.items()}
    torch.cuda.synchronize()
    ptr = {"host": {k: v.ctypes.data for k, v in groups.items()}, "device": {k: int(v.data_ptr()) for k, v in dgroups.items()}}
    faces = (_ffi.FdtFace * (n * mf))()
    counts = np.zeros(n, np.int32)
    cp = counts.ctypes.data_as(_ffi.i32p)
    mesh = np.zeros((n, mf, 468, 3), np.float32)
    frame_bytes = sum(w * hh * 3 for (w, hh), _ in order)

    def frames_of(mem):
        return (_ffi.FdtFrame * n)(*[_ffi.FdtFrame(ptr[mem][s] + j * s[0] * s[1] * 3, s[0], s[1], s[0] * 3, BGR) for s, j in order])

    descs = {mem: frames_of(mem) for mem in ("host", "device")}

    def run(variant, mode, mem):
        mk = 0 if mem == "host" else 1
        mp = mesh.ctypes.data_as(_ffi.f32p) if mode else None
        t0 = time.perf_counter()
        if variant == "per_frame":
            for i, (s, j) in enumerate(order):
                check(lib.fdt_detect_batch(h, ptr[mem][s] + j * s[0] * s[1] * 3, 1, s[0], s[1], s[0] * 3, BGR, mode, mk, faces,
                                           cp, mp, None))
        elif variant == "per_size":
            for s, g in groups.items():
                check(lib.fdt_detect_batch(h, ptr[mem][s], len(g), s[0], s[1], s[0] * 3, BGR, mode, mk, faces, cp, mp, None))
        else:
            check(lib.fdt_detect_frames(h, descs[mem], n, mode, mk, faces, cp, mp, None))
        return time.perf_counter() - t0

    variants = ("per_frame", "per_size", "mixed")
    combos = [(mode, mem) for mode in (0, 1) for mem in ("host", "device")]
    for mode, mem in combos:                       # warm-up: every shape the timed rounds use
        for v in variants:
            run(v, mode, mem)
    # the mixed call finds the faces the per-frame calls find
    ref = []
    for s, j in order:
        check(lib.fdt_detect_batch(h, ptr["host"][s] + j * s[0] * s[1] * 3, 1, s[0], s[1], s[0] * 3, BGR, 0, 0, faces, cp, None, None))
        ref.append(int(counts[0]))
    check(lib.fdt_detect_frames(h, descs["host"], n, 0, 0, faces, cp, None, None))
    assert counts.tolist() == ref, "fdt_detect_frames disagrees with per-frame calls"
    photo_faces = int(sum(ref))

    rounds = []
    for r in range(args.rounds):
        row = {"round": r}
        for mode, mem in combos:
            key = "%s_%s" % ("fast" if mode == 0 else "standard", mem)
            row[key] = {v: n / run(v, mode, mem) for v in variants}
        rounds.append(row)
        print(json.dumps(row), flush=True)
    photo = {}
    for mode, mem in combos:
        key = "%s_%s" % ("fast" if mode == 0 else "standard", mem)
        photo[key] = {v: {"img_s_median": statistics.median(x[key][v] for x in rounds),
                          "img_s_range": [min(x[key][v] for x in rounds), max(x[key][v] for x in rounds)]} for v in variants}
        photo[key]["mixed_over_per_size"] = photo[key]["mixed"]["img_s_median"] / photo[key]["per_size"]["img_s_median"]
        photo[key]["mixed_over_per_frame"] = photo[key]["mixed"]["img_s_median"] / photo[key]["per_frame"]["img_s_median"]

    # ---- JPEG workload
    jpegs = []
    for i in range(args.jpegs):
        s, j = order[i % n]
        jpegs.append(cv2.imencode(".jpg", groups[s][j], [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes())
    bufs = [np.frombuffer(b, np.uint8) for b in jpegs]
    nj = len(bufs)
    info = (C.c_int32 * 8)()
    t0 = time.perf_counter()
    for b in bufs:
        check(lib.fdt_host_jpeg_info(b.ctypes.data, b.size, info))
    host_decode_s = time.perf_counter() - t0
    jptrs = (C.c_void_p * nj)(*[b.ctypes.data for b in bufs])
    jsizes = (C.c_size_t * nj)(*[b.size for b in bufs])
    wh = np.zeros((nj, 2), np.int32)
    status = np.zeros(nj, np.int32)
    one_wh = (C.c_int32 * 2)()

    def run_jpeg(variant, mode):
        mp = mesh.ctypes.data_as(_ffi.f32p) if mode else None
        t0 = time.perf_counter()
        if variant == "per_image":
            for b in bufs:
                check(lib.fdt_detect_jpeg(h, b.ctypes.data, b.size, mode, faces, cp, mp, None, one_wh))
        else:
            check(lib.fdt_detect_jpeg_batch(h, jptrs, jsizes, nj, mode, faces, cp, mp, None, wh.ctypes.data_as(_ffi.i32p),
                                            status.ctypes.data_as(_ffi.i32p)))
            assert not status.any()
        return time.perf_counter() - t0

    for mode in (0, 1):
        for v in ("per_image", "batch"):
            run_jpeg(v, mode)
    jrounds = []
    for r in range(args.rounds):
        row = {"round": r}
        for mode in (0, 1):
            row["fast" if mode == 0 else "standard"] = {v: nj / run_jpeg(v, mode) for v in ("per_image", "batch")}
        jrounds.append(row)
        print(json.dumps(row), flush=True)
    jpeg = {m: {v: statistics.median(x[m][v] for x in jrounds) for v in ("per_image", "batch")} for m in ("fast", "standard")}
    jpeg["host_decode_one_thread_s"] = host_decode_s
    jpeg["host_decode_one_thread_img_s"] = nj / host_decode_s
    jpeg["host_threads"] = os.cpu_count()

    # ---- letterbox cost on a uniform C2 chunk
    det2 = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=1024)
    h2 = det2._h
    import bench
    base = bench.synth_base("c2")
    W, H, B = 1280, 720, 1024
    dev = torch.from_numpy(base).cuda()[torch.arange(B, device="cuda") % len(base)].contiguous()
    torch.cuda.synchronize()
    f2 = (_ffi.FdtFace * (B * mf))()
    c2 = np.zeros(B, np.int32)
    d2 = (_ffi.FdtFrame * B)(*[_ffi.FdtFrame(int(dev.data_ptr()) + i * W * H * 3, W, H, W * 3, BGR) for i in range(B)])
    lib.fdt_set_stage_timing(h2, 1)
    ms = C.c_float()
    lb = {"k_letterbox": [], "k_letterbox_multi": []}
    for r in range(2 + 10):
        for k in lb:
            if k == "k_letterbox":
                rc = lib.fdt_detect_batch(h2, int(dev.data_ptr()), B, W, H, W * 3, BGR, 0, 1, f2, c2.ctypes.data_as(_ffi.i32p), None, None)
            else:
                rc = lib.fdt_detect_frames(h2, d2, B, 0, 1, f2, c2.ctypes.data_as(_ffi.i32p), None, None)
            if rc != 0:
                raise RuntimeError(lib.fdt_last_error(h2).decode())
            lib.fdt_get_stage_ms(h2, 0, C.byref(ms), None)
            if r >= 2:
                lb[k].append(float(ms.value))
    lib.fdt_set_stage_timing(h2, 0)
    letterbox = {k: {"ms_median": statistics.median(v), "ms_range": [min(v), max(v)]} for k, v in lb.items()}
    letterbox["multi_over_uniform"] = letterbox["k_letterbox_multi"]["ms_median"] / letterbox["k_letterbox"]["ms_median"]

    result = {"workload": {"photos": "%d frames over %d sizes (640x480 .. 4032x3024, landscape and portrait), %d unique per size, "
                                     "%.2f GB of BGR; short-range detector, maxBatch 256, %d faces in fast mode"
                                     % (n, len(SIZES), UNIQUE, frame_bytes / 1e9, photo_faces),
                           "jpeg": "%d photos of the same sizes re-encoded at quality 90" % nj,
                           "letterbox": "C2 chunk: 1024 device frames of 1280x720 BGR, maxBatch 1024, stage timing stage 0"},
              "card": card(), "rounds": args.rounds, "photo": photo, "photo_rounds": rounds, "jpeg": jpeg, "jpeg_rounds": jrounds,
              "letterbox": letterbox,
              "how": "host clock around calls that return results on the host (each ends in a device synchronise); host frames "
                     "are pageable numpy arrays; variants alternate within each round after one warm-up pass of each"}
    print(json.dumps(result), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")
    det.dispose()
    det2.dispose()


if __name__ == "__main__":
    main()
