"""Frames stored sideways (EXIF orientation 6) against the same work on upright frames, one process, one GPU.

Workload: --batch synthetic 1280x720 frames (synth.face_frames, 64 unique, tiled), short-range detector, fast mode, chunks of
1024.  Each frame is stored sideways, as a 720 x 1280 image whose upright image (orientation 6) is the 1280x720 frame.  Variants:
  upright_o1  the upright frames, fdt_detect_batch (what orientation 6 must reproduce, bit for bit)
  stored_o1   the stored frames read as they are (a 720 x 1280 portrait letterbox, the same rows read as orientation 6)
  stored_o3   the stored frames rotated 180 degrees (orientation 3: flipped taps, plain kernels)
  stored_o6   the stored frames, fdt_detect_batch_oriented(6): the transposed gather
Device-resident: frames in device memory, results to the host, library timer (fdt_timer_begin / end); letterbox stage time per
1024 frames from fdt_set_stage_timing in a separate pass.  End to end: --e2e-batch frames in pinned host memory, BGR and NV12,
h2d bytes per frame from fdt_last_h2d_bytes, max(library timer, wall clock).  Status quo (BGR): the caller rotates every frame
with cv2.rotate on a host thread pool, then calls fdt_detect_batch on the upright frames.  Standard mode, C4-shaped (1024
frames, at most 4 faces, chunks of 512): stored_o6 against upright_o1.  Variants alternate within each of --rounds rounds.

    python tools/bench_orient.py [--rounds 3] [--out profiles/r05a_bench_orient.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_yuv import card, nv12_of  # noqa: E402

BGR, NV12 = 16, 0x1000


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--e2e-batch", type=int, default=2048)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import cv2
    import torch
    import bench
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi, build
    from oracle.jpeg_ops import exif_transform

    build.build()
    lib = _ffi.load()
    W, H, P = 1280, 720, bench.PERIOD
    up = bench.synth_base("c2")                                       # [P][720][1280][3] upright
    st = np.ascontiguousarray(np.stack([exif_transform(f, 8) for f in up]))   # [P][1280][720][3] stored: exif_transform(st, 6) == up
    assert np.array_equal(exif_transform(st[0], 6), up[0])
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=1024)
    h, mf = det._h, det._max_faces

    def check(rc, hh=h):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(hh).decode())

    # (frames, stored width, height, orientation) of each variant; the frames arrays are [P] unique frames
    geo = {"upright_o1": (W, H, 1), "stored_o1": (H, W, 1), "stored_o3": (H, W, 3), "stored_o6": (H, W, 6)}
    src = {"upright_o1": up, "stored_o1": st, "stored_o3": st, "stored_o6": st}

    # ---- device-resident
    B = args.batch
    idx = torch.arange(B, device="cuda") % P
    dev = {"up": torch.from_numpy(up).cuda()[idx].contiguous(), "st": torch.from_numpy(st).cuda()[idx].contiguous()}
    torch.cuda.synchronize()
    faces = (_ffi.FdtFace * (B * mf))()
    counts = np.zeros(B, np.int32)
    cp = counts.ctypes.data_as(_ffi.i32p)
    ms = C.c_float()

    def dev_call(v, n=B):
        w, hh, o = geo[v]
        ptr = dev["up" if v == "upright_o1" else "st"].data_ptr()
        check(lib.fdt_detect_batch_oriented(h, ptr, n, w, hh, w * 3, BGR, o, 0, 1, faces, cp, None, None))

    def device_rate(v):
        for _ in range(args.warmup):
            dev_call(v)
        lib.fdt_timer_begin(h)
        for _ in range(args.steps):
            dev_call(v)
        lib.fdt_timer_end(h, C.byref(ms))
        return B * args.steps / (ms.value / 1e3), int(counts.sum())

    def letterbox_ms(v):
        lib.fdt_set_stage_timing(h, 1)
        vals = []
        for r in range(2 + 5):
            dev_call(v)
            lib.fdt_get_stage_ms(h, 0, C.byref(ms), None)
            if r >= 2:
                vals.append(float(ms.value) * 1024 / B)
        lib.fdt_set_stage_timing(h, 0)
        return statistics.median(vals)

    # the oriented call reproduces the upright one
    dev_call("upright_o1")
    ref = counts.copy()
    dev_call("stored_o6")
    assert np.array_equal(counts, ref), "orientation 6 disagrees with the upright frames"
    dev_faces = int(ref.sum())

    # ---- end to end from pinned host memory
    E = args.e2e_batch
    pins, hosts = [], {}

    def pinned(frames):
        fb = frames[0].nbytes
        p = C.c_void_p()
        if lib.fdt_alloc_pinned(E * fb, C.byref(p)) != 0:
            raise RuntimeError("pinned allocation of %d bytes failed" % (E * fb))
        pins.append(p)
        arr = np.ctypeslib.as_array((C.c_uint8 * (E * fb)).from_address(p.value)).reshape((E,) + frames.shape[1:])
        for r0 in range(0, E, P):
            arr[r0:r0 + P] = frames[:min(P, E - r0)]
        return arr

    hosts[("bgr", "up")] = pinned(up)
    hosts[("bgr", "st")] = pinned(st)
    hosts[("nv12", "up")] = pinned(np.stack([nv12_of(f) for f in up]))
    hosts[("nv12", "st")] = pinned(np.stack([nv12_of(f) for f in st]))
    rot = pinned(up)                                                  # the status quo's rotation target
    ef = (_ffi.FdtFace * (E * mf))()
    ec = np.zeros(E, np.int32)
    ecp = ec.ctypes.data_as(_ffi.i32p)
    pool = ThreadPoolExecutor(os.cpu_count() or 8)

    def e2e_call(fmt, v):
        w, hh, o = geo[v]
        arr = hosts[(fmt, "up" if v == "upright_o1" else "st")]
        mt, stride = (BGR, w * 3) if fmt == "bgr" else (NV12, w)
        check(lib.fdt_detect_batch_oriented(h, arr.ctypes.data, E, w, hh, stride, mt, o, 0, 0, ef, ecp, None, None))

    def status_quo():
        s = hosts[("bgr", "st")]

        def one(i):
            cv2.rotate(s[i], cv2.ROTATE_90_CLOCKWISE, dst=rot[i])
        list(pool.map(one, range(E)))
        check(lib.fdt_detect_batch(h, rot.ctypes.data, E, W, H, W * 3, BGR, 0, 0, ef, ecp, None, None))

    def timed(fn, steps):
        for _ in range(max(1, args.warmup // 2)):
            fn()
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        return E * steps / (max(float(ms.value), wall) / 1e3)

    status_quo()
    assert np.array_equal(exif_transform(hosts[("bgr", "st")][5], 6), rot[5])

    # ---- standard mode, C4-shaped
    det4 = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withIris=False, maxBatch=512, maxFaces=4)
    h4 = det4._h
    up4 = bench.synth_base("c4")
    st4 = np.ascontiguousarray(np.stack([exif_transform(f, 8) for f in up4]))
    B4 = 1024
    i4 = torch.arange(B4, device="cuda") % P
    dev4 = {"upright_o1": torch.from_numpy(up4).cuda()[i4].contiguous(), "stored_o6": torch.from_numpy(st4).cuda()[i4].contiguous()}
    torch.cuda.synchronize()
    f4 = (_ffi.FdtFace * (B4 * 4))()
    c4 = np.zeros(B4, np.int32)
    m4 = np.zeros((B4, 4, 468, 3), np.float32)

    def std_call(v):
        w, hh, o = geo[v]
        check(lib.fdt_detect_batch_oriented(h4, dev4[v].data_ptr(), B4, w, hh, w * 3, BGR, o, 1, 1, f4, c4.ctypes.data_as(_ffi.i32p),
                                            m4.ctypes.data_as(_ffi.f32p), None), h4)

    def std_rate(v):
        std_call(v)
        lib.fdt_timer_begin(h4)
        t0 = time.perf_counter()
        for _ in range(max(2, args.steps // 2)):
            std_call(v)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h4, C.byref(ms))
        return B4 * max(2, args.steps // 2) / (max(float(ms.value), wall) / 1e3)

    std_call("upright_o1")
    ref4 = (c4.copy(), m4.copy())
    std_call("stored_o6")
    assert np.array_equal(c4, ref4[0]) and np.array_equal(m4, ref4[1]), "standard mode: orientation 6 disagrees with upright"
    std_faces = int(ref4[0].sum())

    rounds = []
    for r in range(args.rounds):
        row = {"round": r, "device_img_s": {}, "letterbox_ms_per_1024": {}, "e2e_img_s": {}, "h2d_bytes_per_frame": {},
               "standard_img_s": {}}
        for v in geo:
            row["device_img_s"][v] = device_rate(v)[0]
        for v in geo:
            row["letterbox_ms_per_1024"][v] = letterbox_ms(v)
        for fmt in ("bgr", "nv12"):
            for v in ("upright_o1", "stored_o1", "stored_o6"):
                k = "%s_%s" % (fmt, v)
                row["e2e_img_s"][k] = timed(lambda: e2e_call(fmt, v), args.steps)
                row["h2d_bytes_per_frame"][k] = int(lib.fdt_last_h2d_bytes(h)) / E
        row["e2e_img_s"]["bgr_status_quo_cv2_rotate"] = timed(status_quo, max(2, args.steps // 5))
        for v in ("upright_o1", "stored_o6"):
            row["standard_img_s"][v] = std_rate(v)
        rounds.append(row)
        print(json.dumps(row), flush=True)

    def summary(key):
        ks = rounds[0][key].keys()
        return {k: {"median": statistics.median(x[key][k] for x in rounds),
                    "range": [min(x[key][k] for x in rounds), max(x[key][k] for x in rounds)]} for k in ks}

    dv, lb, e2e, std = summary("device_img_s"), summary("letterbox_ms_per_1024"), summary("e2e_img_s"), summary("standard_img_s")
    ratios = {
        "device_o6_over_upright_o1": dv["stored_o6"]["median"] / dv["upright_o1"]["median"],
        "device_o6_over_stored_o1": dv["stored_o6"]["median"] / dv["stored_o1"]["median"],
        "letterbox_o6_over_stored_o1": lb["stored_o6"]["median"] / lb["stored_o1"]["median"],
        "letterbox_o6_over_upright_o1": lb["stored_o6"]["median"] / lb["upright_o1"]["median"],
        "e2e_nv12_o6_over_upright_o1": e2e["nv12_stored_o6"]["median"] / e2e["nv12_upright_o1"]["median"],
        "e2e_bgr_o6_over_upright_o1": e2e["bgr_stored_o6"]["median"] / e2e["bgr_upright_o1"]["median"],
        "e2e_bgr_o6_over_status_quo": e2e["bgr_stored_o6"]["median"] / e2e["bgr_status_quo_cv2_rotate"]["median"],
        "standard_o6_over_upright_o1": std["stored_o6"]["median"] / std["upright_o1"]["median"],
    }
    result = {"workload": "short-range BlazeFace 128x128, fast mode, synthetic 1280x720 frames (64 unique, tiled) stored sideways as "
                          "720x1280 (orientation 6); device: %d frames, chunks of 1024; end to end: %d pinned host frames; "
                          "standard: C4-shaped, 1024 frames, <= 4 faces, chunks of 512; %d faces per device pass, %d in standard"
                          % (B, E, dev_faces, std_faces),
              "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": rounds,
              "summary": {"device_img_s": dv, "letterbox_ms_per_1024": lb, "e2e_img_s": e2e,
                          "h2d_bytes_per_frame": rounds[-1]["h2d_bytes_per_frame"], "standard_img_s": std, "ratios": ratios},
              "host_threads": os.cpu_count(),
              "how": "device: fdt_detect_batch_oriented on device frames (fast-mode results copied to the host), fdt_timer_begin/end; "
                     "letterbox: fdt_set_stage_timing stage 0, median of 5 calls, scaled to 1024 frames; end to end: pinned host "
                     "frames, max(library timer, wall clock); status quo: cv2.rotate of every stored frame on a thread pool of "
                     "host_threads threads into pinned memory, then fdt_detect_batch; variants alternate within each round"}
    print(json.dumps(result), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")
    pool.shutdown()
    for p in pins:
        lib.fdt_free_pinned(p)
    det.dispose()
    det4.dispose()


if __name__ == "__main__":
    main()
