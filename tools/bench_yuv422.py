"""BGR against packed YUV 4:2:2 input (YUYV, UYVY) on the C2 workload, one process, one GPU.

The 64 unique frames of bench.synth_base("c2") (1280x720) are converted once, before any timing, to YUYV with
cv2.cvtColor(COLOR_BGR2YUV_YUYV); the UYVY frames are the same samples in UYVY byte order, and the BGR frames are
cv2.cvtColor(yuyv, COLOR_YUV2BGR_YUYV), so every variant detects the same image.  Frames are tiled to --batch and detected by the
short-range detector in fast mode, chunks of --chunk.  Variants alternate within each of --rounds rounds:
  * device-resident images/s (fdt_detect_batch_device, library timer fdt_timer_begin / end) for bgr, yuyv, uyvy, and
    caller_route_device: the YUYV frames converted by the caller with the same BT.601 fixed-point arithmetic written in torch,
    one chunk at a time inside the timed window (on torch's stream, synchronised before each call), then detected as BGR;
  * end to end from pinned host memory (--e2e-batch frames, fdt_detect_batch, max(library timer, wall clock)) for bgr and yuyv,
    with fdt_last_h2d_bytes per frame and the same round's plain pinned cudaMemcpyAsync rate, and caller_route_host:
    cv2.cvtColor(COLOR_YUV2BGR_YUYV) of every frame on a host thread pool into a pinned BGR buffer, then fdt_detect_batch;
  * standard mode, C4-shaped (1024 frames, at most 4 faces, chunks of 512): bgr against yuyv.
Once per format: the letterbox kernel time of one chunk (fdt_profile_chunk launch 0, mean of 20 passes).  Before timing, every
variant's face records are checked bitwise against BGR's.

    python tools/bench_yuv422.py [--rounds 3] [--out profiles/r09a_bench_yuv422.json]
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

from bench_yuv import card  # noqa: E402

BGR, YUYV, UYVY = 16, 0x1020, 0x1021


def to_uyvy(yuyv: np.ndarray) -> np.ndarray:
    """The same samples in UYVY byte order (Y0 U Y1 V -> U Y0 V Y1)."""
    q = yuyv.reshape(yuyv.shape[:-2] + (-1, 4))
    return np.ascontiguousarray(q[..., [1, 0, 3, 2]]).reshape(yuyv.shape)


def torch_yuyv_to_bgr(t):
    """cv2.cvtColor(COLOR_YUV2BGR_YUYV) in torch: [N, H, W, 2] uint8 -> [N, H, W, 3] uint8 (BT.601, 20-bit fixed point)."""
    import torch
    x = t.to(torch.int32)
    y = x[..., 0]
    m = x.reshape(x.shape[0], x.shape[1], -1, 4)                      # macropixels Y0 U Y1 V
    u = m[..., 1].repeat_interleave(2, dim=-1) - 128
    v = m[..., 3].repeat_interleave(2, dim=-1) - 128
    yy = (y - 16).clamp_(min=0) * 1220542 + (1 << 19)
    b = (yy + 2116026 * u) >> 20
    g = (yy - 852492 * v - 409993 * u) >> 20
    r = (yy + 1673527 * v) >> 20
    return torch.stack([b, g, r], -1).clamp_(0, 255).to(torch.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--chunk", type=int, default=1024)
    ap.add_argument("--e2e-batch", type=int, default=2048)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import cv2
    import torch
    import bench
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi, build

    build.build()
    lib = _ffi.load()
    W, H, B, P, E = 1280, 720, args.batch, bench.PERIOD, args.e2e_batch
    src = bench.synth_base("c2")                                           # [P][720][1280][3] BGR
    yuyv = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_YUYV) for f in src])   # [P][720][1280][2]
    uyvy = to_uyvy(yuyv)
    base = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_YUYV) for f in yuyv])
    assert np.array_equal(cv2.cvtColor(uyvy[3], cv2.COLOR_YUV2BGR_UYVY), base[3])
    fmts = {"bgr": (BGR, W * 3, base), "yuyv": (YUYV, W * 2, yuyv), "uyvy": (UYVY, W * 2, uyvy)}
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=args.chunk)
    h, mf = det._h, det._max_faces

    def check(rc, hh=h):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(hh).decode())

    idx = torch.arange(B, device="cuda") % P
    dev = {k: torch.from_numpy(f).cuda()[idx].contiguous() for k, (_, _, f) in fmts.items()}
    torch.cuda.synchronize()
    assert torch.equal(torch_yuyv_to_bgr(dev["yuyv"][:8]), dev["bgr"][:8])
    pf, pc = C.c_void_p(), C.c_void_p()
    ms = C.c_float()

    def dev_call(mt, stride, ptr, n=B):
        check(lib.fdt_detect_batch_device(h, ptr, n, W, H, stride, mt, 0, C.byref(pf), C.byref(pc)))

    def dev_records():
        counts = np.empty(B, np.int32)
        faces = np.empty(B * mf * C.sizeof(_ffi.FdtFace), np.uint8)
        check(lib.fdt_copy_to_host(h, counts.ctypes.data, pc.value, counts.nbytes))
        check(lib.fdt_copy_to_host(h, faces.ctypes.data, pf.value, faces.nbytes))
        rec = faces.reshape(B, mf, -1)
        return counts, [rec[b, :counts[b]].tobytes() for b in range(B)]

    conv = torch.empty((B, H, W, 3), dtype=torch.uint8, device="cuda")

    def caller_steps(n):
        for _ in range(n):
            lib.fdt_synchronize(h)                               # the previous call may still read conv
            for c0 in range(0, B, args.chunk):
                conv[c0:c0 + args.chunk] = torch_yuyv_to_bgr(dev["yuyv"][c0:c0 + args.chunk])
            torch.cuda.synchronize()
            dev_call(BGR, W * 3, conv.data_ptr())
        lib.fdt_synchronize(h)

    def device_rate(k):
        def steps(n):
            if k == "caller_route_device":
                caller_steps(n)
            else:
                mt, stride, _ = fmts[k]
                for _ in range(n):
                    dev_call(mt, stride, dev[k].data_ptr())
        steps(args.warmup)
        lib.fdt_synchronize(h)
        torch.cuda.synchronize()
        lib.fdt_timer_begin(h)
        steps(args.steps)
        lib.fdt_timer_end(h, C.byref(ms))
        return B * args.steps / (ms.value / 1e3)

    # bitwise agreement of every variant's face records with BGR's
    dev_call(BGR, W * 3, dev["bgr"].data_ptr())
    ref_counts, ref = dev_records()
    for k in ("yuyv", "uyvy"):
        mt, stride, _ = fmts[k]
        dev_call(mt, stride, dev[k].data_ptr())
        assert dev_records()[1] == ref, k
    caller_steps(1)
    assert dev_records()[1] == ref, "caller_route_device"
    dev_faces = int(ref_counts.sum())

    # ---- end to end from pinned host memory
    pins, hosts = [], {}

    def pinned(shape):
        nb = int(np.prod(shape))
        p = C.c_void_p()
        if lib.fdt_alloc_pinned(nb, C.byref(p)) != 0:
            raise RuntimeError("pinned allocation of %d bytes failed" % nb)
        pins.append(p)
        return np.ctypeslib.as_array((C.c_uint8 * nb).from_address(p.value)).reshape(shape)

    for k in ("bgr", "yuyv"):
        frames = fmts[k][2]
        arr = pinned((E,) + frames.shape[1:])
        for r0 in range(0, E, P):
            arr[r0:r0 + P] = frames[:min(P, E - r0)]
        hosts[k] = arr
    conv_host = pinned((E, H, W, 3))
    pool = ThreadPoolExecutor(max_workers=os.cpu_count() or 8)
    ef = (_ffi.FdtFace * (E * mf))()
    ec = np.zeros(E, np.int32)
    ecp = ec.ctypes.data_as(_ffi.i32p)

    def host_convert(i):
        cv2.cvtColor(hosts["yuyv"][i], cv2.COLOR_YUV2BGR_YUYV, dst=conv_host[i])

    def e2e_call(k):
        if k == "caller_route_host":
            list(pool.map(host_convert, range(E)))
            check(lib.fdt_detect_batch(h, conv_host.ctypes.data, E, W, H, W * 3, BGR, 0, 0, ef, ecp, None, None))
            return
        mt, stride, _ = fmts[k]
        check(lib.fdt_detect_batch(h, hosts[k].ctypes.data, E, W, H, stride, mt, 0, 0, ef, ecp, None, None))

    def e2e_rate(k):
        for _ in range(max(1, args.warmup // 2)):
            e2e_call(k)
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_call(k)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        return E * args.steps / (max(float(ms.value), wall) / 1e3), int(lib.fdt_last_h2d_bytes(h)) / E

    e2e_call("bgr")
    e2e_ref = bytes(ef)
    for k in ("yuyv", "caller_route_host"):
        e2e_call(k)
        assert bytes(ef) == e2e_ref, "end to end: %s disagrees with bgr" % k

    def memcpy_ceiling():
        nb = 512 << 20
        hp = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        dp = torch.empty(nb, dtype=torch.uint8, device="cuda")
        dp.copy_(hp, non_blocking=True)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(4):
            dp.copy_(hp, non_blocking=True)
        ev1.record()
        torch.cuda.synchronize()
        return 4 * nb / (ev0.elapsed_time(ev1) * 1e-3) / 1e9

    # ---- standard mode, C4-shaped
    det4 = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withIris=False, maxBatch=512, maxFaces=4)
    h4 = det4._h
    y4 = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_YUYV) for f in bench.synth_base("c4")])
    b4 = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_YUYV) for f in y4])
    B4 = 1024
    i4 = torch.arange(B4, device="cuda") % P
    dev4 = {"bgr": torch.from_numpy(b4).cuda()[i4].contiguous(), "yuyv": torch.from_numpy(y4).cuda()[i4].contiguous()}
    torch.cuda.synchronize()
    f4 = (_ffi.FdtFace * (B4 * 4))()
    c4 = np.zeros(B4, np.int32)
    m4 = np.zeros((B4, 4, 468, 3), np.float32)

    def std_call(k):
        mt, stride = (BGR, W * 3) if k == "bgr" else (YUYV, W * 2)
        check(lib.fdt_detect_batch(h4, dev4[k].data_ptr(), B4, W, H, stride, mt, 1, 1, f4, c4.ctypes.data_as(_ffi.i32p),
                                   m4.ctypes.data_as(_ffi.f32p), None), h4)

    def std_rate(k):
        std_call(k)
        n = max(2, args.steps // 2)
        lib.fdt_timer_begin(h4)
        t0 = time.perf_counter()
        for _ in range(n):
            std_call(k)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h4, C.byref(ms))
        return B4 * n / (max(float(ms.value), wall) / 1e3)

    std_call("bgr")
    std_ref = (bytes(f4), c4.copy(), m4.copy())
    std_call("yuyv")
    assert bytes(f4) == std_ref[0] and np.array_equal(c4, std_ref[1]) and np.array_equal(m4, std_ref[2]), "standard: yuyv != bgr"
    std_faces = int(std_ref[1].sum())

    rounds = []
    for r in range(args.rounds):
        row = {"round": r, "device_img_s": {}, "e2e_img_s": {}, "h2d_bytes_per_frame": {}, "standard_img_s": {},
               "h2d_ceiling_gbs": memcpy_ceiling()}
        for k in ("bgr", "yuyv", "uyvy", "caller_route_device"):
            row["device_img_s"][k] = device_rate(k)
        for k in ("bgr", "yuyv", "caller_route_host"):
            row["e2e_img_s"][k], row["h2d_bytes_per_frame"][k] = e2e_rate(k)
        for k in ("bgr", "yuyv"):
            row["standard_img_s"][k] = std_rate(k)
        rounds.append(row)
        print(json.dumps(row), flush=True)

    letterbox = {}
    for k, (mt, stride, _) in fmts.items():
        arr = (C.c_float * 512)()
        nl = C.c_int32()
        check(lib.fdt_profile_chunk(h, dev[k].data_ptr(), args.chunk, W, H, stride, mt, 20, arr, 512, C.byref(nl)))
        letterbox[k] = {"kernel": "k_letterbox" if k == "bgr" else "k_letterbox_rgb<false, true>", "ms_per_chunk": float(arr[0]),
                        "chunk": args.chunk}

    def summary(key):
        ks = rounds[0][key].keys()
        return {k: {"median": statistics.median(x[key][k] for x in rounds),
                    "range": [min(x[key][k] for x in rounds), max(x[key][k] for x in rounds)]} for k in ks}

    dv, e2e, std = summary("device_img_s"), summary("e2e_img_s"), summary("standard_img_s")
    ratios = {
        "device_yuyv_over_bgr": dv["yuyv"]["median"] / dv["bgr"]["median"],
        "device_uyvy_over_bgr": dv["uyvy"]["median"] / dv["bgr"]["median"],
        "device_yuyv_over_caller_route": dv["yuyv"]["median"] / dv["caller_route_device"]["median"],
        "letterbox_yuyv_over_bgr": letterbox["yuyv"]["ms_per_chunk"] / letterbox["bgr"]["ms_per_chunk"],
        "letterbox_uyvy_over_bgr": letterbox["uyvy"]["ms_per_chunk"] / letterbox["bgr"]["ms_per_chunk"],
        "e2e_yuyv_over_bgr": e2e["yuyv"]["median"] / e2e["bgr"]["median"],
        "e2e_yuyv_over_caller_route": e2e["yuyv"]["median"] / e2e["caller_route_host"]["median"],
        "standard_yuyv_over_bgr": std["yuyv"]["median"] / std["bgr"]["median"],
    }
    result = {"workload": "C2: short-range BlazeFace 128x128, fast mode, synthetic 1280x720 frames (64 unique, tiled); device: %d "
                          "frames, chunks of %d; end to end: %d pinned host frames; standard: C4-shaped, 1024 frames, <= 4 faces, "
                          "chunks of 512; %d faces per device pass, %d in standard" % (B, args.chunk, E, dev_faces, std_faces),
              "card": card(), "steps": args.steps, "warmup": args.warmup, "host_threads": os.cpu_count(), "rounds": rounds,
              "letterbox": letterbox,
              "summary": {"device_img_s": dv, "e2e_img_s": e2e, "h2d_bytes_per_frame": rounds[-1]["h2d_bytes_per_frame"],
                          "h2d_ceiling_gbs_median": statistics.median(x["h2d_ceiling_gbs"] for x in rounds),
                          "standard_img_s": std, "ratios": ratios},
              "how": "device: fdt_detect_batch_device on device-resident frames, fdt_timer_begin/end (caller_route_device: the "
                     "torch conversion of every step inside that window, torch.cuda.synchronize() before each library call); "
                     "letterbox: fdt_profile_chunk launch 0, mean of 20 passes over one chunk; end to end: fdt_detect_batch on "
                     "pinned host frames, max(library timer, wall clock) (caller_route_host: cv2.cvtColor per frame on a thread pool "
                     "of host_threads workers inside the window); ceiling: cudaMemcpyAsync of a 512 MiB pinned buffer x 4, CUDA "
                     "events, same round; standard: fdt_detect_batch mode 1 on device frames, results to the host; variants "
                     "alternate within each round; every variant's records checked bitwise against bgr first"}
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
