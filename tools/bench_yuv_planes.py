"""Separate-plane YUV 4:2:0 frames (fdt_detect_yuv_planes) against the caller's alternatives, one process, one GPU.

Workloads (synthetic 1920x1080 face frames, 64 unique, tiled; short-range detector):
  * device, NVDEC-shaped: --batch pitched NV12 surfaces (pitch 2048, chroma at 2048 * 1088, each its own pointer), fast mode,
    chunks of --chunk, library timer (fdt_timer_begin / end).  Variants, alternating within each of --rounds rounds:
      planes          fdt_detect_yuv_planes on the surfaces (U, V one stride and 1 byte apart: the FrameD route);
      repack_batch    the caller's route today: a torch copy of every surface into one contiguous [N, 1620, 1920] NV12 tensor
                      inside the timed window (torch.cuda.synchronize() before the library call), then fdt_detect_batch;
      frames_ceiling  fdt_detect_frames on already contiguous NV12 copies (the same kernels without the pitch).
    Letterbox stage ms per 1024 frames (fdt_set_stage_timing, stage 0) for planes on the surfaces (k_letterbox_multi), and on
    the same samples with U and V in two allocations of their own (the plane-table variant, k_letterbox_multi<., ., true>).
  * host, FFmpeg-shaped: --host-batch I420 frames with padded linesizes 1984 / 1024 / 1056 in pinned memory, fast mode:
      planes          fdt_detect_yuv_planes (each plane's sampled columns uploaded, 2-D copies);
      repack_batch    a numpy repack into one contiguous pinned I420 buffer inside the timed window, then fdt_detect_batch
                      (whose fast-mode upload is sparse: the tap rows only).
    max(library timer, wall clock).
  * standard mode, C4-shaped (1280x720, at most 4 faces, 1024 device frames, chunks of 512): planes on pitched NV12 surfaces
    against fdt_detect_batch on contiguous NV12.
Also the host-side argument checks of one 4096-frame device call, for both calls (a call whose last frame points at host memory
runs every check and launches nothing).  Every variant's face records are checked bitwise against the contiguous NV12 / I420 call
first.

    python tools/bench_yuv_planes.py [--rounds 3] [--out profiles/r07a_bench_yuv_planes.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_yuv import card  # noqa: E402

NV12, I420 = 0x1000, 0x1002


def i420(bgr):
    import cv2
    return np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in bgr])       # [P][3H/2][W]


def nv12(yuv, w, h):
    out = yuv.copy()
    u = yuv[:, h:].reshape(len(yuv), -1)[:, : w * h // 4]
    v = yuv[:, h:].reshape(len(yuv), -1)[:, w * h // 4:]
    out[:, h:] = np.stack([u, v], -1).reshape(len(yuv), h // 2, w)
    return out


def summary(rounds, key):
    ks = rounds[0][key].keys()
    return {k: {"median": statistics.median(x[key][k] for x in rounds),
                "range": [min(x[key][k] for x in rounds), max(x[key][k] for x in rounds)]} for k in ks}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--chunk", type=int, default=1024)
    ap.add_argument("--host-batch", type=int, default=2048)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import torch
    import bench
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi, build, synth

    build.build()
    lib = _ffi.load()
    W, H, P, B, E = 1920, 1080, bench.PERIOD, args.batch, args.host_batch
    PITCH, SH = 2048, 1088
    base = np.concatenate([synth.face_frames(P - 8, W, H), synth.noise_frames(8, W, H)])
    yuv = i420(base)                                                              # [P][1620][1920]
    nv = nv12(yuv, W, H)
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=args.chunk)
    h, mf = det._h, det._max_faces
    ms = C.c_float()

    def check(rc, hh=h):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(hh).decode())

    faces = (_ffi.FdtFace * (B * mf))()
    counts = np.zeros(B, np.int32)
    cp = counts.ctypes.data_as(_ffi.i32p)

    # ---- device, NVDEC-shaped surfaces: [B][SH * 3 / 2][PITCH], each surface its own pointer
    idx = torch.arange(B, device="cuda") % P
    nv_dev = torch.from_numpy(nv).cuda()
    surf = torch.randint(0, 256, (P, SH * 3 // 2, PITCH), dtype=torch.uint8, device="cuda")
    surf[:, :H, :W] = nv_dev[:, :H]
    surf[:, SH:SH + H // 2, :W] = nv_dev[:, H:]
    surf = surf[idx].contiguous()
    contig = nv_dev[idx].contiguous()                                             # [B][1620][1920]
    del nv_dev
    torch.cuda.synchronize()
    sb, cb = SH * 3 // 2 * PITCH, H * 3 // 2 * W

    def planes_arr(ptrs):
        arr = (_ffi.FdtYuvPlanes * len(ptrs))()
        for i, (y, u, v, sy, su, sv, ps) in enumerate(ptrs):
            arr[i].plane = (C.c_void_p * 3)(y, u, v)
            arr[i].row_stride = (C.c_int32 * 3)(sy, su, sv)
            arr[i].width, arr[i].height, arr[i].pixel_stride = W, H, ps
        return arr

    s0 = surf.data_ptr()
    surf_desc = planes_arr([(s0 + i * sb, s0 + i * sb + SH * PITCH, s0 + i * sb + SH * PITCH + 1, PITCH, PITCH, PITCH, 2)
                            for i in range(B)])
    c0 = contig.data_ptr()
    frames_desc = (_ffi.FdtFrame * B)(*[_ffi.FdtFrame(c0 + i * cb, W, H, W, NV12) for i in range(B)])
    repacked = torch.empty_like(contig)

    def run(k):
        if k == "planes":
            check(lib.fdt_detect_yuv_planes(h, surf_desc, None, B, 0, 1, faces, cp, None, None))
        elif k == "frames_ceiling":
            check(lib.fdt_detect_frames(h, frames_desc, B, 0, 1, faces, cp, None, None))
        elif k == "repack_batch":
            repacked[:, :H] = surf[:, :H, :W]
            repacked[:, H:] = surf[:, SH:SH + H // 2, :W]
            torch.cuda.synchronize()
            check(lib.fdt_detect_batch(h, repacked.data_ptr(), B, W, H, W, NV12, 0, 1, faces, cp, None, None))

    def rate(k):
        for _ in range(args.warmup):
            run(k)
        torch.cuda.synchronize()
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            run(k)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        return B * args.steps / (max(float(ms.value), wall) / 1e3)

    run("frames_ceiling")
    ref = (bytes(faces), counts.copy())
    for k in ("planes", "repack_batch"):
        run(k)
        assert bytes(faces) == ref[0] and np.array_equal(counts, ref[1]), k
    dev_faces = int(ref[1].sum())

    # the plane-table route: the same samples with U and V in allocations of their own (V's rows 64 bytes longer)
    NT = args.chunk
    y_t = contig[:NT, :H].contiguous()
    u_t = torch.from_numpy(np.ascontiguousarray(yuv[:, H:].reshape(P, -1)[:, : W * H // 4].reshape(P, H // 2, W // 2))).cuda()
    v_t = torch.zeros((P, H // 2, W // 2 + 64), dtype=torch.uint8, device="cuda")
    v_t[:, :, : W // 2] = torch.from_numpy(np.ascontiguousarray(yuv[:, H:].reshape(P, -1)[:, W * H // 4:].reshape(P, H // 2, W // 2))).cuda()
    u_t, v_t = u_t[idx[:NT]].contiguous(), v_t[idx[:NT]].contiguous()
    torch.cuda.synchronize()
    yb, ub, vb = H * W, H // 2 * W // 2, H // 2 * (W // 2 + 64)
    table_desc = planes_arr([(y_t.data_ptr() + i * yb, u_t.data_ptr() + i * ub, v_t.data_ptr() + i * vb, W, W // 2, W // 2 + 64, 1)
                             for i in range(NT)])
    check(lib.fdt_detect_yuv_planes(h, table_desc, None, NT, 0, 1, faces, cp, None, None))
    assert bytes(faces)[: NT * mf * C.sizeof(_ffi.FdtFace)] == ref[0][: NT * mf * C.sizeof(_ffi.FdtFace)], "plane table"

    def letterbox_ms(desc, n, reps=10):
        check(lib.fdt_detect_yuv_planes(h, desc, None, n, 0, 1, faces, cp, None, None))
        lib.fdt_set_stage_timing(h, 1)
        tot = 0.0
        for _ in range(reps):
            check(lib.fdt_detect_yuv_planes(h, desc, None, n, 0, 1, faces, cp, None, None))
            lb = C.c_float()
            lib.fdt_get_stage_ms(h, 0, C.byref(lb), None)
            tot += lb.value
        lib.fdt_set_stage_timing(h, 0)
        return tot / reps * 1024 / n

    # host-side argument checks of one device call (the descriptors, and cudaPointerGetAttributes on every frame pointer: three per
    # separate-plane frame, one per fdt_frame): a call whose last frame points at host memory runs them all and launches nothing
    hostbuf = np.zeros(16, np.uint8)

    def check_ms(k, reps=5):
        if k == "planes":
            last = surf_desc[B - 1]
            keep = last.plane[2]
            surf_desc[B - 1].plane[2] = hostbuf.ctypes.data
            call = lambda: lib.fdt_detect_yuv_planes(h, surf_desc, None, B, 0, 1, faces, cp, None, None)
        else:
            keep = frames_desc[B - 1].data
            frames_desc[B - 1].data = hostbuf.ctypes.data
            call = lambda: lib.fdt_detect_frames(h, frames_desc, B, 0, 1, faces, cp, None, None)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            rc = call()
            ts.append((time.perf_counter() - t0) * 1e3)
            assert rc == _ffi.FDT_ERR_BAD_ARG and b"frame %d" % (B - 1) in lib.fdt_last_error(h), k
        if k == "planes":
            surf_desc[B - 1].plane[2] = keep
        else:
            frames_desc[B - 1].data = keep
        return statistics.median(ts)

    # ---- host, FFmpeg-shaped I420 in pinned memory: linesizes 1984 / 1024 / 1056
    LY, LU, LV = 1984, 1024, 1056
    fb = H * LY + H // 2 * (LU + LV)
    pin = C.c_void_p()
    check(lib.fdt_alloc_pinned(E * fb + E * cb, C.byref(pin)))
    pbuf = np.ctypeslib.as_array((C.c_uint8 * (E * fb + E * cb)).from_address(pin.value))
    hf = pbuf[: E * fb].reshape(E, fb)
    hrep = pbuf[E * fb:].reshape(E, cb)
    rng = np.random.default_rng(0)
    for i in range(E):
        f, src = hf[i], yuv[i % P]
        f[:] = rng.integers(0, 256, fb, dtype=np.uint8) if i < P else hf[i % P]
        if i < P:
            f[: H * LY].reshape(H, LY)[:, :W] = src[:H]
            f[H * LY: H * LY + H // 2 * LU].reshape(H // 2, LU)[:, : W // 2] = src[H:].reshape(-1)[: W * H // 4].reshape(H // 2, W // 2)
            f[H * LY + H // 2 * LU:].reshape(H // 2, LV)[:, : W // 2] = src[H:].reshape(-1)[W * H // 4:].reshape(H // 2, W // 2)
    hp = hf.ctypes.data
    host_desc = planes_arr([(hp + i * fb, hp + i * fb + H * LY, hp + i * fb + H * LY + H // 2 * LU, LY, LU, LV, 1) for i in range(E)])
    hfaces = (_ffi.FdtFace * (E * mf))()
    hcounts = np.zeros(E, np.int32)
    hcp = hcounts.ctypes.data_as(_ffi.i32p)

    def host_run(k):
        if k == "planes":
            check(lib.fdt_detect_yuv_planes(h, host_desc, None, E, 0, 0, hfaces, hcp, None, None))
        else:
            y = hf[:, : H * LY].reshape(E, H, LY)[:, :, :W]
            u = hf[:, H * LY: H * LY + H // 2 * LU].reshape(E, H // 2, LU)[:, :, : W // 2]
            v = hf[:, H * LY + H // 2 * LU:].reshape(E, H // 2, LV)[:, :, : W // 2]
            hrep[:, : H * W].reshape(E, H, W)[:] = y
            hrep[:, H * W: H * W + W * H // 4].reshape(E, H // 2, W // 2)[:] = u
            hrep[:, H * W + W * H // 4:].reshape(E, H // 2, W // 2)[:] = v
            check(lib.fdt_detect_batch(h, hrep.ctypes.data, E, W, H, W, I420, 0, 0, hfaces, hcp, None, None))

    def host_rate(k):
        host_run(k)
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        n = max(2, args.steps // 2)
        for _ in range(n):
            host_run(k)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        return E * n / (max(float(ms.value), wall) / 1e3), int(lib.fdt_last_h2d_bytes(h)) / E

    host_run("repack_batch")
    href = (bytes(hfaces), hcounts.copy())
    host_run("planes")
    assert bytes(hfaces) == href[0] and np.array_equal(hcounts, href[1]), "host planes"
    assert int(lib.fdt_last_h2d_bytes(h)) == E * (W * H + 2 * (H // 2) * (W // 2)), "host upload bytes"

    # ---- standard mode, C4-shaped
    det4 = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withIris=False, maxBatch=512, maxFaces=4)
    h4 = det4._h
    W4, H4, B4, P4 = 1280, 720, 1024, 768
    nv4 = torch.from_numpy(nv12(i420(bench.synth_base("c4")), W4, H4)).cuda()
    i4 = torch.arange(B4, device="cuda") % P
    c4 = nv4[i4].contiguous()
    s4 = torch.zeros((B4, P4 * 3 // 2, 1280 + 256), dtype=torch.uint8, device="cuda")
    s4[:, :H4, :W4] = c4[:, :H4]
    s4[:, P4:P4 + H4 // 2, :W4] = c4[:, H4:]
    torch.cuda.synchronize()
    sb4 = s4[0].numel()
    d4 = (_ffi.FdtYuvPlanes * B4)()
    for i in range(B4):
        p0 = s4.data_ptr() + i * sb4
        d4[i].plane = (C.c_void_p * 3)(p0, p0 + P4 * 1536, p0 + P4 * 1536 + 1)
        d4[i].row_stride = (C.c_int32 * 3)(1536, 1536, 1536)
        d4[i].width, d4[i].height, d4[i].pixel_stride = W4, H4, 2
    f4 = (_ffi.FdtFace * (B4 * 4))()
    n4 = np.zeros(B4, np.int32)
    m4 = np.zeros((B4, 4, 468, 3), np.float32)

    def std_run(k):
        if k == "planes":
            check(lib.fdt_detect_yuv_planes(h4, d4, None, B4, 1, 1, f4, n4.ctypes.data_as(_ffi.i32p), m4.ctypes.data_as(_ffi.f32p), None), h4)
        else:
            check(lib.fdt_detect_batch(h4, c4.data_ptr(), B4, W4, H4, W4, NV12, 1, 1, f4, n4.ctypes.data_as(_ffi.i32p),
                                       m4.ctypes.data_as(_ffi.f32p), None), h4)

    def std_rate(k):
        std_run(k)
        n = max(2, args.steps // 2)
        lib.fdt_timer_begin(h4)
        t0 = time.perf_counter()
        for _ in range(n):
            std_run(k)
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h4, C.byref(ms))
        return B4 * n / (max(float(ms.value), wall) / 1e3)

    std_run("nv12_batch")
    sref = (bytes(f4), n4.copy(), m4.copy())
    std_run("planes")
    assert bytes(f4) == sref[0] and np.array_equal(n4, sref[1]) and np.array_equal(m4, sref[2]), "standard planes"
    std_faces = int(sref[1].sum())

    rounds = []
    for r in range(args.rounds):
        row = {"round": r, "device_img_s": {}, "letterbox_ms_per_1024": {}, "host_img_s": {}, "host_h2d_bytes_per_frame": {},
               "standard_img_s": {}}
        for k in ("planes", "repack_batch", "frames_ceiling"):
            row["device_img_s"][k] = rate(k)
        row["host_check_ms_per_call"] = {k: check_ms(k) for k in ("planes", "frames_ceiling")}
        row["letterbox_ms_per_1024"]["framed_route"] = letterbox_ms(surf_desc, NT)
        row["letterbox_ms_per_1024"]["plane_table_route"] = letterbox_ms(table_desc, NT)
        for k in ("planes", "repack_batch"):
            row["host_img_s"][k], row["host_h2d_bytes_per_frame"][k] = host_rate(k)
        for k in ("planes", "nv12_batch"):
            row["standard_img_s"][k] = std_rate(k)
        rounds.append(row)
        print(json.dumps(row), flush=True)

    dv, lb, hs, st, hc = (summary(rounds, k) for k in ("device_img_s", "letterbox_ms_per_1024", "host_img_s", "standard_img_s",
                                                        "host_check_ms_per_call"))
    ratios = {
        "device_planes_over_frames_ceiling": dv["planes"]["median"] / dv["frames_ceiling"]["median"],
        "device_planes_over_repack_batch": dv["planes"]["median"] / dv["repack_batch"]["median"],
        "letterbox_plane_table_over_framed": lb["plane_table_route"]["median"] / lb["framed_route"]["median"],
        "host_planes_over_repack_batch": hs["planes"]["median"] / hs["repack_batch"]["median"],
        "standard_planes_over_nv12_batch": st["planes"]["median"] / st["nv12_batch"]["median"],
    }
    result = {"workload": "short-range BlazeFace 128x128; device: %d NVDEC-shaped 1920x1080 NV12 surfaces (pitch 2048, chroma at "
                          "row 1088), fast mode, chunks of %d, %d faces per pass; host: %d FFmpeg-shaped I420 frames (linesizes "
                          "1984 / 1024 / 1056) in pinned memory, fast mode; standard: C4-shaped, 1024 1280x720 frames, <= 4 faces, "
                          "chunks of 512, %d faces" % (B, args.chunk, dev_faces, E, std_faces),
              "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": rounds,
              "summary": {"device_img_s": dv, "host_check_ms_per_call": hc, "letterbox_ms_per_1024": lb, "host_img_s": hs,
                          "host_h2d_bytes_per_frame": rounds[-1]["host_h2d_bytes_per_frame"], "standard_img_s": st, "ratios": ratios},
              "how": "device and standard: library timer fdt_timer_begin/end (repack_batch: the torch copy of every step inside that "
                     "window, torch.cuda.synchronize() before each library call), max with the wall clock; letterbox: "
                     "fdt_set_stage_timing stage 0 over %d frames, mean of 10 calls, scaled to 1024; host: max(library timer, wall "
                     "clock), the numpy repack inside the window; host_check: wall clock of one device call of %d frames whose last frame points at host "
                     "memory (every argument and pointer check, no launch), median of 5; variants alternate within each round; every variant's records "
                     "checked bitwise against the contiguous call first" % (NT, B)}
    print(json.dumps(result), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")
    lib.fdt_free_pinned(pin)
    det.dispose()
    det4.dispose()


if __name__ == "__main__":
    main()
