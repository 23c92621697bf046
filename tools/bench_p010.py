"""16-bit YUV 4:2:0 frames (FDT_FMT_P010, fdt_detect_yuv_planes16) against the 8-bit calls and the caller's route, one process,
one GPU.  Variants alternate within each of --rounds rounds; every variant's face records are checked bitwise against its 8-bit
counterpart first.

Workloads (synthetic face frames, 64 unique, tiled; short-range detector; 16-bit words = 8-bit sample << 8 | noise):
  * device, NVDEC-shaped: --batch pitched 1920x1080 surfaces (pitch 2048 samples, chroma at pitch * 1088), fast mode, chunks
    of --chunk, library timer (fdt_timer_begin / end):
      planes16        fdt_detect_yuv_planes16 (sample_bits 16) on P016 surfaces;
      planes8         fdt_detect_yuv_planes on the same frames as 8-bit NV12 surfaces;
      shift_batch     the caller's route today: a torch (surface >> 8).to(uint8) copy into one contiguous [N, 1620, 1920] NV12
                      tensor inside the timed window (torch.cuda.synchronize() before the library call), then fdt_detect_batch.
    Letterbox stage ms per 1024 frames (fdt_set_stage_timing, stage 0): planes16 on the P016 surfaces against the 8-bit
    plane-table letterbox (U and V in allocations of their own).
  * device, C2-shaped: fdt_detect_batch on 4096 contiguous 1280x720 P010 frames against NV12.
  * host, 2048 pinned frames, fast mode, max(library timer, wall clock): uniform 1280x720 P010 (sparse row upload) against NV12,
    and 1920x1080 yuv420p10le planes (FFmpeg linesizes 3968 / 1984 / 2048 bytes) through fdt_detect_yuv_planes16 against the
    8-bit planes through fdt_detect_yuv_planes.
  * standard mode, C4-shaped (1024 device 1280x720 frames, <= 4 faces, chunks of 512): P010 against NV12.

    python tools/bench_p010.py [--rounds 5] [--out profiles/r10a_bench_p010.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_yuv import card  # noqa: E402
from bench_yuv_planes import i420, nv12, summary  # noqa: E402

NV12, I420, P010 = 0x1000, 0x1002, 0x1003


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
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
    PITCH, SH = 2048, 1088                                                        # samples, rows
    ms = C.c_float()

    def check(rc, hh):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(hh).decode())

    def widen(t8):
        """16-bit words of 8-bit samples: t8 << 8 | noise (a torch uint8 tensor on the device -> int16 bits of uint16 words)."""
        noise = torch.randint(0, 256, t8.shape, dtype=torch.int32, device=t8.device)
        return ((t8.to(torch.int32) << 8) | noise).to(torch.int16)               # the bits of uint16 words

    def timed(run, n_frames, hh, steps):
        for _ in range(args.warmup):
            run()
        torch.cuda.synchronize()
        lib.fdt_timer_begin(hh)
        t0 = time.perf_counter()
        for _ in range(steps):
            run()
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(hh, C.byref(ms))
        return n_frames * steps / (max(float(ms.value), wall) / 1e3)

    def planes_arr(ptrs, w, h):
        arr = (_ffi.FdtYuvPlanes * len(ptrs))()
        for i, (y, u, v, sy, su, sv, ps) in enumerate(ptrs):
            arr[i].plane = (C.c_void_p * 3)(y, u, v)
            arr[i].row_stride = (C.c_int32 * 3)(sy, su, sv)
            arr[i].width, arr[i].height, arr[i].pixel_stride = w, h, ps
        return arr

    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=args.chunk)
    h, mf = det._h, det._max_faces
    faces = (_ffi.FdtFace * (B * mf))()
    counts = np.zeros(B, np.int32)
    cp = counts.ctypes.data_as(_ffi.i32p)

    # ---- device, NVDEC-shaped surfaces
    base = np.concatenate([synth.face_frames(P - 8, W, H), synth.noise_frames(8, W, H)])
    yuv = i420(base)
    nv = torch.from_numpy(nv12(yuv, W, H)).cuda()                                # [P][1620][1920]
    idx = torch.arange(B, device="cuda") % P
    s8 = torch.randint(0, 256, (P, SH * 3 // 2, PITCH), dtype=torch.uint8, device="cuda")
    s8[:, :H, :W] = nv[:, :H]
    s8[:, SH:SH + H // 2, :W] = nv[:, H:]
    s16 = widen(s8)
    s8, s16 = s8[idx].contiguous(), s16[idx].contiguous()
    torch.cuda.synchronize()
    sb8, sb16 = SH * 3 // 2 * PITCH, SH * 3 // 2 * PITCH * 2
    p8, p16 = s8.data_ptr(), s16.data_ptr()
    d8 = planes_arr([(p8 + i * sb8, p8 + i * sb8 + SH * PITCH, p8 + i * sb8 + SH * PITCH + 1, PITCH, PITCH, PITCH, 2)
                     for i in range(B)], W, H)
    d16 = planes_arr([(p16 + i * sb16, p16 + i * sb16 + SH * PITCH * 2, p16 + i * sb16 + SH * PITCH * 2 + 2, 2 * PITCH, 2 * PITCH,
                       2 * PITCH, 2) for i in range(B)], W, H)
    repacked = torch.empty((B, H * 3 // 2, W), dtype=torch.uint8, device="cuda")

    def dev_run(k):
        if k == "planes16":
            check(lib.fdt_detect_yuv_planes16(h, d16, None, B, 16, 0, 1, faces, cp, None, None), h)
        elif k == "planes8":
            check(lib.fdt_detect_yuv_planes(h, d8, None, B, 0, 1, faces, cp, None, None), h)
        elif k == "shift_batch":
            # (t >> 8).to(uint8) on the words' int16 bits: the arithmetic shift keeps the high byte's bits, the cast wraps
            repacked[:, :H] = (s16[:, :H, :W] >> 8).to(torch.uint8)
            repacked[:, H:] = (s16[:, SH:SH + H // 2, :W] >> 8).to(torch.uint8)
            torch.cuda.synchronize()
            check(lib.fdt_detect_batch(h, repacked.data_ptr(), B, W, H, W, NV12, 0, 1, faces, cp, None, None), h)

    dev_run("planes8")
    ref = (bytes(faces), counts.copy())
    for k in ("planes16", "shift_batch"):
        dev_run(k)
        assert bytes(faces) == ref[0] and np.array_equal(counts, ref[1]), k
    dev_faces = int(ref[1].sum())

    # the 8-bit plane-table letterbox: U and V in allocations of their own (V's rows 64 bytes longer)
    NT = args.chunk
    y_t = nv[idx[:NT], :H].contiguous()
    u_t = nv[idx[:NT], H:, 0::2].contiguous()
    v_t = torch.zeros((NT, H // 2, W // 2 + 64), dtype=torch.uint8, device="cuda")
    v_t[:, :, :W // 2] = nv[idx[:NT], H:, 1::2]
    torch.cuda.synchronize()
    yb, ub, vb = H * W, H // 2 * W // 2, H // 2 * (W // 2 + 64)
    table8 = planes_arr([(y_t.data_ptr() + i * yb, u_t.data_ptr() + i * ub, v_t.data_ptr() + i * vb, W, W // 2, W // 2 + 64, 1)
                         for i in range(NT)], W, H)
    sz = NT * mf * C.sizeof(_ffi.FdtFace)
    check(lib.fdt_detect_yuv_planes(h, table8, None, NT, 0, 1, faces, cp, None, None), h)
    assert bytes(faces)[:sz] == ref[0][:sz], "8-bit plane table"

    def letterbox_ms(call, reps=10):
        call()
        lib.fdt_set_stage_timing(h, 1)
        tot = 0.0
        for _ in range(reps):
            call()
            lb = C.c_float()
            lib.fdt_get_stage_ms(h, 0, C.byref(lb), None)
            tot += lb.value
        lib.fdt_set_stage_timing(h, 0)
        return tot / reps

    lb_calls = {"planes16": lambda: check(lib.fdt_detect_yuv_planes16(h, d16, None, NT, 16, 0, 1, faces, cp, None, None), h),
                "plane_table8": lambda: check(lib.fdt_detect_yuv_planes(h, table8, None, NT, 0, 1, faces, cp, None, None), h)}

    # ---- device, C2-shaped uniform batches
    W2, H2 = 1280, 720
    nv2 = torch.from_numpy(nv12(i420(bench.synth_base("c2")), W2, H2)).cuda()
    c2_8 = nv2[idx].contiguous()                                                  # [B][1080][1280]
    c2_16 = widen(c2_8)
    torch.cuda.synchronize()

    def c2_run(k):
        t, mt, stride = (c2_16, P010, 2 * W2) if k == "p010" else (c2_8, NV12, W2)
        check(lib.fdt_detect_batch(h, t.data_ptr(), B, W2, H2, stride, mt, 0, 1, faces, cp, None, None), h)

    c2_run("nv12")
    cref = (bytes(faces), counts.copy())
    c2_run("p010")
    assert bytes(faces) == cref[0] and np.array_equal(counts, cref[1]), "c2 p010"

    # ---- host, pinned: uniform 1280x720 P010 / NV12, and 1920x1080 yuv420p10le planes / their 8-bit planes
    fb16, fb8 = H2 * W2 * 3, H2 * W2 * 3 // 2
    LY, LU, LV = 3968, 1984, 2048                                                 # bytes, FFmpeg-style linesizes
    pf16 = H * LY + H // 2 * (LU + LV)
    pf8 = H * W + 2 * (H // 2) * (W // 2)
    total = E * (fb16 + fb8 + pf16 + pf8)
    pin = C.c_void_p()
    check(lib.fdt_alloc_pinned(total, C.byref(pin)), h)
    pbuf = np.ctypeslib.as_array((C.c_uint8 * total).from_address(pin.value))
    o = 0
    hp16 = pbuf[o:o + E * fb16]; o += E * fb16
    hp8 = pbuf[o:o + E * fb8]; o += E * fb8
    hq16 = pbuf[o:o + E * pf16].reshape(E, pf16); o += E * pf16
    hq8 = pbuf[o:o + E * pf8].reshape(E, pf8)
    hidx = np.arange(E) % P
    hp8.reshape(E, fb8)[:] = nv2.cpu().numpy().reshape(P, fb8)[hidx]
    hp16.view(np.int16).reshape(E, fb8)[:] = widen(torch.from_numpy(hp8.reshape(E, fb8)[:P].copy()).cuda()).cpu().numpy()[hidx]
    rng = np.random.default_rng(0)
    for i in range(P):
        src = yuv[i]
        f = hq16[i]
        f.view(np.uint16)[:] = rng.integers(0, 1 << 16, pf16 // 2, dtype=np.uint16)
        for plane, off, ls, rows, cols in ((src[:H], 0, LY, H, W),
                                           (src[H:].reshape(-1)[:W * H // 4].reshape(H // 2, W // 2), H * LY, LU, H // 2, W // 2),
                                           (src[H:].reshape(-1)[W * H // 4:].reshape(H // 2, W // 2), H * LY + H // 2 * LU, LV,
                                            H // 2, W // 2)):
            words = (plane.astype(np.uint16) << 2) | rng.integers(0, 4, plane.shape, dtype=np.uint16) \
                | (rng.integers(0, 64, plane.shape, dtype=np.uint16) << 10)
            f[off:off + rows * ls].view(np.uint16).reshape(rows, ls // 2)[:, :cols] = words
        g = hq8[i]
        g[:H * W] = src[:H].reshape(-1)
        g[H * W:] = src[H:].reshape(-1)
    hq16[P:] = hq16[hidx[P:]]
    hq8[P:] = hq8[hidx[P:]]
    q16 = hq16.ctypes.data
    q8 = hq8.ctypes.data
    hd16 = planes_arr([(q16 + i * pf16, q16 + i * pf16 + H * LY, q16 + i * pf16 + H * LY + H // 2 * LU, LY, LU, LV, 1)
                       for i in range(E)], W, H)
    hd8 = planes_arr([(q8 + i * pf8, q8 + i * pf8 + H * W, q8 + i * pf8 + H * W + H // 2 * W // 2, W, W // 2, W // 2, 1)
                      for i in range(E)], W, H)
    hfaces = (_ffi.FdtFace * (E * mf))()
    hcounts = np.zeros(E, np.int32)
    hcp = hcounts.ctypes.data_as(_ffi.i32p)

    def host_run(k):
        if k == "p010":
            check(lib.fdt_detect_batch(h, hp16.ctypes.data, E, W2, H2, 2 * W2, P010, 0, 0, hfaces, hcp, None, None), h)
        elif k == "nv12":
            check(lib.fdt_detect_batch(h, hp8.ctypes.data, E, W2, H2, W2, NV12, 0, 0, hfaces, hcp, None, None), h)
        elif k == "planes16_p10":
            check(lib.fdt_detect_yuv_planes16(h, hd16, None, E, 10, 0, 0, hfaces, hcp, None, None), h)
        else:
            check(lib.fdt_detect_yuv_planes(h, hd8, None, E, 0, 0, hfaces, hcp, None, None), h)

    host_bytes = {}
    for a, b in (("nv12", "p010"), ("planes8", "planes16_p10")):
        host_run(a)
        hr = (bytes(hfaces), hcounts.copy())
        host_run(b)
        assert bytes(hfaces) == hr[0] and np.array_equal(hcounts, hr[1]), b
        host_bytes[b] = int(lib.fdt_last_h2d_bytes(h)) / E
        host_run(a)
        host_bytes[a] = int(lib.fdt_last_h2d_bytes(h)) / E
    assert host_bytes["p010"] == 552960 and host_bytes["planes16_p10"] == 2 * host_bytes["planes8"], host_bytes

    # ---- standard mode, C4-shaped
    det4 = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withIris=False, maxBatch=512, maxFaces=4)
    h4 = det4._h
    B4 = 1024
    c4_8 = torch.from_numpy(nv12(i420(bench.synth_base("c4")), W2, H2)).cuda()[torch.arange(B4, device="cuda") % P].contiguous()
    c4_16 = widen(c4_8)
    torch.cuda.synchronize()
    f4 = (_ffi.FdtFace * (B4 * 4))()
    n4 = np.zeros(B4, np.int32)
    m4 = np.zeros((B4, 4, 468, 3), np.float32)

    def std_run(k):
        t, mt, stride = (c4_16, P010, 2 * W2) if k == "p010" else (c4_8, NV12, W2)
        check(lib.fdt_detect_batch(h4, t.data_ptr(), B4, W2, H2, stride, mt, 1, 1, f4, n4.ctypes.data_as(_ffi.i32p),
                                   m4.ctypes.data_as(_ffi.f32p), None), h4)

    std_run("nv12")
    sref = (bytes(f4), n4.copy(), m4.copy())
    std_run("p010")
    assert bytes(f4) == sref[0] and np.array_equal(n4, sref[1]) and np.array_equal(m4, sref[2]), "standard p010"

    rounds = []
    for r in range(args.rounds):
        row = {"round": r, "device_img_s": {}, "letterbox_ms_per_1024": {}, "c2_img_s": {}, "host_img_s": {}, "standard_img_s": {}}
        for k in ("planes16", "planes8", "shift_batch"):
            row["device_img_s"][k] = timed(lambda: dev_run(k), B, h, args.steps)
        for k in ("planes16", "plane_table8"):
            row["letterbox_ms_per_1024"][k] = letterbox_ms(lb_calls[k]) * 1024 / NT
        for k in ("p010", "nv12"):
            row["c2_img_s"][k] = timed(lambda: c2_run(k), B, h, args.steps)
        for k in ("p010", "nv12", "planes16_p10", "planes8"):
            row["host_img_s"][k] = timed(lambda: host_run(k), E, h, max(2, args.steps // 2))
        for k in ("p010", "nv12"):
            row["standard_img_s"][k] = timed(lambda: std_run(k), B4, h4, max(2, args.steps // 2))
        rounds.append(row)
        print(json.dumps(row), flush=True)

    keys = ("device_img_s", "letterbox_ms_per_1024", "c2_img_s", "host_img_s", "standard_img_s")
    sm = {k: summary(rounds, k) for k in keys}
    med = lambda k, v: sm[k][v]["median"]
    ratios = {
        "device_planes16_over_planes8": med("device_img_s", "planes16") / med("device_img_s", "planes8"),
        "device_planes16_over_shift_batch": med("device_img_s", "planes16") / med("device_img_s", "shift_batch"),
        "letterbox_planes16_over_plane_table8": med("letterbox_ms_per_1024", "planes16") / med("letterbox_ms_per_1024", "plane_table8"),
        "c2_p010_over_nv12": med("c2_img_s", "p010") / med("c2_img_s", "nv12"),
        "host_p010_over_nv12": med("host_img_s", "p010") / med("host_img_s", "nv12"),
        "host_planes16_p10_over_planes8": med("host_img_s", "planes16_p10") / med("host_img_s", "planes8"),
        "standard_p010_over_nv12": med("standard_img_s", "p010") / med("standard_img_s", "nv12"),
    }
    result = {"workload": "short-range BlazeFace 128x128; device: %d NVDEC-shaped 1920x1080 surfaces (pitch 2048 samples, chroma at "
                          "row 1088), fast mode, chunks of %d, %d faces per pass; c2: %d device 1280x720 frames, fast mode; host: "
                          "%d pinned frames, fast mode (1280x720 P010 / NV12; 1920x1080 yuv420p10le planes with linesizes 3968 / "
                          "1984 / 2048 bytes and random bits above bit 10 / contiguous 8-bit I420 planes); standard: C4-shaped, "
                          "1024 1280x720 device frames, <= 4 faces, chunks of 512" % (B, args.chunk, dev_faces, B, E),
              "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": rounds,
              "summary": dict(sm, ratios=ratios, host_h2d_bytes_per_frame=host_bytes),
              "how": "library timer fdt_timer_begin/end around --steps calls after --warmup calls, max with the wall clock (shift_batch: "
                     "the torch >> 8 copy of every step inside that window, torch.cuda.synchronize() before each library call); "
                     "letterbox: fdt_set_stage_timing stage 0 over %d frames, mean of 10 calls, scaled to 1024; variants alternate "
                     "within each round; medians and [min, max] over rounds; every variant's records checked bitwise against its 8-bit "
                     "counterpart first" % NT}
    print(json.dumps(result), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")
    lib.fdt_free_pinned(pin)
    det.dispose()
    det4.dispose()


if __name__ == "__main__":
    main()
