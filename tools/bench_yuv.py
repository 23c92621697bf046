"""BGR against NV12 input on the C2 workload (short-range detector, 1280x720 frames, fast mode), one process, one GPU.

The 64 unique frames of bench.synth_base("c2") are tiled to a batch of 4096 and detected in chunks of 1024; each BGR frame
is converted to NV12 once, before any timing.  The two formats alternate for --rounds rounds; every round measures
  * device-resident images/s (frames already on the GPU, fdt_detect_batch_device, fdt_timer_* events),
  * end-to-end images/s from pinned host frames (fdt_detect_batch, H2D + D2H inside the timed region),
  * the H2D bytes per frame the library uploaded (fdt_last_h2d_bytes) and the plain pinned cudaMemcpyAsync rate of the
    same round (the ceiling an upload of those bytes can reach),
and once per format the letterbox kernel time of a 1024-frame chunk (fdt_profile_chunk, launch 0).

    python tools/bench_yuv.py [--rounds 3] [--steps 10] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

NV12 = 0x1000
BGR = 16


def nv12_of(bgr):
    import cv2
    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    flat = i420[h:].reshape(-1)
    uv = np.stack([flat[:w * h // 4], flat[w * h // 4:]], -1).reshape(h // 2, w)
    return np.concatenate([i420[:h], uv])


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as ex:
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % str(ex)[:80]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--chunk", type=int, default=1024)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import torch
    import bench
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi, build

    build.build()
    lib = _ffi.load()
    W, H, B, P = 1280, 720, args.batch, bench.PERIOD
    base = bench.synth_base("c2")
    fmts = {"bgr": (BGR, W * 3, W * H * 3, base),
            "nv12": (NV12, W, W * H * 3 // 2, np.stack([nv12_of(f) for f in base]))}
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=False, maxBatch=args.chunk)
    h = det._h
    mf = det._max_faces

    def check(rc):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(h).decode())

    idx = np.arange(B) % P
    dev, pins, hosts = {}, {}, {}
    for k, (mt, stride, fb, frames) in fmts.items():
        dev[k] = torch.from_numpy(frames).cuda()[torch.from_numpy(idx).cuda()].contiguous()
        pins[k] = C.c_void_p()
        if lib.fdt_alloc_pinned(B * fb, C.byref(pins[k])) != 0:
            raise RuntimeError("pinned allocation of %d bytes failed" % (B * fb))
        arr = np.ctypeslib.as_array((C.c_uint8 * (B * fb)).from_address(pins[k].value)).reshape(B, -1)
        for r0 in range(0, B, P):
            arr[r0:r0 + P] = frames.reshape(P, -1)[idx[r0:r0 + P]]
        hosts[k] = arr
    torch.cuda.synchronize()
    out_faces, out_counts = C.c_void_p(), C.c_void_p()
    lib.fdt_alloc_pinned(B * mf * C.sizeof(_ffi.FdtFace), C.byref(out_faces))
    lib.fdt_alloc_pinned(B * 4, C.byref(out_counts))
    fptr, cptr = C.cast(out_faces, C.POINTER(_ffi.FdtFace)), C.cast(out_counts, _ffi.i32p)
    pf, pc = C.c_void_p(), C.c_void_p()
    ms = C.c_float()

    def device_rate(k):
        mt, stride, _, _ = fmts[k]
        step = lambda: check(lib.fdt_detect_batch_device(h, dev[k].data_ptr(), B, W, H, stride, mt, 0, C.byref(pf), C.byref(pc)))
        for _ in range(args.warmup):
            step()
        lib.fdt_synchronize(h)
        lib.fdt_timer_begin(h)
        for _ in range(args.steps):
            step()
        lib.fdt_timer_end(h, C.byref(ms))
        counts = np.empty(B, np.int32)
        check(lib.fdt_copy_to_host(h, counts.ctypes.data, pc.value, B * 4))
        return B * args.steps / (ms.value / 1e3), int(counts.sum())

    def e2e_rate(k):
        mt, stride, _, _ = fmts[k]
        step = lambda: check(lib.fdt_detect_batch(h, pins[k].value, B, W, H, stride, mt, 0, 0, fptr, cptr, None, None))
        for _ in range(max(1, args.warmup // 2)):
            step()
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        e_ms = max(float(ms.value), wall)
        h2d = int(lib.fdt_last_h2d_bytes(h))
        counts = np.ctypeslib.as_array(cptr, (B,)).copy()
        return B * args.steps / (e_ms / 1e3), h2d / B, int(counts.sum())

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

    rounds = []
    for r in range(args.rounds):
        row = {"round": r, "h2d_ceiling_gbs": memcpy_ceiling()}
        for k in fmts:
            dv, dfaces = device_rate(k)
            ev, bpf, efaces = e2e_rate(k)
            assert efaces == dfaces, "host and device paths disagree on the face count (%s)" % k
            row[k] = {"device_img_s": dv, "e2e_img_s": ev, "h2d_bytes_per_frame": bpf, "faces": dfaces,
                      "e2e_frac_of_ceiling": ev * bpf / 1e9 / row["h2d_ceiling_gbs"]}
        rounds.append(row)
        print(json.dumps(row), flush=True)

    letterbox = {}
    for k, (mt, stride, _, _) in fmts.items():
        cap = 512
        arr = (C.c_float * cap)()
        nl = C.c_int32()
        check(lib.fdt_profile_chunk(h, dev[k].data_ptr(), args.chunk, W, H, stride, mt, 20, arr, cap, C.byref(nl)))
        letterbox[k] = {"kernel": "k_letterbox" if k == "bgr" else "k_letterbox_yuv", "ms_per_chunk": float(arr[0]),
                        "chunk": args.chunk, "detector_chunk_ms": float(sum(arr[i] for i in range(nl.value)))}

    def med(k, f):
        return statistics.median(x[k][f] for x in rounds)

    summary = {k: {"device_img_s_median": med(k, "device_img_s"), "e2e_img_s_median": med(k, "e2e_img_s"),
                   "device_img_s_range": [min(x[k]["device_img_s"] for x in rounds), max(x[k]["device_img_s"] for x in rounds)],
                   "e2e_img_s_range": [min(x[k]["e2e_img_s"] for x in rounds), max(x[k]["e2e_img_s"] for x in rounds)],
                   "e2e_frac_of_ceiling_median": med(k, "e2e_frac_of_ceiling"),
                   "h2d_bytes_per_frame": rounds[-1][k]["h2d_bytes_per_frame"]} for k in fmts}
    summary["nv12_over_bgr"] = {"device": summary["nv12"]["device_img_s_median"] / summary["bgr"]["device_img_s_median"],
                                "e2e": summary["nv12"]["e2e_img_s_median"] / summary["bgr"]["e2e_img_s_median"]}
    result = {"workload": "C2: short-range BlazeFace 128x128, batch %d synthetic 1280x720 frames (64 unique, tiled), chunks of %d, "
                          "fast mode; NV12 frames converted from the BGR ones once before timing" % (B, args.chunk),
              "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": rounds, "letterbox": letterbox,
              "summary": summary,
              "how": "device: fdt_detect_batch_device on device-resident frames, fdt_timer_begin/end; e2e: fdt_detect_batch on "
                     "pinned host frames, max(events, wall clock); ceiling: cudaMemcpyAsync of a 512 MiB pinned buffer x 4, "
                     "CUDA events, same round; letterbox: fdt_profile_chunk launch 0, mean of 20 passes"}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")
    for p in pins.values():
        lib.fdt_free_pinned(p)
    lib.fdt_free_pinned(out_faces); lib.fdt_free_pinned(out_counts)
    det.dispose()


if __name__ == "__main__":
    main()
