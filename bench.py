#!/usr/bin/env python
"""bench.py — BlazeFace detect throughput (preprocess + infer + decode + NMS) on N B200s.

  python bench.py --gpus 1 --steps 5 --warmup 3                      # BASELINE.json configs[1] (default, "c2")
  python bench.py --config c3                                         # full-range 192x192, 2048 x 1920x1080
  python bench.py --config c4                                         # detect + warp + 468-point mesh, 1024 frames, <= 4 faces
  python bench.py --scaling strong --gpus 8                           # the config's batch split across the ranks (shard_range)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...   # the reference's CPU pipeline (real cv2 calls + cv2.dnn) on the host cores
  python bench.py --dump-outputs DIR ... # also writes the results of the last timed step as DIR/<name>.npy

Frames are independent, so the batch shards across ranks with no collective on the data path.  Default scaling is
weak (the config's batch PER GPU); `--scaling strong` keeps the config's batch as the job total.

One JSON line on stdout (rank 0).  `value` = throughput with frames resident in HBM (CUDA events on the library's
streams, max over ranks); `e2e` = the same metric through fdt_detect_batch with pinned HOST frames, H2D + D2H inside
the timed region.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "images/sec BlazeFace detect (pre+infer+NMS)"
PERIOD = 64            # unique synthetic frames; the batch tiles them
DUMP_BYTES = 64 * 10**6 - 64 * 1024    # --dump-outputs budget, less room for the .npy headers

CONFIGS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "c2": dict(model="shortRange", file="face_detection_short_range.tflite", w=1280, h=720, batch=4096, mode="fast", S=128, anchors=896,
               sides=(160, 560), max_faces=0,
               workload="configs[1]: short-range BlazeFace 128x128 (896 anchors), batch %d synthetic 1280x720 BGR frames per GPU, "
                        "letterbox->detect->weighted NMS"),
    "c3": dict(model="full", file="face_detection_full_range.tflite", w=1920, h=1080, batch=2048, mode="fast", S=192, anchors=2304,
               sides=(120, 700), max_faces=0,
               workload="configs[2]: full-range BlazeFace 192x192 (2304 anchors), batch %d synthetic 1920x1080 BGR frames per GPU, "
                        "letterbox->detect->weighted NMS"),
    "c4": dict(model="shortRange", file="face_detection_short_range.tflite", w=1280, h=720, batch=1024, mode="standard", S=128, anchors=896,
               sides=(160, 560), max_faces=4,
               workload="configs[3]: short-range detection + warpAffine crops -> face_landmark 468-point mesh, up to 4 faces/frame, "
                        "batch %d synthetic 1280x720 BGR frames per GPU"),
}


def synth_base(name: str = "c2"):
    """The PERIOD unique frames of a config: 56 composited-face frames + 8 noise frames (SURVEY.md 8d)."""
    from face_detection_tflite_b200 import synth
    c = CONFIGS[name or "c2"]
    return np.concatenate([synth.face_frames(PERIOD - 8, c["w"], c["h"], min_side=c["sides"][0], max_side=c["sides"][1]),
                           synth.noise_frames(8, c["w"], c["h"])])


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons, pw = [], None, set(), []
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not f[0].isdigit() or int(f[0]) != self.idx:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2]); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, pw) if p > 200] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "samples_under_load": len(busy)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_outputs(out_dir: Path, counts: np.ndarray, faces: np.ndarray, mesh=None):
    """Writes one step's results as .npy files: counts [B] and the valid slots of `faces` (fdt_face records, [B, max_faces])
    and `mesh` ([B, max_faces, 468, 3] or None), in frame then slot order.  When the faces of every frame could exceed
    DUMP_BYTES, only those of a seeded sample of frames are written; the sample depends on B and max_faces alone, so
    two builds given the same arguments write the same frames."""
    B, mf = faces.shape
    per_face = 19 * 8 + (8 + mesh[0, 0].nbytes if mesh is not None else 0)
    k = min(B, max(0, (DUMP_BYTES - 16 * B) // (mf * per_face)))
    frames = np.arange(B) if k == B else np.sort(np.random.default_rng(0).choice(B, k, replace=False))
    fi, slot = np.nonzero(np.arange(mf)[None, :] < counts[frames][:, None])
    fb = frames[fi]
    f = faces[fb, slot]
    out = {"counts": counts.astype(np.float64),                        # faces per frame, every frame of the step
           "sample_frames": frames.astype(np.float64),                 # the frames whose faces follow
           "face_frame": fb.astype(np.float64),
           "face_box": np.stack([f["xmin"], f["ymin"], f["xmax"], f["ymax"]], 1),
           "face_score": f["score"],
           "face_keypoints": f["keypoints"].reshape(-1, 6, 2),
           "face_anchor_index": f["anchor_index"].astype(np.float64)}
    if mesh is not None:
        out["face_mesh_score"] = f["mesh_score"]
        out["face_mesh"] = mesh[fb, slot]
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(out_dir / (name + ".npy"), np.ascontiguousarray(a))
    return sum(a.nbytes for a in out.values())


def cpu_reference(cfg_name: str, steps: int, warmup: int, sample: int):
    """The reference's CPU path (oracle/cpu_bench.py: real cv2 resize / copyMakeBorder / warpAffine + cv2.dnn forward +
    vectorised candidate scan + restated decode / NMS) on all host cores."""
    from oracle.cpu_bench import CpuPipeline
    c = CONFIGS[cfg_name]
    det = (ROOT / "assets/models" / c["file"]).read_bytes()
    mesh = (ROOT / "assets/models/face_landmark.tflite").read_bytes() if c["mode"] == "standard" else None
    cp = CpuPipeline(det, c["model"], "bench", "synth_base", cfg_name, mesh_bytes=mesh)
    for _ in range(warmup):
        cp.run(min(sample, 4 * cp.workers))
    times = []
    for _ in range(steps):
        t, _faces = cp.run(sample)
        times.append(t)
    cp.close()
    total = sum(times)
    return {"value": sample * steps / total, "ms_per_step": 1e3 * total / steps, "cores": cp.workers,
            "sample": "%d of the same synthetic %dx%d frames per step, %d steps, one cv2 / cv2.dnn fp32 worker per core (cv2.resize + "
                      "copyMakeBorder + blobFromImage + net.forward%s; stand-in for TFLite/XNNPACK)"
                      % (sample, c["w"], c["h"], steps, " + warpAffine + face_landmark forward" if mesh else "")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (weak) / per job (strong); 0 = the config's batch")
    ap.add_argument("--chunk", type=int, default=0, help="frames per internal chunk (fdt_config.max_batch); 0 = 1024 (c2), 512 (c4), 256 (c3)")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="after the timed steps, write what the last one returned (rank 0's frames) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm returns face counts only)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = CONFIGS[args.config]
    W, H = cfg["w"], cfg["h"]
    Bcfg = args.batch or cfg["batch"]
    # measured on the final kernels: c2 763 k / 778 k / 782 k images/s at chunks of 512 / 1024 / 2048; c3 106 k / 110 k at 256 / 512 (256 kept: the
    # committed ncu capture of c3 is per 256 frames); c4 133 k / 142 k / 146 k at 256 / 512 / 1024 (512: two chunks keep the upload overlapped)
    chunk = args.chunk or {"c2": 1024, "c4": 512}.get(args.config, 256)
    standard = cfg["mode"] == "standard"

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    config = {"workload": cfg["workload"] % Bcfg + (" [strong scaling: that batch is the job total]" if args.scaling == "strong" else ""),
              "name": args.config, "frames_per_gpu": Bcfg if args.scaling == "weak" else "%d / %d ranks" % (Bcfg, world),
              "frame": "%dx%dx3 u8 BGR" % (W, H), "sharding": "frames split across ranks, no collective",
              "l2": "inputs_exceed_l2 (%.1f GB of frames per step and GPU)" % ((Bcfg if args.scaling == "weak" else Bcfg / world) * W * H * 3 / 1e9),
              "chunk": "%d frames per internal chunk (fdt_config.max_batch), chunks alternate over two streams" % chunk}

    if args.impl == "reference":
        if rank != 0:
            return
        sample = args.cpu_sample or {"c2": 2048, "c3": 512, "c4": 512}[args.config]
        r = cpu_reference(args.config, args.steps, max(args.warmup, 1), sample)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "images/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    import torch
    import torch.distributed as dist
    from face_detection_tflite_b200 import _ffi, build, sharding
    import face_detection_tflite_b200 as fdt

    if rank == 0:
        build.build()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    torch.cuda.set_device(local)
    lib = _ffi.load()
    det = fdt.FaceDetector.create(fdt.FaceDetectionModel[cfg["model"]], withMesh=standard, withIris=False, device=local, maxBatch=chunk,
                                  maxFaces=cfg["max_faces"])
    h = det._h
    mf = det._max_faces
    mode = 1 if standard else 0
    if args.scaling == "strong":
        lo, hi = sharding.shard_range(Bcfg, rank, world)
        B, B_job = hi - lo, Bcfg
    else:
        lo, B, B_job = 0, Bcfg, Bcfg * world
    frame_bytes = W * H * 3
    base = synth_base(args.config)
    idx = (np.arange(B) + lo) % PERIOD                      # frame k of the job is unique frame k mod PERIOD
    dev = torch.from_numpy(base).cuda()[torch.from_numpy(idx).cuda()].contiguous()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    face_sz = C.sizeof(_ffi.FdtFace)
    out_faces = C.c_void_p(); out_counts = C.c_void_p(); out_mesh = C.c_void_p()
    lib.fdt_alloc_pinned(max(B, 1) * mf * face_sz, C.byref(out_faces))
    lib.fdt_alloc_pinned(max(B, 1) * 4, C.byref(out_counts))
    if standard:
        lib.fdt_alloc_pinned(max(B, 1) * mf * _ffi.FDT_MESH_FLOATS * 4, C.byref(out_mesh))
    fptr = C.cast(out_faces, C.POINTER(_ffi.FdtFace)); cptr = C.cast(out_counts, _ffi.i32p)
    mptr = C.cast(out_mesh, _ffi.f32p) if standard else None
    pf, pc = C.c_void_p(), C.c_void_p()

    def check(rc):
        if rc != 0:
            raise RuntimeError(lib.fdt_last_error(h).decode())

    def step_device():
        if standard:      # results (faces + meshes) land on the host: the mesh stage needs the host between its device stages
            check(lib.fdt_detect_batch(h, dev.data_ptr(), B, W, H, W * 3, 16, mode, 1, fptr, cptr, mptr, None))
        else:
            check(lib.fdt_detect_batch_device(h, dev.data_ptr(), B, W, H, W * 3, 16, mode, C.byref(pf), C.byref(pc)))

    # ---- device-resident throughput -----------------------------------------------------------------
    # nvidia-smi needs ~100 ms per sample: it runs from the warm-up to the end of the e2e phase (the same
    # kernels under the same load) so that even a short timed region yields under-load samples
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step_device()
    lib.fdt_synchronize(h)
    launches_per_step = int(lib.fdt_last_launch_count(h))
    barrier()
    ms = C.c_float()
    lib.fdt_timer_begin(h)
    for _ in range(args.steps):
        step_device()
    lib.fdt_timer_end(h, C.byref(ms))
    barrier()
    t_ms = sharding.max_over_ranks(float(ms.value), world, torch.device("cuda", local))
    value = B_job * args.steps / (t_ms / 1e3)
    # face count of the last step (also proves the work was done)
    host_counts = np.empty(max(B, 1), np.int32)
    if standard:
        host_counts[:] = np.ctypeslib.as_array(cptr, (max(B, 1),))
    else:
        check(lib.fdt_copy_to_host(h, host_counts.ctypes.data, pc.value, B * 4))
    faces_found = int(host_counts[:B].sum())
    dumped = None
    if args.dump_outputs is not None and rank == 0:
        face_dtype = np.dtype(_ffi.FdtFace)
        if standard:      # fdt_detect_batch filled the pinned host buffers of the last step
            faces = np.ctypeslib.as_array(C.cast(out_faces, C.POINTER(C.c_uint8)), (B * mf * face_sz,)).view(face_dtype)
            mesh = np.ctypeslib.as_array(mptr, (B * mf * _ffi.FDT_MESH_FLOATS,)).reshape(B, mf, -1, 3)
        else:             # the device buffers fdt_detect_batch_device returned hold it until the next call
            faces = np.empty(B * mf, face_dtype)
            check(lib.fdt_copy_to_host(h, faces.ctypes.data, pf.value, B * mf * face_sz))
            mesh = None
        nbytes = dump_outputs(args.dump_outputs, host_counts[:B], faces.reshape(B, mf), mesh)
        dumped = {"dir": str(args.dump_outputs), "bytes": nbytes}

    # ---- end to end: pinned host frames -> fdt_detect_batch -> host results ------------------------------
    e2e = None
    if not args.no_e2e:
        # Host frames live in pinned memory (c2: B x 2.76 MB = 11.3 GB per rank).  When the box cannot pin that much for every
        # rank, the step is issued as `split` calls over a pinned buffer of B / split frames (same bytes uploaded per step).
        split = int(os.environ.get("FDT_BENCH_E2E_SPLIT", "0"))
        if split <= 0:
            split = 1
            try:
                avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
                while split < 8 and (B // split) * frame_bytes * world * 1.5 > avail:
                    split *= 2
            except Exception:
                pass
        Bc = B // split
        pin = C.c_void_p()
        if lib.fdt_alloc_pinned(Bc * frame_bytes, C.byref(pin)) != 0:
            raise RuntimeError("pinned allocation failed")
        harr = np.ctypeslib.as_array((C.c_uint8 * (Bc * frame_bytes)).from_address(pin.value)).reshape(Bc, H, W, 3)
        # (with split > 1 every call re-reads the first B / split frames of the shard: same bytes, same face mix)
        for r0 in range(0, Bc, PERIOD):
            harr[r0:r0 + PERIOD] = base[idx[r0:min(r0 + PERIOD, Bc)]]

        def step_e2e():
            for k in range(split):
                fo = C.cast(C.c_void_p(out_faces.value + k * Bc * mf * face_sz), C.POINTER(_ffi.FdtFace))
                co = C.cast(C.c_void_p(out_counts.value + k * Bc * 4), _ffi.i32p)
                mo = C.cast(C.c_void_p(out_mesh.value + k * Bc * mf * _ffi.FDT_MESH_FLOATS * 4), _ffi.f32p) if standard else None
                check(lib.fdt_detect_batch(h, pin.value, Bc, W, H, W * 3, 16, mode, 0, fo, co, mo, None))

        for _ in range(2):
            step_e2e()
        barrier()
        e_steps = args.steps
        lib.fdt_timer_begin(h)
        t0 = time.perf_counter()
        for _ in range(e_steps):
            step_e2e()
        wall = (time.perf_counter() - t0) * 1e3
        lib.fdt_timer_end(h, C.byref(ms))
        barrier()
        e_ms = sharding.max_over_ranks(max(float(ms.value), wall), world, torch.device("cuda", local))
        e2e_counts = np.ctypeslib.as_array(cptr, (max(B, 1),))[:Bc * split].copy()
        # the host path must return what the device path returned: per-frame counts, and the boxes of a sample of frames
        want_counts = np.tile(host_counts[:Bc], split) if split > 1 else host_counts[:Bc * split]
        assert np.array_equal(e2e_counts, want_counts), "host and device paths disagree on per-frame face counts"
        if not standard and B > 0:
            dfaces = (_ffi.FdtFace * (min(B, 64) * mf))()
            check(lib.fdt_copy_to_host(h, C.addressof(dfaces), pf.value, min(B, 64) * mf * face_sz))
            for b in range(min(Bc, 64)):
                for j in range(int(e2e_counts[b])):
                    a, d = fptr[b * mf + j], dfaces[b * mf + j]
                    assert (a.xmin, a.ymin, a.xmax, a.ymax, a.score, a.anchor_index) == (d.xmin, d.ymin, d.xmax, d.ymax, d.score, d.anchor_index), \
                        "host and device paths disagree on frame %d" % b
        h2d = int(lib.fdt_last_h2d_bytes(h)) * split
        eager = min(4, mf)
        d2h = B * 4 + B * eager * face_sz + (faces_found * _ffi.FDT_MESH_FLOATS * 4 + faces_found * 8 if standard else 0)
        e2e = {"value": B_job * e_steps / (e_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
               "host_frame_bytes_per_step": B * frame_bytes, "d2h_bytes_per_step": d2h, "steps": e_steps, "calls_per_step": split,
               "note": "fdt_detect_batch on pinned host frames" +
                       ("; only the source rows the INTER_LINEAR taps read (2 of every 10) are uploaded, by one strided DMA per chunk; "
                        "results leave compacted (counts + the first 4 slots per frame, more on demand)" if not standard else
                        "; whole frames are uploaded (the crop-warp gathers from the full-resolution frame)")}
        lib.fdt_free_pinned(pin)
        # PCIe ceiling next to it: plain cudaMemcpyAsync of one contiguous pinned buffer, all ranks at the same time (what the
        # host can feed N GPUs at once).  The e2e step uploads h2d bytes per step; achieved / ceiling says how close it runs to the link.
        try:
            nb = 512 << 20
            hp = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            dp = torch.empty(nb, dtype=torch.uint8, device="cuda")
            dp.copy_(hp, non_blocking=True)
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(4):
                dp.copy_(hp, non_blocking=True)
            ev1.record()
            torch.cuda.synchronize()
            ceil_gbs = 4 * nb / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
            tot = torch.tensor([ceil_gbs], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tot)
            ach = h2d * e_steps / (e_ms / 1e3) / 1e9 * world          # every rank uploads its own shard
            e2e["pcie"] = {"h2d_ceiling_gbs_this_gpu": ceil_gbs, "h2d_ceiling_gbs_all_ranks": float(tot.item()),
                           "h2d_achieved_gbs_all_ranks": ach, "frac_of_ceiling": ach / float(tot.item()),
                           "how": "cudaMemcpyAsync of one contiguous 512 MiB pinned buffer x 4, CUDA events, every rank at the same time"}
            del hp, dp
        except Exception as ex:                      # the measurement is informative only
            e2e["pcie"] = {"error": str(ex)[:200]}

    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed steps + e2e steps"

    # ---- per-kernel timing + roofline of the dominant kernel (rank 0) ----------------------------------------
    roofline, kernels = None, None
    if rank == 0 and B > 0:
        n = min(int(det.maxBatch), B)
        cap = 512
        arr = (C.c_float * cap)()
        nl = C.c_int32()
        kn, tn = C.create_string_buffer(64), C.create_string_buffer(160)
        macs, byt = C.c_double(), C.c_double()
        rc = lib.fdt_profile_chunk(h, dev.data_ptr(), n, W, H, W * 3, 16, 20, arr, cap, C.byref(nl))
        if rc == 0:
            kernels = []
            nw, nh = (cfg["S"], round(H * cfg["S"] / W))
            for i in range(nl.value):
                lib.fdt_get_step_info(h, i, kn, tn, 160, C.byref(macs), C.byref(byt))
                b = byt.value
                if i == 0:
                    b = nw * nh * 4 * 3 + cfg["S"] * cfg["S"] * 3   # unique source bytes of INTER_LINEAR taps + u8 output (SURVEY.md 8d)
                kernels.append({"launch": i, "net": "detector", "kernel": kn.value.decode(), "tensor": tn.value.decode(), "ms": arr[i],
                                "macs_per_unit": macs.value, "bytes_per_unit": b, "units_per_launch": n, "unit": "image"})
            ndet = len(kernels)
            if standard:
                # mesh net: per-step timing over the crops the last call left in the stage buffers (units = faces)
                ns, got = C.c_int32(), C.c_int32()
                lib.fdt_debug_get_mesh_stage(h, 0, None, None, None, C.byref(got))     # crops the last mesh pass left in the stage buffers
                nf = got.value
                if nf > 0 and lib.fdt_profile_net(h, 1, nf, 10, arr, cap, C.byref(ns)) == 0:
                    for i in range(ns.value):
                        lib.fdt_get_net_step_info(h, 1, i, kn, tn, 160, C.byref(macs), C.byref(byt))
                        kernels.append({"launch": ndet + i, "net": "face_landmark", "kernel": kn.value.decode(), "tensor": tn.value.decode(),
                                        "ms": arr[i], "macs_per_unit": macs.value, "bytes_per_unit": byt.value, "units_per_launch": nf,
                                        "unit": "face"})
            for k in kernels:
                k["gbs"] = k["bytes_per_unit"] * k["units_per_launch"] / (k["ms"] * 1e-3) / 1e9 if k["ms"] > 0 else None
                k["tflops"] = 2 * k["macs_per_unit"] * k["units_per_launch"] / (k["ms"] * 1e-3) / 1e12 if k["ms"] > 0 else None
            # Kernels whose activations never leave the SM between layers (the image-resident chains) or that are pure latency
            # (one block per image, one GEMM tile per CTA) have no meaningful HBM roofline: their algorithmic HBM bytes are only
            # the chain's input and outputs.  The roofline object is quoted for the dominant HBM-streaming kernel; the on-chip
            # ones are listed beside it with their share of the step.
            on_chip = ("k_tail_ws", "k_fc_tc", "k_decode_nms")
            stream_k = [k for k in kernels if k["kernel"] not in on_chip]
            top = max(stream_k, key=lambda k: k["ms"])
            peak, how = peaks()
            total_ms = sum(k["ms"] for k in kernels)
            # DRAM traffic of the same launch from the committed ncu --set full capture (profiles/), when the kernel matches
            traffic, traffic_src = None, None
            tfile = sorted((ROOT / "profiles").glob("r*_%s_traffic.json" % args.config))
            if tfile:
                tj = json.loads(tfile[-1].read_text())
                ent = [e for e in tj["launches"] if e["launch"] == top["launch"]]      # (launch 0 = k_letterbox in both numberings)
                if ent and ent[0]["kernel"].split("<")[0] == top["kernel"] and ent[0]["images_per_launch"] == n:
                    traffic, traffic_src = ent[0]["dram_bytes_per_launch"], "profiles/" + tfile[-1].name
            det_k = kernels[1:ndet - 1]
            roofline = {"kernel": "%s[%s]" % (top["kernel"], top["tensor"]), "bound": "hbm", "achieved": top["gbs"], "peak": peak,
                        "unit": "GB/s", "frac": top["gbs"] / peak, "traffic": traffic, "traffic_source": traffic_src,
                        "algorithmic_bytes_per_launch": top["bytes_per_unit"] * top["units_per_launch"], "peak_source": how,
                        "share_of_step": top["ms"] / total_ms, "units_per_launch": "%d %ss" % (top["units_per_launch"], top["unit"]),
                        "note": "dominant HBM-streaming kernel by device time; achieved = algorithmic activation bytes (inputs read once + "
                                "outputs written once, fp32 NHWC) / CUDA-event duration of that launch",
                        "on_chip_kernels": [{"kernel": "%s[%s]" % (k["kernel"], k["tensor"]), "ms": k["ms"], "share_of_step": k["ms"] / total_ms,
                                             "tflops": k["tflops"], "hbm_gbs": k["gbs"], "frac_hbm": (k["gbs"] or 0) / peak,
                                             "bound": "shared-memory pipe + layer-to-layer latency: activations stay in shared memory / TMEM "
                                                      "between layers, HBM sees only the chain's input and outputs"}
                                            for k in kernels if k["kernel"] in ("k_tail_ws", "k_fc_tc")],
                        "step": {"ms": total_ms, "algorithmic_gbs": sum(k["bytes_per_unit"] * k["units_per_launch"] for k in kernels) / (total_ms * 1e-3) / 1e9,
                                 "frac_hbm": sum(k["bytes_per_unit"] * k["units_per_launch"] for k in kernels) / (total_ms * 1e-3) / 1e9 / peak},
                        "stages": {
                            "letterbox": {"ms": kernels[0]["ms"], "gbs": kernels[0]["gbs"], "frac_hbm": kernels[0]["gbs"] / peak},
                            "conv_stack": {"ms": sum(k["ms"] for k in det_k),
                                           "gbs": sum(k["bytes_per_unit"] for k in det_k) * n / (sum(k["ms"] for k in det_k) * 1e-3) / 1e9,
                                           "tflops": 2 * sum(k["macs_per_unit"] for k in det_k) * n / (sum(k["ms"] for k in det_k) * 1e-3) / 1e12},
                            "decode_nms": {"ms": kernels[ndet - 1]["ms"], "gbs": kernels[ndet - 1]["gbs"], "frac_hbm": kernels[ndet - 1]["gbs"] / peak}}}
            roofline["stages"]["conv_stack"]["frac_hbm"] = roofline["stages"]["conv_stack"]["gbs"] / peak
            if standard and len(kernels) > ndet:
                mk = kernels[ndet:]
                nf = mk[0]["units_per_launch"]
                roofline["stages"]["mesh_net"] = {"ms": sum(k["ms"] for k in mk), "faces": nf,
                                                  "gbs": sum(k["bytes_per_unit"] for k in mk) * nf / (sum(k["ms"] for k in mk) * 1e-3) / 1e9,
                                                  "tflops": 2 * sum(k["macs_per_unit"] for k in mk) * nf / (sum(k["ms"] for k in mk) * 1e-3) / 1e12}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        det.dispose()
        r = cpu_reference(args.config, 2, 1, args.cpu_sample or {"c2": 2048, "c3": 512, "c4": 512}[args.config])
        cpu = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e,
                "gpu_launches": launches_per_step * args.steps, "faces_per_step": faces_found,
                "faces_per_s": faces_found * (world if args.scaling == "weak" else 1) * args.steps / (t_ms / 1e3) if standard else None,
                "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels}
        if dumped:
            line["outputs"] = dumped
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
