"""Face crops of the detect calls (fdt_set_face_crops) against their absence and against the caller's routes, one process, one GPU.

Workloads (synthetic 1280x720 face frames of the (F) distribution, <= 4 faces, in device memory; short-range detector):
  * C4-shaped: --c4-batch frames, standard mode, chunks of 512 (bench.py c4).  Variants, alternating within each of --rounds
    rounds: crops off, and 112x112 embedding crops as float32 RGB CHW, v / 127.5 - 1 (a recognition net's input).  Wall clock
    around each call (the call returns with its results on the host).  Stage 9 (the crop warps) ms per chunk in a separate
    timed pass (fdt_set_stage_timing).
  * C2-shaped: --c2-batch frames, fast mode, chunks of 1024 (bench.py c2), crops off against on.  Both through
    fdt_detect_batch with host results: with crops on, fast mode adds a host stage per chunk (faces to the host, the ROIs, the
    crop warp).
  * The caller's route today for the same crops: every frame with faces downloaded as host BGR (the crops need it), then
    FaceDetector.embeddingCrop per face (one upload, warp and download per face), on --route-frames frames; the library's
    route is costed as the C4 call with crops on minus crops off, per face.
  * Informative: torch affine_grid + grid_sample (bilinear, zeros padding, align_corners=False) on the device frames with the
    same inverse maps, 128 faces per batch, into float32 RGB CHW.  Not bit-equal to extractAlignedSquare (float sampling
    instead of OpenCV's fixed-point taps); the fraction of equal u8 values is reported.
Every crops-on call's face records are checked bitwise against the crops-off call first.

    python tools/bench_face_crops.py [--rounds 3] [--out profiles/r08a_bench_face_crops.json]
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


def frames(n, unique=64):
    from face_detection_tflite_b200.synth import face_frames
    base = face_frames(unique, 1280, 720)
    return np.ascontiguousarray(np.concatenate([base] * ((n + unique - 1) // unique))[:n])


def med(xs):
    return {"median": statistics.median(xs), "range": [min(xs), max(xs)], "runs": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--c4-batch", type=int, default=1024)
    ap.add_argument("--c2-batch", type=int, default=4096)
    ap.add_argument("--route-frames", type=int, default=64)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import torch
    import face_detection_tflite_b200 as fdt
    from face_detection_tflite_b200 import _ffi
    from oracle import geometry as geo
    from oracle.cv_ops import aligned_square_matrix, invert_affine

    result = {"card": card(), "rounds": args.rounds, "steps": args.steps}
    spec = fdt.FaceCropSpec("embedding", 112, "rgb", True, np.float32, 1 / 127.5, -1.0)
    W, H = 1280, 720

    def run(d, dev, n, mode):
        """(seconds per call, records bytes, faces) of `steps` calls on n device frames."""
        f, c = None, None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            f, c, _ = d.detectBatchRaw(dev.data_ptr(), count=n, width=W, height=H, mode=mode, memKind=_ffi.FDT_MEM_DEVICE)
        dt = (time.perf_counter() - t0) / args.steps
        return dt, bytes(f)[: n * d._max_faces * C.sizeof(_ffi.FdtFace)], int(c.sum()), f, c

    for name, n, mode, chunk in (("c4_standard", args.c4_batch, 1, 512), ("c2_fast", args.c2_batch, 0, 1024)):
        d = fdt.FaceDetector.create(fdt.FaceDetectionModel.shortRange, withMesh=mode == 1, withIris=False, maxBatch=chunk, maxFaces=4)
        host = frames(n)
        dev = torch.from_numpy(host.reshape(-1)).cuda()
        d.setFaceCrops(None); run(d, dev, n, mode)
        d.setFaceCrops(spec); run(d, dev, n, mode)          # warm-up of both shapes (arena, staging)
        off, on = [], []
        for r in range(args.rounds):
            d.setFaceCrops(None)
            t_off, rec_off, faces, f_off, c_off = run(d, dev, n, mode)
            d.setFaceCrops(spec)
            t_on, rec_on, faces_on, f_on, c_on = run(d, dev, n, mode)
            assert faces_on == faces and np.array_equal(c_on, c_off)
            assert all(bytes(f_on[b * 4 + j]) == bytes(f_off[b * 4 + j]) for b in range(n) for j in range(int(c_off[b])))
            off.append(n / t_off); on.append(n / t_on)
            print(json.dumps({"workload": name, "round": r, "off_images_s": n / t_off, "on_images_s": n / t_on}), flush=True)
        row = {"frames": n, "faces_per_call": faces, "chunk": chunk, "crops_off_images_s": med(off), "crops_on_images_s": med(on),
               "ratio_on_over_off": med([a / b for a, b in zip(on, off)])}
        got, ok = d.faceCrops()
        assert got.shape == (faces, 3, 112, 112) and ok.all()
        # stage 9: the crop warps, per chunk (fdt_get_stage_ms sums over the last call)
        d._lib.fdt_set_stage_timing(d._h, 1)
        ms9, nl = [], C.c_int32()
        for _ in range(args.steps):
            d.detectBatchRaw(dev.data_ptr(), count=n, width=W, height=H, mode=mode, memKind=_ffi.FDT_MEM_DEVICE)
            ms = C.c_float()
            d._lib.fdt_get_stage_ms(d._h, 9, C.byref(ms), C.byref(nl))
            ms9.append(ms.value)
        d._lib.fdt_set_stage_timing(d._h, 0)
        nchunks = (n + chunk - 1) // chunk
        row["stage9_ms_per_chunk"] = med([m / nchunks for m in ms9])
        row["stage9_launches_per_call"] = nl.value
        row["stage9_crops_per_s"] = faces / (statistics.median(ms9) / 1e3)
        if name == "c4_standard":
            # the library's route: the crops-on call minus the crops-off call, per face
            lib_face_s = statistics.median([faces / (n / a - n / b) for a, b in zip(on, off)]) if all(a < b for a, b in zip(on, off)) else None
            # the caller's route: download each frame with faces, embeddingCrop per face
            nf = args.route_frames
            kf = [(b, j) for b in range(nf) for j in range(int(c_on[b]))]
            dets = d._faces_per_frame(f_on, c_on, None, None, [(W, H)] * n)[:nf]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            route = []
            for b in range(nf):
                if not dets[b]:
                    continue
                img = dev[b * W * H * 3:(b + 1) * W * H * 3].cpu().numpy().reshape(H, W, 3)
                for face in dets[b]:
                    route.append(d.embeddingCrop(face, img))
            route_s = time.perf_counter() - t0
            k0 = sum(int(c_on[b]) for b in range(nf))
            lib_u8 = np.round((got[:k0].transpose(0, 2, 3, 1)[..., ::-1] + 1.0) * 127.5).astype(np.uint8)
            row["caller_route"] = {"frames": nf, "faces": len(kf), "faces_per_s": len(kf) / route_s,
                                   "crops_equal": bool(len(route) == k0 and all(np.array_equal(a, b) for a, b in zip(lib_u8, route))),
                                   "library_faces_per_s_incremental": lib_face_s,
                                   "library_faces_per_s_stage9": row["stage9_crops_per_s"],
                                   "speedup_incremental": lib_face_s / (len(kf) / route_s) if lib_face_s else None,
                                   "speedup_stage9": row["stage9_crops_per_s"] / (len(kf) / route_s)}
            # torch affine_grid + grid_sample on the device frames (informative, not bit-equal)
            import torch.nn.functional as F
            mats, idx = [], []
            for b in range(n):
                for j in range(int(c_on[b])):
                    kp = f_on[b * 4 + j].keypoints
                    theta, cx, cy, size = geo.compute_embedding_alignment((kp[0] * W, kp[1] * H), (kp[2] * W, kp[3] * H))
                    M = invert_affine(aligned_square_matrix(cx, cy, size, -theta, 112)[0])   # dst -> src pixel map
                    # pixel centres -> normalised coordinates (align_corners=False): src_n = (2 * src + 1) / size - 1
                    Sd = np.array([[112 / 2, 0, 112 / 2 - 0.5], [0, 112 / 2, 112 / 2 - 0.5], [0, 0, 1]])
                    Ss = np.array([[2 / W, 0, 1 / W - 1], [0, 2 / H, 1 / H - 1]])
                    mats.append(Ss @ np.vstack([M, [0, 0, 1]]) @ Sd)
                    idx.append(b)
            th = torch.tensor(np.stack(mats), dtype=torch.float32, device="cuda")
            ix = torch.tensor(idx, device="cuda")
            fr = dev.view(n, H, W, 3)
            scale = torch.tensor([1 / 127.5], device="cuda")

            def grid_route():
                outs = []
                for s in range(0, len(idx), 128):
                    src = fr[ix[s:s + 128]].permute(0, 3, 1, 2).flip(1).float()
                    g = F.affine_grid(th[s:s + 128], (src.shape[0], 3, 112, 112), align_corners=False)
                    outs.append(F.grid_sample(src, g, mode="bilinear", padding_mode="zeros", align_corners=False) * scale - 1.0)
                return torch.cat(outs)

            grid_route()
            gt = []
            for _ in range(args.rounds):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                for _ in range(args.steps):
                    gout = grid_route()
                torch.cuda.synchronize(); gt.append(len(idx) * args.steps / (time.perf_counter() - t0))
            g8 = torch.round((gout + 1.0) * 127.5).clamp(0, 255).to(torch.uint8).cpu().numpy()
            l8 = np.round((got + 1.0) * 127.5).astype(np.uint8)
            row["torch_grid_sample"] = {"faces_per_s": med(gt), "equal_u8_fraction": float((g8 == l8).mean()),
                                        "max_abs_u8_diff": int(np.abs(g8.astype(int) - l8.astype(int)).max()),
                                        "note": "float bilinear sampling, not OpenCV's fixed-point taps: not bit-equal"}
        result[name] = row
        print(json.dumps({name: {k: v for k, v in row.items()}}, default=str), flush=True)
        d.dispose()
        del dev
        torch.cuda.empty_cache()
    print(json.dumps(result), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
