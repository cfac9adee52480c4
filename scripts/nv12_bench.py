#!/usr/bin/env python
"""NV12 batch step against the BGR batch step on bench.py's C2 / C5 inputs.

The frames of bench.py's workload are converted to NV12 the way a decoder hands them over (cv2 COLOR_BGR2YUV_I420, U and V
interleaved), and the BGR step runs on what cv2.cvtColor(COLOR_YUV2BGR_NV12) gives back (the round trip is lossy, so the
original BGR frames are never the comparison).  Parity first: tensor, det_scale, detections, crops and modes of
    NV12 step: preprocess_batch_nv12 -> detect_batch -> align_detections_nv12
    BGR step:  preprocess_batch      -> detect_batch -> align_detections
must be byte-identical.  Then both steps are timed with CUDA events, alternating in one process, and profiled per kernel
(fd_ctx_profile) in a separate pass.  One JSON file per workload goes to --out-dir.

    python scripts/nv12_bench.py --workloads c2,c5 --steps 100 --rounds 3 --out-dir profiles
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBS = 7.7   # B200 data-sheet HBM3e bandwidth, for the least time a conversion pass could take


def y_rows(dy, scale_y, h):
    """the source rows (and whether the second has weight) of destination row dy of cv::resize INTER_LINEAR (fd_resize.cuh)"""
    fy = np.float32((dy + 0.5) * scale_y - 0.5)
    sy = int(np.floor(fy))
    fr = np.float32(fy - np.float32(sy))
    two = int(np.rint(np.float32(fr * np.float32(2048.0)))) != 0
    return min(max(sy, 0), h - 1), min(max(sy + 1, 0), h - 1), two


def preprocess_bytes(h, w, new_h, nv12):
    """bytes the preprocess kernel reads per frame (whole staged rows) plus the 640x640x3 f32 tensor it writes"""
    scale_y = 1.0 / (new_h / h)
    total = 0
    for dy in range(new_h):
        y0, y1, two = y_rows(dy, scale_y, h)
        if nv12:
            total += w * (2 if two else 1) + w * (2 if two and (y1 >> 1) != (y0 >> 1) else 1)
        else:
            total += 3 * w * (2 if two else 1)
    return total + 3 * 640 * 640 * 4


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
    except Exception as e:   # reported, not guessed
        pl = "unavailable (%s)" % type(e).__name__
    return name, pl


def run(wl, args):
    import cv2
    import torch
    import bench
    from rs_face_detection_b200 import Context
    ctx = Context(0)
    w = bench.Workload(ctx, wl, 0, 0)
    B, H, W = w.B, w.H, w.W
    # NV12 planes and the BGR frames cvtColor makes of them
    ys, uvs, bgrs = [], [], []
    for t in w.frames_t:
        bgr = t.cpu().numpy()
        i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
        uv = np.empty((H // 2, W), np.uint8)
        c, n = i420[H:].reshape(-1), (H // 2) * (W // 2)   # U then V planes
        uv[:, 0::2] = c[:n].reshape(H // 2, W // 2)
        uv[:, 1::2] = c[n:2 * n].reshape(H // 2, W // 2)
        y = i420[:H]
        back = cv2.cvtColor(np.concatenate([y, uv], 0), cv2.COLOR_YUV2BGR_NV12)
        ys.append(torch.from_numpy(np.ascontiguousarray(y)).cuda())
        uvs.append(torch.from_numpy(uv).cuda())
        bgrs.append(torch.from_numpy(back).cuda())
    w.frames_t = bgrs
    w.frames_l = ctx.frame_table([(t.data_ptr(), H, W, W * 3) for t in bgrs])
    nv_l = ctx.frame_table_nv12([(y.data_ptr(), uv.data_ptr(), H, W, W, W) for y, uv in zip(ys, uvs)])
    tensor_nv = torch.empty_like(w.tensor_t)
    crops_nv = torch.empty_like(w.crops_t)
    mode_bgr = torch.empty(w.cap_faces, dtype=torch.uint8, device="cuda")
    mode_nv = torch.empty_like(mode_bgr)

    def step_bgr():
        ds = ctx.preprocess_batch(w.frames_l, w.tensor_t)
        ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
        ctx.align_detections(w.frames_l, w.crops_t, w.cap_faces, None, mode_bgr)
        return ds

    def step_nv():
        ds = ctx.preprocess_batch_nv12(nv_l, tensor_nv)
        ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
        ctx.align_detections_nv12(nv_l, crops_nv, w.cap_faces, None, mode_nv)
        return ds

    # ---- parity
    res = []
    for fn, tensor, crops, mode in ((step_bgr, w.tensor_t, w.crops_t, mode_bgr), (step_nv, tensor_nv, crops_nv, mode_nv)):
        ds = fn()
        counts, det, lmk = ctx.detect_fetch(B)
        ctx.synchronize()
        n = int(counts.sum())
        res.append(dict(ds=ds, counts=counts, det=det, lmk=lmk, tensor=tensor.cpu().numpy(), crops=crops[:n].cpu().numpy(),
                        modes=mode[:n].cpu().numpy()))
    for k in res[0]:
        if not np.array_equal(res[0][k], res[1][k]):
            raise SystemExit("%s: NV12 step differs from the BGR step on the converted frames in %s" % (wl, k))
    faces = int(res[0]["counts"].sum())

    # ---- timing: alternating rounds of `steps` steps, CUDA events
    for _ in range(args.warmup):
        step_bgr()
        step_nv()
    ctx.synchronize()
    times = {"bgr": [], "nv12": []}
    for _ in range(args.rounds):
        for kind, fn in (("bgr", step_bgr), ("nv12", step_nv)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s = torch.cuda.ExternalStream(ctx.stream())
            e0.record(s)
            for _ in range(args.steps):
                fn()
            e1.record(s)
            e1.synchronize()
            times[kind].append(e0.elapsed_time(e1) / args.steps)
    ctx.detect_fetch(B)

    # ---- per-kernel profile, a pass of its own
    prof = {}
    for kind, fn in (("bgr", step_bgr), ("nv12", step_nv)):
        ctx.profile(True)
        for _ in range(args.steps):
            fn()
        p = ctx.profile_fetch()
        ctx.profile(False)
        prof[kind] = {k: dict(launches=n, us_per_launch=us / max(n, 1)) for k, (n, us) in p.items()}
    ctx.detect_fetch(B)
    name, power = gpu_identity()
    new_h = int(ctx.letterbox_geometry(H, W)[1])
    pre = {"bgr": preprocess_bytes(H, W, new_h, False) * B, "nv12": preprocess_bytes(H, W, new_h, True) * B}
    conv_us = 4.5 * H * W * B / (HBM_TBS * 1e12) * 1e6    # read 1.5 B + write 3 B per pixel
    best = {k: min(v) for k, v in times.items()}
    out = {
        "workload": wl, "gpu": name, "power_limit": power, "batch": B, "frame": "%dx%d" % (W, H), "faces": faces,
        "ms_per_step": times, "frames_per_s": {k: B / (v * 1e-3) for k, v in best.items()},
        "preprocess_bytes_per_step": pre,
        "preprocess_us": {k: prof[k].get(n, {}).get("us_per_launch") for k, n in (("bgr", "preprocess_tma_kernel"), ("nv12", "preprocess_tma_kernel_nv12"))},
        "profile": prof,
        "least_conversion_pass_us": conv_us,
        "nv12_beats_bgr_plus_conversion": best["nv12"] * 1e3 < best["bgr"] * 1e3 + conv_us,
        "parity": "tensor, det_scale, detections, crops and modes byte-identical to the BGR step on the cvtColor frames",
        "steps": args.steps, "rounds": args.rounds, "warmup": args.warmup,
    }
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="c2,c5")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out-dir", default=None, help="write r4_nv12_<workload>.json here")
    args = ap.parse_args()
    for wl in args.workloads.split(","):
        out = run(wl, args)
        print(json.dumps(out))
        if args.out_dir:
            os.makedirs(args.out_dir, exist_ok=True)
            with open(os.path.join(args.out_dir, "r4_nv12_%s.json" % wl), "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
