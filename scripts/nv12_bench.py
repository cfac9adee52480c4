#!/usr/bin/env python
"""4:2:0 batch steps (NV12, NV21, I420, YV12) against the BGR batch step on bench.py's C2 / C5 inputs.

The frames of bench.py's workload are converted to 4:2:0 the way a decoder hands them over (cv2 COLOR_BGR2YUV_I420), and
the BGR step runs on what cv2.cvtColor(COLOR_YUV2BGR_I420) gives back (the round trip is lossy, so the original BGR frames
are never the comparison; every layout of the same chroma converts to the same BGR frame).  Each layout case keeps its
planes in one layout: nv12 / nv21 (chroma pitch W), i420 / yv12 (tight chroma pitch W/2) and i420_padded / yv12_padded
(chroma pitch W/2 rounded up to 64 bytes, plus 64).  Parity first: tensor, det_scale, detections, crops and modes of
    layout step: preprocess_batch_nv12 / _yuv420 -> detect_batch -> align_detections_nv12 / _yuv420
    BGR step:    preprocess_batch                -> detect_batch -> align_detections
must be byte-identical.  Then the steps are timed with CUDA events, alternating in one process, and profiled per kernel
(fd_ctx_profile) in a separate pass.  The NV12 case calls the *_nv12 entry points.  One JSON file per workload goes to
--out-dir: r4_nv12_<workload>.json for the NV12 case alone (the default), r5_yuv420_<workload>.json otherwise.  'i420' is
the tight chroma pitch only; name 'i420_padded' as well to measure the padded one.

    python scripts/nv12_bench.py --workloads c2,c5 --steps 100 --rounds 3 --out-dir profiles
    python scripts/nv12_bench.py --layouts nv12,nv21,i420,i420_padded --workloads c2,c5 --out-dir profiles
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


# case -> (FD_YUV420_* layout, chroma pitch from the width)
LAYOUTS = {"nv12": (0, lambda W: W), "nv21": (1, lambda W: W), "i420": (2, lambda W: W // 2), "yv12": (3, lambda W: W // 2),
           "i420_padded": (2, lambda W: -(-(W // 2) // 64) * 64 + 64), "yv12_padded": (3, lambda W: -(-(W // 2) // 64) * 64 + 64)}
KERNEL_SUFFIX = {0: "_nv12", 1: "_nv21", 2: "_i420", 3: "_i420"}   # I420 and YV12 share the planar kernels


def preprocess_bytes(h, w, new_h, kind):
    """bytes the preprocess kernel reads per frame (whole staged rows: Y rows and one or two chroma rows, a planar chroma row
    as a U and a V row of w/2 bytes) plus the 640x640x3 f32 tensor it writes"""
    scale_y = 1.0 / (new_h / h)
    total = 0
    for dy in range(new_h):
        y0, y1, two = y_rows(dy, scale_y, h)
        if kind == "bgr":
            total += 3 * w * (2 if two else 1)
        else:
            total += w * (2 if two else 1) + w * (2 if two and (y1 >> 1) != (y0 >> 1) else 1)
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
    cases = args.layouts.split(",")
    # one I420 conversion per frame; every layout case holds the same Y, U, V bytes
    ys, us, vs, bgrs = [], [], [], []
    for t in w.frames_t:
        i420 = cv2.cvtColor(t.cpu().numpy(), cv2.COLOR_BGR2YUV_I420)
        c, n = i420[H:].reshape(-1), (H // 2) * (W // 2)   # U then V planes
        ys.append(np.ascontiguousarray(i420[:H]))
        us.append(c[:n].reshape(H // 2, W // 2))
        vs.append(c[n:2 * n].reshape(H // 2, W // 2))
        bgrs.append(torch.from_numpy(cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420)).cuda())
    w.frames_t = bgrs
    w.frames_l = ctx.frame_table([(t.data_ptr(), H, W, W * 3) for t in bgrs])
    ys_t = [torch.from_numpy(y).cuda() for y in ys]
    tables, keep = {}, []
    for case in cases:
        layout, pitch_of = LAYOUTS[case]
        puv = pitch_of(W)
        desc = []
        for y_t, u, v in zip(ys_t, us, vs):
            if layout in (0, 1):
                c = np.zeros((H // 2, puv), np.uint8)
                c[:, 0::2], c[:, 1::2] = (u, v) if layout == 0 else (v, u)
            else:
                c = np.zeros((H, puv), np.uint8)
                c[:H // 2, :W // 2], c[H // 2:, :W // 2] = (u, v) if layout == 2 else (v, u)
            c_t = torch.from_numpy(c).cuda()
            keep.append(c_t)
            desc.append((y_t.data_ptr(), c_t.data_ptr(), H, W, W, puv))
        tables[case] = (layout, ctx.frame_table_nv12(desc), puv)
    tensors = {k: torch.empty_like(w.tensor_t) for k in ["bgr"] + cases}
    crops = {k: torch.empty_like(w.crops_t) for k in ["bgr"] + cases}
    modes = {k: torch.empty(w.cap_faces, dtype=torch.uint8, device="cuda") for k in ["bgr"] + cases}
    tensors["bgr"], crops["bgr"] = w.tensor_t, w.crops_t

    def step_bgr():
        ds = ctx.preprocess_batch(w.frames_l, w.tensor_t)
        ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
        ctx.align_detections(w.frames_l, w.crops_t, w.cap_faces, None, modes["bgr"])
        return ds

    def make_step(case):
        layout, tab, _ = tables[case]
        if case == "nv12":   # the *_nv12 entry points
            def step():
                ds = ctx.preprocess_batch_nv12(tab, tensors[case])
                ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
                ctx.align_detections_nv12(tab, crops[case], w.cap_faces, None, modes[case])
                return ds
        else:
            def step():
                ds = ctx.preprocess_batch_yuv420(tab, layout, tensors[case])
                ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
                ctx.align_detections_yuv420(tab, layout, crops[case], w.cap_faces, None, modes[case])
                return ds
        return step

    steps = [("bgr", step_bgr)] + [(case, make_step(case)) for case in cases]

    # ---- parity
    res = {}
    for kind, fn in steps:
        ds = fn()
        counts, det, lmk = ctx.detect_fetch(B)
        ctx.synchronize()
        n = int(counts.sum())
        res[kind] = dict(ds=ds, counts=counts, det=det, lmk=lmk, tensor=tensors[kind].cpu().numpy(), crops=crops[kind][:n].cpu().numpy(),
                         modes=modes[kind][:n].cpu().numpy())
    for case in cases:
        for k in res["bgr"]:
            if not np.array_equal(res["bgr"][k], res[case][k]):
                raise SystemExit("%s: %s step differs from the BGR step on the converted frames in %s" % (wl, case, k))
    faces = int(res["bgr"]["counts"].sum())

    # ---- timing: alternating rounds of `steps` steps, CUDA events
    for _ in range(args.warmup):
        for _, fn in steps:
            fn()
    ctx.synchronize()
    times = {k: [] for k, _ in steps}
    for _ in range(args.rounds):
        for kind, fn in steps:
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
    for kind, fn in steps:
        ctx.profile(True)
        for _ in range(args.steps):
            fn()
        p = ctx.profile_fetch()
        ctx.profile(False)
        prof[kind] = {k: dict(launches=n, us_per_launch=us / max(n, 1)) for k, (n, us) in p.items()}
    ctx.detect_fetch(B)
    name, power = gpu_identity()
    new_h = int(ctx.letterbox_geometry(H, W)[1])
    pre = {k: preprocess_bytes(H, W, new_h, k) * B for k, _ in steps}
    conv_us = 4.5 * H * W * B / (HBM_TBS * 1e12) * 1e6    # read 1.5 B + write 3 B per pixel
    best = {k: min(v) for k, v in times.items()}
    kname = {"bgr": ""}
    kname.update({c: KERNEL_SUFFIX[tables[c][0]] for c in cases})
    out = {
        "workload": wl, "gpu": name, "power_limit": power, "batch": B, "frame": "%dx%d" % (W, H), "faces": faces,
        "chroma_pitch": {c: tables[c][2] for c in cases},
        "ms_per_step": times, "frames_per_s": {k: B / (v * 1e-3) for k, v in best.items()},
        "preprocess_bytes_per_step": pre,
        "preprocess_us": {k: prof[k].get("preprocess_tma_kernel" + kname[k], {}).get("us_per_launch") for k, _ in steps},
        "warp_us": {k: prof[k].get("warp_fixed_kernel" + kname[k], {}).get("us_per_launch") for k, _ in steps},
        "profile": prof,
        "least_conversion_pass_us": conv_us,
        "beats_bgr_plus_conversion": {c: best[c] * 1e3 < best["bgr"] * 1e3 + conv_us for c in cases},
        "parity": "tensor, det_scale, detections, crops and modes of every layout byte-identical to the BGR step on the cvtColor frames",
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
    ap.add_argument("--layouts", default="nv12", help="comma-separated cases: " + ", ".join(LAYOUTS))
    ap.add_argument("--out-dir", default=None, help="write --out-name (%%s: the workload) here")
    ap.add_argument("--out-name", default=None, help="default: r4_nv12_%%s.json for --layouts nv12, else r5_yuv420_%%s.json")
    args = ap.parse_args()
    if args.out_name is None:
        args.out_name = "r4_nv12_%s.json" if args.layouts == "nv12" else "r5_yuv420_%s.json"
    for wl in args.workloads.split(","):
        out = run(wl, args)
        print(json.dumps(out))
        if args.out_dir:
            os.makedirs(args.out_dir, exist_ok=True)
            with open(os.path.join(args.out_dir, args.out_name % wl), "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
