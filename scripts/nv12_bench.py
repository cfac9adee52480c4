#!/usr/bin/env python
"""4:2:0 (NV12, NV21, I420, YV12), packed 4:2:2 (YUY2, UYVY, YVYU) and interleaved RGB-family (RGB24, RGBA, BGRA, GRAY8)
batch steps against the BGR batch step on bench.py's C2 / C5 inputs.

The frames of bench.py's workload are converted to 4:2:0 the way a decoder hands them over (cv2 COLOR_BGR2YUV_I420), and
the BGR step runs on what cv2.cvtColor(COLOR_YUV2BGR_I420) gives back (the round trip is lossy, so the original BGR frames
are never the comparison; every layout of the same chroma converts to the same BGR frame).  Each layout case keeps its
planes in one layout: nv12 / nv21 (chroma pitch W), i420 / yv12 (tight chroma pitch W/2) and i420_padded / yv12_padded
(chroma pitch W/2 rounded up to 64 bytes, plus 64).  The packed cases yuy2 / uyvy / yvyu (pitch 2W) carry the same bytes:
each macropixel holds its two Y values and the U, V of its 2x2 block, so cv2.cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY / _YVYU)
gives the same BGR frame as well.  The RGB-family cases rgb24 / rgba / bgra (tight pitch, a noisy fourth byte) hold the BGR
frames themselves (when no YUV case is named, bench.py's own frames); gray8 holds cv2 COLOR_BGR2GRAY of them, and is compared
with a BGR step of its own (bgr_gray8) on what cv2.cvtColor(COLOR_GRAY2BGR) gives back.  Parity first: tensor, det_scale,
detections, crops and modes of
    layout step: preprocess_batch_nv12 / _yuv420 / _yuv422 / _rgb -> detect_batch -> align_detections_nv12 / _yuv420 / _yuv422 / _rgb
    BGR step:    preprocess_batch                       -> detect_batch -> align_detections
must be byte-identical.  Then the steps are timed with CUDA events, alternating in one process, and profiled per kernel
(fd_ctx_profile) in a separate pass.  The NV12 case calls the *_nv12 entry points.  One JSON file per workload goes to
--out-dir: r4_nv12_<workload>.json for the NV12 case alone (the default), r6_yuv422_<workload>.json when every case named
with --layouts is packed, r7_rgb_<workload>.json when every case is RGB-family, r5_yuv420_<workload>.json otherwise.  'i420' is the tight chroma pitch only; name 'i420_padded' as
well to measure the padded one.

    python scripts/nv12_bench.py --workloads c2,c5 --steps 100 --rounds 3 --out-dir profiles
    python scripts/nv12_bench.py --layouts nv12,nv21,i420,i420_padded --workloads c2,c5 --out-dir profiles
    python scripts/nv12_bench.py --layouts yuy2,uyvy,yvyu --workloads c2,c5 --out-dir profiles
    python scripts/nv12_bench.py --layouts rgb24,rgba,bgra,gray8 --workloads c2,c5 --out-dir profiles
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
# packed 4:2:2 case -> FD_YUV422_* layout and the byte positions of Y0, U, Y1, V in a macropixel
PACKED = {"yuy2": (0, (0, 1, 2, 3)), "uyvy": (1, (1, 0, 3, 2)), "yvyu": (2, (0, 3, 2, 1))}
# RGB-family case -> FD_RGB_* layout, bytes per pixel, kernel name suffix (RGBA and BGRA share the 4-byte kernels)
RGB = {"rgb24": (0, 3, "_rgb24"), "rgba": (1, 4, "_rgba"), "bgra": (2, 4, "_rgba"), "gray8": (3, 1, "_gray8")}


def preprocess_bytes(h, w, new_h, kind):
    """bytes the preprocess kernel reads per frame (whole staged rows: BGR rows of 3w bytes, packed 4:2:2 rows of 2w bytes,
    RGB-family rows of 3w, 4w or w bytes, or Y rows and one or two chroma rows, a planar chroma row as a U and a V row of w/2
    bytes) plus the 640x640x3 f32 tensor it writes"""
    scale_y = 1.0 / (new_h / h)
    total = 0
    for dy in range(new_h):
        y0, y1, two = y_rows(dy, scale_y, h)
        if kind in ("bgr", "bgr_gray8"):
            total += 3 * w * (2 if two else 1)
        elif kind in RGB:
            total += RGB[kind][1] * w * (2 if two else 1)
        elif kind in PACKED:
            total += 2 * w * (2 if two else 1)
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
    for t in (w.frames_t if any(c not in RGB for c in cases) else []):
        i420 = cv2.cvtColor(t.cpu().numpy(), cv2.COLOR_BGR2YUV_I420)
        c, n = i420[H:].reshape(-1), (H // 2) * (W // 2)   # U then V planes
        ys.append(np.ascontiguousarray(i420[:H]))
        us.append(c[:n].reshape(H // 2, W // 2))
        vs.append(c[n:2 * n].reshape(H // 2, W // 2))
        bgrs.append(torch.from_numpy(cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420)).cuda())
    if bgrs:
        w.frames_t = bgrs
        w.frames_l = ctx.frame_table([(t.data_ptr(), H, W, W * 3) for t in bgrs])
    ys_t = [torch.from_numpy(y).cuda() for y in ys]
    tables, keep = {}, []
    rng = np.random.default_rng(7)
    gray_bgr = None
    for case in cases:
        if case in RGB:   # the BGR frames in the case's layout (gray8: their cv2 grey, against its own BGR step)
            layout, bpp, _ = RGB[case]
            desc = []
            for t in w.frames_t:
                bgr = t.cpu().numpy()
                if case == "gray8":
                    px = cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY)
                else:
                    px = np.empty((H, W, bpp), np.uint8)
                    px[..., :3] = bgr[..., ::-1] if case in ("rgb24", "rgba") else bgr
                    if bpp == 4:
                        px[..., 3] = rng.integers(0, 256, (H, W), np.uint8)
                p_t = torch.from_numpy(np.ascontiguousarray(px).reshape(H, bpp * W)).cuda()
                keep.append(p_t)
                desc.append((p_t.data_ptr(), H, W, bpp * W))
                if case == "gray8":
                    keep.append(torch.from_numpy(cv2.cvtColor(px, cv2.COLOR_GRAY2BGR)).cuda())
                    gray_bgr = (gray_bgr or []) + [(keep[-1].data_ptr(), H, W, 3 * W)]
            tables[case] = (layout, ctx.frame_table(desc), bpp * W)
            continue
        if case in PACKED:   # each macropixel: its two Y values and the U, V of its 2x2 block
            layout, order = PACKED[case]
            desc = []
            for y_t, y, u, v in zip(ys_t, ys, us, vs):
                m = np.empty((H, W // 2, 4), np.uint8)
                m[..., order[0]], m[..., order[2]] = y[:, 0::2], y[:, 1::2]
                m[..., order[1]], m[..., order[3]] = np.repeat(u, 2, 0), np.repeat(v, 2, 0)
                p_t = torch.from_numpy(m.reshape(H, 2 * W)).cuda()
                keep.append(p_t)
                desc.append((p_t.data_ptr(), H, W, 2 * W))
            tables[case] = (layout, ctx.frame_table(desc), 2 * W)
            continue
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
    refs = ["bgr"] + (["bgr_gray8"] if gray_bgr else [])
    tensors = {k: torch.empty_like(w.tensor_t) for k in refs + cases}
    crops = {k: torch.empty_like(w.crops_t) for k in refs + cases}
    modes = {k: torch.empty(w.cap_faces, dtype=torch.uint8, device="cuda") for k in refs + cases}
    tensors["bgr"], crops["bgr"] = w.tensor_t, w.crops_t

    def step_bgr():
        ds = ctx.preprocess_batch(w.frames_l, w.tensor_t)
        ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
        ctx.align_detections(w.frames_l, w.crops_t, w.cap_faces, None, modes["bgr"])
        return ds

    def make_bgr_step(kind, tab):
        def step():
            ds = ctx.preprocess_batch(tab, tensors[kind])
            ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
            ctx.align_detections(tab, crops[kind], w.cap_faces, None, modes[kind])
            return ds
        return step

    def make_step(case):
        layout, tab, _ = tables[case]
        if case in RGB:
            def step():
                ds = ctx.preprocess_batch_rgb(tab, layout, tensors[case])
                ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
                ctx.align_detections_rgb(tab, layout, crops[case], w.cap_faces, None, modes[case])
                return ds
        elif case in PACKED:
            def step():
                ds = ctx.preprocess_batch_yuv422(tab, layout, tensors[case])
                ctx.detect_batch(w.heads_c, B, ds, bench.CONF_THR, bench.IOU_THR)
                ctx.align_detections_yuv422(tab, layout, crops[case], w.cap_faces, None, modes[case])
                return ds
        elif case == "nv12":   # the *_nv12 entry points
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

    steps = [("bgr", step_bgr)] + ([("bgr_gray8", make_bgr_step("bgr_gray8", ctx.frame_table(gray_bgr)))] if gray_bgr else [])
    steps += [(case, make_step(case)) for case in cases]
    ref_of = {c: "bgr_gray8" if c == "gray8" else "bgr" for c in cases}   # the BGR step on the case's converted frames

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
            if not np.array_equal(res[ref_of[case]][k], res[case][k]):
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
    conv_packed_us = 5.0 * H * W * B / (HBM_TBS * 1e12) * 1e6    # read 2 B + write 3 B per pixel
    conv_rgb_us = {c: (RGB[c][1] + 3) * H * W * B / (HBM_TBS * 1e12) * 1e6 for c in cases if c in RGB}   # read bpp + write 3 B
    conv_of = {c: conv_rgb_us[c] if c in RGB else conv_packed_us if c in PACKED else conv_us for c in cases}
    best = {k: min(v) for k, v in times.items()}
    kname = {"bgr": "", "bgr_gray8": ""}
    kname.update({c: RGB[c][2] if c in RGB else "_yuv422" if c in PACKED else KERNEL_SUFFIX[tables[c][0]] for c in cases})
    out = {
        "workload": wl, "gpu": name, "power_limit": power, "batch": B, "frame": "%dx%d" % (W, H), "faces": faces,
        "chroma_pitch": {c: tables[c][2] for c in cases if c not in PACKED and c not in RGB},
        "ms_per_step": times, "frames_per_s": {k: B / (v * 1e-3) for k, v in best.items()},
        "preprocess_bytes_per_step": pre,
        "preprocess_us": {k: prof[k].get("preprocess_tma_kernel" + kname[k], {}).get("us_per_launch") for k, _ in steps},
        "warp_us": {k: prof[k].get("warp_fixed_kernel" + kname[k], {}).get("us_per_launch") for k, _ in steps},
        "profile": prof,
        "least_conversion_pass_us": conv_us,
        "beats_bgr_plus_conversion": {c: best[c] * 1e3 < best[ref_of[c]] * 1e3 + conv_of[c] for c in cases},
        "parity": "tensor, det_scale, detections, crops and modes of every layout byte-identical to the BGR step on the cvtColor frames",
        "steps": args.steps, "rounds": args.rounds, "warmup": args.warmup,
    }
    if any(c in PACKED for c in cases):
        out["packed_pitch"] = {c: tables[c][2] for c in cases if c in PACKED}
        out["least_conversion_pass_us_packed"] = conv_packed_us
    if conv_rgb_us:
        out["rgb_pitch"] = {c: tables[c][2] for c in cases if c in RGB}
        out["least_conversion_pass_us_rgb"] = conv_rgb_us
        out["reference_step"] = {c: ref_of[c] for c in cases if c in RGB}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="c2,c5")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--layouts", default="nv12", help="comma-separated cases: " + ", ".join(list(LAYOUTS) + list(PACKED) + list(RGB)))
    ap.add_argument("--out-dir", default=None, help="write --out-name (%%s: the workload) here")
    ap.add_argument("--out-name", default=None,
                    help="default: r4_nv12_%%s.json for --layouts nv12, r6_yuv422_%%s.json for packed cases only, r7_rgb_%%s.json for "
                         "RGB-family cases only, else r5_yuv420_%%s.json")
    args = ap.parse_args()
    if args.out_name is None:
        packed_only = all(c in PACKED for c in args.layouts.split(","))
        rgb_only = all(c in RGB for c in args.layouts.split(","))
        args.out_name = ("r4_nv12_%s.json" if args.layouts == "nv12" else "r6_yuv422_%s.json" if packed_only
                         else "r7_rgb_%s.json" if rgb_only else "r5_yuv420_%s.json")
    for wl in args.workloads.split(","):
        out = run(wl, args)
        print(json.dumps(out))
        if args.out_dir:
            os.makedirs(args.out_dir, exist_ok=True)
            with open(os.path.join(args.out_dir, args.out_name % wl), "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
