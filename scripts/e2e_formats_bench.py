#!/usr/bin/env python
"""fd_pipeline_host on host frames in other layouts (fd_pipeline_host_yuv420 / _yuv422 / _rgb) against the BGR call, on
bench.py's C2 inputs (64 x 1080p, its head tensors).

The frames are converted as scripts/nv12_bench.py does: cv2 COLOR_BGR2YUV_I420, and the BGR leg runs on what
cv2.cvtColor(COLOR_YUV2BGR_I420) gives back.  nv12 and i420 (tight chroma pitch W/2) hold those Y, U, V planes, yuy2 the same
bytes packed (each macropixel: its two Y values and the U, V of its 2x2 block), rgba the BGR leg's frames with a noisy fourth
byte, gray8 cv2 COLOR_BGR2GRAY of them (its parity reference is the BGR call on COLOR_GRAY2BGR of the grey frames).  Every
frame sits in pinned host memory with tight rows.  Each leg runs bench.py's e2e setup: 3 host threads, one fd_ctx each,
alternating batches, heads_zero_copy, in two modes: every face aligned with FD_UPLOAD_FULL, and FacePipeline::extract's
select flow with FD_UPLOAD_ON_DEMAND.  Parity first: every output of a layout leg must be byte-identical to its BGR reference.
Then the legs are timed in alternating rounds; per leg: frames/s, ms/step, H2D and D2H MB/step, with the GPU's name and power
limit read in the same run.

    python scripts/e2e_formats_bench.py --steps 48 --rounds 3 --out profiles/r8_e2e_formats.json
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

LEGS = ("bgr", "nv12", "i420", "yuy2", "rgba", "gray8")
MODES = {"all_full": dict(heads_zero_copy=True), "select_on_demand": dict(select=True, upload=1, heads_zero_copy=True)}


def build_frames(w):
    """leg -> (kind, layout, host descriptors, BGR reference frames); keeps every buffer alive in the returned list"""
    import cv2
    import torch
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    H, W = w.H, w.W
    rng = np.random.default_rng(7)
    legs, keep = {}, []
    bgr, ys, cs_nv12, cs_i420, packed, rgba, gray, gray_bgr = [], [], [], [], [], [], [], []
    for t in w.frames_t:
        i420 = cv2.cvtColor(t.cpu().numpy(), cv2.COLOR_BGR2YUV_I420)
        c, n = i420[H:].reshape(-1), (H // 2) * (W // 2)
        y, u, v = i420[:H], c[:n].reshape(H // 2, W // 2), c[n:2 * n].reshape(H // 2, W // 2)
        b = cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420)
        bgr.append(pin(b))
        ys.append(pin(y))
        uv = np.empty((H // 2, W), np.uint8)
        uv[:, 0::2], uv[:, 1::2] = u, v
        cs_nv12.append(pin(uv))
        cs_i420.append(pin(np.concatenate([u, v], 0)))
        m = np.empty((H, W // 2, 4), np.uint8)
        m[..., 0], m[..., 2] = y[:, 0::2], y[:, 1::2]
        m[..., 1], m[..., 3] = np.repeat(u, 2, 0), np.repeat(v, 2, 0)
        packed.append(pin(m.reshape(H, 2 * W)))
        px = np.empty((H, W, 4), np.uint8)
        px[..., :3] = b[..., ::-1]
        px[..., 3] = rng.integers(0, 256, (H, W), np.uint8)
        rgba.append(pin(px.reshape(H, 4 * W)))
        g = cv2.cvtColor(b, cv2.COLOR_BGR2GRAY)
        gray.append(pin(g))
        gray_bgr.append(pin(cv2.cvtColor(g, cv2.COLOR_GRAY2BGR)))
    keep += [bgr, ys, cs_nv12, cs_i420, packed, rgba, gray, gray_bgr]
    legs["bgr"] = ("bgr", None, bgr, bgr)
    legs["nv12"] = ("yuv420", 0, [(y.ctypes.data, c.ctypes.data, H, W, W, W) for y, c in zip(ys, cs_nv12)], bgr)
    legs["i420"] = ("yuv420", 2, [(y.ctypes.data, c.ctypes.data, H, W, W, W // 2) for y, c in zip(ys, cs_i420)], bgr)
    legs["yuy2"] = ("yuv422", 0, [(p.ctypes.data, H, W, 2 * W) for p in packed], bgr)
    legs["rgba"] = ("rgb", 1, [(p.ctypes.data, H, W, 4 * W) for p in rgba], bgr)
    legs["gray8"] = ("rgb", 3, [(p.ctypes.data, H, W, W) for p in gray], gray_bgr)
    return legs, keep


def call(ctx, leg, heads, cap, bufs, kw):
    import bench
    kind, layout, frames, _ = leg
    if kind == "bgr":
        return ctx.pipeline_host(frames, heads, cap, bench.CONF_THR, bench.IOU_THR, bufs=bufs, **kw)
    tab = ctx.frame_table_nv12(frames) if kind == "yuv420" else ctx.frame_table(frames)
    return getattr(ctx, "pipeline_host_" + kind)(tab, layout, heads, cap, conf_thr=bench.CONF_THR, iou_thr=bench.IOU_THR, bufs=bufs, **kw)


def same(a, b):
    (ba, ta, _, _), (bb, tb, _, _) = a, b
    if ta != tb or ba["n_crops"] != bb["n_crops"]:
        return False
    n = ba["n_crops"]
    return (all(np.array_equal(ba[k], bb[k]) for k in ("counts", "det_scale", "sel"))
            and all(np.array_equal(ba[k][:ta], bb[k][:ta]) for k in ("det", "lmk"))
            and all(np.array_equal(ba[k][:n], bb[k][:n]) for k in ("crops", "align_mode")))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=48, help="timed batches per leg and round (a multiple of the lanes)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--lanes", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_e2e_formats.json"))
    args = ap.parse_args()
    import torch
    import bench
    from nv12_bench import gpu_identity
    from rs_face_detection_b200 import Context
    ctxs = [Context(0) for _ in range(args.lanes)]
    for c in ctxs:
        c.set_sharing(args.lanes)
    w = bench.Workload(ctxs[0], "c2", 0, 0)
    B, cap = w.B, w.cap_faces
    legs, keep = build_frames(w)
    heads = [torch.from_numpy(h).pin_memory().numpy() for h in w.heads_np]
    pinb = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    mkbufs = lambda: dict(counts=pinb((B,), torch.int32), det=pinb((cap, 5), torch.float32), lmk=pinb((cap, 10), torch.float32),
                          crops=pinb((cap, 112, 112, 3), torch.uint8), det_scale=pinb((B,), torch.float32),
                          align_mode=pinb((cap,), torch.uint8), sel=pinb((B, 2), torch.int32), tensor=None)
    bufs = [mkbufs() for _ in ctxs]
    name, power = gpu_identity()

    parity = {}
    for mode, kw in MODES.items():
        for leg in LEGS[1:]:
            kind, layout, _, ref_frames = legs[leg]
            ref = ctxs[0].pipeline_host(ref_frames, heads, cap, bench.CONF_THR, bench.IOU_THR, bufs=mkbufs(), **kw)
            got = call(ctxs[1], legs[leg], heads, cap, mkbufs(), kw)
            parity["%s/%s" % (leg, mode)] = same(got, ref)
    if not all(parity.values()):
        print(json.dumps({"parity": parity}))
        sys.exit("parity failed")

    res = [None] * len(ctxs)

    def run(leg, kw, n_each):
        def worker(i):
            torch.cuda.set_device(0)
            for _ in range(n_each):
                res[i] = call(ctxs[i], legs[leg], heads, cap, bufs[i], kw)
        th = [threading.Thread(target=worker, args=(i,)) for i in range(len(ctxs))]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        return time.perf_counter() - t0

    steps = max(2 * len(ctxs), args.steps) // len(ctxs) * len(ctxs)
    times = {(leg, mode): [] for leg in LEGS for mode in MODES}
    traffic = {}
    for mode, kw in MODES.items():
        for leg in LEGS:
            run(leg, kw, 2)   # warm-up: workspaces, pinned staging, first launches
    for r in range(args.rounds):
        for mode, kw in MODES.items():
            for leg in (LEGS if r % 2 == 0 else LEGS[::-1]):
                times[(leg, mode)].append(run(leg, kw, steps // len(ctxs)))
                traffic[(leg, mode)] = (res[0][2], res[0][3], res[0][1], bufs[0]["n_crops"])
    out = {"gpu": name, "power_limit": power, "workload": "c2 (64 x 1080p, bench.py's head tensors)", "lanes": len(ctxs),
           "steps_per_round": steps, "rounds": args.rounds, "parity": parity, "legs": {}}
    for (leg, mode), ts in times.items():
        best = min(ts)
        h2d, d2h, total, n_crops = traffic[(leg, mode)]
        out["legs"]["%s/%s" % (leg, mode)] = {
            "frames_per_s": B * steps / best, "frames_per_s_rounds": [B * steps / t for t in ts], "ms_per_step": 1e3 * best / steps,
            "h2d_mb_per_step": h2d / 1e6, "d2h_mb_per_step": d2h / 1e6, "detections_per_step": int(total), "crops_per_step": int(n_crops)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for k, v in out["legs"].items():
        print("%-24s %8.0f frames/s  %6.2f ms/step  H2D %7.1f MB/step" % (k, v["frames_per_s"], v["ms_per_step"], v["h2d_mb_per_step"]))
    print("%s, power limit %s" % (name, power))
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()
