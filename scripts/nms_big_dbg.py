"""A/B of the big NMS path between this tree's library and another build's (say, the parent commit's, built in-tree).

  python scripts/nms_big_dbg.py --other DIR [--rounds 3] [--reps 30] [--out FILE]

Rows, each host-timed from the call to its end (the calls synchronise, or are followed by a synchronise):
  detect_K*     fd_detect_batch + fd_detect_fetch of an 8-image 640 x 640 batch; image 0 holds K planted candidates (small
                boxes around their anchors), so its NMS is deferred to nms_big_kernel on the decode kernel's keys
  argsort_*     fd_argsort_descending (host scores in, order out)
  nms_100k_*    fd_nms_device on 100 000 device-resident boxes: the bench's crowd (grid path), and the same with every 13th box
                zero-width (not "fast": the radix sort + peel fallback)
  nms_4096_mid  fd_nms_device at 4 096 boxes (the mid path, which shares the decision sweeps)
Every round runs one worker process per tree, alternating which goes first; median and p10 / p90 are over all rounds'
samples.  Each row's outputs are hashed, and the two trees must agree.  The card's name and power limit are read in the
same run."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
A, FEAT, AOFF = 2, (20, 40, 80), (0, 800, 4000)   # anchors per cell, feature sides of strides 32 / 16 / 8, first anchor id of each


def _batch_heads(rng, K, B=8, others=30):
    """image 0: K candidates on random anchors, images 1..B-1: `others` each.  Scores U(0.75, 0.99), boxes 8..40 px"""
    from rs_face_detection_b200.utils import synth
    aw = synth.BASE_ANCHORS[..., 2] - synth.BASE_ANCHORS[..., 0] + 1
    heads = []
    for n in FEAT:
        fg = np.full((B, A, n, n), 0.1, np.float32)
        heads += [np.concatenate([1 - fg, fg], 1), np.zeros((B, 4 * A, n, n), np.float32), np.zeros((B, 10 * A, n, n), np.float32)]
    for b in range(B):
        ids = rng.choice(AOFF[2] + 2 * FEAT[2] ** 2, K if b == 0 else others, replace=False)
        s = np.searchsorted(AOFF, ids, side="right") - 1
        local = ids - np.asarray(AOFF)[s]
        a, cell = local % A, local // A
        n = np.asarray(FEAT)[s]
        h, w = cell // n, cell % n
        score = rng.uniform(0.75, 0.99, len(ids)).astype(np.float32)
        side = rng.uniform(8, 40, len(ids))
        for i in range(len(ids)):
            si, ai, hi, wi, wa = s[i], a[i], h[i], w[i], aw[s[i], a[i]]
            heads[3 * si][b, ai, hi, wi] = 1 - score[i]
            heads[3 * si][b, A + ai, hi, wi] = score[i]
            heads[3 * si + 1][b, 4 * ai:4 * ai + 4, hi, wi] = [rng.normal(0, 2) / wa, rng.normal(0, 2) / wa, np.log(side[i] / wa),
                                                               np.log(side[i] * rng.uniform(0.9, 1.1) / wa)]
    return heads


def _time(fn, reps, warm=5):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e6 * (time.perf_counter() - t0))
    return ts


def worker(root, reps):
    sys.path.insert(0, root)
    from rs_face_detection_b200 import Context
    from rs_face_detection_b200.utils import synth
    ctx = Context(0)
    rows = {}

    def row(name, fn, result):
        ts = _time(fn, reps)
        rows[name] = {"us": ts, "hash": hashlib.sha256(result()).hexdigest()}

    for K in (4097, 8000, 16000):
        heads = _batch_heads(np.random.default_rng(K), K)
        devs = [ctx.to_device(h) for h in heads]
        ds = np.ones(8, np.float32)
        out = {}

        def step():
            ctx.detect_batch(devs, 8, ds, 0.7, 0.4)
            out["r"] = ctx.detect_fetch(8)
        row("detect_K%d" % K, step, lambda: b"".join(np.ascontiguousarray(x).tobytes() for x in out["r"]))
        for d in devs:
            d.free()
    for n in (4097, 20000, 100000):
        rng = np.random.default_rng(n)
        s = (np.round(rng.uniform(0, 1, n) * 1000) / 1000).astype(np.float32)
        out = {}
        row("argsort_%d" % n, lambda: out.__setitem__("o", ctx.argsort_descending(s)), lambda: out["o"].tobytes())
    crowd = synth.make_crowd_boxes(100000, seed=42)
    zero_width = crowd.copy()
    zero_width[::13, 2] = zero_width[::13, 0] - 1.0
    for name, dets in (("nms_100k_crowd", crowd), ("nms_100k_zero_width", zero_width),
                       ("nms_4096_mid", synth.make_crowd_boxes(4096, seed=7, n_faces=200))):
        N = len(dets)
        d, keep, num = ctx.to_device(dets), ctx.alloc(4 * N), ctx.alloc(16)

        def call():
            ctx.nms_device(d, N, 0.4, keep, num)
            ctx.synchronize()

        def result():
            k = int(num.download((2,), np.int32)[0])
            return keep.download((N,), np.int32)[:k].tobytes()
        row(name, call, result)
    ctx.close()
    print(json.dumps(rows))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="root of another in-tree build to compare with")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out")
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker, args.reps)
    trees = {"this": HERE}
    if args.other:
        trees["other"] = os.path.abspath(args.other)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    samples = {t: {} for t in trees}
    hashes = {t: {} for t in trees}
    round_medians = {t: {} for t in trees}
    for r in range(args.rounds):
        order = list(trees) if r % 2 == 0 else list(trees)[::-1]
        for t in order:
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", trees[t], "--reps", str(args.reps)],
                                 capture_output=True, text=True, check=True)
            for name, v in json.loads(res.stdout.strip().splitlines()[-1]).items():
                samples[t].setdefault(name, []).extend(v["us"])
                round_medians[t].setdefault(name, []).append(round(float(np.median(v["us"])), 1))
                assert hashes[t].setdefault(name, v["hash"]) == v["hash"], (t, name, "outputs differ between rounds")
    report = {"gpu": card[0] if card else None, "rounds": args.rounds, "reps": args.reps, "rows": {}}
    for name in samples["this"]:
        entry = {}
        for t in trees:
            x = np.asarray(samples[t][name])
            entry[t] = {"median_us": round(float(np.median(x)), 1), "p10_us": round(float(np.percentile(x, 10)), 1),
                        "p90_us": round(float(np.percentile(x, 90)), 1), "round_medians_us": round_medians[t][name]}
        if args.other:
            entry["same_outputs"] = hashes["this"][name] == hashes["other"][name]
            entry["this_over_other"] = round(entry["this"]["median_us"] / entry["other"]["median_us"], 3)
        report["rows"][name] = entry
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if args.other and not all(e["same_outputs"] for e in report["rows"].values()):
        sys.exit("outputs differ between the trees")


if __name__ == "__main__":
    main()
