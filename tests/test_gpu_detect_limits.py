"""The fused detect kernel (fd_detect_fused.cu) at its internal limits, against the oracle and against its other builds.

Head tensors are planted rather than sampled, so each image has an exact candidate set and a kept count known by
construction: the rank sort's regimes (K = 1 .. 1024, parts = 32 / nruns), the general single-CTA NMS and the deferral
beyond it, the estimate loop's later passes (faces 64.. of an image), empty estimates (the bbox fallback of the align warp),
the exact-IEEE NMS for zero-area boxes, and the threshold / signed-zero edges of the score scan.  Every scenario runs on
both register builds (fd_ctx_set_sharing 1 and 2), and in subprocesses behind FD_NO_FUSED=1 (the three-kernel path) and
FD_FUSED_GENERAL=1; all must give the same bytes.  The oracle (detect_post, align_face) is the judge of every value; the
builder only chooses which path runs.
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from detect_ref import assert_rows_exact, decode_rows
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONF, IOU = 0.7, 0.4
A = 2
FEAT = (20, 40, 80)              # feature map side of strides 32, 16, 8 at 640 x 640
AOFF = (0, 800, 4000)            # first anchor id of each stride in the 32|16|8 concatenation
AW = synth.BASE_ANCHORS[..., 2] - synth.BASE_ANCHORS[..., 0] + 1   # [stride][anchor] widths: 512 256 | 128 64 | 32 16
TN = (synth.ARCFACE_TEMPLATE - 56.0) / 112.0
FRAME_H, FRAME_W = 1080, 1920
DS = np.float32(1 / 3)           # 1920 x 1080 letterboxed into 640 x 360
CROP = 112 * 112 * 3
SWEEP_K = (0, 1, 2, 31, 32, 33, 64, 65, 96, 97, 160, 352, 513, 1023, 1024, 1025, 2048, 4095, 4096, 4097)
PATTERNS = ("distinct", "tied", "reversed")
KEPT = (1, 63, 64, 65, 128, 1023, 1024)


# ---------------------------------------------------------------- planted heads
def _blank(B, bg_fg):
    heads = []
    for n in FEAT:
        fg = np.full((B, A, n, n), bg_fg, np.float32)
        heads += [np.concatenate([1 - fg, fg], 1), np.zeros((B, 4 * A, n, n), np.float32), np.zeros((B, 10 * A, n, n), np.float32)]
    return heads


def _members(h8, w8):
    """the anchors whose centre is the centre of stride-8 cell (h8, w8): every base anchor is centred at 7.5 + stride * cell"""
    m = [(2, h8, w8, 1), (2, h8, w8, 0)]
    if h8 % 2 == 0 and w8 % 2 == 0:
        m += [(1, h8 // 2, w8 // 2, 1), (1, h8 // 2, w8 // 2, 0)]
    if h8 % 4 == 0 and w8 % 4 == 0:
        m += [(0, h8 // 4, w8 // 4, 1), (0, h8 // 4, w8 // 4, 0)]
    return m


def _groups(rng, n_sites, g, rows=80, cells=None):
    """n_sites groups of g anchors; the members of a group share a centre and are given the same 4 x 4 px box, so exactly
    one per group survives NMS.  Sites are stride-8 cells 8 px apart (16 / 32 px for g > 2 / g > 4): boxes of different
    groups never touch."""
    step = 1 if g <= 2 else (2 if g <= 4 else 4)
    if cells is None:
        cells = [(h, w) for h in range(0, rows, step) for w in range(0, 80, step)]
        cells = [cells[i] for i in rng.choice(len(cells), n_sites, replace=False)]
    out = []
    for h8, w8 in cells:
        m = _members(h8, w8)
        out.append([m[i] for i in rng.choice(len(m), g, replace=False)])
    return out


def _anchor_id(c):
    s, h, w, a = c
    return AOFF[s] + (h * FEAT[s] + w) * A + a


def _scores(rng, cands, pattern):
    K = len(cands)
    if pattern == "distinct":
        r = rng.permutation(K)
    elif pattern == "tied":
        return np.full(K, 0.875, np.float32)
    elif pattern == "reversed":   # increasing with anchor id: the sorted order is the reverse of the concatenation order
        r = np.argsort(np.argsort([_anchor_id(c) for c in cands], kind="stable"), kind="stable")
    else:
        raise ValueError(pattern)
    return (0.75 + 0.2 * (r + 1) / (K + 1)).astype(np.float32)


def _plant(heads, b, rng, groups, scores="distinct", lmk="tmpl", box=(4.0, 4.0)):
    """writes one image's candidates; returns K.  lmk per candidate: 'tmpl' (template-shaped, the estimate succeeds), 'zero'
    (five equal points: empty estimate), 'nan', 'inf'; box: the (w, h) in detector pixels, 0 for a zero-area box"""
    cands = [c for grp in groups for c in grp]
    sc = scores if isinstance(scores, np.ndarray) else _scores(rng, cands, scores)
    kinds = [lmk] * len(cands) if isinstance(lmk, str) else lmk
    boxes = [box] * len(cands) if isinstance(box, tuple) else box
    for (s, h, w, a), score, kind, (bw, bh) in zip(cands, sc, kinds, boxes):
        aw = AW[s, a]
        heads[3 * s][b, a, h, w] = np.float32(1) - score
        heads[3 * s][b, A + a, h, w] = score
        with np.errstate(divide="ignore"):
            heads[3 * s + 1][b, 4 * a:4 * a + 4, h, w] = [0.0, 0.0, np.log(bw / aw), np.log(bh / aw)]
        size, th = rng.uniform(24, 60), rng.uniform(-0.5, 0.5)   # drawn for every kind: the rng stream does not depend on it
        rot = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        pts = (TN * size) @ rot.T / aw
        if kind == "zero":
            pts[:] = 0.0
        elif kind == "nan":
            pts[:] = np.nan
        elif kind == "inf":
            pts[2, 0] = np.inf
        heads[3 * s + 2][b, 10 * a:10 * a + 10, h, w] = pts.reshape(10)
    return len(cands)


@functools.lru_cache(maxsize=None)   # (callers only read the arrays)
def _sweep_batch(seed=1):
    """every K of SWEEP_K with every score pattern, one image each; groups of 1 / 2 / 4 keep at most 1024 faces up to K = 4096"""
    rng = np.random.default_rng(seed)
    heads = _blank(len(SWEEP_K) * len(PATTERNS), 0.1)
    meta, b = [], 0
    for K in SWEEP_K:
        g = 1 if K <= 1024 else (2 if K <= 2048 else 4)
        n = -(-K // g)
        for p in PATTERNS:
            grp = _groups(rng, n, g)
            if n:
                grp[-1] = grp[-1][:K - g * (n - 1)]
            assert _plant(heads, b, rng, grp, p) == K
            meta.append(dict(K=K, kept=n))
            b += 1
    return heads, meta


@functools.lru_cache(maxsize=None)
def _kept_batch(seed=2, lmk="tmpl"):
    """one image per kept count of KEPT; some as coincident pairs (K = 2 x kept).  Rows < 44: every centre inside 1080p"""
    rng = np.random.default_rng(seed)
    heads = _blank(len(KEPT), 0.1)
    meta = []
    for b, kept in enumerate(KEPT):
        g = 2 if kept in (63, 65, 128) else 1
        K = _plant(heads, b, rng, _groups(rng, kept, g, rows=44), "distinct" if b % 2 else "reversed", lmk)
        meta.append(dict(K=K, kept=kept))
    return heads, meta


@functools.lru_cache(maxsize=None)
def _crowded_kept_batch(seed=3, lmk="tmpl"):
    """image 0: 1500 coincident pairs (K = 3000, 1500 kept: more than the fused kernel's rows hold); image 1: 20 faces"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, 0.1)
    meta = []
    for b, (kept, g) in enumerate(((1500, 2), (20, 1))):
        K = _plant(heads, b, rng, _groups(rng, kept, g, rows=44), "distinct", lmk)
        meta.append(dict(K=K, kept=kept))
    return heads, meta


@functools.lru_cache(maxsize=None)
def _empty_estimate_batch(seed=4, warm=False):
    """two images of 150 faces (three estimate passes) mixing template, all-zero and non-finite landmark deltas; boxes near
    the right and bottom borders of the frame make the fallback crop fail (mode 0) as well as succeed (mode 2).  warm: the
    same boxes with template and empty landmarks swapped, so transforms left over from it cannot pass for the real ones"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, 0.1)
    meta = []
    for b in range(2):
        inner = [(h, w) for h in range(44) for w in range(78)]
        edge = [(h, w) for h in range(46) for w in (78, 79)] + [(h, w) for h in (44, 45) for w in range(78)]
        cells = [inner[i] for i in rng.choice(len(inner), 100, replace=False)] + [edge[i] for i in rng.choice(len(edge), 50, replace=False)]
        kinds = list(rng.choice(["tmpl", "tmpl", "zero", "zero", "nan", "inf"], len(cells)))
        if warm:
            kinds = ["zero" if k == "tmpl" else "tmpl" for k in kinds]
        K = _plant(heads, b, rng, _groups(rng, len(cells), 1, cells=cells), "distinct", kinds)
        meta.append(dict(K=K, kept=K))
    return heads, meta


@functools.lru_cache(maxsize=None)
def _threshold_batch(seed=5):
    """conf 0.7: per image 40 scores exactly at the threshold, 40 one ulp below it (dropped), 40 above, on disjoint boxes"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, 0.1)
    at, below = np.float32(CONF), np.nextafter(np.float32(CONF), np.float32(0))
    for b in range(2):
        sc = np.concatenate([np.full(40, at), np.full(40, below), rng.uniform(0.71, 0.99, 40)]).astype(np.float32)
        perm = rng.permutation(120)
        _plant(heads, b, rng, _groups(rng, 120, 1), sc[perm])
    return heads, [dict(K=80, kept=80)] * 2


@functools.lru_cache(maxsize=None)
def _signed_zero_batch(seed=6):
    """conf 0 with background -1: +0.0 and -0.0 foreground scores pass and tie (one key), on disjoint boxes and on coincident
    pairs whose members differ only in the sign of their zero score"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, -1.0)
    for b in range(2):
        single = _groups(rng, 60, 1, rows=40)
        pairs = _groups(rng, 30, 2, cells=[(h, w) for h in range(40, 80, 2) for w in range(0, 80, 2)][:30])
        sc = np.where(rng.uniform(0, 1, 120) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
        sc[::7] = rng.uniform(0.0, 0.5, len(sc[::7]))
        _plant(heads, b, rng, single + pairs, sc)
    return heads, [dict(K=120, kept=90)] * 2


@functools.lru_cache(maxsize=None)
def _zero_area_batch(seed=7):
    """zero-area boxes (dw = -inf gives x2 - x1 + 1 == 0) among ordinary ones: the fused kernel must leave its fast IoU test
    for the exact IEEE one, where 0 / 0 is NaN and `!(ovr <= thr)` suppresses every zero-area box after the first kept one"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, 0.1)
    for b in range(2):
        cells = [(h, w) for h in range(79) for w in range(79) if w != 41]   # (the far borders would clip a zero side to 1)
        grp = _groups(rng, 80, 1, cells=[cells[i] for i in rng.choice(len(cells), 80, replace=False)])
        grp += _groups(rng, 10, 2, cells=[(h, 41) for h in range(1, 80, 8)])
        grp = [grp[i] for i in rng.permutation(len(grp))]
        boxes = []
        for i, g in enumerate(grp):
            boxes += [(0.0, 4.0) if i % 3 == 0 else ((4.0, 0.0) if i % 3 == 1 else (4.0, 4.0))] * len(g)
        _plant(heads, b, rng, grp, "distinct", "tmpl", boxes)
    return heads, None


@functools.lru_cache(maxsize=None)
def _big_fallback_batch(seed=8, zero_width=False):
    """image 0: K = 4097 candidates with one tied score (groups of 4, as in the sweep), so the anchor id decides every order;
    with zero_width every other group has zero-width boxes.  image 1: 20 faces"""
    rng = np.random.default_rng(seed)
    heads = _blank(2, 0.1)
    K, g = 4097, 4
    n = -(-K // g)
    grp = _groups(rng, n, g)
    grp[-1] = grp[-1][:K - g * (n - 1)]
    boxes = [(0.0, 4.0) if zero_width and i % 2 == 0 else (4.0, 4.0) for i, members in enumerate(grp) for _ in members]
    assert _plant(heads, 0, rng, grp, "tied", "tmpl", boxes) == K
    _plant(heads, 1, rng, _groups(rng, 20, 1, rows=44), "distinct")
    return heads, n


# ---------------------------------------------------------------- running a step
@functools.lru_cache(maxsize=None)
def _frames_host(B):
    return tuple(synth.make_frame(FRAME_H, FRAME_W, 500 + i) for i in range(B))


def _step(c, heads, ds, conf=CONF, iou=IOU, frames=None, cap=0):
    """detect (and align into fresh buffers) one batch; returns the fetched outputs and the path the step took"""
    B = heads[0].shape[0]
    devs = [c.to_device(h) for h in heads]
    c.detect_batch(devs, B, np.full(B, ds, np.float32), conf, iou)
    st = c.detect_last_stats()
    crops = modes = None
    if frames is not None:
        crops, modes = c.alloc(cap * CROP), c.alloc(cap)
        n0 = c.launch_count()
        c.align_detections(frames, crops, cap, ok_dev=modes)
        st["align_launches"] = c.launch_count() - n0
    counts, det, lmk = c.detect_fetch(B)
    out = dict(counts=counts, det=det, lmk=lmk.reshape(-1, 10), stats=st)
    if frames is not None:
        n = len(det)
        assert n <= cap, (n, cap)
        c.synchronize()
        out["crops"] = crops.download((n, 112, 112, 3), np.uint8) if n else np.zeros((0, 112, 112, 3), np.uint8)
        out["modes"] = modes.download((n,), np.uint8) if n else np.zeros(0, np.uint8)
    for d in devs:
        d.free()
    return out


def _upload_frames(c, B):
    bufs = [c.to_device(f) for f in _frames_host(B)]
    return bufs, [(d.ptr, FRAME_H, FRAME_W, FRAME_W * 3) for d in bufs]


def _aligned_steps(c, warm_heads, heads, cap):
    """the real batch after a warm-up batch of the same geometry: the first align call sizes the ctx's transform buffers
    (est_cap), so the second one reads the transforms the fused kernel estimated; the warm-up's landmarks differ, so stale
    transforms do not reproduce the expected crops"""
    bufs, frames = _upload_frames(c, heads[0].shape[0])
    _step(c, warm_heads, DS, frames=frames, cap=cap)
    out = _step(c, heads, DS, frames=frames, cap=cap)
    del bufs
    return out


def _run_sweep(c):
    heads, meta = _sweep_batch()
    fresh = _step(c, heads, 1.0)        # first meeting: every image with K > 1024 is deferred; the fetch makes the ctx crowded
    crowded = _step(c, heads, 1.0)      # from now on 1024 < K <= 4096 stays on the device
    return heads, meta, dict(fresh=fresh, crowded=crowded)


def _run_kept(c):
    heads, meta = _kept_batch()
    warm, _ = _kept_batch(lmk="zero")
    return heads, meta, dict(kept=_aligned_steps(c, warm, heads, sum(m["kept"] for m in meta)))


def _run_crowded_kept(c):
    heads, meta = _crowded_kept_batch()
    bufs, frames = _upload_frames(c, 2)
    cap = sum(m["kept"] for m in meta)
    first = _step(c, heads, DS, frames=frames, cap=cap)
    again = _step(c, heads, DS, frames=frames, cap=cap)
    del bufs
    return heads, meta, dict(first=first, again=again)


def _run_empty(c):
    heads, meta = _empty_estimate_batch()
    warm, _ = _empty_estimate_batch(warm=True)
    return heads, meta, dict(empty=_aligned_steps(c, warm, heads, sum(m["kept"] for m in meta)))


def _run_big_fallback(c):
    tied, _ = _big_fallback_batch()
    zero_width, _ = _big_fallback_batch(zero_width=True)
    return dict(negative_iou=_step(c, tied, 1.0, iou=-1.0), zero_width=_step(c, zero_width, 1.0))


def _run_edges(c):
    th, _ = _threshold_batch()
    sz, _ = _signed_zero_batch()
    za, _ = _zero_area_batch()
    return dict(threshold=_step(c, th, 1.0), signed_zero=_step(c, sz, 1.0, conf=0.0), zero_area=_step(c, za, 1.0))


SCENARIOS = dict(sweep=_run_sweep, kept=_run_kept, crowded_kept=_run_crowded_kept, empty=_run_empty, big_fallback=_run_big_fallback)
ARRAYS = ("counts", "det", "lmk", "crops", "modes")


def _both_builds(scenario):
    """runs a scenario on a fresh ctx with the 64-register build, then on another with the 32-register build; every output
    array must be byte-identical between them.  Returns the first run."""
    from rs_face_detection_b200 import Context
    runs = []
    for sharing in (1, 2):
        c = Context(0)
        try:
            c.set_sharing(sharing)
            runs.append(scenario(c))
        finally:
            c.set_sharing(1)
            c.close()
    outs = [r[-1] if isinstance(r, tuple) else r for r in runs]
    for name in outs[0]:
        for k in ARRAYS:
            if k in outs[0][name]:
                assert outs[0][name][k].tobytes() == outs[1][name][k].tobytes(), "%s/%s differs between the register builds" % (name, k)
        assert outs[0][name]["stats"] == outs[1][name]["stats"], name
    return runs[0]


def _check(oracle, heads, meta, out, ds, conf=CONF, iou=IOU, frames=None):
    """rows vs the oracle bit for bit (tests/detect_ref.py: boxes against a correctly rounded exp), and with frames every crop and mode vs
    oracle.align_face(frame, landmark row, bbox=detection row).  Returns the oracle's per-image (K, kept)."""
    cfg = oracle.make_det_cfg(conf_thr=conf, iou_thr=iou)
    B = heads[0].shape[0]
    assert len(out["counts"]) == B and out["counts"].sum() == len(out["det"])
    off, got = 0, []
    for b in range(B):
        edet, elmk, K = oracle.detect_post(cfg, [h[b] for h in heads], ds)
        n = int(out["counts"][b])
        assert n == len(edet), (b, n, len(edet))
        det, lmk = out["det"][off:off + n], out["lmk"][off:off + n]
        assert_rows_exact(det, lmk, (edet, elmk), decode_rows([h[b] for h in heads], cfg, ds, conf, iou), "image %d" % b)
        if meta is not None:
            assert (K, n) == (meta[b]["K"], meta[b]["kept"]), (b, K, n, meta[b])   # the builder planted what it meant to
        if frames is not None:
            for i in range(off, off + n):
                ecrop, _, emode = oracle.align_face(frames[b], out["lmk"][i], bbox=out["det"][i], with_mode=True)
                assert int(out["modes"][i]) == emode, (b, i - off, int(out["modes"][i]), emode)
                np.testing.assert_array_equal(out["crops"][i], ecrop if ecrop is not None else np.zeros((112, 112, 3), np.uint8),
                                              err_msg="image %d face %d" % (b, i - off))
        got.append((K, n))
        off += n
    return got


# ---------------------------------------------------------------- tests
def test_candidate_count_sweep(oracle):
    """K from 0 to 4097 in one batch, with distinct, tied and reversed scores: the rank sort at every parts = 32 / nruns regime
    (K = 1024 fills the head / row union), the general single-CTA NMS for 1024 < K <= 4096 once the ctx is crowded, the
    deferral beyond — on a fresh and on a crowded ctx, in both register builds."""
    heads, meta, outs = _both_builds(_run_sweep)
    fresh, crowded = outs["fresh"]["stats"], outs["crowded"]["stats"]
    n_pat = len(PATTERNS)
    assert fresh["fused"] and not fresh["crowded"] and fresh["max_candidates"] == 4097
    assert fresh["deferred_images"] == n_pat * sum(K > 1024 for K in SWEEP_K)
    assert crowded["fused"] and crowded["crowded"] and crowded["deferred_images"] == n_pat * sum(K > 4096 for K in SWEEP_K)
    _check(oracle, heads, meta, outs["fresh"], 1.0)
    for k in ("counts", "det", "lmk"):
        assert outs["fresh"][k].tobytes() == outs["crowded"][k].tobytes()


def test_kept_count_sweep_every_crop_from_fused_transforms(oracle):
    """1 .. 1024 kept faces per image: the fused kernel's estimate loop writes the transforms of every face, in all of its
    passes of 64; the align call then launches the warp kernel alone, and every crop and mode matches the oracle."""
    heads, meta, outs = _both_builds(_run_kept)
    out = outs["kept"]
    st = out["stats"]
    assert st["fused"] and st["deferred_images"] == 0 and st["max_candidates"] == 1024
    assert st["align_launches"] == 1, st     # no estimate_kernel: the crops come from the detect kernel's transforms
    _check(oracle, heads, meta, out, DS, frames=_frames_host(len(KEPT)))
    assert (out["modes"] == 1).all()


def test_crowded_image_with_more_kept_faces_than_rows_is_deferred(oracle):
    """K = 3000 with 1500 kept on a crowded ctx: the general NMS runs in the fused kernel, finds more kept faces than its rows
    hold, and gives the image up; the fetch completes it and re-aligns.  Same rows and crops as on the fresh ctx."""
    heads, meta, outs = _both_builds(_run_crowded_kept)
    first, again = outs["first"], outs["again"]
    assert first["stats"]["fused"] and not first["stats"]["crowded"] and first["stats"]["deferred_images"] == 1
    assert again["stats"]["crowded"] and again["stats"]["deferred_images"] == 1 and again["stats"]["max_candidates"] == 3000
    _check(oracle, heads, meta, again, DS, frames=_frames_host(2))
    for k in ARRAYS:
        assert first[k].tobytes() == again[k].tobytes(), k


def test_empty_estimates_take_the_bbox_fallback(oracle):
    """Faces whose landmarks give no transform (five equal points, NaN, inf) in the fused path: ok = 0 from the detect kernel,
    then the warp kernel's bbox fallback from the detection rows (stride 5): a fallback crop (mode 2), or the reference's Err
    (mode 0, zero crop) where the padded box leaves the frame; the other faces warp (mode 1)."""
    heads, meta, outs = _both_builds(_run_empty)
    out = outs["empty"]
    assert out["stats"]["fused"] and out["stats"]["deferred_images"] == 0 and out["stats"]["align_launches"] == 1
    _check(oracle, heads, meta, out, DS, frames=_frames_host(2))
    assert set(out["modes"].tolist()) == {0, 1, 2}
    assert (out["modes"][150:] != 1).sum() > 0   # also among the second image's faces (a later offset)


def test_threshold_equality_and_signed_zeros(oracle):
    """`score >= conf_thr`: a score equal to the threshold passes, one ulp below does not.  At conf_thr = 0, +0.0 and -0.0
    both pass, share one sort key and keep the concatenation order; their rows keep the sign bit."""
    outs = _both_builds(_run_edges)
    th, sz = outs["threshold"], outs["signed_zero"]
    for o in (th, sz):
        assert o["stats"]["fused"] and o["stats"]["deferred_images"] == 0
    assert th["stats"]["max_candidates"] == 80
    _check(oracle, *_threshold_batch(), th, 1.0)
    assert (th["det"][:, 4] >= np.float32(CONF)).all() and (th["det"][:, 4] == np.float32(CONF)).sum() > 0
    assert sz["stats"]["max_candidates"] == 120
    _check(oracle, *_signed_zero_batch(), sz, 1.0, conf=0.0)
    signs = np.signbit(sz["det"][:, 4])[sz["det"][:, 4] == 0]
    assert signs.any() and not signs.all()


def test_zero_area_boxes_take_the_exact_nms(oracle):
    """Zero-area candidate boxes: IoU 0 / 0 is NaN and the reference suppresses every zero-area box after the first kept
    one.  Only the fused kernel's exact-IEEE greedy reproduces that; its division-free fast test would keep them all."""
    outs = _both_builds(_run_edges)
    o = outs["zero_area"]
    assert o["stats"]["fused"] and o["stats"]["deferred_images"] == 0
    heads = _zero_area_batch()[0]
    got = _check(oracle, heads, None, o, 1.0)
    boxes = o["det"][:, :4]
    area0 = (boxes[:, 2] - boxes[:, 0] + 1) * (boxes[:, 3] - boxes[:, 1] + 1) == 0
    off = 0
    for b, (K, n) in enumerate(got):
        assert K == 100 and n == 31 and area0[off:off + n].sum() == 1, (b, K, n)   # one zero-area box of 60 groups survives
        off += n


def test_deferred_image_through_the_big_fallback_with_ties(oracle):
    """A deferred image with K = 4097 tied candidates runs nms_big_kernel on the decode kernel's keys (slot order, anchor ids
    up to the total anchor count).  A negative IoU threshold and zero-width boxes each make its grid decline, so it sorts those
    keys by anchor id, then score, and runs the peel: the anchor id decides which member of a group is kept, and which one
    zero-width box survives (IoU 0 / 0 suppresses every later one).  The other image's count must stay its own."""
    outs = _both_builds(_run_big_fallback)
    n_groups = _big_fallback_batch()[1]
    neg, zw = outs["negative_iou"], outs["zero_width"]
    for o in (neg, zw):
        assert o["stats"]["deferred_images"] == 1 and o["stats"]["max_candidates"] == 4097
    _check(oracle, _big_fallback_batch()[0], [dict(K=4097, kept=1), dict(K=20, kept=1)], neg, 1.0, iou=-1.0)
    _check(oracle, _big_fallback_batch(zero_width=True)[0], [dict(K=4097, kept=n_groups // 2 + 1), dict(K=20, kept=20)], zw, 1.0)


def test_pipelined_shared_contexts_match_serial(oracle):
    """bench.py's pipelined pattern: two contexts with fd_ctx_set_sharing(2) alternate detect + align steps on their own
    streams with no host synchronisation in between; each ends with the same rows, crops and modes as a serial run."""
    from rs_face_detection_b200 import Context
    hx, mx = _kept_batch()
    hy, my = _empty_estimate_batch()
    cx, cy = sum(m["kept"] for m in mx), sum(m["kept"] for m in my)
    serial = {}
    c = Context(0)
    try:
        for name, h, cap in (("x", hx, cx), ("y", hy, cy)):
            bufs, frames = _upload_frames(c, h[0].shape[0])
            serial[name] = _step(c, h, DS, frames=frames, cap=cap)
            del bufs
    finally:
        c.close()
    ctxs = [Context(0), Context(0)]
    try:
        lanes = []
        for c in ctxs:
            c.set_sharing(2)
            res = dict(crops=c.alloc(max(cx, cy) * CROP), modes=c.alloc(max(cx, cy)))
            for name, h in (("x", hx), ("y", hy)):
                res[name + "_heads"] = [c.to_device(t) for t in h]
                res[name + "_frames"] = _upload_frames(c, h[0].shape[0])
            lanes.append(res)
        plan = [(0, "x"), (1, "y"), (0, "y"), (1, "x"), (0, "x"), (1, "y"), (0, "y"), (1, "x")]
        for lane, name in plan:
            c, r = ctxs[lane], lanes[lane]
            B = (hx if name == "x" else hy)[0].shape[0]
            c.detect_batch(r[name + "_heads"], B, np.full(B, DS, np.float32), CONF, IOU)
            c.align_detections(r[name + "_frames"][1], r["crops"], cx if name == "x" else cy, ok_dev=r["modes"])
        for lane, name in ((0, "y"), (1, "x")):
            c, r = ctxs[lane], lanes[lane]
            counts, det, lmk = c.detect_fetch(len(serial[name]["counts"]))
            c.synchronize()
            n = len(det)
            np.testing.assert_array_equal(counts, serial[name]["counts"])
            assert det.tobytes() == serial[name]["det"].tobytes() and lmk.reshape(-1, 10).tobytes() == serial[name]["lmk"].tobytes()
            assert r["crops"].download((n, 112, 112, 3), np.uint8).tobytes() == serial[name]["crops"].tobytes(), name
            assert r["modes"].download((n,), np.uint8).tobytes() == serial[name]["modes"].tobytes(), name
    finally:
        for c in ctxs:
            c.set_sharing(1)
            c.close()
    _check(oracle, hx, mx, serial["x"], DS, frames=_frames_host(len(KEPT)))


# ---------------------------------------------------------------- the environment switches
def _replay(path=None):
    """every scenario on fresh contexts of this process; outputs (and the paths taken) as one dict, optionally saved"""
    from rs_face_detection_b200 import Context
    flat = {}
    scen = dict(SCENARIOS, edges=_run_edges)
    for key, fn in scen.items():
        c = Context(0)
        try:
            r = fn(c)
        finally:
            c.close()
        outs = r[-1] if isinstance(r, tuple) else r
        for name, o in outs.items():
            for k in ARRAYS:
                if k in o:
                    flat["%s/%s/%s" % (key, name, k)] = o[k]
            st = o["stats"]
            flat["%s/%s/path" % (key, name)] = np.array([st["fused"], st["crowded"], st["deferred_images"], st.get("align_launches", -1)])
    if path:
        np.savez(path, **flat)
    return flat


@functools.lru_cache(maxsize=None)
def _replay_here():
    return _replay()


@pytest.mark.parametrize("env", ["FD_NO_FUSED", "FD_FUSED_GENERAL"])
def test_switches_replay_byte_identical(tmp_path, env):
    """FD_NO_FUSED=1 (decode / nms_cta_kernel / finalize, estimate_kernel at align time: the A/B reference) and
    FD_FUSED_GENERAL=1 (the general single-CTA NMS in the fused kernel from the first call) are read once per process: each
    replays every scenario in a subprocess, and every output, crops and modes included, must equal this process's bytes."""
    path = str(tmp_path / "replay.npz")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "from test_gpu_detect_limits import _replay\n"
            "_replay(%r); print('ok')\n" % (ROOT, os.path.join(ROOT, "tests"), path))
    env_vars = {k: v for k, v in os.environ.items() if k not in ("FD_NO_FUSED", "FD_FUSED_GENERAL")}
    env_vars[env] = "1"
    res = subprocess.run([sys.executable, "-c", code], env=env_vars, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "ok" in res.stdout, res.stderr[-2000:]
    here = _replay_here()
    got = dict(np.load(path))
    assert sorted(got) == sorted(here)
    for k in here:
        if k.endswith("/path"):
            continue
        assert got[k].dtype == here[k].dtype and got[k].tobytes() == here[k].tobytes(), k
    paths = {k[:-5]: v for k, v in got.items() if k.endswith("/path")}
    if env == "FD_NO_FUSED":
        assert not any(v[0] for v in paths.values())
        assert paths["kept/kept"][3] == 2            # estimate_kernel + warp
    else:
        assert all(v[0] for v in paths.values())
        n_pat = len(PATTERNS)
        assert here["sweep/fresh/path"][2] == n_pat * sum(K > 1024 for K in SWEEP_K)
        assert paths["sweep/fresh"][2] == n_pat * sum(K > 4096 for K in SWEEP_K)   # no first meeting needed
        assert paths["crowded_kept/first"][2] == 1
