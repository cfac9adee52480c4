"""Every path that writes detection rows, bit for bit: landmarks and scores against the oracle, boxes against a restatement
with a correctly rounded exp (tests/detect_ref.py).  Configurations use box stds 0.1 / 0.1 / 0.2 / 0.2, landmark std 0.2 and
det_scales that are not powers of two, so that a reordered multiply or a reciprocal in place of a division changes bits."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from detect_ref import F, assert_bitwise, box_geom, box_pred, check_image, exp32_cr, libm_expf, log32_cr, nonlinear_transform_ref, pred_ref
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STDS, LSTD = (0.1, 0.1, 0.2, 0.2), 0.2
SCALES = np.array([1.0, 0.5, 0.33333334, 0.59259259, 2.0, 0.1], np.float32)
# the floats whose float64 exp lies within 4 double ulps of a float32 rounding midpoint, over the whole domain [-104, 89]
NEAR_MIDPOINT = [float.fromhex(s) for s in ("0x1.fdff02p-17", "0x1.cd3982p-14", "0x1.8d7cb6p-12", "-0x1p-25", "-0x1.c1c4b8p-10",
                                            "-0x1.e1dbe2p-8", "-0x1.d2259ap+3")]
AW = synth.BASE_ANCHORS[..., 2] - synth.BASE_ANCHORS[..., 0] + 1      # [stride][anchor]: 512 256 | 128 64 | 32 16
FEAT = (20, 40, 80)


def _cfgs(oracle, conf, iou, stds=STDS, lstd=LSTD, geometry=None):
    """(library config, oracle config) of one detector"""
    from rs_face_detection_b200 import default_config
    cfg = default_config()
    kw = {}
    if geometry is not None:
        image_wh, strides, base = geometry
        cfg.image_w, cfg.image_h = image_wh
        cfg.n_strides = len(strides)
        cfg.num_anchors = base.shape[1]
        for i, st in enumerate(strides):
            cfg.strides[i] = st
            for a in range(base.shape[1]):
                for k in range(4):
                    cfg.base_anchors[(i * 4 + a) * 4 + k] = float(base[i, a, k])
        kw = dict(image_size=image_wh, strides=strides, base_anchors=base)
    for k in range(4):
        cfg.bbox_stds[k] = stds[k]
    cfg.landmark_std = lstd
    return cfg, oracle.make_det_cfg(conf_thr=conf, iou_thr=iou, bbox_stds=stds, landmark_std=lstd, **kw)


def _check_batch(oracle, ocfg, heads, ds, counts, det, lmk, what=""):
    det, lmk = np.asarray(det).reshape(-1, 5), np.asarray(lmk).reshape(-1, 10)
    assert int(np.sum(counts)) == len(det), (what, np.sum(counts), len(det))
    off, Ks = 0, []
    for b in range(len(counts)):
        n = int(counts[b])
        Ks.append(check_image(oracle, ocfg, [h[b] for h in heads], ds[b], det[off:off + n], lmk[off:off + n], what="%s image %d" % (what, b)))
        off += n
    return Ks


def _run(c, heads, ds, conf, iou):
    devs = [c.to_device(h) for h in heads]
    B = heads[0].shape[0]
    c.detect_batch(devs, B, ds, conf, iou)
    st = c.detect_last_stats()
    counts, det, lmk = c.detect_fetch(B)
    for d in devs:
        d.free()
    return counts, det, lmk, st


def _scales(B):
    return SCALES[np.arange(B) % len(SCALES)]


# ---------------------------------------------------------------- chosen delta values
@functools.lru_cache(maxsize=None)
def _libm_misrounded(n=20):
    """inputs in [-4, 4] whose libm expf differs from the correctly rounded exp, from a seeded sample of 10^6 floats"""
    import ctypes.util
    m = C.CDLL(ctypes.util.find_library("m"))
    m.expf.restype, m.expf.argtypes = C.c_float, [C.c_float]
    x = np.random.default_rng(2024).uniform(-4, 4, 10 ** 6).astype(F)
    cr = exp32_cr(x)
    lib = np.fromiter((m.expf(v) for v in x.tolist()), F, len(x))
    bad = x[lib != cr]
    assert len(bad) >= n, len(bad)
    return tuple(float(v) for v in bad[:n])


def chosen_values():
    return (NEAR_MIDPOINT + list(_libm_misrounded()) + [88.5, 88.72283, 88.72284, 89.0, 100.0, 1e30]
            + [-87.5, -95.0, -103.9, -110.0] + [0.0, -0.0, np.inf, -np.inf, np.nan])


def chosen_heads(values):
    """one image, default geometry, stds 1 (so dw and dh equal the values): each value on its own anchor as dw and on another
    as dh, the anchor picked so that exp(value) * width lies in [0.5, 1279) where one does (x2 = (pw - 1) / 2 then keeps every
    bit of the exp), and dx, dy chosen to put the box centre at 0.  Ten more anchors carry +-0, +-inf and NaN landmark
    deltas.  Scores: distinct, all above 0.7.  -> heads, planted scores, and per planted anchor whether its box is zero-area"""
    rng = np.random.default_rng(11)
    heads = []
    for n in FEAT:
        fg = np.full((1, 2, n, n), 0.1, F)
        heads += [np.concatenate([1 - fg, fg], 1), np.zeros((1, 8, n, n), F), rng.normal(0, 0.3, (1, 20, n, n)).astype(F)]
    free = {(s, a): [(h, w) for h in range(FEAT[s]) for w in range(FEAT[s])] for s in range(3) for a in range(2)}
    for k in free:
        rng.shuffle(free[k])
    sizes = sorted(free, key=lambda k: AW[k])
    specials = [0.0, -0.0, np.inf, -np.inf, np.nan]
    plan = [(v, 0) for v in values] + [(v, 1) for v in values] + [(None, j) for j in range(10)]
    scores = (0.75 + 0.2 * (rng.permutation(len(plan)) + 1) / (len(plan) + 1)).astype(F)
    zero_area = []
    for (v, j), score in zip(plan, scores):
        e = np.float64(exp32_cr(np.array([0.0 if v is None else v], F))[0])
        s, a = next((k for k in sizes if 0.5 <= e * AW[k] < 1279), sizes[0])
        h, w = free[(s, a)].pop()
        aw = F(AW[s, a])
        cx, cy = F(synth.BASE_ANCHORS[s, a, 0] + w * 8 * 2 ** (2 - s)) + F(0.5) * (aw - F(1)), \
            F(synth.BASE_ANCHORS[s, a, 1] + h * 8 * 2 ** (2 - s)) + F(0.5) * (aw - F(1))
        heads[3 * s][0, a, h, w], heads[3 * s][0, 2 + a, h, w] = F(1) - score, score
        visible = 0.5 <= e * AW[s, a]
        d = np.array([-cx / aw if visible else 0.0, -cy / aw if visible else 0.0, 0.0, 0.0], F)
        if v is not None:
            d[2 + j] = v
        heads[3 * s + 1][0, 4 * a:4 * a + 4, h, w] = d
        if v is None:
            heads[3 * s + 2][0, 10 * a:10 * a + 10, h, w] = [specials[(j + k) % 5] for k in range(10)]
        with np.errstate(all="ignore"):
            box = box_pred(np.array([aw]), np.array([aw]), np.array([cx]), np.array([cy]), d[None])[0]
            box = np.fmax(np.fmin(box, F(639)), F(0))
            zero_area.append(bool((box[2] - box[0] + F(1)) * (box[3] - box[1] + F(1)) == 0))
    return heads, scores, np.array(zero_area)


def check_chosen(oracle, counts, det, lmk, heads, scores, zero_area, ocfg, what):
    _check_batch(oracle, ocfg, heads, np.ones(1, F), counts, det, lmk, what)
    kept = set(det[:, 4].tolist())
    missing = [i for i, s in enumerate(scores) if float(s) not in kept]
    # zero-area boxes meet each other with IoU 0 / 0 = NaN, which the reference's `ovr <= thr` removes: the first survives
    assert all(zero_area[i] for i in missing) and len(missing) == max(int(zero_area.sum()) - 1, 0), (what, missing)


# ---------------------------------------------------------------- scenarios replayed behind FD_NO_FUSED
@functools.lru_cache(maxsize=None)
def _scenarios():
    """name -> (heads, det_scales, conf, iou, stds, landmark std); deterministic, so a subprocess rebuilds the same inputs"""
    out = {}
    for B in (1, 5, 150):
        out["fused_b%d" % B] = (synth.make_heads(B, seed=40 + B, n_faces=8)[0], _scales(B), 0.7, 0.4, STDS, LSTD)
    out["crowded"] = (synth.make_heads(2, seed=21, n_faces=60)[0], _scales(2), 0.2, 0.4, STDS, LSTD)
    out["big"] = (synth.make_heads(2, seed=21, n_faces=60)[0], SCALES[2:4], 0.05, 0.4, STDS, LSTD)
    heads, _, _ = chosen_heads(chosen_values())
    out["chosen"] = (heads, np.ones(1, F), 0.7, 1.0, (1, 1, 1, 1), 1.0)
    return out


def replay(path, sharing=1):
    """runs every scenario on a fresh ctx of this process and saves the rows (and whether the fused kernel ran)"""
    from rs_face_detection_b200 import Context
    from oracle import oracle
    flat = {}
    for name, (heads, ds, conf, iou, stds, lstd) in _scenarios().items():
        c = Context(0, _cfgs(oracle, conf, iou, stds, lstd)[0])
        try:
            c.set_sharing(sharing)
            counts, det, lmk, st = _run(c, heads, ds, conf, iou)
        finally:
            c.close()
        flat.update({name + "/counts": counts, name + "/det": det, name + "/lmk": lmk, name + "/fused": np.array(st["fused"])})
    np.savez(path, **flat)
    return flat


def _check_replay(oracle, flat, what):
    for name, (heads, ds, conf, iou, stds, lstd) in _scenarios().items():
        ocfg = _cfgs(oracle, conf, iou, stds, lstd)[1]
        counts, det, lmk = flat[name + "/counts"], flat[name + "/det"], flat[name + "/lmk"]
        if name == "chosen":
            _, scores, zero_area = chosen_heads(chosen_values())
            check_chosen(oracle, counts, det.reshape(-1, 5), lmk, heads, scores, zero_area, ocfg, what + " " + name)
        else:
            _check_batch(oracle, ocfg, heads, ds, counts, det, lmk, what + " " + name)


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("sharing", [1, 2])
@pytest.mark.parametrize("B", [1, 5, 150])
def test_fused_kernel_rows(oracle, sharing, B):
    """the fused detect kernel, in its 64- and 32-register builds, with one image, a few, and more images than SMs"""
    from rs_face_detection_b200 import Context
    heads, ds, conf, iou, stds, lstd = _scenarios()["fused_b%d" % B]
    cfg, ocfg = _cfgs(oracle, conf, iou)
    c = Context(0, cfg)
    try:
        c.set_sharing(sharing)
        counts, det, lmk, st = _run(c, heads, ds, conf, iou)
    finally:
        c.close()
    assert st["fused"] and st["deferred_images"] == 0
    Ks = _check_batch(oracle, ocfg, heads, ds, counts, det, lmk, "fused")
    assert min(Ks) > 8 and counts.sum() > 5 * B


@pytest.mark.parametrize("sharing", [1, 2])
def test_chosen_delta_values(oracle, sharing):
    """near-midpoint exps, inputs libm's expf misrounds, overflow, subnormal and zero widths, +-0 / +-inf / NaN deltas"""
    from rs_face_detection_b200 import Context
    values = chosen_values()
    heads, scores, zero_area = chosen_heads(values)
    cfg, ocfg = _cfgs(oracle, 0.7, 1.0, (1, 1, 1, 1), 1.0)
    c = Context(0, cfg)
    try:
        c.set_sharing(sharing)
        counts, det, lmk, st = _run(c, heads, np.ones(1, F), 0.7, 1.0)
    finally:
        c.close()
    assert st["fused"] and st["max_candidates"] == len(scores)
    check_chosen(oracle, counts, det.reshape(-1, 5), lmk, heads, scores, zero_area, ocfg, "chosen")
    assert zero_area.sum() >= 4
    # libm misrounds some of these: the oracle's boxes differ on them, the kernel's must not differ from exp32_cr
    assert sum(libm_expf(v) != exp32_cr(np.array([v], F))[0] for v in values[7:27]) == 20


def test_three_kernel_path_without_128bit_score_rows(oracle):
    """41 x 41 positions: the fused kernel declines the geometry (decode, NMS CTA, finalize)"""
    from rs_face_detection_b200 import Context
    base = np.array([[[-8, -8, 15, 15], [-20, -20, 27, 27]]], F)
    cfg, ocfg = _cfgs(oracle, 0.7, 0.4, geometry=((328, 328), (8,), base))
    rng = np.random.default_rng(5)
    fg = rng.uniform(0, 0.6, (3, 2, 41, 41)).astype(F)
    hot = rng.uniform(0, 1, fg.shape) < 0.03
    fg[hot] = rng.uniform(0.7, 0.999, int(hot.sum())).astype(F)
    heads = [np.concatenate([1 - fg, fg], 1), rng.normal(0, 0.3, (3, 8, 41, 41)).astype(F), rng.normal(0, 0.3, (3, 20, 41, 41)).astype(F)]
    c = Context(0, cfg)
    try:
        counts, det, lmk, st = _run(c, heads, SCALES[3:6], 0.7, 0.4)
    finally:
        c.close()
    assert not st["fused"] and counts.sum() > 30
    _check_batch(oracle, ocfg, heads, SCALES[3:6], counts, det, lmk, "41x41")


def test_three_kernel_path_for_a_misaligned_score_tensor(oracle):
    """a score tensor 4 bytes off a 16-byte boundary: the fused kernel declines it and the three kernels run"""
    from rs_face_detection_b200 import Context, ffi
    heads, _ = synth.make_heads(3, seed=77, n_faces=10)
    ds = SCALES[1:4]
    cfg, ocfg = _cfgs(oracle, 0.7, 0.4)
    c = Context(0, cfg)
    try:
        bufs, ptrs = [], []
        for i, h in enumerate(heads):
            h = np.ascontiguousarray(h)
            b = c.alloc(h.nbytes + 16)
            off = 4 if i == 3 else 0
            ffi._chk(ffi.load().fd_memcpy_h2d(c.handle, C.c_void_p(b.ptr + off), h.ctypes.data_as(C.c_void_p), C.c_size_t(h.nbytes)))
            bufs.append(b)
            ptrs.append(b.ptr + off)
        c.detect_batch(ptrs, 3, ds, 0.7, 0.4)
        st = c.detect_last_stats()
        counts, det, lmk = c.detect_fetch(3)
    finally:
        c.close()
    assert not st["fused"]
    _check_batch(oracle, ocfg, heads, ds, counts, det, lmk, "misaligned")


def test_three_kernel_path_replay(oracle, tmp_path):
    """FD_NO_FUSED=1 in a subprocess: the fused-kernel scenarios and the chosen values through decode / NMS / finalize"""
    path = str(tmp_path / "rows.npz")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "from test_gpu_decode_exact import replay\n"
            "replay(%r); print('ok')\n" % (ROOT, os.path.join(ROOT, "tests"), path))
    env = {k: v for k, v in os.environ.items() if k not in ("FD_NO_FUSED", "FD_FUSED_GENERAL")}
    env["FD_NO_FUSED"] = "1"
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "ok" in res.stdout, res.stderr[-2000:]
    flat = dict(np.load(path))
    assert not any(v for k, v in flat.items() if k.endswith("/fused"))
    _check_replay(oracle, flat, "FD_NO_FUSED")


def test_deferred_images_fresh_and_crowded(oracle):
    """1024 < K <= 4096: deferred on a fresh ctx (rows from finalize after fd_detect_fetch), run by the fused kernel's general
    NMS once the ctx is crowded (an image with more kept faces than its rows hold is still deferred); K > 4096: the big path;
    every anchor above conf 0.02"""
    from rs_face_detection_b200 import Context
    sc = _scenarios()
    cfg, ocfg_c = _cfgs(oracle, 0.2, 0.4)
    c = Context(0, cfg)
    try:
        heads, ds, conf, iou = sc["crowded"][:4]
        fresh = _run(c, heads, ds, conf, iou)
        crowded = _run(c, heads, ds, conf, iou)
        big_heads, big_ds = sc["big"][:2]
        big = _run(c, big_heads, big_ds, 0.05, 0.4)
        dense = synth.make_dense_heads(2, seed=3)
        dense_out = _run(c, dense, SCALES[4:6], 0.02, 0.4)
    finally:
        c.close()
    assert fresh[3]["deferred_images"] > 0 and not fresh[3]["crowded"]
    assert crowded[3]["crowded"] and crowded[3]["deferred_images"] <= fresh[3]["deferred_images"]
    assert big[3]["deferred_images"] > 0 and big[3]["max_candidates"] > 4096
    Ks = _check_batch(oracle, ocfg_c, heads, ds, *fresh[:3], what="fresh")
    assert max(Ks) > 1024 and max(Ks) <= 4096
    _check_batch(oracle, ocfg_c, heads, ds, *crowded[:3], what="crowded")
    _check_batch(oracle, _cfgs(oracle, 0.05, 0.4)[1], big_heads, big_ds, *big[:3], what="big")
    Ks = _check_batch(oracle, _cfgs(oracle, 0.02, 0.4)[1], dense, SCALES[4:6], *dense_out[:3], what="dense")
    assert Ks == [16800, 16800]


def test_other_entry_points(oracle):
    """fd_detect (one image from host arrays), fd_detect_batch_raw, the device rows of fd_detect_view, fd_pipeline_host"""
    from rs_face_detection_b200 import Context, ffi
    cfg, ocfg = _cfgs(oracle, 0.7, 0.4)
    heads, _ = synth.make_heads(3, seed=90, n_faces=12, content_hw=(360, 640))
    ds = SCALES[2:5]
    c = Context(0, cfg)
    try:
        for b in range(3):
            det, lmk = c.detect([h[b] for h in heads], ds[b], 0.7, 0.4)
            check_image(oracle, ocfg, [h[b] for h in heads], ds[b], det, lmk, what="fd_detect %d" % b)
        raw = [np.frombuffer(h.astype("<f4").tobytes(), np.uint8) for h in heads]
        c.detect_batch_raw(raw, [h.shape for h in heads], ds, 0.7, 0.4)
        _check_batch(oracle, ocfg, heads, ds, *c.detect_fetch(3), what="raw")
        crowd, _ = synth.make_heads(2, seed=21, n_faces=60)
        for hh, conf in ((heads, 0.7), (crowd, 0.2)):
            B = hh[0].shape[0]
            devs = [c.to_device(h) for h in hh]
            c.detect_batch(devs, B, ds[:B], conf, 0.4)
            v = c.detect_view()
            offs = np.empty(B + 1, np.int32)
            lib = ffi.load()
            ffi._chk(lib.fd_memcpy_d2h(c.handle, offs.ctypes.data_as(C.c_void_p), C.c_void_p(v.offsets_dev), C.c_size_t(offs.nbytes)))
            n = int(offs[B])
            det, lmk = np.empty((max(n, 1), 5), F), np.empty((max(n, 1), 10), F)
            ffi._chk(lib.fd_memcpy_d2h(c.handle, det.ctypes.data_as(C.c_void_p), C.c_void_p(v.det_dev), C.c_size_t(20 * n)))
            ffi._chk(lib.fd_memcpy_d2h(c.handle, lmk.ctypes.data_as(C.c_void_p), C.c_void_p(v.landmarks_dev), C.c_size_t(40 * n)))
            _check_batch(oracle, _cfgs(oracle, conf, 0.4)[1], hh, ds[:B], np.diff(offs), det[:n], lmk[:n], what="view")
            c.detect_fetch(B)
            for d in devs:
                d.free()
        frames = [synth.make_frame(1080, 1920, 31), synth.make_frame(720, 1280, 32), synth.make_frame(1081, 1923, 33)]
        bufs, total, _, _ = c.pipeline_host(frames, heads, cap_rows=3 * 64, conf_thr=0.7, iou_thr=0.4)
        assert total > 15
        _check_batch(oracle, ocfg, heads, bufs["det_scale"], bufs["counts"], bufs["det"][:total], bufs["lmk"][:total], what="pipeline_host")
    finally:
        c.close()


def _geometry(image_wh, strides, A):
    base = np.zeros((len(strides), A, 4), F)
    for i, st in enumerate(strides):
        for a in range(A):
            half = st * (a + 1) * 1.5
            base[i, a] = [-half + st / 2, -half + st / 2, half + st / 2 - 1, half + st / 2 - 1]
    return image_wh, strides, base


@pytest.mark.parametrize("image_wh,strides,A", [((480, 320), (16, 8), 1), ((640, 640), (32, 16, 8), 3), ((328, 328), (8,), 2)])
def test_other_detector_geometries(oracle, image_wh, strides, A):
    from rs_face_detection_b200 import Context
    geo = _geometry(image_wh, strides, A)
    cfg, ocfg = _cfgs(oracle, 0.7, 0.4, geometry=geo)
    rng = np.random.default_rng(image_wh[0] + A)
    heads = []
    for st in strides:
        fh, fw = (image_wh[1] + st - 1) // st, (image_wh[0] + st - 1) // st
        fg = rng.uniform(0, 0.6, (3, A, fh, fw)).astype(F)
        hot = rng.uniform(0, 1, fg.shape) < 0.02
        fg[hot] = rng.uniform(0.7, 0.999, int(hot.sum())).astype(F)
        heads += [np.ascontiguousarray(np.concatenate([1 - fg, fg], 1)), rng.normal(0, 0.3, (3, 4 * A, fh, fw)).astype(F),
                  rng.normal(0, 0.3, (3, 10 * A, fh, fw)).astype(F)]
    c = Context(0, cfg)
    try:
        counts, det, lmk, st = _run(c, heads, SCALES[[3, 2, 5]], 0.7, 0.4)
    finally:
        c.close()
    Ks = _check_batch(oracle, ocfg, heads, SCALES[[3, 2, 5]], counts, det, lmk, "geometry")
    assert min(Ks) > 5 and counts.sum() > 0


def _op_boxes(values):
    """one box per value whose width w = 2^k makes exp(value) * w land in [0.5, 2) where it can, centred on 0 (dx = 0) or,
    past 2^23, at w / 2 with dx = -0.5: x2 = (pw - 1) / 2 then holds every bit of the exp"""
    boxes, dx = [], []
    for v in values:
        k = int(np.clip(np.round(-v / np.log(2)), 0, 126)) if np.isfinite(v) else 0
        if k <= 23:
            r = (2.0 ** k - 1) / 2
            boxes.append([-r, -r, r, r])
            dx.append(0.0)
        else:
            boxes.append([0, 0, 2.0 ** k, 2.0 ** k])
            dx.append(-0.5)
    return np.array(boxes, F), np.array(dx, F)


def test_standalone_box_ops_bitwise(ctx):
    """fd_bbox_pred / fd_nonlinear_pred against the exp32_cr restatement on the chosen values and on random deltas;
    fd_nonlinear_transform against the log32_cr restatement"""
    values = np.array(chosen_values(), F)
    b, dx = _op_boxes(values)
    d = np.zeros((len(values), 8), F)
    d[:, 0], d[:, 1], d[:, 2], d[:, 3] = dx, dx, values, values[::-1]
    d[:, 4:] = np.random.default_rng(1).normal(0, 0.4, (len(values), 4))
    d[:, 6] = values[::-1]
    for fn, all_groups in ((ctx.bbox_pred, False), (ctx.nonlinear_pred, True)):
        assert_bitwise(fn(b, d), pred_ref(b, d, all_groups), "chosen %s" % all_groups)
    w = box_geom(b)[0]
    vis = np.isfinite(values) & (exp32_cr(values) * w >= 0.5) & (exp32_cr(values) * w < 2 ** 24)
    assert vis[:7].all()        # every near-midpoint exp shows in x2 to its last bit
    got = ctx.nonlinear_pred(b, d)
    assert_bitwise(got[vis, 2], (F(0.5) * (exp32_cr(values[vis]) * w[vis] - F(1))).astype(F))
    rng = np.random.default_rng(0)
    n = 5000
    x, y = rng.uniform(-50, 600, n), rng.uniform(-50, 600, n)
    rb = np.stack([x, y, x + rng.uniform(1, 300, n), y + rng.uniform(1, 300, n)], 1).astype(F)
    rd = rng.normal(0, 0.4, (n, 8)).astype(F)
    assert_bitwise(ctx.bbox_pred(rb, rd), pred_ref(rb, rd, False), "bbox_pred")
    assert_bitwise(ctx.nonlinear_pred(rb, rd), pred_ref(rb, rd, True), "nonlinear_pred")
    g = np.stack([x + rng.normal(0, 5, n), y + rng.normal(0, 5, n), rb[:, 2] + rng.normal(0, 20, n), rb[:, 3] + rng.normal(0, 20, n)], 1).astype(F)
    g[:7] = [[0, 0, -1, -1], [0, 0, -2, 5], [0, 0, 1e30, 1e-30], [0, 0, 1e-30, 1e30], [0, 0, np.inf, np.nan], [0, 0, 0, 0], [5, 5, 4, 4]]
    assert_bitwise(ctx.nonlinear_transform(rb, g), nonlinear_transform_ref(rb, g), "nonlinear_transform")
