"""Reference for the detection rows (boxes, scores, landmarks) and the bitwise check every detect test uses.

The detector's decode is written to be bit-exact: every operation rounded separately in the reference's order, no
contraction.  Two things can still make a GPU row differ from the oracle's:

- nothing, for the landmarks and the scores: no transcendental touches them, so they must equal the oracle's bit for bit;
- the box exp.  The oracle computes `expf(dw) * w` with the platform's libm, which is not correctly rounded (glibc 2.39
  misrounds about 7 in 100 000 floats of [-20, 20], and picks its variant per CPU).  The kernels round exp correctly, so
  the boxes are compared bit for bit with a numpy restatement that uses a correctly rounded exp (`exp32_cr`), and may
  differ from the oracle's only on rows whose `dw` or `dh` is one of the inputs libm's `expf` misrounds.

"Bitwise" compares `.view(np.uint32)`, so a sign-of-zero change fails; a NaN equals any NaN (the payload of a NaN is
not part of what the reference defines).
"""
import ctypes
import ctypes.util

import numpy as np

F = np.float32
_ULPS = 4          # float64 results this many double ulps from a float32 rounding midpoint are settled with mpmath


def _round_cr(x, fn64, fn_mp):
    """float32(fn(x)) correctly rounded: the float64 result rounded to float32, except where it lies within _ULPS double ulps
    of a float32 midpoint, where the exact value (mpmath, 200 bits) decides the side"""
    shape = np.shape(x)
    x = np.asarray(x, F).ravel()
    with np.errstate(all="ignore"):
        y = fn64(x.astype(np.float64))
        r = y.astype(F)
        r64 = r.astype(np.float64)
        toward = np.where(y > r64, np.nextafter(r, F(np.inf)), np.nextafter(r, F(-np.inf))).astype(np.float64)
        mid = np.where(np.isinf(r) & np.isfinite(y), np.sign(y) * (2.0 ** 128 - 2.0 ** 103), (r64 + toward) / 2)
        near = np.isfinite(y) & (np.abs(y - mid) <= _ULPS * np.spacing(np.abs(y)))
    if not near.any():
        return r.reshape(shape)
    import mpmath
    out = r.copy()
    with mpmath.workprec(200):
        for i in np.nonzero(near)[0]:
            exact = fn_mp(mpmath.mpf(float(x[i])))
            lo, hi = sorted((float(r64[i]), float(toward[i])))
            out[i] = F(hi) if exact > mpmath.mpf(float(mid[i])) else F(lo)
    return out.reshape(shape)


def exp32_cr(x):
    """float32 exp, correctly rounded (round to nearest even), elementwise"""
    import mpmath
    return _round_cr(x, np.exp, mpmath.exp)


def log32_cr(x):
    """float32 natural log, correctly rounded, elementwise (log 0 = -inf, log of a negative number = NaN)"""
    import mpmath
    return _round_cr(x, np.log, mpmath.log)


_libm = None


def libm_expf(x):
    """the oracle's expf: the same libm the oracle links, through ctypes (one call per value)"""
    global _libm
    if _libm is None:
        _libm = ctypes.CDLL(ctypes.util.find_library("m"))
        _libm.expf.restype = ctypes.c_float
        _libm.expf.argtypes = [ctypes.c_float]
    return F(_libm.expf(float(F(x))))


def _same(a, b):
    """bitwise equality, elementwise; NaN equals NaN"""
    a, b = np.asarray(a, F), np.asarray(b, F)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def _cfg_fields(cfg):
    strides = [int(cfg.strides[s]) for s in range(cfg.n_strides)]
    A = int(cfg.num_anchors)
    base = np.array(cfg.base_anchors[:], F).reshape(8, 4, 4)[:len(strides), :A]
    return strides, A, base, np.array(cfg.bbox_stds[:], F), F(cfg.landmark_std), int(cfg.image_w), int(cfg.image_h)


def box_pred(w, h, cx, cy, d, exp=exp32_cr):
    """bbox_pred on the anchor (or box) geometry, in the reference's order (face_detection.rs:516-549)"""
    pcx = ((d[:, 0] * w).astype(F) + cx).astype(F)
    pcy = ((d[:, 1] * h).astype(F) + cy).astype(F)
    pw = (exp(d[:, 2]) * w).astype(F)
    ph = (exp(d[:, 3]) * h).astype(F)
    hx = (F(0.5) * (pw - F(1)).astype(F)).astype(F)
    hy = (F(0.5) * (ph - F(1)).astype(F)).astype(F)
    return np.stack([(pcx - hx).astype(F), (pcy - hy).astype(F), (pcx + hx).astype(F), (pcy + hy).astype(F)], 1)


def box_geom(b):
    """width, height and centre of boxes (x1, y1, x2, y2) as face_detection.rs:522-525 computes them"""
    b = np.asarray(b, F)
    w = ((b[:, 2] - b[:, 0]).astype(F) + F(1)).astype(F)
    h = ((b[:, 3] - b[:, 1]).astype(F) + F(1)).astype(F)
    cx = (b[:, 0] + (F(0.5) * (w - F(1)).astype(F)).astype(F)).astype(F)
    cy = (b[:, 1] + (F(0.5) * (h - F(1)).astype(F)).astype(F)).astype(F)
    return w, h, cx, cy


def decode_rows(heads, cfg, det_scale, conf, iou):
    """The post-CNN half (face_detection.rs:319-493) restated in numpy float32 for ONE image: every anchor decoded and
    clipped, `score >= conf` selects, strides stacked in config order, stable descending sort, oracle.nms, rows gathered,
    divided by det_scale.  heads: 3 arrays (scores (2A,H,W), boxes (4A,H,W), landmarks (10A,H,W)) per stride; cfg: an
    oracle DetCfg (geometry, anchors, stds).  -> det (M,5), landmarks (M,5,2), dwh (M,2): each kept row's box deltas
    dw, dh after bbox_stds, i.e. the arguments of its two exps."""
    from oracle import oracle
    strides, A, base, bstd, lstd, img_w, img_h = _cfg_fields(cfg)
    conf, ds = F(conf), F(det_scale)
    boxes, scores, lmks, dwh = [], [], [], []
    for s, stride in enumerate(strides):
        sc, bb, lm = (np.asarray(heads[3 * s + k], F) for k in range(3))
        H, W = bb.shape[-2:]
        sc, bb, lm = sc.reshape(2 * A, H, W), bb.reshape(4 * A, H, W), lm.reshape(10 * A, H, W)
        sw = (np.arange(W) * stride).astype(F)[None, :, None]
        sh = (np.arange(H) * stride).astype(F)[:, None, None]
        an = np.empty((H, W, A, 4), F)
        an[..., 0] = base[s][None, None, :, 0] + sw
        an[..., 1] = base[s][None, None, :, 1] + sh
        an[..., 2] = base[s][None, None, :, 2] + sw
        an[..., 3] = base[s][None, None, :, 3] + sh
        w, h, cx, cy = box_geom(an.reshape(-1, 4))
        fg = sc[A:].transpose(1, 2, 0).reshape(-1)                                  # (H,W,A) order
        sel = np.nonzero(fg >= conf)[0]
        d = (bb.reshape(A, 4, H, W).transpose(2, 3, 0, 1).reshape(-1, 4)[sel] * bstd).astype(F)
        ld = (lm.reshape(A, 10, H, W).transpose(2, 3, 0, 1).reshape(-1, 5, 2)[sel] * lstd).astype(F)
        w, h, cx, cy = w[sel], h[sel], cx[sel], cy[sel]
        with np.errstate(all="ignore"):
            box = box_pred(w, h, cx, cy, d)
            box[:, 0::2] = np.fmax(np.fmin(box[:, 0::2], F(img_w - 1)), F(0))       # fminf / fmaxf: a NaN side is clipped
            box[:, 1::2] = np.fmax(np.fmin(box[:, 1::2], F(img_h - 1)), F(0))
            l = np.empty_like(ld)
            l[:, :, 0] = ((ld[:, :, 0] * w[:, None]).astype(F) + cx[:, None]).astype(F)
            l[:, :, 1] = ((ld[:, :, 1] * h[:, None]).astype(F) + cy[:, None]).astype(F)
        boxes.append(box), scores.append(fg[sel]), lmks.append(l), dwh.append(d[:, 2:4])
    box, sc, lm, dwh = (np.concatenate(v) for v in (boxes, scores, lmks, dwh))
    if len(box) == 0:
        return np.zeros((0, 5), F), np.zeros((0, 5, 2), F), np.zeros((0, 2), F)
    order = np.argsort(-sc.astype(np.float64), kind="stable")
    pre = np.concatenate([box[order], sc[order, None]], 1).astype(F)
    keep = oracle.nms(pre, F(iou))
    det = pre[keep].copy()
    with np.errstate(all="ignore"):
        det[:, :4] = (det[:, :4] / ds).astype(F)
        lmk = (lm[order][keep] / ds).astype(F)
    return det, lmk, dwh[order][keep].copy()


def assert_rows_exact(got_det, got_lmk, oracle_rows, ref_rows, what=""):
    """The check of one image's detection rows.  oracle_rows: (det, landmarks) from oracle.detect_post; ref_rows: the
    result of decode_rows.  Row count and scores equal; landmarks bitwise equal to the oracle's; boxes bitwise equal to
    the restatement's, and different from the oracle's only on rows where libm's expf misrounds dw or dh."""
    edet, elmk = (np.asarray(a, F) for a in oracle_rows[:2])
    rdet, rlmk, dwh = ref_rows
    got_det, got_lmk = np.asarray(got_det, F).reshape(-1, 5), np.asarray(got_lmk, F).reshape(-1, 10)
    edet, elmk, rlmk = edet.reshape(-1, 5), elmk.reshape(-1, 10), np.asarray(rlmk, F).reshape(-1, 10)
    assert len(got_det) == len(got_lmk) == len(edet) == len(rdet), ("row count", what, len(got_det), len(edet), len(rdet))
    assert _same(rdet[:, 4], edet[:, 4]).all(), ("the restatement's scores differ from the oracle's", what)
    assert _same(rlmk, elmk).all(), ("the restatement's landmarks differ from the oracle's", what)
    bad = np.nonzero(~_same(got_det[:, 4], edet[:, 4]))[0]
    assert len(bad) == 0, ("score", what, bad[:5], got_det[bad[:5], 4], edet[bad[:5], 4])
    bad = np.nonzero(~_same(got_lmk, elmk).all(1))[0]
    assert len(bad) == 0, ("landmarks differ from the oracle's", what, bad[:5], got_lmk[bad[:1]], elmk[bad[:1]])
    bad = np.nonzero(~_same(got_det[:, :4], rdet[:, :4]).all(1))[0]
    assert len(bad) == 0, ("boxes differ from the correctly rounded restatement", what, bad[:5], got_det[bad[:1]], rdet[bad[:1]],
                           dwh[bad[:1]])
    for i in np.nonzero(~_same(rdet[:, :4], edet[:, :4]).all(1))[0]:
        dw, dh = dwh[i]
        assert not (_same(libm_expf(dw), exp32_cr(dw)) and _same(libm_expf(dh), exp32_cr(dh))), \
            ("box differs from the oracle's on a row libm's expf rounds correctly", what, i, rdet[i], edet[i], dwh[i])


def pred_ref(boxes, deltas, all_groups):
    """fd_nonlinear_pred (all_groups) / fd_bbox_pred (first 4 columns regressed, the rest copied) with exp32_cr"""
    boxes, deltas = np.asarray(boxes, F), np.asarray(deltas, F)
    w, h, cx, cy = box_geom(boxes)
    out = np.zeros_like(deltas) if all_groups else deltas.copy()
    with np.errstate(all="ignore"):
        for j in range(0, deltas.shape[1] - 3, 4) if all_groups else (0,):
            out[:, j:j + 4] = box_pred(w, h, cx, cy, deltas[:, j:j + 4])
    return out


def nonlinear_transform_ref(ex, gt):
    """fd_nonlinear_transform (bbox_transform.rs:67-88) with log32_cr"""
    ew, eh, ecx, ecy = box_geom(ex)
    gw, gh, gcx, gcy = box_geom(gt)
    with np.errstate(all="ignore"):
        return np.stack([((gcx - ecx).astype(F) / (ew + F(1e-14)).astype(F)).astype(F),
                         ((gcy - ecy).astype(F) / (eh + F(1e-14)).astype(F)).astype(F),
                         log32_cr((gw / ew).astype(F)), log32_cr((gh / eh).astype(F))], 1)


def assert_bitwise(got, want, what=""):
    """bitwise equality (NaN equals NaN), reporting the first differing elements"""
    got, want = np.asarray(got, F), np.asarray(want, F)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.argwhere(~_same(got, want))
    assert len(bad) == 0, (what, len(bad), [(tuple(i), got[tuple(i)], want[tuple(i)]) for i in bad[:5]])


def check_image(oracle,cfg, heads_b, det_scale, det, lmk, conf=None, iou=None, what=""):
    """assert_rows_exact for one image's rows against oracle.detect_post and decode_rows; returns the oracle's K"""
    conf = cfg.conf_thr if conf is None else conf
    iou = cfg.iou_thr if iou is None else iou
    edet, elmk, K = oracle.detect_post(cfg, heads_b, det_scale)
    assert_rows_exact(det, lmk, (edet, elmk), decode_rows(heads_b, cfg, det_scale, conf, iou), what)
    return K
