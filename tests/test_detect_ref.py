"""The detection-row reference (tests/detect_ref.py) against the oracle, on the CPU: decode_rows must give the oracle's rows,
scores and landmarks bit for bit and boxes except where libm's expf misrounds; exp32_cr and log32_cr must be correctly
rounded where a float64 evaluation alone cannot tell."""
import numpy as np
import pytest

from detect_ref import (F, assert_bitwise, assert_rows_exact, decode_rows, exp32_cr, libm_expf, log32_cr, nonlinear_transform_ref,
                        pred_ref)
from rs_face_detection_b200.utils import synth

# the floats whose float64 exp lies within 4 double ulps of a float32 rounding midpoint, over the whole domain [-104, 89]
NEAR_MIDPOINT = [float.fromhex(s) for s in ("0x1.fdff02p-17", "0x1.cd3982p-14", "0x1.8d7cb6p-12", "-0x1p-25", "-0x1.c1c4b8p-10",
                                            "-0x1.e1dbe2p-8", "-0x1.d2259ap+3")]
SCALES = (1.0, 0.5, 0.33333334, 0.59259259, 2.0, 0.1)


def _mp_round(x, fn):
    """float32 nearest to fn(x), from a 200-bit evaluation and the two float32 neighbours of its float64 rounding"""
    import mpmath
    with mpmath.workprec(200):
        v = fn(mpmath.mpf(float(F(x))))
        with np.errstate(over="ignore"):
            c = F(float(v))
        cands = [np.nextafter(c, F(-np.inf)), c, np.nextafter(c, F(np.inf))]
        return min(cands, key=lambda t: abs(mpmath.mpf(float(t)) - v))


def test_exp32_cr_at_the_near_midpoint_inputs():
    import mpmath
    x = np.array(NEAR_MIDPOINT, F)
    got = exp32_cr(x)
    for xi, gi in zip(x, got):
        assert gi.view(np.uint32) == _mp_round(xi, mpmath.exp).view(np.uint32), float(xi).hex()
    # each of them really is a hard case: the float64 result lies within a few double ulps of a float32 midpoint
    y = np.exp(x.astype(np.float64))
    r = y.astype(F).astype(np.float64)
    other = np.where(y > r, np.nextafter(y.astype(F), F(np.inf)), np.nextafter(y.astype(F), F(-np.inf))).astype(np.float64)
    assert (np.abs(y - (r + other) / 2) <= 4 * np.spacing(y)).all()


def test_exp32_and_log32_against_mpmath_on_a_sample():
    import mpmath
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.uniform(-104, 89, 300), rng.uniform(-1, 1, 300), [0.0, -0.0, 88.72283, 88.72284, -103.97, -87.33655]]).astype(F)
    e = exp32_cr(x)
    for xi, ei in zip(x, e):
        assert ei.view(np.uint32) == _mp_round(xi, mpmath.exp).view(np.uint32) or (np.isinf(ei) and xi > 88), float(xi).hex()
    p = np.concatenate([rng.uniform(1e-3, 3, 300), np.exp(rng.uniform(-80, 80, 300))]).astype(F)
    lg = log32_cr(p)
    for pi, li in zip(p, lg):
        assert li.view(np.uint32) == _mp_round(pi, mpmath.log).view(np.uint32), float(pi).hex()
    assert np.isneginf(log32_cr(np.array([0.0], F)))[0] and np.isnan(log32_cr(np.array([-1.0], F)))[0]
    assert np.isinf(exp32_cr(np.array([np.inf, 89.0], F))).all() and exp32_cr(np.array([-np.inf, -110.0], F)).tolist() == [0.0, 0.0]


@pytest.mark.parametrize("stds,lstd", [((1, 1, 1, 1), 1.0), ((0.1, 0.1, 0.2, 0.2), 0.2)])
@pytest.mark.parametrize("seed,faces,conf", [(21, 12, 0.7), (22, 30, 0.5), (23, 0, 0.7), (24, 6, 0.02)])
def test_decode_rows_against_the_oracle(oracle, stds, lstd, seed, faces, conf):
    heads, _ = synth.make_heads(1, seed=seed, n_faces=faces)
    hb = [h[0] for h in heads]
    cfg = oracle.make_det_cfg(conf_thr=conf, iou_thr=0.4, bbox_stds=stds, landmark_std=lstd)
    for ds in SCALES:
        edet, elmk, K = oracle.detect_post(cfg, hb, ds)
        ref = decode_rows(hb, cfg, ds, conf, 0.4)
        assert_rows_exact(ref[0], ref[1], (edet, elmk), ref, "seed %d ds %r" % (seed, ds))
        assert faces == 0 or len(edet) > 0


def test_decode_rows_other_geometry(oracle):
    """A = 3, two strides, a non-square image: the reference follows the configuration"""
    strides, A, image_wh = (16, 8), 3, (480, 320)
    base = np.zeros((len(strides), A, 4), F)
    for i, st in enumerate(strides):
        for a in range(A):
            half = st * (a + 1) * 1.5
            base[i, a] = [-half + st / 2, -half + st / 2, half + st / 2 - 1, half + st / 2 - 1]
    rng = np.random.default_rng(3)
    heads = []
    for st in strides:
        fh, fw = (image_wh[1] + st - 1) // st, (image_wh[0] + st - 1) // st
        fg = rng.uniform(0, 1, (A, fh, fw)).astype(F)
        heads += [np.concatenate([1 - fg, fg]), rng.normal(0, 0.3, (4 * A, fh, fw)).astype(F), rng.normal(0, 0.3, (10 * A, fh, fw)).astype(F)]
    cfg = oracle.make_det_cfg(conf_thr=0.6, iou_thr=0.4, image_size=image_wh, strides=strides, base_anchors=base,
                              bbox_stds=(0.1, 0.1, 0.2, 0.2), landmark_std=0.2)
    for ds in (1.0, 0.59259259):
        edet, elmk, K = oracle.detect_post(cfg, heads, ds)
        ref = decode_rows(heads, cfg, ds, 0.6, 0.4)
        assert K > 100 and len(edet) > 10
        assert_rows_exact(ref[0], ref[1], (edet, elmk), ref)


def test_libm_expf_differs_from_correct_rounding_only_rarely():
    """the premise of the box rule: libm's expf is the oracle's and may misround, but only on a small fraction of inputs"""
    rng = np.random.default_rng(7)
    x = rng.uniform(-4, 4, 20000).astype(F)
    cr = exp32_cr(x)
    diff = sum(libm_expf(v) != c for v, c in zip(x, cr))
    assert diff <= 20


def test_standalone_restatements_against_the_oracle(oracle):
    """pred_ref / nonlinear_transform_ref against the oracle's bbox_transform functions: equal wherever libm rounds exp / log
    correctly"""
    import ctypes
    import ctypes.util
    rng = np.random.default_rng(8)
    n = 3000
    x1, y1 = rng.uniform(-50, 600, n), rng.uniform(-50, 600, n)
    b = np.stack([x1, y1, x1 + rng.uniform(1, 300, n), y1 + rng.uniform(1, 300, n)], 1).astype(F)
    d = rng.normal(0, 0.4, (n, 8)).astype(F)
    for all_groups, fn in ((False, oracle.bbox_pred), (True, oracle.nonlinear_pred)):
        want, got = pred_ref(b, d, all_groups), fn(b, d)
        ok = exp32_cr(d) == np.array([[libm_expf(v) for v in row] for row in d], F)
        for j in range(0, 8 if all_groups else 4, 4):
            rows = ok[:, j + 2] & ok[:, j + 3]
            assert_bitwise(got[rows, j:j + 4], want[rows, j:j + 4])
        assert_bitwise(got[:, 4:] if not all_groups else got[:, :0], want[:, 4:] if not all_groups else want[:, :0])
    g = np.stack([x1 + rng.normal(0, 5, n), y1 + rng.normal(0, 5, n), b[:, 2] + rng.normal(0, 9, n), b[:, 3] + rng.normal(0, 9, n)], 1).astype(F)
    want, got = nonlinear_transform_ref(b, g), oracle.nonlinear_transform(b, g)
    assert_bitwise(got[:, :2], want[:, :2])
    m = ctypes.CDLL(ctypes.util.find_library("m"))
    m.logf.restype, m.logf.argtypes = ctypes.c_float, [ctypes.c_float]
    w = (g[:, 2] - g[:, 0] + F(1)) / (b[:, 2] - b[:, 0] + F(1))
    ok = np.array([F(m.logf(float(v))) for v in w.astype(F)]) == log32_cr(w.astype(F))
    assert ok.mean() > 0.8             # glibc's logf is within 1 ulp, not correctly rounded: a few percent differ
    assert_bitwise(got[ok, 2], want[ok, 2])
