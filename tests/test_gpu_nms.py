"""NMS parity (bit-exact keep lists) through the C ABI vs the oracle restatement of processing/nms.rs."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu


def _random_dets(n, seed, canvas=640, side=(8, 120), quant=None, score_levels=None):
    rng = np.random.default_rng(seed)
    s = rng.uniform(*side, n)
    x = rng.uniform(0, canvas, n)
    y = rng.uniform(0, canvas, n)
    sc = rng.uniform(0.02, 1, n)
    if score_levels:
        sc = np.round(sc * score_levels) / score_levels      # many exact ties -> stable ordering matters
    d = np.stack([x, y, x + s, y + s * rng.uniform(0.7, 1.3, n), sc], 1).astype(np.float32)
    if quant:
        d[:, :4] = np.round(d[:, :4] / quant) * quant          # IoUs land exactly on thresholds more often
    return d


def test_reference_vectors(ctx, oracle):
    dets = np.array([[100, 100, 210, 210, 0.72], [250, 250, 420, 420, 0.8], [220, 220, 320, 330, 0.92],
                     [100, 100, 210, 210, 0.6]], np.float32)          # nms.rs:76-83
    assert ctx.nms(dets, 0.4).tolist() == [2, 1, 0]
    assert ctx.cpu_nms(dets, 0.3).tolist() == [2, 1, 0]               # cpu_nms.rs:65-72
    from rs_face_detection_b200.processing.nms import nms
    from rs_face_detection_b200.rcnn.gpu_nms import gpu_nms
    assert nms(dets, 0.4, ctx).tolist() == [2, 1, 0]
    assert gpu_nms(dets, 0.3).tolist() == [2, 1, 0]                   # gpu_nms.rs test, via the literal `_nms` symbol


@pytest.mark.parametrize("n", [0, 1, 2, 63, 64, 65, 127, 1000, 1023, 1024, 1025, 2048, 4095, 4096])
def test_small_path_sizes(ctx, oracle, n):
    dets = _random_dets(n, 100 + n)
    for thr in (0.4, 0.45):
        np.testing.assert_array_equal(ctx.nms(dets, thr), oracle.nms(dets, thr))


@pytest.mark.parametrize("n", [4097, 5000, 16800, 100000])
def test_big_path_sizes(ctx, oracle, n):
    dets = _random_dets(n, 7 + n, canvas=2000, side=(8, 64))
    np.testing.assert_array_equal(ctx.nms(dets, 0.4), oracle.nms(dets, 0.4))


@pytest.mark.parametrize("n", [1025, 2561, 4096, 8192, 12287, 12288, 12289])
def test_mid_path_sizes(ctx, oracle, n):
    """A single problem of a few thousand boxes: rank sort + brute-force predecessor lists over all SMs (fd_nms.cu, mid path)."""
    dets = _random_dets(n, 31 + n, canvas=1200, side=(8, 90), score_levels=500)       # ties: the rank sort must be stable
    for thr in (0.4, 0.3):
        np.testing.assert_array_equal(ctx.nms(dets, thr), oracle.nms(dets, thr))
    np.testing.assert_array_equal(ctx.cpu_nms(dets, 0.4), oracle.cpu_nms(dets, 0.4))


def test_mid_path_crowded_clusters_overflow_the_lists(ctx, oracle):
    """300 jittered candidates per face: most boxes have more predecessors than a list holds (96) and rescan every earlier box."""
    dets = synth.make_crowd_boxes(6000, seed=9, n_faces=20)
    got, exp = ctx.nms(dets, 0.4), oracle.nms(dets, 0.4)
    np.testing.assert_array_equal(got, exp)
    n = 5000                                                   # chain: box i overlaps only i-1 -> worst-case decision depth
    x = np.arange(n, dtype=np.float32) * 6
    chain = np.stack([x, np.zeros(n, np.float32), x + 10, np.full(n, 10, np.float32), np.linspace(0.99, 0.01, n, dtype=np.float32)], 1)
    np.testing.assert_array_equal(ctx.nms(chain, 0.2), oracle.nms(chain, 0.2))


def test_dense_crowd_c3(ctx, oracle):
    """BASELINE config 3: ~100k candidates, 5000 faces x 20 jittered boxes, 1% duplicated scores."""
    dets = synth.make_crowd_boxes(100000, seed=42)
    got, exp = ctx.nms(dets, 0.4), oracle.nms(dets, 0.4)
    np.testing.assert_array_equal(got, exp)
    assert 3000 < len(got) < 30000


def test_many_kept_boxes(ctx, oracle):
    """Sparse boxes: almost everything is kept (> 16 384), so the one-launch path orders its kept keys with the radix passes
    (index bits, then score bits) instead of all-pairs counting; quantised scores make the index tie-break matter."""
    dets = _random_dets(40000, 123, canvas=9000, side=(8, 60), score_levels=500)
    got, exp = ctx.nms(dets, 0.4), oracle.nms(dets, 0.4)
    assert len(exp) > 20000
    np.testing.assert_array_equal(got, exp)
    order = oracle.argsort_descending(dets[:, 4])
    srt = np.ascontiguousarray(dets[order])
    np.testing.assert_array_equal(ctx.nms_sorted(srt, 0.4), oracle.nms_sorted(srt, 0.4))


@pytest.mark.parametrize("n,levels", [(500, 10), (3000, 50), (20000, 100)])
def test_ties_and_quantised_boxes(ctx, oracle, n, levels):
    dets = _random_dets(n, 11 + n, canvas=400, quant=4.0, score_levels=levels)
    for thr in (0.25, 0.4, 0.5):
        np.testing.assert_array_equal(ctx.nms(dets, thr), oracle.nms(dets, thr))
        np.testing.assert_array_equal(ctx.cpu_nms(dets, thr), oracle.cpu_nms(dets, thr))


def test_all_identical_and_all_disjoint(ctx, oracle):
    same = np.tile(np.array([[10, 10, 50, 50, 0.5]], np.float32), (3000, 1))
    assert ctx.nms(same, 0.4).tolist() == [0]
    g = np.arange(70, dtype=np.float32)
    xs, ys = np.meshgrid(g * 20, g * 20)
    dis = np.stack([xs.ravel(), ys.ravel(), xs.ravel() + 10, ys.ravel() + 10, np.linspace(0.1, 0.9, 4900, dtype=np.float32)], 1)
    np.testing.assert_array_equal(ctx.nms(dis, 0.4), oracle.nms(dis, 0.4))
    assert len(ctx.nms(dis, 0.4)) == 4900


def test_chain_dependency(ctx, oracle):
    """box i overlaps only i-1: the keep set alternates and the parallel rounds need their worst-case depth."""
    n = 1500
    x = np.arange(n, dtype=np.float32) * 6
    dets = np.stack([x, np.zeros(n, np.float32), x + 10, np.full(n, 10, np.float32), np.linspace(0.99, 0.01, n, dtype=np.float32)], 1)
    np.testing.assert_array_equal(ctx.nms(dets, 0.2), oracle.nms(dets, 0.2))


def test_degenerate_boxes_and_thresholds(ctx, oracle):
    rng = np.random.default_rng(5)
    dets = _random_dets(600, 77)
    dets[::7, 2] = dets[::7, 0] - 1.0          # zero width  -> area 0 -> 0/0 = NaN overlap -> box removed (nms.rs:58 `<=`)
    dets[::11, 3] = dets[::11, 1] - 5.0        # negative height
    for thr in (0.4, 0.0, -0.1, 1.0, 1.5):
        np.testing.assert_array_equal(ctx.nms(dets, thr), oracle.nms(dets, thr))
        np.testing.assert_array_equal(ctx.cpu_nms(dets, thr), oracle.cpu_nms(dets, thr))
    big = _random_dets(6000, 78, canvas=900)
    big[::13, 2] = big[::13, 0] - 1.0
    np.testing.assert_array_equal(ctx.nms(big, 0.4), oracle.nms(big, 0.4))
    np.testing.assert_array_equal(ctx.nms(big, -1.0), oracle.nms(big, -1.0))


def test_nan_score_is_an_error(ctx):
    from rs_face_detection_b200 import FdError, ffi
    dets = _random_dets(100, 1)
    dets[5, 4] = np.nan
    with pytest.raises(FdError) as e:
        ctx.nms(dets, 0.4)
    assert e.value.code == ffi.FD_ERR_NAN_SCORE
    dets = _random_dets(9000, 2)
    dets[5, 4] = np.nan
    with pytest.raises(FdError):
        ctx.nms(dets, 0.4)


@pytest.mark.parametrize("n", [10, 3000, 50000])
def test_nms_sorted_contract(ctx, oracle, n):
    """`_nms` contract (gpu_nms.hpp:6-8): boxes pre-sorted; keep indexes the sorted array."""
    dets = _random_dets(n, 31 + n, canvas=1500)
    order = oracle.argsort_descending(dets[:, 4])
    srt = np.ascontiguousarray(dets[order])
    np.testing.assert_array_equal(ctx.nms_sorted(srt, 0.4), oracle.nms_sorted(srt, 0.4))
    np.testing.assert_array_equal(order[ctx.nms_sorted(srt, 0.4)], oracle.nms(dets, 0.4))
    np.testing.assert_array_equal(ctx.nms_sorted(np.ascontiguousarray(srt[:, :4]), 0.4), oracle.nms_sorted(srt, 0.4))


@pytest.mark.parametrize("n,kind", [pytest.param(n, "quantised", id=str(n)) for n in (1, 77, 4096, 4097, 100000)]
                         + [pytest.param(n, k, id="%d-%s" % (n, k)) for n, k in ((4097, "nan"), (100000, "nan"), (100000, "equal"))])
def test_argsort_descending(ctx, oracle, n, kind):
    """Above 4 096 scores argsort_kernel sorts over the differing score bits: none when every score is equal."""
    from rs_face_detection_b200 import FdError, ffi
    rng = np.random.default_rng(n)
    s = (np.round(rng.uniform(0, 1, n) * 1000) / 1000).astype(np.float32)
    s[::17] = -s[::17]
    if kind == "equal":
        s[:] = np.float32(0.375)
    if kind == "nan":
        s[n // 3] = np.nan
        with pytest.raises(FdError) as e:
            ctx.argsort_descending(s)
        assert e.value.code == ffi.FD_ERR_NAN_SCORE
        return
    np.testing.assert_array_equal(ctx.argsort_descending(s), oracle.argsort_descending(s))


def reference_cuda_nms(srt, thresh):
    """Keep list of the reference's own CUDA NMS (`_nms`, src/nms_kernel.cu) on score-sorted boxes, or None when
    oracle/_ref has not been built from a reference checkout (`make -C oracle ref REF=<checkout>`)."""
    path = os.path.join(ROOT, "oracle", "_ref", "libref_gpu_nms.so")
    if not os.path.exists(path):
        return None
    ref = C.CDLL(path)
    # nms_kernel.cu:91 defines _nms(.., const float*, ..) while gpu_nms.hpp:7 declares float*: the definition is a
    # C++ overload, not the extern "C" symbol, so look the mangled name up.
    import subprocess
    names = [l.split()[-1] for l in subprocess.check_output(["nm", "-D", "--defined-only", path], text=True).splitlines()
             if "_nms" in l and "kernel" not in l]
    assert names, "no _nms symbol in oracle/_ref"
    ref_nms = getattr(ref, names[0])
    srt = np.ascontiguousarray(srt, np.float32)
    keep = np.zeros(len(srt), np.int32)
    num = C.c_int(0)
    ref_nms(keep.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(num), srt.ctypes.data_as(C.POINTER(C.c_float)), len(srt), 5,
            C.c_float(thresh), 0)
    return keep[:num.value]


def test_vs_reference_cuda_nms(ctx):
    """The reference's own (vestigial, never built) CUDA NMS: an A/B cross-check on non-degenerate data, where
    `ovr > thr` == `!(ovr <= thr)`.  Its keep list is stored in tests/golden/ref_nms_golden.npz
    (tests/golden/make_ref_nms_golden.py); when oracle/_ref is built, the stored list is checked against the library too."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_nms_golden.npz"))
    srt, keep, thresh = g["dets_sorted"], g["keep"], float(g["thresh"])
    np.testing.assert_array_equal(ctx.nms_sorted(srt, thresh), keep)
    live = reference_cuda_nms(srt, thresh)
    if live is not None:
        np.testing.assert_array_equal(live, keep)


def test_property_random_small(ctx, oracle):
    hypothesis = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(st.integers(0, 300), st.integers(0, 10 ** 6), st.sampled_from([0.3, 0.4, 0.45, 0.5]), st.sampled_from([None, 2.0, 8.0]))
    def prop(n, seed, thr, quant):
        dets = _random_dets(n, seed, canvas=200, quant=quant, score_levels=20)
        np.testing.assert_array_equal(ctx.nms(dets, thr), oracle.nms(dets, thr))

    prop()


def test_single_cta_and_spatial_paths_behind_the_switches():
    """FD_NMS_CROSS=4096 FD_NMS_MID_CAP=0: the single-CTA general path (what the fused detect kernel runs for crowded images)
    and the spatial path at the sizes the mid path normally takes — same keep lists."""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import numpy as np\n"
            "from rs_face_detection_b200 import Context\n"
            "from oracle import oracle as O\n"
            "from test_gpu_nms import _random_dets\n"
            "O.build(); c = Context(0)\n"
            "for n in (1025, 2048, 4096, 4097, 6000):\n"
            "    d = _random_dets(n, 5 + n, canvas=1200, side=(8, 90), score_levels=300)\n"
            "    np.testing.assert_array_equal(c.nms(d, 0.4), O.nms(d, 0.4))\n"
            "    np.testing.assert_array_equal(c.cpu_nms(d, 0.3), O.cpu_nms(d, 0.3))\n"
            "print('ok')\n" % (ROOT, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, FD_NMS_CROSS="4096", FD_NMS_MID_CAP="0"), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-1500:]


def test_one_launch_big_path_behind_the_switch():
    """FD_NMS_MID_CAP=0 sends every problem above 1 024 boxes through nms_big_kernel (the spatial path as one cooperative launch):
    its sort (0-4 digit passes, several tiles per CTA), the peel fallback for irregular boxes / one-cell grids, the `_nms`
    (presorted) contract, cpu_nms's comparison, the NaN flag."""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import numpy as np\n"
            "from rs_face_detection_b200 import Context, FdError\n"
            "from rs_face_detection_b200.utils import synth\n"
            "from oracle import oracle as O\n"
            "from test_gpu_nms import _random_dets\n"
            "O.build(); c = Context(0)\n"
            "for n in (1025, 5000, 13000, 40000):\n"
            "    d = _random_dets(n, 5 + n, canvas=1500, side=(8, 90), score_levels=300)\n"
            "    np.testing.assert_array_equal(c.nms(d, 0.4), O.nms(d, 0.4))\n"
            "    np.testing.assert_array_equal(c.cpu_nms(d, 0.3), O.cpu_nms(d, 0.3))\n"
            "d = synth.make_crowd_boxes(200000, seed=4, n_faces=10000)\n"          # more tiles than CTAs
            "np.testing.assert_array_equal(c.nms(d, 0.4), O.nms(d, 0.4))\n"
            "d = synth.make_crowd_boxes(30000, seed=9, n_faces=100)\n"           # 300 candidates per face: every list overflows
            "np.testing.assert_array_equal(c.nms(d, 0.4), O.nms(d, 0.4))\n"
            "np.testing.assert_array_equal(c.cpu_nms(d, 0.5), O.cpu_nms(d, 0.5))\n"
            "d = _random_dets(6000, 78, canvas=900); d[::13, 2] = d[::13, 0] - 1.0\n"   # zero-width boxes: not 'fast' -> peel
            "for thr in (0.4, -1.0, 1.5):\n"
            "    np.testing.assert_array_equal(c.nms(d, thr), O.nms(d, thr))\n"
            "same = np.tile(np.array([[10, 10, 50, 50, 0.5]], np.float32), (3000, 1))\n"   # no differing key bit, one grid cell
            "assert c.nms(same, 0.4).tolist() == [0]\n"
            "n = 5000; x = np.arange(n, dtype=np.float32) * 6\n"
            "chain = np.stack([x, np.zeros(n, np.float32), x + 10, np.full(n, 10, np.float32), np.linspace(0.99, 0.01, n, dtype=np.float32)], 1)\n"
            "np.testing.assert_array_equal(c.nms(chain, 0.2), O.nms(chain, 0.2))\n"
            "d = _random_dets(30000, 3, canvas=2000); order = O.argsort_descending(d[:, 4]); srt = np.ascontiguousarray(d[order])\n"
            "np.testing.assert_array_equal(c.nms_sorted(srt, 0.4), O.nms_sorted(srt, 0.4))\n"
            "d = _random_dets(9000, 2); d[5, 4] = np.nan\n"
            "try:\n"
            "    c.nms(d, 0.4); raise SystemExit('NaN score not reported')\n"
            "except FdError:\n"
            "    pass\n"
            "d = _random_dets(9000, 2)\n"
            "np.testing.assert_array_equal(c.nms(d, 0.4), O.nms(d, 0.4))\n"          # the flag of the failed call does not stick
            "print('ok')\n" % (ROOT, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, FD_NMS_MID_CAP="0"), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-1500:]
