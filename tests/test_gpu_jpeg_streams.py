"""The GPU JPEG decoder (fd_imdecode / fd_decode_jpeg_batch) against cv2.imdecode on stream layouts other encoders write
(tests/jpeg_streams.py): RGB-tagged streams, rearranged tables and segments, data after EOI, a missing EOI, 1..33 x 1..33
images and libjpeg's largest aspect ratios; through each entropy decoder (one restart interval per thread, self-synchronising
with and without restart markers as boundaries, the host Huffman pass, the host marker scan).  Bytes, never a tolerance."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

import jpeg_streams as J  # noqa: E402
from rs_face_detection_b200.utils import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SAMPLINGS = ("420", "422", "444")
# restart intervals of the three device entropy paths: none (self-synchronising decoder), short (one interval per thread),
# long (self-synchronising decoder with the restart markers as boundaries)
RST_PATHS = (0, 4, 40)
EXTREME = ((65500, 8), (8, 65500), (65500, 17))


def variant_cases(rst):
    """[(id, stream, expected BGR)] of every colour-space and layout variant at this restart interval"""
    img = synth.make_frame(83, 117, 21 + rst)
    out = []
    for ss in SAMPLINGS:
        out += [(n, s, J.decode_cv2(s)) for n, s, _ in J.colour_space_variants(img, ss, rst=rst)]
        out += [(n, s, J.decode_cv2(ref)) for n, s, ref in J.layout_variants(img, ss, rst=rst, seed=rst)]
    return out


def tiny_cases():
    """[(id, stream, expected BGR)]: the 1..33 x 1..33 sweep (4:2:0 / 4:2:2 / 4:4:4, with and without restart markers) and
    an RGB-tagged copy of every stream without them"""
    out = []
    for n, s in J.tiny_streams():
        out.append((n, s, J.decode_cv2(s)))
        if n.endswith("rst0"):
            r = J.as_rgb(s)
            out.append((n + "-rgb", r, J.decode_cv2(r)))
    return out


def rst_of(name):
    return int(re.search(r"-rst(\d+)", name).group(1))


def selfsync(name):
    """the default paths: streams without restart markers or with long intervals take the self-synchronising decoder"""
    r = rst_of(name)
    return r == 0 or r >= 32


def read_frame(ctx, fr):
    """a device frame of decode_jpeg_batch, read back at its pitch -> (h, w, 3)"""
    rows = np.empty((fr.height, fr.pitch), np.uint8)
    ctx.lib.fd_memcpy_d2h(ctx.handle, rows.ctypes.data_as(C.c_void_p), C.c_void_p(fr.data), C.c_size_t(rows.nbytes))
    return rows[:, :fr.width * 3].reshape(fr.height, fr.width, 3)


def check_batch(ctx, cases, n_threads=2):
    """decodes the streams of `cases` in one decode_jpeg_batch call; every frame equal to its expected BGR"""
    frames = ctx.decode_jpeg_batch([np.frombuffer(s, np.uint8) for _, s, _ in cases], n_threads=n_threads)
    ctx.synchronize()
    stats = ctx.jpeg_last_stats()
    for fr, (name, _, want) in zip(frames, cases):
        np.testing.assert_array_equal(read_frame(ctx, fr), want, err_msg=name)
    return stats


def check_all_paths(ctx, switch):
    """every variant and the tiny sweep in batches, with the entropy path each batch must take under `switch` (None, or the
    environment switch this process was started with)"""
    groups = [("rst%d" % r, variant_cases(r), r) for r in RST_PATHS]
    tiny = tiny_cases()
    groups += [("tiny-rst%d" % r, [c for c in tiny if rst_of(c[0]) == r], r) for r in (0, 1)]
    for name, cases, rst in groups:
        for b0 in range(0, len(cases), 1200):
            part = cases[b0:b0 + 1200]
            st = check_batch(ctx, part)
            B = len(part)
            if switch == "FD_JPEG_HOST_HUFFMAN":
                assert st["host_entropy_images"] == B, (name, st)
            elif switch == "FD_JPEG_RST_SYNC_MIN":          # every restart interval is a boundary of the self-synchronising chain
                assert st["selfsync_images"] == B and st["host_entropy_images"] == 0, (name, st)
            else:                                           # default, or the host locates the restart markers
                assert st["device_entropy_images"] == B and st["host_entropy_images"] == 0, (name, st)
                assert st["selfsync_images"] == sum(selfsync(n) for n, _, _ in part), (name, st)


@pytest.fixture(scope="module")
def tiny():
    return tiny_cases()


@pytest.fixture(scope="module")
def variants():
    return {r: variant_cases(r) for r in RST_PATHS}


@pytest.mark.parametrize("rst", RST_PATHS)
def test_variants_through_imdecode(ctx, variants, rst):
    for name, s, want in variants[rst]:
        np.testing.assert_array_equal(ctx.imdecode(s), want, err_msg=name)
        st = ctx.jpeg_last_stats()
        assert st["device_entropy_images"] == 1 and st["selfsync_images"] == selfsync(name), (name, st)


def test_variants_mixed_in_one_batch(ctx, variants, tiny):
    """all variants of all three entropy paths, 4:2:0 / 4:2:2 / 4:4:4, RGB and YCbCr, and tiny images in one call"""
    cases = [c for r in RST_PATHS for c in variants[r]] + tiny[::37]
    rng = np.random.default_rng(5)
    cases = [cases[i] for i in rng.permutation(len(cases))]
    st = check_batch(ctx, cases, n_threads=3)
    assert st["device_entropy_images"] == len(cases) and st["host_entropy_images"] == 0, st
    assert st["selfsync_images"] == sum(selfsync(n) for n, _, _ in cases), st


def test_tiny_sizes(ctx, tiny):
    for b0 in range(0, len(tiny), 1500):
        part = tiny[b0:b0 + 1500]
        st = check_batch(ctx, part)
        assert st["device_entropy_images"] == len(part), st
    for name, s, want in tiny[::11]:                              # exact-size grids of the single-image call
        np.testing.assert_array_equal(ctx.imdecode(s), want, err_msg=name)


def test_extreme_aspect_ratios(ctx):
    """libjpeg's 65 500 limit: one image row per grid row of jpeg_color_kernel, near the grid's y limit"""
    cases = []
    for h, w in EXTREME:
        img = synth.make_frame(h, w, h + w)
        for rst in RST_PATHS:
            s = J.encode(img, "420", 90, rst)
            cases.append(("%dx%d-rst%d" % (h, w, rst), s, J.decode_cv2(s)))
        r = J.as_rgb(J.encode(img, "420", 90))
        cases.append(("%dx%d-rgb" % (h, w), r, J.decode_cv2(r)))
    for name, s, want in cases:
        np.testing.assert_array_equal(ctx.imdecode(s), want, err_msg=name)
    check_batch(ctx, cases)


def test_out_of_scope_streams_are_errors_and_the_context_keeps_decoding(ctx):
    from rs_face_detection_b200 import FdError
    img = synth.make_frame(64, 96, 13)
    good = J.as_rgb(J.encode(img, "422", 90, 4))
    want = J.decode_cv2(good)
    for name, bad in J.error_streams(img):
        with pytest.raises(FdError):
            ctx.imdecode(bad)
            pytest.fail(name)
        np.testing.assert_array_equal(ctx.imdecode(good), want, err_msg=name)
        with pytest.raises(FdError):
            ctx.decode_jpeg_batch([good, bad])
            pytest.fail(name)
        assert check_batch(ctx, [(name, good, want)])["device_entropy_images"] == 1


def test_pipeline_host_jpeg_with_an_rgb_tagged_stream(ctx):
    """fd_pipeline_host_jpeg on an RGB-tagged stream next to ordinary ones == fd_pipeline_host on cv2.imdecode of the bytes"""
    B = 3
    frames = [synth.make_frame(720, 1280, 2700 + i) for i in range(B)]
    streams = [J.encode(frames[0], "420", 88), J.as_rgb(J.encode(frames[1], "420", 88)), J.encode(frames[2], "444", 85, rst=8)]
    arrays = [np.frombuffer(s, np.uint8).copy() for s in streams]
    decoded = [J.decode_cv2(s) for s in streams]
    heads, _ = synth.make_heads(B, seed=3500, n_faces=8, content_hw=(360, 640))
    ref, total, _, _ = ctx.pipeline_host(decoded, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, want_tensor=True)
    got, total2, _, _ = ctx.pipeline_host(arrays, heads, cap_rows=B * 64, conf_thr=0.7, iou_thr=0.4, want_tensor=True, jpeg=True, jpeg_threads=2)
    assert total2 == total > 0
    for k in ("counts", "tensor", "det_scale"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
    for k in ("det", "lmk", "crops", "align_mode"):
        np.testing.assert_array_equal(got[k][:total], ref[k][:total], err_msg=k)


@pytest.mark.parametrize("switch", ["FD_JPEG_HOST_HUFFMAN", "FD_JPEG_RST_SYNC_MIN", "FD_JPEG_HOST_MARKER_SCAN"])
def test_every_variant_under_each_decoder_switch(switch):
    """the switches are read once per process: one process each, all variants and the tiny sweep"""
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_jpeg_streams as T\n"
            "from rs_face_detection_b200 import Context\n"
            "c = Context(0)\n"
            "T.check_all_paths(c, %r)\n"
            "c.close()\n"
            "print('ok')\n" % (ROOT, HERE, switch))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **{switch: "1"}), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-3000:]


def test_every_variant_default_paths(ctx):
    check_all_paths(ctx, None)
