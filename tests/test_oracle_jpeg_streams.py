"""The CPU JPEG oracle (oracle/fd_jpeg_oracle.c) against cv2.imdecode on stream layouts other encoders write
(tests/jpeg_streams.py): RGB-tagged streams, rearranged tables and segments, data after EOI, 1..33 x 1..33 images and
libjpeg's largest aspect ratios.  Bit-exact: the oracle is the second pin of the GPU decoder's tests."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

import jpeg_streams as J  # noqa: E402
from rs_face_detection_b200.utils import synth  # noqa: E402

SAMPLINGS = ("420", "422", "444")


def _check(oracle, name, stream, reference=None):
    want = J.decode_cv2(stream if reference is None else reference)
    assert want is not None, "%s: cv2 cannot decode the stream" % name
    got = oracle.jpeg_decode(stream)
    assert got.shape == want.shape, name
    if not np.array_equal(got, want):
        d = np.abs(got.astype(int) - want.astype(int))
        raise AssertionError("%s: %d bytes differ, max %d" % (name, int((d > 0).sum()), int(d.max())))
    return want


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_colour_space_signalling(oracle, sampling):
    img = synth.make_frame(70, 101, 7)
    for rst in (0, 3):
        plain = J.decode_cv2(J.encode(img, sampling, 90, rst))
        for name, s, rgb in J.colour_space_variants(img, sampling, rst=rst):
            want = _check(oracle, name, s)
            # an RGB stream's output is the YCbCr decode with the colour conversion left out, so it differs from it
            assert np.array_equal(want, plain) != rgb, name


def test_rgb_output_is_upsampled_components_reordered(oracle):
    """jdcolor.c's YCbCr -> BGR integer formula applied to the RGB-tagged decode gives back the ordinary decode: 'fancy
    upsampling, then no colour conversion' is the whole rule"""
    img = synth.make_frame(48, 80, 9)
    for sampling in SAMPLINGS:
        s = J.encode(img, sampling, 90)
        comp = oracle.jpeg_decode(J.as_rgb(s)).astype(np.int64)
        y, cb, cr = comp[..., 2], comp[..., 1] - 128, comp[..., 0] - 128
        r = y + ((91881 * cr + 32768) >> 16)
        g = y + ((-22554 * cb + 32768 - 46802 * cr) >> 16)
        b = y + ((116130 * cb + 32768) >> 16)
        np.testing.assert_array_equal(np.clip(np.stack([b, g, r], -1), 0, 255), J.decode_cv2(s), err_msg=sampling)


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_tables_segments_and_stream_end(oracle, sampling):
    img = synth.make_frame(83, 117, 11)
    for rst in (0, 2, 40):
        for name, s, ref in J.layout_variants(img, sampling, rst=rst, seed=rst):
            want = _check(oracle, name, s, ref)
            assert want.shape == img.shape, name          # EXIF orientation is ignored by IMREAD_UNCHANGED


def test_tiny_sizes(oracle):
    for name, s in J.tiny_streams():
        _check(oracle, name, s)
        if name.endswith("rst0"):
            _check(oracle, name + "-rgb", J.as_rgb(s))


def test_extreme_aspect_ratios(oracle):
    for h, w in ((65500, 8), (8, 65500), (65500, 17)):
        img = synth.make_frame(h, w, h + w)
        for rst in (0, 5):
            _check(oracle, "%dx%d-rst%d" % (h, w, rst), J.encode(img, "420", 90, rst))


def test_out_of_scope_streams_are_errors(oracle):
    for name, s in J.error_streams(synth.make_frame(64, 96, 13)):
        with pytest.raises(ValueError):
            oracle.jpeg_decode(s)
            pytest.fail(name)
