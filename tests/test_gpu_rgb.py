"""Interleaved RGB-family frames (RGB24, RGBA, BGRA, GRAY8) through the batched *_rgb calls.

Every *_rgb call must give, byte for byte, what its BGR counterpart gives on cv2.cvtColor(COLOR_RGB2BGR / RGBA2BGR /
BGRA2BGR / GRAY2BGR) of the same frame, in the same ctx (tensor, det_scale, crops, M, modes, selections); the BGR results are
also checked against the CPU oracle on the converted frames (tests/rgb_ref.py restates the conversion and is pinned against
cv2).  The frames live in pitched buffers whose padding, leading and trailing bytes, and the fourth byte of RGBA / BGRA
pixels, are noise: aligned (bulk-copy preprocess, interior warp reads), word-aligned (row-staging preprocess, interior warp
reads for 4-byte pixels) and unaligned (row-staging preprocess, per-tap warp reads for 3- and 4-byte pixels)."""
import numpy as np
import pytest

from rs_face_detection_b200.utils import synth
from rgb_ref import BGRA, BPP, GRAY8, NAMES, RGB24, RGBA, bgr_to_rgb, rgb_to_bgr
from test_gpu_yuv420 import _caller_faces, _heads
from test_gpu_yuv422 import _assert_steps_equal, _planted_heads, _step

pytestmark = pytest.mark.gpu
CONF, IOU = 0.7, 0.4
SIZES = [(1, 1), (3, 5), (361, 645), (1081, 1920), (1080, 1920), (2160, 3840), (1920, 1080), (100, 641)]
LAYOUTS = [RGB24, RGBA, BGRA, GRAY8]
MODES = ("aligned", "word", "unaligned")
CASES = [(l, m) for l in LAYOUTS for m in MODES]


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _pitch(W, bpp, i, mode):
    """(pitch, start offset) of frame i"""
    if mode == "aligned":
        return -(-bpp * W // 64) * 64, 0
    if mode == "word":
        return -(-bpp * W // 4) * 4 + 4, 4
    return bpp * W + 1 + 2 * (i % 2), 1 + i % 3


class RgbFrames:
    """B frames in `layout` in noisy pitched device buffers, and the BGR frames cvtColor makes of them"""

    def __init__(self, torch, ctx, sizes, seed, layout, mode="aligned", alpha="noise"):
        rng = np.random.default_rng(seed)
        bpp = BPP[layout]
        self.bufs, self.desc, self.bgr_np, self.bgr_t = [], [], [], []
        for i, (H, W) in enumerate(sizes):
            a = rng.integers(0, 256, (H, W), np.uint8) if alpha == "noise" else alpha
            rows = bgr_to_rgb(synth.make_frame(H, W, seed + i), layout, alpha=a)
            pitch, off = _pitch(W, bpp, i, mode)
            buf = rng.integers(0, 256, off + H * pitch + 64, np.uint8)
            buf[off:off + H * pitch].reshape(H, pitch)[:, :bpp * W] = rows
            bgr = rgb_to_bgr(buf[off:], layout, H, W, pitch)
            t = torch.from_numpy(buf).cuda()
            self.bufs.append(t)
            self.desc.append((t.data_ptr() + off, H, W, pitch))
            self.bgr_np.append(bgr)
            self.bgr_t.append(torch.from_numpy(bgr).cuda())
        self.rgb = ctx.frame_table(self.desc)
        self.bgr = ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(self.bgr_t, sizes)])
        self.sizes, self.layout = sizes, layout

    def bgr_of(self, layout):
        """the BGR frames cvtColor makes of the same buffers read in another layout of the same size"""
        return [rgb_to_bgr(t.cpu().numpy()[p - t.data_ptr():], layout, H, W, pitch) for t, (p, H, W, pitch) in zip(self.bufs, self.desc)]


def _bgr_table(torch, ctx, frames, keep):
    keep += [torch.from_numpy(np.ascontiguousarray(b)).cuda() for b in frames]
    return ctx.frame_table([(t.data_ptr(), b.shape[0], b.shape[1], b.shape[1] * 3) for t, b in zip(keep[-len(frames):], frames)])


def _preprocess_both(torch, ctx, fr):
    B = len(fr.sizes)
    ta = torch.empty((B, 3, 640, 640), dtype=torch.float32, device="cuda")
    tb = torch.full((B, 3, 640, 640), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    dsa = ctx.preprocess_batch(fr.bgr, ta)
    dsb = ctx.preprocess_batch_rgb(fr.rgb, fr.layout, tb)
    ctx.synchronize()
    np.testing.assert_array_equal(dsb, dsa)
    a, b = ta.cpu().numpy(), tb.cpu().numpy()
    for i in range(B):
        np.testing.assert_array_equal(b[i], a[i], err_msg="%s frame %d %s" % (NAMES[fr.layout], i, fr.sizes[i]))
    return a, dsa


@pytest.mark.parametrize("layout,mode", CASES)
def test_preprocess_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    fr = RgbFrames(torch, ctx, SIZES, 10 + layout, layout, mode)
    try:
        for sharing in (1, 2):
            ctx.set_sharing(sharing)
            tensor, ds = _preprocess_both(torch, ctx, fr)
    finally:
        ctx.set_sharing(1)
    for i, bgr in enumerate(fr.bgr_np):
        det_img, sc = oracle.preprocess_letterbox(bgr)
        np.testing.assert_array_equal(tensor[i], oracle.to_tensor(det_img)[0])
        assert ds[i] == sc


def test_preprocess_with_normalisation_table(torch):
    """a non-identity pixel normalisation takes the table path of both preprocess kernels; a GRAY8 frame still gives three
    different planes"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.pixel_means[:] = (104.0, 117.0, 123.0)
    cfg.pixel_stds[:] = (57.0, 57.5, 58.0)
    c = Context(0, cfg)
    try:
        for layout, mode in CASES:
            t, _ = _preprocess_both(torch, c, RgbFrames(torch, c, SIZES[2:6], 30, layout, mode))
            if layout == GRAY8:
                assert not np.array_equal(t[0, 0], t[0, 1]) and not np.array_equal(t[0, 1], t[0, 2])
    finally:
        c.close()


def test_preprocess_row_staging_for_wide_rows(torch, ctx, oracle):
    """an aligned 8K RGBA row (30 720 B) does not fit the bulk-copy ring: the row-staging kernel takes it"""
    fr = RgbFrames(torch, ctx, [(4320, 7680), (40, 7680)], 35, BGRA, "aligned")
    tensor, _ = _preprocess_both(torch, ctx, fr)
    det_img, _ = oracle.preprocess_letterbox(fr.bgr_np[1])
    np.testing.assert_array_equal(tensor[1], oracle.to_tensor(det_img)[0])


@pytest.mark.parametrize("layout,mode", CASES)
def test_align_detections_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    sizes = [(1080, 1920)] * 4
    fr = RgbFrames(torch, ctx, sizes, 40 + layout, layout, mode)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _planted_heads(B, np.random.default_rng(41 + layout))]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    cap = 128
    out = []
    for rgb in (False, True):
        crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((cap, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if rgb:
            ctx.align_detections_rgb(fr.rgb, layout, crops, cap, M, ok)
        else:
            ctx.align_detections(fr.bgr, crops, cap, M, ok)
        out.append((crops, M, ok))
    counts, det, lmk = ctx.detect_fetch(B)
    ctx.synchronize()
    n = int(counts.sum())
    (ca, Ma, oka), (cb, Mb, okb) = [(c[:n].cpu().numpy(), M[:n].cpu().numpy(), o[:n].cpu().numpy()) for c, M, o in out]
    np.testing.assert_array_equal(okb, oka)
    np.testing.assert_array_equal(Mb, Ma)
    np.testing.assert_array_equal(cb, ca)
    assert {0, 1, 2} <= set(oka.tolist())
    off, crossing = 0, 0
    for b, bgr in enumerate(fr.bgr_np):
        H, W = sizes[b]
        for i in range(off, off + int(counts[b])):
            crop, M_, mode_ = oracle.align_face(bgr, lmk[i], bbox=det[i], with_mode=True)
            assert oka[i] == mode_
            np.testing.assert_array_equal(ca[i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
            if mode_ == 1:   # the crop's corners mapped back to the frame
                inv = np.linalg.inv(np.vstack([np.asarray(Ma[i]).reshape(2, 3), [0, 0, 1]]))
                xy = inv @ np.array([[0, 111, 0, 111], [0, 0, 111, 111], [1, 1, 1, 1]], np.float64)
                crossing |= (xy[0].min() < 0) | ((xy[0].max() > W - 1) << 1) | ((xy[1].min() < 0) << 2) | ((xy[1].max() > H - 1) << 3)
        off += int(counts[b])
    assert crossing == 15, crossing   # left, right, top and bottom


@pytest.mark.parametrize("crop", [(112, 112), (96, 112)])
@pytest.mark.parametrize("layout,mode", [(RGB24, "aligned"), (RGBA, "unaligned"), (BGRA, "word"), (GRAY8, "unaligned"),
                                         (RGB24, "unaligned"), (GRAY8, "aligned")])
def test_align_batch_caller_faces(torch, oracle, crop, layout, mode):
    """fd_align_batch_rgb with caller landmarks, with boxes and with bbox == None; 112x112 runs the fixed-size warp, 96x112
    the general one"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.crop_w, cfg.crop_h = crop
    c = Context(0, cfg)
    try:
        sizes = [(1080, 1920), (361, 645), (241, 320), (1, 1)]
        fr = RgbFrames(torch, c, sizes, 50 + layout, layout, mode)
        rng = np.random.default_rng(51)
        F = 140
        lmk, box, fidx = _caller_faces(rng, sizes, F)
        lmk_t, box_t, fidx_t = (torch.from_numpy(a).cuda() for a in (lmk, box, fidx))
        for sharing in (1, 2):
            c.set_sharing(sharing)
            for with_box in (True, False):
                res = []
                for rgb in (False, True):
                    crops = torch.full((F, crop[1], crop[0], 3), 77, dtype=torch.uint8, device="cuda")
                    M = torch.zeros((F, 6), dtype=torch.float64, device="cuda")
                    ok = torch.full((F,), 9, dtype=torch.uint8, device="cuda")
                    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                    bb = box_t if with_box else None
                    if rgb:
                        c.align_batch_rgb(fr.rgb, layout, lmk_t, fidx_t, F, crops, M, ok, bb)
                    else:
                        c.align_batch(fr.bgr, lmk_t, fidx_t, F, crops, M, ok, bb)
                    c.synchronize()
                    res.append((crops.cpu().numpy(), M.cpu().numpy(), ok.cpu().numpy()))
                (ca, Ma, oka), (cb, Mb, okb) = res
                np.testing.assert_array_equal(okb, oka)
                np.testing.assert_array_equal(Mb, Ma)
                np.testing.assert_array_equal(cb, ca)
                assert {0, 1, 2} <= set(oka.tolist()) or not with_box
                if sharing == 1:
                    for f in range(0, F, 5):
                        out, _, mode_ = oracle.align_face(fr.bgr_np[fidx[f]], lmk[f], bbox=box[f] if with_box else None, dsize=crop,
                                                          with_mode=True)
                        assert oka[f] == mode_
                        np.testing.assert_array_equal(ca[f], out if out is not None else np.zeros_like(ca[f]))
    finally:
        c.close()


@pytest.mark.parametrize("layout,mode", [(RGB24, "unaligned"), (RGBA, "aligned"), (BGRA, "word"), (GRAY8, "aligned")])
def test_select_and_align_selected(torch, ctx, oracle, layout, mode):
    sizes = [(1080, 1920)] * 5 + [(721, 1281)]
    fr = RgbFrames(torch, ctx, sizes, 60 + layout, layout, mode)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 61, n_faces=8)]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    enroll = layout in (RGBA, GRAY8)
    res = []
    for rgb in (False, True):
        sel = ctx.select_detections_rgb(fr.rgb, layout, enroll) if rgb else ctx.select_detections(fr.bgr, enroll)
        crops = torch.full((B, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((B, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((B,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if rgb:
            ctx.align_selected_rgb(fr.rgb, layout, crops, M, ok)
        else:
            ctx.align_selected(fr.bgr, crops, M, ok)
        ctx.synchronize()
        res.append((sel, crops.cpu().numpy(), M.cpu().numpy(), ok.cpu().numpy()))
    for a, b in zip(*res):
        np.testing.assert_array_equal(b, a)
    assert (res[0][0][:, 0] >= 0).any()
    sel, crops, _, ok = res[0]   # the BGR side against the oracle
    counts, det, lmk = ctx.detect_fetch(B)
    off = 0
    for b in range(B):
        n = int(counts[b])
        d, l = det[off:off + n], lmk[off:off + n].reshape(-1, 5, 2)
        bi, ki = oracle.face_selection(sizes[b], d, l, enroll) if n else (-1, -1)
        assert tuple(sel[b]) == (off + bi if bi >= 0 else -1, off + ki if ki >= 0 else -1)
        crop, mode_ = (None, 0)
        if bi >= 0 and ki >= 0:
            crop, _, mode_ = oracle.align_face(fr.bgr_np[b], l[ki], bbox=d[bi], with_mode=True)
        assert ok[b] == mode_
        np.testing.assert_array_equal(crops[b], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += n


@pytest.mark.parametrize("view", [False, True])
def test_deferred_image_replays_the_warp_in_the_recorded_layout(torch, view):
    """an image with K > 4096 candidates is completed at fd_detect_fetch / fd_detect_view; the align enqueued before it is
    replayed on the frames in the layout of the align call"""
    from rs_face_detection_b200 import Context
    from test_gpu_detect_limits import _blank, _groups, _plant
    c = Context(0)
    try:
        rng = np.random.default_rng(70)
        heads = _blank(2, 0.1)
        grp = _groups(rng, 1025, 4)
        grp[-1] = grp[-1][:4097 - 4 * 1024]
        assert _plant(heads, 0, rng, grp, "distinct") == 4097
        _plant(heads, 1, rng, _groups(rng, 20, 1, rows=44), "distinct")
        sizes = [(1080, 1920)] * 2
        heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in heads]
        for layout, mode in [(RGB24, "aligned"), (RGBA, "unaligned"), (BGRA, "aligned"), (GRAY8, "word")]:
            fr = RgbFrames(torch, c, sizes, 71 + layout, layout, mode)
            res = []
            for rgb in (False, True):
                out = torch.empty((2, 3, 640, 640), device="cuda")
                ds = c.preprocess_batch_rgb(fr.rgb, layout, out) if rgb else c.preprocess_batch(fr.bgr, out)
                c.detect_batch(c.head_table(heads_t), 2, ds, CONF, IOU)
                cap = 2048
                crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
                ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                if rgb:
                    c.align_detections_rgb(fr.rgb, layout, crops, cap, None, ok)
                else:
                    c.align_detections(fr.bgr, crops, cap, None, ok)
                assert c.detect_last_stats()["deferred_images"] == 1
                if view:
                    c.detect_view()
                counts, det, _ = c.detect_fetch(2)
                c.synchronize()
                n = int(counts.sum())
                res.append((counts, det, crops[:n].cpu().numpy(), ok[:n].cpu().numpy()))
            for a, b in zip(*res):
                np.testing.assert_array_equal(b, a, err_msg=NAMES[layout])
            assert int(res[0][0][0]) == 1025
    finally:
        c.close()


def test_same_buffers_as_rgb24_then_bgr_and_as_rgba_then_bgra(torch, ctx):
    """one set of 3-byte buffers stepped as RGB24 and at once as BGR (byte-identical frame tables: only the recorded format
    differs), and one set of 4-byte buffers as RGBA and at once as BGRA: each step matches the BGR step on its own frames"""
    sizes = [(1080, 1920)] * 4
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 76, n_faces=10)]
    keep = []
    fr3 = RgbFrames(torch, ctx, sizes, 75, RGB24)
    got = [_step(torch, ctx, heads_t, B, "rgb", fr3.rgb, RGB24), _step(torch, ctx, heads_t, B, None, fr3.rgb)]
    refs = [_step(torch, ctx, heads_t, B, None, _bgr_table(torch, ctx, fr3.bgr_of(RGB24), keep)),
            _step(torch, ctx, heads_t, B, None, _bgr_table(torch, ctx, [b[..., ::-1] for b in fr3.bgr_of(RGB24)], keep))]
    for g, r, what in zip(got, refs, ("rgb24", "bgr")):
        _assert_steps_equal(g, r, what)
    assert not np.array_equal(got[0][0], got[1][0])
    fr4 = RgbFrames(torch, ctx, sizes, 77, RGBA)
    got = [_step(torch, ctx, heads_t, B, "rgb", fr4.rgb, RGBA), _step(torch, ctx, heads_t, B, "rgb", fr4.rgb, BGRA)]
    for layout, g in zip((RGBA, BGRA), got):
        _assert_steps_equal(g, _step(torch, ctx, heads_t, B, None, _bgr_table(torch, ctx, fr4.bgr_of(layout), keep)), NAMES[layout])
    assert not np.array_equal(got[0][0], got[1][0])


def test_rgb_after_nv12_yuy2_and_bgr(torch, ctx):
    """the ctx records each call's format: BGR, GRAY8, NV12, RGBA, YUY2, RGBA on one ctx"""
    from yuv420_ref import NV12, bgr_to_yuv420
    from yuv422_ref import YUY2, bgr_to_yuv422
    sizes = [(1080, 1920)] * 3 + [(362, 646)]
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 86, n_faces=10)]
    fr = RgbFrames(torch, ctx, sizes, 85, RGBA, "aligned")
    gray = RgbFrames(torch, ctx, sizes, 87, GRAY8, "unaligned")
    planes, nv, yuy = [], [], []
    for i, (H, W) in enumerate(sizes):   # NV12 and YUY2 frames of other content
        y, uv = bgr_to_yuv420(synth.make_frame(H, W, 90 + i), NV12)
        planes += [torch.from_numpy(np.ascontiguousarray(y)).cuda(), torch.from_numpy(np.ascontiguousarray(uv)).cuda()]
        nv.append((planes[-2].data_ptr(), planes[-1].data_ptr(), H, W, W, W))
        planes.append(torch.from_numpy(np.ascontiguousarray(bgr_to_yuv422(synth.make_frame(H, W, 95 + i), YUY2))).cuda())
        yuy.append((planes[-1].data_ptr(), H, W, 2 * W))
    ref = _step(torch, ctx, heads_t, B, None, fr.bgr)
    ref_gray = _step(torch, ctx, heads_t, B, None, gray.bgr)
    _assert_steps_equal(_step(torch, ctx, heads_t, B, "rgb", gray.rgb, GRAY8), ref_gray, "gray8")
    nv_step = _step(torch, ctx, heads_t, B, "yuv420", ctx.frame_table_nv12(nv), NV12)
    _assert_steps_equal(_step(torch, ctx, heads_t, B, "rgb", fr.rgb, RGBA), ref, "rgba after nv12")
    yuy_step = _step(torch, ctx, heads_t, B, "yuv422", ctx.frame_table(yuy), YUY2)
    _assert_steps_equal(_step(torch, ctx, heads_t, B, "rgb", fr.rgb, RGBA), ref, "rgba after yuy2")
    assert not np.array_equal(nv_step[0], ref[0]) and not np.array_equal(yuy_step[0], ref[0])


def test_frames_that_differ_only_in_alpha_give_identical_outputs(torch, ctx):
    sizes = [(1080, 1920), (361, 645)]
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 96, n_faces=10)]
    for layout, mode in [(RGBA, "aligned"), (BGRA, "unaligned")]:
        a = RgbFrames(torch, ctx, sizes, 97, layout, mode, alpha=0)
        b = RgbFrames(torch, ctx, sizes, 97, layout, mode, alpha="noise")
        assert not np.array_equal(a.bufs[0].cpu().numpy(), b.bufs[0].cpu().numpy())
        _assert_steps_equal(_step(torch, ctx, heads_t, B, "rgb", b.rgb, layout), _step(torch, ctx, heads_t, B, "rgb", a.rgb, layout),
                            NAMES[layout])


@pytest.mark.parametrize("layout", [RGB24, BGRA, GRAY8])
def test_write_before_preprocess_is_seen(torch, ctx, oracle, layout):
    """a torch kernel on the ctx stream rewrites the frames right before the call"""
    sizes = [(1080, 1920)] * 4
    fr = RgbFrames(torch, ctx, sizes, 80, layout)
    new = RgbFrames(torch, ctx, sizes, 90, layout)
    out = torch.empty((4, 3, 640, 640), device="cuda")
    ctx.preprocess_batch_rgb(fr.rgb, layout, out)      # the descriptor table is on the device: the next call enqueues no copy
    ctx.synchronize()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):
        for dst, src in zip(fr.bufs, new.bufs):
            torch.bitwise_or(src, 0, out=dst)
    ctx.preprocess_batch_rgb(fr.rgb, layout, out)
    ctx.synchronize()
    got = out.cpu().numpy()
    for i, bgr in enumerate(new.bgr_np):
        det_img, _ = oracle.preprocess_letterbox(bgr)
        np.testing.assert_array_equal(got[i], oracle.to_tensor(det_img)[0])


def test_bad_descriptors_are_rejected(torch, ctx):
    from rs_face_detection_b200 import FdError, ffi
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    p = buf.data_ptr()
    out = torch.empty((1, 3, 640, 640), device="cuda")
    bad = []
    for l in LAYOUTS:
        bpp = BPP[l]
        bad += [(l, d) for d in [(p, 12, 0, 64), (p, 0, 16, 64), (p, -1, 16, 64), (p, 12, -2, 64), (p, 12, 16, bpp * 16 - 1), (0, 12, 16, 64)]]
    bad += [(l, (p, 12, 16, 64)) for l in (4, -1, 1 << 20)]
    # a detect on B = 1 so that the calls taking the last detections reach their descriptor check
    ds = ctx.preprocess_batch_rgb([(p, 13, 15, 45)], RGB24, out)   # odd sizes, pitch = 3W: accepted
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(1, 5, n_faces=2)]
    ctx.detect_batch(ctx.head_table(heads_t), 1, ds, CONF, IOU)
    ctx.select_detections_rgb([(p, 13, 15, 15)], GRAY8)
    for layout, d in bad:
        calls = [lambda: ctx.preprocess_batch_rgb([d], layout, out),
                 lambda: ctx.align_batch_rgb([d], layout, buf, buf, 1, buf),
                 lambda: ctx.align_detections_rgb([d], layout, buf, 1),
                 lambda: ctx.select_detections_rgb([d], layout),
                 lambda: ctx.align_selected_rgb([d], layout, buf)]
        for k, call in enumerate(calls):
            with pytest.raises(FdError) as e:
                call()
            assert e.value.code == ffi.FD_ERR_INVALID, (layout, d, k)
    ctx.synchronize()
    # an unknown layout is rejected also where there is nothing to do (B == 0, F == 0)
    for call in (lambda: ctx.preprocess_batch_rgb([], 4, out),
                 lambda: ctx.align_batch_rgb([(p, 12, 16, 64)], -1, buf, buf, 0, buf)):
        with pytest.raises(FdError) as e:
            call()
        assert e.value.code == ffi.FD_ERR_INVALID
    ctx.preprocess_batch_rgb([], BGRA, out)
