"""Packed 4:2:2 camera frames (YUY2, UYVY, YVYU) through the batched *_yuv422 calls.

Every *_yuv422 call must give, byte for byte, what its BGR counterpart gives on cv2.cvtColor(COLOR_YUV2BGR_<layout>) of the
same frame, in the same ctx (tensor, det_scale, crops, M, modes, selections); the BGR results are also checked against the
CPU oracle on the converted frames (tests/yuv422_ref.py restates the conversion and is pinned against cv2).  The packed
planes live in pitched buffers whose padding, leading and trailing bytes are noise: aligned (bulk-copy preprocess, interior
warp reads), word-aligned (row-staging preprocess, interior warp reads) and unaligned (row-staging preprocess, per-tap warp
reads)."""
import numpy as np
import pytest

from rs_face_detection_b200.utils import synth
from test_gpu_yuv420 import _caller_faces, _heads
from yuv422_ref import NAMES, UYVY, YUY2, YVYU, bgr_to_yuv422, yuv422_to_bgr

pytestmark = pytest.mark.gpu
CONF, IOU = 0.7, 0.4
SIZES = [(1, 2), (3, 4), (361, 646), (1081, 1920), (1080, 1920), (2160, 3840), (1920, 1080), (100, 642)]
LAYOUTS = [YUY2, UYVY, YVYU]
CASES = [(l, m) for l in LAYOUTS for m in ("aligned", "unaligned")]


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _pitch(W, i, mode):
    """(pitch, start offset) of frame i"""
    if mode == "aligned":
        return -(-2 * W // 64) * 64, 0
    if mode == "word":
        return 2 * W + 4, 4
    return 2 * W + 1 + 2 * (i % 2), 1 + i % 3


class PackedFrames:
    """B frames in `layout` in noisy pitched device buffers, and the BGR frames cvtColor makes of them"""

    def __init__(self, torch, ctx, sizes, seed, layout, mode="aligned"):
        rng = np.random.default_rng(seed)
        self.bufs, self.desc, self.bgr_np, self.bgr_t = [], [], [], []
        for i, (H, W) in enumerate(sizes):
            rows = bgr_to_yuv422(synth.make_frame(H, W, seed + i), layout)
            pitch, off = _pitch(W, i, mode)
            buf = rng.integers(0, 256, off + H * pitch + 64, np.uint8)
            buf[off:off + H * pitch].reshape(H, pitch)[:, :2 * W] = rows
            bgr = yuv422_to_bgr(buf[off:], layout, H, W, pitch)
            t = torch.from_numpy(buf).cuda()
            self.bufs.append(t)
            self.desc.append((t.data_ptr() + off, H, W, pitch))
            self.bgr_np.append(bgr)
            self.bgr_t.append(torch.from_numpy(bgr).cuda())
        self.packed = ctx.frame_table(self.desc)
        self.bgr = ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(self.bgr_t, sizes)])
        self.sizes, self.layout = sizes, layout

    def bgr_of(self, layout):
        """the BGR frames cvtColor makes of the same buffers read in another layout"""
        out = []
        for t, (p, H, W, pitch) in zip(self.bufs, self.desc):
            out.append(yuv422_to_bgr(t.cpu().numpy()[p - t.data_ptr():], layout, H, W, pitch))
        return out


def _preprocess_both(torch, ctx, fr):
    B = len(fr.sizes)
    ta = torch.empty((B, 3, 640, 640), dtype=torch.float32, device="cuda")
    tb = torch.full((B, 3, 640, 640), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    dsa = ctx.preprocess_batch(fr.bgr, ta)
    dsb = ctx.preprocess_batch_yuv422(fr.packed, fr.layout, tb)
    ctx.synchronize()
    np.testing.assert_array_equal(dsb, dsa)
    a, b = ta.cpu().numpy(), tb.cpu().numpy()
    for i in range(B):
        np.testing.assert_array_equal(b[i], a[i], err_msg="%s frame %d %s" % (NAMES[fr.layout], i, fr.sizes[i]))
    return a, dsa


@pytest.mark.parametrize("layout,mode", CASES + [(YUY2, "word")])
def test_preprocess_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    fr = PackedFrames(torch, ctx, SIZES, 10 + layout, layout, mode)
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
    """a non-identity pixel normalisation takes the table path of both preprocess kernels"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.pixel_means[:] = (104.0, 117.0, 123.0)
    cfg.pixel_stds[:] = (57.0, 57.5, 58.0)
    c = Context(0, cfg)
    try:
        for layout, mode in CASES:
            _preprocess_both(torch, c, PackedFrames(torch, c, SIZES[2:6], 30, layout, mode))
    finally:
        c.close()


def _planted_heads(B, rng):
    """per image: template faces at the corners and edges of the 1080p content (their crops cross every border) and inside,
    and five-equal-point faces (empty estimate) inside, where the reference takes the bbox-crop fallback, and at the right
    edge, where its ROI leaves the image and the reference errs.  Boxes of 4 to 7 px give fallback ROIs of both parities."""
    from test_gpu_detect_limits import _blank, _groups, _plant
    heads = _blank(B, 0.1)
    edge = [(0, 0), (0, 40), (0, 79), (22, 0), (44, 0), (44, 40), (44, 79), (10, 10), (30, 50)]
    empty = [(20, 30), (12, 46), (34, 22), (26, 62), (22, 79)]
    for b in range(B):
        grp = _groups(rng, 0, 1, cells=edge + empty)
        kinds = ["tmpl"] * len(edge) + ["zero"] * len(empty)
        boxes = [(4.0, 4.0)] * len(edge) + [(4.0 + k + b % 2, 4.0 + k) for k in range(len(empty))]
        _plant(heads, b, rng, grp, "distinct", lmk=kinds, box=boxes)
    return heads


@pytest.mark.parametrize("layout,mode", CASES)
def test_align_detections_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    sizes = [(1080, 1920)] * 4
    fr = PackedFrames(torch, ctx, sizes, 40 + layout, layout, mode)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _planted_heads(B, np.random.default_rng(41 + layout))]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    cap = 128
    out = []
    for packed in (False, True):
        crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((cap, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if packed:
            ctx.align_detections_yuv422(fr.packed, layout, crops, cap, M, ok)
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
    off, odd_roi, crossing = 0, False, 0
    for b, bgr in enumerate(fr.bgr_np):
        H, W = sizes[b]
        for i in range(off, off + int(counts[b])):
            crop, M_, mode_ = oracle.align_face(bgr, lmk[i], bbox=det[i], with_mode=True)
            assert oka[i] == mode_
            np.testing.assert_array_equal(ca[i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
            if mode_ == 2:
                odd_roi |= int(np.float32(det[i][0]) - np.float32(22)) % 2 == 1
            if mode_ == 1:   # the crop's corners mapped back to the frame
                inv = np.linalg.inv(np.vstack([np.asarray(Ma[i]).reshape(2, 3), [0, 0, 1]]))
                xy = inv @ np.array([[0, 111, 0, 111], [0, 0, 111, 111], [1, 1, 1, 1]], np.float64)
                crossing |= (xy[0].min() < 0) | ((xy[0].max() > W - 1) << 1) | ((xy[1].min() < 0) << 2) | ((xy[1].max() > H - 1) << 3)
        off += int(counts[b])
    assert odd_roi
    assert crossing == 15, crossing   # left, right, top and bottom


@pytest.mark.parametrize("crop", [(112, 112), (96, 112)])
@pytest.mark.parametrize("layout,mode", [(YUY2, "aligned"), (UYVY, "unaligned"), (YVYU, "word"), (UYVY, "aligned")])
def test_align_batch_caller_faces(torch, oracle, crop, layout, mode):
    """fd_align_batch_yuv422 with caller landmarks, with boxes and with bbox == None; 112x112 runs the fixed-size warp, 96x112
    the general one; the bbox-crop fallback (mode 2) meets odd ROI origins"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.crop_w, cfg.crop_h = crop
    c = Context(0, cfg)
    try:
        sizes = [(1080, 1920), (361, 646), (241, 320), (1, 2)]
        fr = PackedFrames(torch, c, sizes, 50 + layout, layout, mode)
        rng = np.random.default_rng(51)
        F = 140
        lmk, box, fidx = _caller_faces(rng, sizes, F)
        lmk_t, box_t, fidx_t = (torch.from_numpy(a).cuda() for a in (lmk, box, fidx))
        for sharing in (1, 2):
            c.set_sharing(sharing)
            for with_box in (True, False):
                res = []
                for packed in (False, True):
                    crops = torch.full((F, crop[1], crop[0], 3), 77, dtype=torch.uint8, device="cuda")
                    M = torch.zeros((F, 6), dtype=torch.float64, device="cuda")
                    ok = torch.full((F,), 9, dtype=torch.uint8, device="cuda")
                    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                    bb = box_t if with_box else None
                    if packed:
                        c.align_batch_yuv422(fr.packed, layout, lmk_t, fidx_t, F, crops, M, ok, bb)
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


@pytest.mark.parametrize("layout,mode", [(YUY2, "unaligned"), (UYVY, "aligned"), (YVYU, "word")])
def test_select_and_align_selected(torch, ctx, oracle, layout, mode):
    sizes = [(1080, 1920)] * 5 + [(721, 1280)]
    fr = PackedFrames(torch, ctx, sizes, 60 + layout, layout, mode)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 61, n_faces=8)]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    enroll = layout == UYVY
    res = []
    for packed in (False, True):
        sel = ctx.select_detections_yuv422(fr.packed, layout, enroll) if packed else ctx.select_detections(fr.bgr, enroll)
        crops = torch.full((B, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((B, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((B,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if packed:
            ctx.align_selected_yuv422(fr.packed, layout, crops, M, ok)
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
        for layout, mode in [(YUY2, "aligned"), (UYVY, "unaligned"), (YVYU, "aligned")]:
            fr = PackedFrames(torch, c, sizes, 71 + layout, layout, mode)
            res = []
            for packed in (False, True):
                out = torch.empty((2, 3, 640, 640), device="cuda")
                ds = c.preprocess_batch_yuv422(fr.packed, layout, out) if packed else c.preprocess_batch(fr.bgr, out)
                c.detect_batch(c.head_table(heads_t), 2, ds, CONF, IOU)
                cap = 2048
                crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
                ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                if packed:
                    c.align_detections_yuv422(fr.packed, layout, crops, cap, None, ok)
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


def _step(torch, ctx, heads_t, B, call, frames, layout=None, cap=256):
    """preprocess, detect and align_detections through the BGR (call None), _yuv420 or _yuv422 calls"""
    out = torch.empty((B, 3, 640, 640), device="cuda")
    crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
    ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    if call is None:
        ds = ctx.preprocess_batch(frames, out)
    else:
        ds = getattr(ctx, "preprocess_batch_" + call)(frames, layout, out)
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    if call is None:
        ctx.align_detections(frames, crops, cap, None, ok)
    else:
        getattr(ctx, "align_detections_" + call)(frames, layout, crops, cap, None, ok)
    counts, det, _ = ctx.detect_fetch(B)
    ctx.synchronize()
    n = int(counts.sum())
    return [out.cpu().numpy(), counts, det, crops[:n].cpu().numpy(), ok[:n].cpu().numpy()]


def _assert_steps_equal(got, ref, what):
    assert len(got[3]) > 10
    for a, b in zip(got, ref):
        np.testing.assert_array_equal(a, b, err_msg=what)


def test_same_buffers_as_yuy2_then_uyvy_back_to_back(torch, ctx):
    """one set of packed buffers stepped as YUY2 and at once as UYVY: each step matches the BGR step on its own cvtColor
    frames"""
    sizes = [(1080, 1920)] * 4
    fr = PackedFrames(torch, ctx, sizes, 75, YUY2)
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 76, n_faces=10)]
    got = [_step(torch, ctx, heads_t, B, "yuv422", fr.packed, YUY2), _step(torch, ctx, heads_t, B, "yuv422", fr.packed, UYVY)]
    for layout, g in zip((YUY2, UYVY), got):
        bgr_t = [torch.from_numpy(b).cuda() for b in fr.bgr_of(layout)]
        ref = _step(torch, ctx, heads_t, B, None, ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(bgr_t, sizes)]))
        _assert_steps_equal(g, ref, NAMES[layout])
    assert not np.array_equal(got[0][0], got[1][0])


def test_packed_after_nv12_and_after_bgr(torch, ctx):
    """the ctx records each call's format: BGR, packed, packed again (the device table is reused), NV12, packed, on one ctx"""
    from yuv420_ref import NV12, bgr_to_yuv420
    sizes = [(1080, 1920)] * 3 + [(361, 646)]
    fr = PackedFrames(torch, ctx, sizes, 85, YVYU, "aligned")
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 86, n_faces=10)]
    planes, nv = [], []
    for i, (H, W) in enumerate(sizes):   # NV12 frames of other content (H even)
        H -= H % 2
        y, uv = bgr_to_yuv420(synth.make_frame(H, W, 90 + i), NV12)
        planes += [torch.from_numpy(np.ascontiguousarray(y)).cuda(), torch.from_numpy(np.ascontiguousarray(uv)).cuda()]
        nv.append((planes[-2].data_ptr(), planes[-1].data_ptr(), H, W, W, W))
    nv_table = ctx.frame_table_nv12(nv)
    ref = _step(torch, ctx, heads_t, B, None, fr.bgr)
    seq = [_step(torch, ctx, heads_t, B, "yuv422", fr.packed, YVYU), _step(torch, ctx, heads_t, B, "yuv422", fr.packed, YVYU)]
    nv_step = _step(torch, ctx, heads_t, B, "yuv420", nv_table, NV12)
    seq.append(_step(torch, ctx, heads_t, B, "yuv422", fr.packed, YVYU))
    for g in seq:
        _assert_steps_equal(g, ref, "yvyu")
    assert not np.array_equal(nv_step[0], ref[0])


@pytest.mark.parametrize("layout", [YUY2, UYVY])
def test_write_before_preprocess_is_seen(torch, ctx, oracle, layout):
    """a torch kernel on the ctx stream rewrites the packed planes right before the call"""
    sizes = [(1080, 1920)] * 4
    fr = PackedFrames(torch, ctx, sizes, 80, layout)
    new = PackedFrames(torch, ctx, sizes, 90, layout)
    out = torch.empty((4, 3, 640, 640), device="cuda")
    ctx.preprocess_batch_yuv422(fr.packed, layout, out)      # the descriptor table is on the device: the next call enqueues no copy
    ctx.synchronize()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):
        for dst, src in zip(fr.bufs, new.bufs):
            torch.bitwise_or(src, 0, out=dst)
    ctx.preprocess_batch_yuv422(fr.packed, layout, out)
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
    common = [(p, 12, 15, 32), (p, 12, 0, 32), (p, 0, 16, 32), (p, -1, 16, 32), (p, 12, -2, 32), (p, 12, 16, 31), (0, 12, 16, 32)]
    bad = [(l, d) for l in LAYOUTS for d in common]
    bad += [(l, (p, 12, 16, 32)) for l in (3, -1, 1 << 20)]
    # a detect on B = 1 so that the calls taking the last detections reach their descriptor check
    ds = ctx.preprocess_batch_yuv422([(p, 13, 16, 32)], UYVY, out)   # odd height, pitch = 2W: accepted
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(1, 5, n_faces=2)]
    ctx.detect_batch(ctx.head_table(heads_t), 1, ds, CONF, IOU)
    ctx.select_detections_yuv422([(p, 13, 16, 32)], YVYU)
    for layout, d in bad:
        calls = [lambda: ctx.preprocess_batch_yuv422([d], layout, out),
                 lambda: ctx.align_batch_yuv422([d], layout, buf, buf, 1, buf),
                 lambda: ctx.align_detections_yuv422([d], layout, buf, 1),
                 lambda: ctx.select_detections_yuv422([d], layout),
                 lambda: ctx.align_selected_yuv422([d], layout, buf)]
        for k, call in enumerate(calls):
            with pytest.raises(FdError) as e:
                call()
            assert e.value.code == ffi.FD_ERR_INVALID, (layout, d, k)
    ctx.synchronize()
    # an unknown layout is rejected also where there is nothing to do (B == 0, F == 0)
    for call in (lambda: ctx.preprocess_batch_yuv422([], 3, out),
                 lambda: ctx.align_batch_yuv422([(p, 12, 16, 32)], -1, buf, buf, 0, buf)):
        with pytest.raises(FdError) as e:
            call()
        assert e.value.code == ffi.FD_ERR_INVALID
    ctx.preprocess_batch_yuv422([], YUY2, out)
