"""NV21, I420 and YV12 video frames through the batched *_yuv420 calls.

Every *_yuv420 call must give, byte for byte, what its BGR counterpart gives on cv2.cvtColor(COLOR_YUV2BGR_<layout>) of the
same frame, in the same ctx (tensor, det_scale, crops, M, modes, selections); the BGR results are also checked against the
CPU oracle on the converted frames (tests/yuv420_ref.py restates the conversions and is pinned against cv2).  The planes live
in pitched buffers whose padding and trailing bytes are noise: aligned (bulk-copy preprocess, interior warp reads),
unaligned (row-staging preprocess, per-tap warp reads) and, for the planar layouts, at the tight pitch_uv = W/2.
Layout NV12 must equal the *_nv12 calls."""
import numpy as np
import pytest

from rs_face_detection_b200.utils import synth
from yuv420_ref import I420, NAMES, NV12, NV21, PLANAR, YV12, bgr_to_yuv420, yuv420_to_bgr

pytestmark = pytest.mark.gpu
CONF, IOU = 0.7, 0.4
SIZES = [(2, 2), (362, 646), (1080, 1920), (2160, 3840), (1920, 1080), (240, 320), (100, 642)]
LAYOUTS = [NV21, I420, YV12]
# (layout, mode): every layout aligned and unaligned, the planar ones also at the tight chroma pitch
CASES = [(l, m) for l in LAYOUTS for m in ("aligned", "unaligned")] + [(I420, "tight"), (YV12, "tight")]


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _pitches(layout, W, i, mode):
    """(pitch_y, pitch_uv, Y start offset, chroma start offset)"""
    cw = W // 2 if layout in PLANAR else W
    if mode == "aligned":
        return -(-W // 64) * 64, -(-cw // 16) * 16 + 16, 0, 0
    if mode == "tight":
        return W, cw, 0, 0
    return W + 3, cw + 1 + 2 * (i % 2), 1 + i % 3, 3


class YuvFrames:
    """B frames in `layout` in noisy pitched device buffers, and the BGR frames cvtColor makes of them"""

    def __init__(self, torch, ctx, sizes, seed, layout, mode="aligned"):
        rng = np.random.default_rng(seed)
        self.bufs, self.desc, self.bgr_np, self.bgr_t = [], [], [], []
        for i, (H, W) in enumerate(sizes):
            y, chroma = bgr_to_yuv420(synth.make_frame(H, W, seed + i), layout)
            py, puv, oy, ouv = _pitches(layout, W, i, mode)
            rows, cw = chroma.shape
            ybuf = rng.integers(0, 256, oy + H * py + 64, np.uint8)
            cbuf = rng.integers(0, 256, ouv + rows * puv + 64, np.uint8)
            ybuf[oy:oy + H * py].reshape(H, py)[:, :W] = y
            cbuf[ouv:ouv + rows * puv].reshape(rows, puv)[:, :cw] = chroma
            bgr = yuv420_to_bgr(ybuf[oy:oy + H * py].reshape(H, py), cbuf[ouv:], layout, H, W, puv)
            yt, ct = torch.from_numpy(ybuf).cuda(), torch.from_numpy(cbuf).cuda()
            self.bufs += [yt, ct]
            self.desc.append((yt.data_ptr() + oy, ct.data_ptr() + ouv, H, W, py, puv))
            self.bgr_np.append(bgr)
            self.bgr_t.append(torch.from_numpy(bgr).cuda())
        self.yuv = ctx.frame_table_nv12(self.desc)
        self.bgr = ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(self.bgr_t, sizes)])
        self.sizes, self.layout = sizes, layout


def _heads(B, seed, n_faces=12):
    return synth.make_heads(B, seed=seed, n_faces=n_faces, content_hw=(360, 640))[0]


def _preprocess_both(torch, ctx, fr):
    B = len(fr.sizes)
    ta = torch.empty((B, 3, 640, 640), dtype=torch.float32, device="cuda")
    tb = torch.full((B, 3, 640, 640), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    dsa = ctx.preprocess_batch(fr.bgr, ta)
    dsb = ctx.preprocess_batch_yuv420(fr.yuv, fr.layout, tb)
    ctx.synchronize()
    np.testing.assert_array_equal(dsb, dsa)
    a, b = ta.cpu().numpy(), tb.cpu().numpy()
    for i in range(B):
        np.testing.assert_array_equal(b[i], a[i], err_msg="%s frame %d %s" % (NAMES[fr.layout], i, fr.sizes[i]))
    return a, dsa


@pytest.mark.parametrize("layout,mode", CASES)
def test_preprocess_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    ctx.set_sharing(2 if mode == "unaligned" else 1)
    try:
        fr = YuvFrames(torch, ctx, SIZES, 10 + layout, layout, mode)
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
            _preprocess_both(torch, c, YuvFrames(torch, c, SIZES[1:4], 30, layout, mode))
    finally:
        c.close()


def _align_detections_both(torch, ctx, fr, cap=512):
    out = []
    for yuv in (False, True):
        crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((cap, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if yuv:
            ctx.align_detections_yuv420(fr.yuv, fr.layout, crops, cap, M, ok)
        else:
            ctx.align_detections(fr.bgr, crops, cap, M, ok)
        out.append((crops, M, ok))
    return out


def _compare_aligned(ctx, out, B):
    counts, det, lmk = ctx.detect_fetch(B)
    ctx.synchronize()
    n = int(counts.sum())
    (ca, Ma, oka), (cb, Mb, okb) = [(c[:n].cpu().numpy(), M[:n].cpu().numpy(), o[:n].cpu().numpy()) for c, M, o in out]
    np.testing.assert_array_equal(okb, oka)
    np.testing.assert_array_equal(Mb, Ma)
    np.testing.assert_array_equal(cb, ca)
    return counts, det, lmk, ca, oka


@pytest.mark.parametrize("layout,mode", [(NV21, "unaligned"), (I420, "aligned"), (YV12, "tight")])
def test_align_detections_matches_bgr_and_oracle(torch, ctx, oracle, layout, mode):
    ctx.set_sharing(2 if layout == I420 else 1)
    try:
        sizes = [(1080, 1920)] * 6
        fr = YuvFrames(torch, ctx, sizes, 40 + layout, layout, mode)
        _, ds = _preprocess_both(torch, ctx, fr)
        heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(len(sizes), 41, n_faces=30)]
        ctx.detect_batch(ctx.head_table(heads_t), len(sizes), ds, CONF, IOU)
        counts, det, lmk, crops, modes = _compare_aligned(ctx, _align_detections_both(torch, ctx, fr), len(sizes))
    finally:
        ctx.set_sharing(1)
    off = 0
    for b, bgr in enumerate(fr.bgr_np):
        for i in range(off, off + int(counts[b])):
            crop, _, mode_ = oracle.align_face(bgr, lmk[i], bbox=det[i], with_mode=True)
            assert modes[i] == mode_
            np.testing.assert_array_equal(crops[i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += int(counts[b])
    assert off > 60


def _caller_faces(rng, sizes, F):
    """landmarks inside, over every border and off the frame, plus empty estimates (all-equal or NaN points)"""
    tmpl = synth.ARCFACE_TEMPLATE.astype(np.float64) - 56.0
    lmk, box, fidx = [], [], []
    for f in range(F):
        b = f % len(sizes)
        H, W = sizes[b]
        cx, cy = rng.uniform(-0.1 * W, 1.1 * W), rng.uniform(-0.1 * H, 1.1 * H)
        size = rng.uniform(0.3, 2.5) * min(H, W) / 4
        th = rng.uniform(-0.6, 0.6)
        rot = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        pts = tmpl / 112.0 * size @ rot.T + [cx, cy]
        kind = f % 7
        if kind == 5:
            pts[:] = [cx, cy]
        elif kind == 6:
            pts[:] = np.nan
        lmk.append(pts.reshape(10))
        x0, y0 = rng.uniform(-30, W), rng.uniform(-30, H)
        box.append([x0, y0, x0 + size, y0 + size])
        fidx.append(b)
    return np.float32(lmk), np.float32(box), np.int32(fidx)


@pytest.mark.parametrize("crop", [(112, 112), (96, 112)])
@pytest.mark.parametrize("layout,mode", [(NV21, "aligned"), (I420, "unaligned"), (YV12, "aligned"), (I420, "tight")])
def test_align_batch_caller_faces(torch, oracle, crop, layout, mode):
    """fd_align_batch_yuv420 with caller landmarks, with boxes and with bbox == None; 112x112 runs the fixed-size warp, 96x112
    the general one; the bbox-crop fallback (mode 2) meets odd ROI origins"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.crop_w, cfg.crop_h = crop
    c = Context(0, cfg)
    try:
        sizes = [(1080, 1920), (362, 646), (240, 320), (2, 2)]
        fr = YuvFrames(torch, c, sizes, 50 + layout, layout, mode)
        rng = np.random.default_rng(51)
        F = 140
        lmk, box, fidx = _caller_faces(rng, sizes, F)
        lmk_t, box_t, fidx_t = (torch.from_numpy(a).cuda() for a in (lmk, box, fidx))
        for sharing in (1, 2):
            c.set_sharing(sharing)
            for with_box in (True, False):
                res = []
                for yuv in (False, True):
                    crops = torch.full((F, crop[1], crop[0], 3), 77, dtype=torch.uint8, device="cuda")
                    M = torch.zeros((F, 6), dtype=torch.float64, device="cuda")
                    ok = torch.full((F,), 9, dtype=torch.uint8, device="cuda")
                    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                    bb = box_t if with_box else None
                    if yuv:
                        c.align_batch_yuv420(fr.yuv, layout, lmk_t, fidx_t, F, crops, M, ok, bb)
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


@pytest.mark.parametrize("layout,mode", [(NV21, "aligned"), (I420, "tight"), (YV12, "unaligned")])
def test_select_and_align_selected(torch, ctx, oracle, layout, mode):
    sizes = [(1080, 1920)] * 5 + [(720, 1280)]
    fr = YuvFrames(torch, ctx, sizes, 60 + layout, layout, mode)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 61, n_faces=8)]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    enroll = layout == I420
    res = []
    for yuv in (False, True):
        sel = ctx.select_detections_yuv420(fr.yuv, layout, enroll) if yuv else ctx.select_detections(fr.bgr, enroll)
        crops = torch.full((B, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((B, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((B,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if yuv:
            ctx.align_selected_yuv420(fr.yuv, layout, crops, M, ok)
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


def test_deferred_image_replays_the_warp_in_the_recorded_layout(torch):
    """an image with K > 4096 candidates is completed at fetch; the align enqueued before it is replayed on the frames in
    the layout of the align call"""
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
        for layout, mode in [(NV21, "aligned"), (I420, "tight"), (YV12, "unaligned")]:
            fr = YuvFrames(torch, c, sizes, 71 + layout, layout, mode)
            res = []
            for yuv in (False, True):
                out = torch.empty((2, 3, 640, 640), device="cuda")
                ds = c.preprocess_batch_yuv420(fr.yuv, layout, out) if yuv else c.preprocess_batch(fr.bgr, out)
                c.detect_batch(c.head_table(heads_t), 2, ds, CONF, IOU)
                cap = 2048
                crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
                ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                if yuv:
                    c.align_detections_yuv420(fr.yuv, layout, crops, cap, None, ok)
                else:
                    c.align_detections(fr.bgr, crops, cap, None, ok)
                assert c.detect_last_stats()["deferred_images"] == 1
                counts, det, _ = c.detect_fetch(2)
                c.synchronize()
                n = int(counts.sum())
                res.append((counts, det, crops[:n].cpu().numpy(), ok[:n].cpu().numpy()))
            for a, b in zip(*res):
                np.testing.assert_array_equal(b, a, err_msg=NAMES[layout])
            assert int(res[0][0][0]) == 1025
    finally:
        c.close()


def test_same_buffers_as_nv12_then_nv21_back_to_back(torch, ctx):
    """one set of interleaved chroma buffers stepped as NV12 and at once as NV21 (byte-equal descriptor tables): each step
    matches the BGR step on its own cvtColor frames"""
    sizes = [(1080, 1920)] * 4
    fr = YuvFrames(torch, ctx, sizes, 75, NV12)
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 76, n_faces=10)]
    cap = 256

    def step(call_yuv, layout, frames):
        out = torch.empty((B, 3, 640, 640), device="cuda")
        crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        ds = ctx.preprocess_batch_yuv420(frames, layout, out) if call_yuv else ctx.preprocess_batch(frames, out)
        ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
        if call_yuv:
            ctx.align_detections_yuv420(frames, layout, crops, cap, None, ok)
        else:
            ctx.align_detections(frames, crops, cap, None, ok)
        counts, det, _ = ctx.detect_fetch(B)
        return out, counts, det, crops, ok

    got = [step(True, NV12, fr.yuv), step(True, NV21, fr.yuv)]   # back to back: the second call reuses the device table
    ctx.synchronize()
    got = [[g.cpu().numpy() if hasattr(g, "cpu") else g for g in r] for r in got]
    for (layout, r) in zip((NV12, NV21), got):
        bgr_np = [yuv420_to_bgr(y, ch, layout, H, W, puv) for y, ch, (H, W, puv) in
                  ((b[0], b[1], (d[2], d[3], d[5])) for b, d in zip(_host_planes(fr), fr.desc))]
        bgr_t = [torch.from_numpy(b).cuda() for b in bgr_np]
        ref = step(False, None, ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(bgr_t, sizes)]))
        ctx.synchronize()
        ref = [g.cpu().numpy() if hasattr(g, "cpu") else g for g in ref]
        n = int(ref[1].sum())
        np.testing.assert_array_equal(r[0], ref[0], err_msg=NAMES[layout])
        np.testing.assert_array_equal(r[1], ref[1])
        np.testing.assert_array_equal(r[2], ref[2])
        np.testing.assert_array_equal(r[3][:n], ref[3][:n])
        np.testing.assert_array_equal(r[4][:n], ref[4][:n])
        assert n > 10
    assert not np.array_equal(got[0][0], got[1][0])


def _host_planes(fr):
    """(Y plane, chroma buffer from its start) of each frame, read back from the device"""
    out = []
    for i, d in enumerate(fr.desc):
        yt, ct = fr.bufs[2 * i], fr.bufs[2 * i + 1]
        H, py = d[2], d[4]
        yo, co = d[0] - yt.data_ptr(), d[1] - ct.data_ptr()
        out.append((yt.cpu().numpy()[yo:yo + H * py].reshape(H, py), ct.cpu().numpy()[co:]))
    return out


def test_layout_nv12_equals_the_nv12_calls(torch, ctx):
    sizes = [(1080, 1920)] * 3 + [(362, 646)]
    fr = YuvFrames(torch, ctx, sizes, 77, NV12, "unaligned")
    B = len(sizes)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 78, n_faces=10)]
    lmk = torch.from_numpy(np.float32(synth.ARCFACE_TEMPLATE.reshape(1, 10) * 3 + 200).repeat(8, 0)).cuda()
    fidx = torch.from_numpy(np.int32(np.arange(8) % B)).cuda()
    res = []
    for yuv in (False, True):
        r = []
        out = torch.empty((B, 3, 640, 640), device="cuda")
        ds = ctx.preprocess_batch_yuv420(fr.yuv, NV12, out) if yuv else ctx.preprocess_batch_nv12(fr.yuv, out)
        ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
        crops = [torch.full((256, 112, 112, 3), 77, dtype=torch.uint8, device="cuda") for _ in range(3)]
        M = [torch.zeros((256, 6), dtype=torch.float64, device="cuda") for _ in range(3)]
        ok = [torch.full((256,), 9, dtype=torch.uint8, device="cuda") for _ in range(3)]
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if yuv:
            ctx.align_detections_yuv420(fr.yuv, NV12, crops[0], 256, M[0], ok[0])
            ctx.align_batch_yuv420(fr.yuv, NV12, lmk, fidx, 8, crops[1], M[1], ok[1])
            sel = ctx.select_detections_yuv420(fr.yuv, NV12, False)
            ctx.align_selected_yuv420(fr.yuv, NV12, crops[2], M[2], ok[2])
        else:
            ctx.align_detections_nv12(fr.yuv, crops[0], 256, M[0], ok[0])
            ctx.align_batch_nv12(fr.yuv, lmk, fidx, 8, crops[1], M[1], ok[1])
            sel = ctx.select_detections_nv12(fr.yuv, False)
            ctx.align_selected_nv12(fr.yuv, crops[2], M[2], ok[2])
        ctx.synchronize()
        r += [out.cpu().numpy(), ds, sel] + [t.cpu().numpy() for t in crops + M + ok]
        res.append(r)
    for a, b in zip(*res):
        np.testing.assert_array_equal(b, a)


@pytest.mark.parametrize("layout", [NV21, I420])
def test_write_before_preprocess_is_seen(torch, ctx, oracle, layout):
    """a torch kernel on the ctx stream rewrites the planes right before the call"""
    sizes = [(1080, 1920)] * 4
    fr = YuvFrames(torch, ctx, sizes, 80, layout)
    new = YuvFrames(torch, ctx, sizes, 90, layout)
    out = torch.empty((4, 3, 640, 640), device="cuda")
    ctx.preprocess_batch_yuv420(fr.yuv, layout, out)      # the descriptor table is on the device: the next call enqueues no copy
    ctx.synchronize()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):
        for dst, src in zip(fr.bufs, new.bufs):
            torch.bitwise_or(src, 0, out=dst)
    ctx.preprocess_batch_yuv420(fr.yuv, layout, out)
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
    u = p + 4096
    common = [(p, u, 11, 16, 16, 16), (p, u, 12, 15, 16, 16), (p, u, 12, 16, 15, 16), (0, u, 12, 16, 16, 16), (p, 0, 12, 16, 16, 16),
              (p, u, 0, 16, 16, 16), (p, u, 12, 0, 16, 16)]
    bad = [(l, d) for l in LAYOUTS for d in common]
    bad += [(NV21, (p, u, 12, 16, 16, 15)), (I420, (p, u, 12, 16, 16, 7)), (YV12, (p, u, 12, 16, 16, 7))]
    bad += [(l, (p, u, 12, 16, 16, 16)) for l in (4, -1, 1 << 20)]
    # a detect on B = 1 so that the calls taking the last detections reach their descriptor check
    ds = ctx.preprocess_batch_yuv420([(p, u, 12, 16, 16, 8)], I420, out)   # planar: pitch_uv = W/2 is accepted
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(1, 5, n_faces=2)]
    ctx.detect_batch(ctx.head_table(heads_t), 1, ds, CONF, IOU)
    ctx.select_detections_yuv420([(p, u, 12, 16, 16, 8)], YV12)
    for layout, d in bad:
        calls = [lambda: ctx.preprocess_batch_yuv420([d], layout, out),
                 lambda: ctx.align_batch_yuv420([d], layout, buf, buf, 1, buf),
                 lambda: ctx.align_detections_yuv420([d], layout, buf, 1),
                 lambda: ctx.select_detections_yuv420([d], layout),
                 lambda: ctx.align_selected_yuv420([d], layout, buf)]
        for k, call in enumerate(calls):
            with pytest.raises(FdError) as e:
                call()
            assert e.value.code == ffi.FD_ERR_INVALID, (layout, d, k)
    ctx.synchronize()
    # an unknown layout is rejected also where there is nothing to do (B == 0, F == 0)
    for call in (lambda: ctx.preprocess_batch_yuv420([], 4, out),
                 lambda: ctx.align_batch_yuv420([(p, u, 12, 16, 16, 16)], -1, buf, buf, 0, buf)):
        with pytest.raises(FdError) as e:
            call()
        assert e.value.code == ffi.FD_ERR_INVALID
    ctx.preprocess_batch_yuv420([], I420, out)
