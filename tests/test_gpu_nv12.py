"""NV12 video frames through the batched calls.

Every *_nv12 call must give, byte for byte, what its BGR counterpart gives on cv2.cvtColor(COLOR_YUV2BGR_NV12) of the same
frame, in the same ctx (tensor, det_scale, crops, M, modes, selections); the BGR results are also checked against the CPU
oracle on the converted frames (tests/nv12_ref.py restates the conversion and is pinned against cv2).  The NV12 planes live
in pitched buffers whose padding and trailing bytes are noise, at aligned and at unaligned pointers and pitches."""
import ctypes as C

import numpy as np
import pytest

from nv12_ref import bgr_to_nv12, nv12_to_bgr
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu
CONF, IOU = 0.7, 0.4
SIZES = [(2, 2), (362, 646), (1080, 1920), (2160, 3840), (1920, 1080), (240, 320), (100, 642)]


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


class Nv12Frames:
    """B frames as NV12 planes in noisy pitched device buffers, and the BGR frames cvtColor makes of them"""

    def __init__(self, torch, ctx, sizes, seed, aligned=True):
        rng = np.random.default_rng(seed)
        self.bufs, self.desc, self.bgr_np, self.bgr_t, self.nv_np = [], [], [], [], []
        for i, (H, W) in enumerate(sizes):
            y, uv = bgr_to_nv12(synth.make_frame(H, W, seed + i))
            bgr = nv12_to_bgr(y, uv)
            if aligned:
                py, puv, oy, ouv = -(-W // 64) * 64, -(-W // 16) * 16 + 16, 0, 0
            else:
                py, puv, oy, ouv = W + 3, W + 1 + 2 * (i % 2), 1 + i % 3, 3
            ybuf = rng.integers(0, 256, oy + H * py + 64, np.uint8)
            uvbuf = rng.integers(0, 256, ouv + (H // 2) * puv + 64, np.uint8)
            ybuf[oy:oy + H * py].reshape(H, py)[:, :W] = y
            uvbuf[ouv:ouv + (H // 2) * puv].reshape(H // 2, puv)[:, :W] = uv
            yt, uvt = torch.from_numpy(ybuf).cuda(), torch.from_numpy(uvbuf).cuda()
            self.bufs += [yt, uvt]
            self.desc.append((yt.data_ptr() + oy, uvt.data_ptr() + ouv, H, W, py, puv))
            self.nv_np.append((y, uv))
            self.bgr_np.append(bgr)
            self.bgr_t.append(torch.from_numpy(bgr).cuda())
        self.nv = ctx.frame_table_nv12(self.desc)
        self.bgr = ctx.frame_table([(t.data_ptr(), h, w, w * 3) for t, (h, w) in zip(self.bgr_t, sizes)])
        self.sizes = sizes


def _heads(B, seed, n_faces=12):
    return synth.make_heads(B, seed=seed, n_faces=n_faces, content_hw=(360, 640))[0]


def _preprocess_both(torch, ctx, fr):
    B = len(fr.sizes)
    ta = torch.empty((B, 3, 640, 640), dtype=torch.float32, device="cuda")
    tb = torch.full((B, 3, 640, 640), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    dsa = ctx.preprocess_batch(fr.bgr, ta)
    dsb = ctx.preprocess_batch_nv12(fr.nv, tb)
    ctx.synchronize()
    np.testing.assert_array_equal(dsb, dsa)
    a, b = ta.cpu().numpy(), tb.cpu().numpy()
    for i in range(B):
        np.testing.assert_array_equal(b[i], a[i], err_msg="frame %d %s" % (i, fr.sizes[i]))
    return a, dsa


@pytest.mark.parametrize("sharing", [1, 2])
@pytest.mark.parametrize("aligned", [True, False])
def test_preprocess_matches_bgr_and_oracle(torch, ctx, oracle, aligned, sharing):
    ctx.set_sharing(sharing)
    try:
        fr = Nv12Frames(torch, ctx, SIZES, 10 + aligned, aligned)
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
        for aligned in (True, False):
            _preprocess_both(torch, c, Nv12Frames(torch, c, SIZES[1:4], 30, aligned))
    finally:
        c.close()


def _detect_align_both(torch, ctx, fr, heads_np, cap=512):
    B = len(fr.sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in heads_np]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    out = []
    for nv in (False, True):
        crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((cap, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        if nv:
            ctx.align_detections_nv12(fr.nv, crops, cap, M, ok)
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
    return counts, det, lmk, ca, oka


@pytest.mark.parametrize("sharing", [1, 2])
@pytest.mark.parametrize("aligned", [True, False])
def test_align_detections_matches_bgr_and_oracle(torch, ctx, oracle, aligned, sharing):
    ctx.set_sharing(sharing)
    try:
        sizes = [(1080, 1920)] * 6
        fr = Nv12Frames(torch, ctx, sizes, 40 + aligned, aligned)
        counts, det, lmk, crops, modes = _detect_align_both(torch, ctx, fr, _heads(len(sizes), 41, n_faces=30))
    finally:
        ctx.set_sharing(1)
    off = 0
    for b, bgr in enumerate(fr.bgr_np):
        for i in range(off, off + int(counts[b])):
            crop, _, mode = oracle.align_face(bgr, lmk[i], bbox=det[i], with_mode=True)
            assert modes[i] == mode
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
@pytest.mark.parametrize("aligned", [True, False])
def test_align_batch_caller_faces(torch, oracle, crop, aligned):
    """fd_align_batch_nv12 with caller landmarks, with boxes and with bbox == None; 112x112 runs the fixed-size warp, 96x112
    the general one"""
    from rs_face_detection_b200 import Context, ffi
    cfg = ffi.default_config()
    cfg.crop_w, cfg.crop_h = crop
    c = Context(0, cfg)
    try:
        for sharing in (1, 2):
            c.set_sharing(sharing)
            sizes = [(1080, 1920), (362, 646), (240, 320), (2, 2)]
            fr = Nv12Frames(torch, c, sizes, 50 + aligned, aligned)
            rng = np.random.default_rng(51)
            F = 140
            lmk, box, fidx = _caller_faces(rng, sizes, F)
            lmk_t, box_t, fidx_t = (torch.from_numpy(a).cuda() for a in (lmk, box, fidx))
            for with_box in (True, False):
                res = []
                for nv in (False, True):
                    crops = torch.full((F, crop[1], crop[0], 3), 77, dtype=torch.uint8, device="cuda")
                    M = torch.zeros((F, 6), dtype=torch.float64, device="cuda")
                    ok = torch.full((F,), 9, dtype=torch.uint8, device="cuda")
                    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
                    fn = c.align_batch_nv12 if nv else c.align_batch
                    fn(fr.nv if nv else fr.bgr, lmk_t, fidx_t, F, crops, M, ok, box_t if with_box else None)
                    c.synchronize()
                    res.append((crops.cpu().numpy(), M.cpu().numpy(), ok.cpu().numpy()))
                (ca, Ma, oka), (cb, Mb, okb) = res
                np.testing.assert_array_equal(okb, oka)
                np.testing.assert_array_equal(Mb, Ma)
                np.testing.assert_array_equal(cb, ca)
                assert {0, 1, 2} <= set(oka.tolist()) or not with_box
                for f in range(0, F, 5):
                    out, _, mode = oracle.align_face(fr.bgr_np[fidx[f]], lmk[f], bbox=box[f] if with_box else None, dsize=crop,
                                                     with_mode=True)
                    assert oka[f] == mode
                    np.testing.assert_array_equal(ca[f], out if out is not None else np.zeros_like(ca[f]))
    finally:
        c.close()


@pytest.mark.parametrize("enroll", [False, True])
def test_select_and_align_selected(torch, ctx, enroll):
    sizes = [(1080, 1920)] * 5 + [(720, 1280)]
    fr = Nv12Frames(torch, ctx, sizes, 60 + enroll)
    B = len(sizes)
    _, ds = _preprocess_both(torch, ctx, fr)
    heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in _heads(B, 61, n_faces=8)]
    ctx.detect_batch(ctx.head_table(heads_t), B, ds, CONF, IOU)
    res = []
    for nv in (False, True):
        sel = (ctx.select_detections_nv12(fr.nv, enroll) if nv else ctx.select_detections(fr.bgr, enroll))
        crops = torch.full((B, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
        M = torch.zeros((B, 6), dtype=torch.float64, device="cuda")
        ok = torch.full((B,), 9, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        (ctx.align_selected_nv12 if nv else ctx.align_selected)(fr.nv if nv else fr.bgr, crops, M, ok)
        ctx.synchronize()
        res.append((sel, crops.cpu().numpy(), M.cpu().numpy(), ok.cpu().numpy()))
    for a, b in zip(*res):
        np.testing.assert_array_equal(b, a)
    assert (res[0][0][:, 0] >= 0).any()


def test_deferred_image_replays_the_nv12_warp(torch):
    """an image with K > 4096 candidates is completed at fetch; the align enqueued before it is replayed on the NV12 frames"""
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
        fr = Nv12Frames(torch, c, sizes, 71)
        heads_t = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in heads]
        res = []
        for nv in (False, True):
            ds = c.preprocess_batch_nv12(fr.nv, torch.empty((2, 3, 640, 640), device="cuda")) if nv else \
                c.preprocess_batch(fr.bgr, torch.empty((2, 3, 640, 640), device="cuda"))
            c.detect_batch(c.head_table(heads_t), 2, ds, CONF, IOU)
            cap = 2048
            crops = torch.full((cap, 112, 112, 3), 77, dtype=torch.uint8, device="cuda")
            ok = torch.full((cap,), 9, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
            (c.align_detections_nv12 if nv else c.align_detections)(fr.nv if nv else fr.bgr, crops, cap, None, ok)
            assert c.detect_last_stats()["deferred_images"] == 1
            counts, det, _ = c.detect_fetch(2)
            c.synchronize()
            n = int(counts.sum())
            res.append((counts, det, crops[:n].cpu().numpy(), ok[:n].cpu().numpy()))
        for a, b in zip(*res):
            np.testing.assert_array_equal(b, a)
        assert int(res[0][0][0]) == 1025
    finally:
        c.close()


def test_bad_descriptors_are_rejected(torch, ctx):
    from rs_face_detection_b200 import FdError, ffi
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
    p = buf.data_ptr()
    out = torch.empty((1, 3, 640, 640), device="cuda")
    bad = [(p, p + 4096, 11, 16, 16, 16), (p, p + 4096, 12, 15, 16, 16), (p, p + 4096, 12, 16, 15, 16), (p, p + 4096, 12, 16, 16, 15),
           (0, p + 4096, 12, 16, 16, 16), (p, 0, 12, 16, 16, 16), (p, p + 4096, 0, 16, 16, 16)]
    for d in bad:
        with pytest.raises(FdError) as e:
            ctx.preprocess_batch_nv12([d], out)
        assert e.value.code == ffi.FD_ERR_INVALID, d
        with pytest.raises(FdError):
            ctx.align_batch_nv12([d], buf, buf, 1, buf)


def test_write_before_preprocess_is_seen(torch, ctx, oracle):
    """a torch kernel on the ctx stream rewrites the NV12 planes right before the call"""
    sizes = [(1080, 1920)] * 4
    fr = Nv12Frames(torch, ctx, sizes, 80)
    new = Nv12Frames(torch, ctx, sizes, 90)
    out = torch.empty((4, 3, 640, 640), device="cuda")
    ctx.preprocess_batch_nv12(fr.nv, out)      # the descriptor table is on the device: the next call enqueues no copy
    ctx.synchronize()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):
        for dst, src in zip(fr.bufs, new.bufs):
            torch.bitwise_or(src, 0, out=dst)
    ctx.preprocess_batch_nv12(fr.nv, out)
    ctx.synchronize()
    got = out.cpu().numpy()
    for i, bgr in enumerate(new.bgr_np):
        det_img, _ = oracle.preprocess_letterbox(bgr)
        np.testing.assert_array_equal(got[i], oracle.to_tensor(det_img)[0])
