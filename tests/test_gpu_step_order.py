"""Ordering of the batch step's kernels on the ctx stream.

The step kernels (preprocess, detect, warp) are launched as programmatic dependent launches: each may be scheduled while
the kernel before it is still running and waits for it before touching global memory.  These tests check that a caller's
kernel that writes the inputs right before a call is seen by that call, and that back-to-back steps over different inputs
with no host synchronisation give the same results as each step run alone."""
import numpy as np
import pytest

from detect_ref import assert_rows_exact, decode_rows
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu
B, H, W = 8, 1080, 1920
CONF, IOU = 0.7, 0.4


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _dev(torch, arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


class Batch:
    def __init__(self, torch, ctx, frames_t, heads_np, cap=B * 64):
        self.ctx, self.frames_t, self.heads_np = ctx, frames_t, heads_np
        self.heads_t = _dev(torch, heads_np)
        self.frames_l = ctx.frame_table([(t.data_ptr(), H, W, W * 3) for t in frames_t])
        self.heads_c = ctx.head_table(self.heads_t)
        self.tensor = torch.empty((B, 3, 640, 640), dtype=torch.float32, device="cuda")
        self.crops = torch.zeros((cap, 112, 112, 3), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()   # torch fills on its own stream, which the ctx's stream does not wait for
        self.cap = cap

    def preprocess(self):
        return self.ctx.preprocess_batch(self.frames_l, self.tensor)

    def detect(self, ds):
        self.ctx.detect_batch(self.heads_c, B, ds, CONF, IOU)

    def align(self):
        self.ctx.align_detections(self.frames_l, self.crops, self.cap)

    def step(self):
        self.detect(self.preprocess())
        self.align()

    def results(self):
        counts, det, lmk = self.ctx.detect_fetch(B)
        self.ctx.synchronize()
        n = int(counts.sum())
        return counts, det, lmk, self.tensor.cpu().numpy(), self.crops[:n].cpu().numpy()


def _frames(torch, seed):
    return _dev(torch, [synth.make_frame(H, W, seed + i) for i in range(B)])


def _heads(seed):
    return synth.make_heads(B, seed=seed, n_faces=12, content_hw=(360, 640))[0]


def _check_vs_oracle(oracle, frames_np, heads_np, res):
    counts, det, lmk, tensor, crops = res
    cfg = oracle.make_det_cfg(conf_thr=CONF, iou_thr=IOU)
    ds = oracle.letterbox_geometry(H, W)[2]
    off = 0
    for b in range(B):
        etensor, edet, elmk, _ = oracle.pipeline_frame(cfg, frames_np[b], [h[b] for h in heads_np])
        np.testing.assert_array_equal(tensor[b], etensor[0])
        n = int(counts[b])
        assert n == len(edet)
        assert_rows_exact(det[off:off + n], lmk[off:off + n], (edet, elmk), decode_rows([h[b] for h in heads_np], cfg, ds, CONF, IOU))
        for i in range(n):
            crop, _, _ = oracle.align_face(frames_np[b], lmk[off + i], bbox=det[off + i], with_mode=True)
            np.testing.assert_array_equal(crops[off + i], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
        off += n
    assert off > B * 4


def test_write_before_preprocess_is_seen(torch, ctx, oracle):
    frames_t = _frames(torch, 500)
    new_t = _frames(torch, 600)
    bt = Batch(torch, ctx, frames_t, _heads(700))
    bt.step()                       # the frame table is on the device: the next preprocess call enqueues no copy
    ctx.synchronize()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):      # an elementwise kernel (not a copy) on the ctx stream, right before the call
        for dst, src in zip(frames_t, new_t):
            torch.bitwise_or(src, 0, out=dst)
    bt.step()
    _check_vs_oracle(oracle, [t.cpu().numpy() for t in new_t], bt.heads_np, bt.results())


def test_write_before_detect_is_seen(torch, ctx, oracle):
    frames_t = _frames(torch, 800)
    bt = Batch(torch, ctx, frames_t, _heads(900))
    new_np = _heads(901)
    new_t = _dev(torch, new_np)
    bt.step()
    ctx.synchronize()
    ds = bt.preprocess()
    s = torch.cuda.ExternalStream(ctx.stream())
    with torch.cuda.stream(s):      # overwrite the heads between the preprocess and the detect call
        for dst, src in zip(bt.heads_t, new_t):
            torch.mul(src, 1.0, out=dst)
    bt.detect(ds)
    bt.align()
    _check_vs_oracle(oracle, [t.cpu().numpy() for t in frames_t], new_np, bt.results())


def test_back_to_back_steps_do_not_interfere(torch, ctx):
    frames_t = _frames(torch, 1000)
    # same frames (one frame table, so nothing but the step kernels is enqueued between steps), different heads
    x = Batch(torch, ctx, frames_t, _heads(1100))
    y = Batch(torch, ctx, frames_t, _heads(1200))
    x.step()
    want_x = x.results()
    y.step()
    want_y = y.results()
    assert int(want_x[0].sum()) != int(want_y[0].sum()) or not np.array_equal(want_x[1], want_y[1])
    x.crops.zero_()
    y.crops.zero_()
    ctx.synchronize()
    for bt in (x, y, x, y):         # no host synchronisation between the steps
        bt.step()
    got_y = y.results()             # the detections of the last step (y) and every step's tensor / crops
    for w, g in zip(want_y, got_y):
        np.testing.assert_array_equal(g, w)
    got_x_crops = x.crops[:int(want_x[0].sum())].cpu().numpy()
    np.testing.assert_array_equal(got_x_crops, want_x[4])
    np.testing.assert_array_equal(x.tensor.cpu().numpy(), want_x[3])
