"""Parity at the sizes BASELINE.json's configs name (VERDICT r1 "parity holes"): the device-resident call sequence over a
full batch — C2 batch-64 1080p, C4 batch-256 with ~50 faces per frame, C5 a shard of 4K frames — against the CPU oracle:
per-image detection counts for EVERY image, rows bit for bit (tests/detect_ref.py), CNN input tensors and aligned crops bit-exact on a
sample, and the size-independent properties (offsets are the prefix sum of the counts, rows sorted by score per image, no
image deferred to the host-completed NMS path)."""
import numpy as np
import pytest

from detect_ref import assert_rows_exact, decode_rows
from rs_face_detection_b200.utils import synth

pytestmark = pytest.mark.gpu


def _run_at_size(ctx, oracle, B, hw, n_faces, n_distinct, tensor_images, crop_sample, seed):
    H, W = hw
    frames = [synth.make_frame(H, W, seed + i) for i in range(n_distinct)]
    heads_d, _ = synth.make_heads(n_distinct, seed=seed + 1000, n_faces=n_faces, content_hw=(360, 640))
    reps = B // n_distinct
    heads = [np.ascontiguousarray(np.tile(h, (reps, 1, 1, 1))) for h in heads_d]
    fdev = [ctx.to_device(f) for f in frames]
    hdev = [ctx.to_device(h) for h in heads]
    fl = ctx.frame_table([(fdev[b % n_distinct].ptr, H, W, W * 3) for b in range(B)])
    tensor = ctx.alloc(B * 3 * 640 * 640 * 4)
    cap = B * max(64, 2 * n_faces)
    crops = ctx.alloc(cap * 112 * 112 * 3)
    for _ in range(2):   # second pass: workspaces sized, `crowded` remembered
        ds = ctx.preprocess_batch(fl, tensor)
        ctx.detect_batch(hdev, B, ds, 0.7, 0.4)
        ctx.align_detections(fl, crops, cap)
        stats = ctx.detect_last_stats()
        counts, det, lmk = ctx.detect_fetch(B)
    assert stats["deferred_images"] == 0 and stats["fused"]
    total = int(counts.sum())
    assert total == len(det) and total > B * n_faces // 2
    got_crops = crops.download((cap, 112, 112, 3), np.uint8)
    cfg = oracle.make_det_cfg(conf_thr=0.7, iou_thr=0.4)
    offs = np.concatenate([[0], np.cumsum(counts)])
    want_scale = oracle.letterbox_geometry(H, W)[2]
    expect = [oracle.detect_post(cfg, [h[i] for h in heads_d], want_scale) for i in range(n_distinct)]
    ref = [decode_rows([h[i] for h in heads_d], cfg, want_scale, 0.7, 0.4) for i in range(n_distinct)]
    rng = np.random.default_rng(seed)
    crop_rows = set(rng.choice(total, size=min(crop_sample, total), replace=False).tolist())
    checked = 0
    for b in range(B):
        edet, elmk, K = expect[b % n_distinct]
        n = int(counts[b])
        assert n == len(edet), "image %d" % b
        d = det[offs[b]:offs[b] + n]
        assert_rows_exact(d, lmk[offs[b]:offs[b] + n], (edet, elmk), ref[b % n_distinct], "image %d" % b)
        assert np.all(np.diff(d[:, 4]) <= 0)                        # descending score within an image
        for i in range(n):
            r = int(offs[b]) + i
            if r in crop_rows:
                crop, _, mode = oracle.align_face(frames[b % n_distinct], lmk[r], bbox=det[r], with_mode=True)
                np.testing.assert_array_equal(got_crops[r], crop if crop is not None else np.zeros((112, 112, 3), np.uint8))
                checked += 1
    assert checked == len(crop_rows)
    t = tensor.download((B, 3, 640, 640), np.float32)
    for b in tensor_images:
        et = oracle.to_tensor(oracle.preprocess_letterbox(frames[b % n_distinct])[0])
        np.testing.assert_array_equal(t[b], et[0] if et.ndim == 4 else et)
    for buf in fdev + hdev + [tensor, crops]:
        buf.free()
    return total


def test_c2_batch64_1080p(ctx, oracle):
    """BASELINE configs[1]: batch-64 1920x1080, ~20 faces per frame, every image distinct; every crop checked."""
    total = _run_at_size(ctx, oracle, B=64, hw=(1080, 1920), n_faces=20, n_distinct=64, tensor_images=[0, 17, 40, 63], crop_sample=4000, seed=7000)
    assert 600 < total < 1400


def test_c4_batch256_50_faces(ctx, oracle):
    """BASELINE configs[3]: batch 256, ~50 faces per frame (32 distinct frames x 8); 200 sampled crops bit-exact."""
    total = _run_at_size(ctx, oracle, B=256, hw=(1080, 1920), n_faces=50, n_distinct=32, tensor_images=[0, 100, 255], crop_sample=200, seed=7100)
    assert total > 5000


def test_c5_4k_shard(ctx, oracle):
    """BASELINE configs[4]: one rank's shard of the 4K stream (16 frames of 3840x2160, ~50 faces per frame)."""
    _run_at_size(ctx, oracle, B=16, hw=(2160, 3840), n_faces=50, n_distinct=8, tensor_images=[0, 9, 15], crop_sample=150, seed=7200)
