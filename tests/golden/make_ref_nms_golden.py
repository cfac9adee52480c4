"""Generates tests/golden/ref_nms_golden.npz for tests/test_gpu_nms.py::test_vs_reference_cuda_nms: 5 000 non-degenerate
boxes (_random_dets(5000, 99, canvas=1200)) sorted by descending score, and the keep list of the reference's own CUDA NMS
(`_nms`, src/nms_kernel.cu, which the reference never builds) on them at IoU 0.4.

With oracle/_ref built from a reference checkout (`make -C oracle ref REF=<checkout>`; calling it needs a GPU) the keep list
comes from that library.  Without it the script writes the CPU oracle's nms_sorted (processing/nms.rs): on non-degenerate
boxes `ovr > thr` == `!(ovr <= thr)`, so the two lists agree, and the committed one equals what the reference's `_nms`
returned for these boxes when the test called the library directly.  `source` in the file says which one wrote it.
Run:  python tests/golden/make_ref_nms_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import oracle as O                                      # noqa: E402
from test_gpu_nms import _random_dets, reference_cuda_nms           # noqa: E402

THRESH = 0.4

if __name__ == "__main__":
    dets = _random_dets(5000, 99, canvas=1200)
    srt = np.ascontiguousarray(dets[O.argsort_descending(dets[:, 4])])
    keep, source = reference_cuda_nms(srt, THRESH), "reference _nms (oracle/_ref)"
    if keep is None:
        keep, source = O.nms_sorted(srt, THRESH), "oracle nms_sorted"
    path = os.path.join(HERE, "ref_nms_golden.npz")
    np.savez_compressed(path, dets_sorted=srt, keep=np.asarray(keep, np.int32), thresh=np.float32(THRESH), source=np.array(source))
    print("wrote", path, "from", source, "kept", len(keep), "of", len(srt))
