"""Generates tests/golden/box_iou_rotated.npz from the REFERENCE's own arithmetic: oracle/_ref/libbox_iou_rotated_ref.so is
/root/reference/torchvision/csrc/ops/box_iou_rotated_utils.h compiled as it lies (oracle/Makefile, target `ref`).  Run in the
build container (the GPU box has no /root/reference):  python tests/golden/gen_golden_rotated.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402


def boxes(rng, n, span=200.0):
    c = rng.uniform(0, span, (n, 2))
    wh = np.exp(rng.uniform(0, 5, (n, 2)))
    a = rng.uniform(-180, 180, (n, 1))
    return np.concatenate([c, wh, a], 1).astype(np.float32)


def main():
    oracle.build()
    rng = np.random.default_rng(1234)
    b1, b2 = boxes(rng, 257), boxes(rng, 193)
    b2[:40] = b1[:40]                                   # identical boxes: IoU 1
    b2[40:70] = b1[40:70]; b2[40:70, 4] += 90.0          # same box rotated by 90 degrees
    b2[70:90, :2] = b1[70:90, :2]                       # concentric
    b2[90:110] = b1[90:110]; b2[90:110, 4] += 1e-3       # nearly coincident edges
    b2[110:115, 2] = 0.0                                # degenerate (zero area)
    b1[200:210, 4] = 0.0; b2[115:125, 4] = 0.0          # axis-aligned
    # test/test_ops.py-style unit boxes
    u1 = np.array([[0.5, 0.5, 1, 1, 0], [0.5, 0.5, 1, 1, 45], [0, 0, 2, 1, 30]], np.float32)
    u2 = np.array([[0.5, 0.5, 1, 1, 0], [1.0, 0.5, 1, 1, 0], [0.5, 0.5, 1, 1, 90], [0, 0, 1, 2, -60]], np.float32)
    # the seeded boxes of tests/test_oracle.py::test_box_iou_rotated_golden_and_ref against themselves in reverse order
    rng = np.random.default_rng(7)
    c = rng.uniform(0, 100, (150, 2)); wh = np.exp(rng.uniform(0, 4, (150, 2))); a = rng.uniform(-360, 360, (150, 1))
    rb = np.concatenate([c, wh, a], 1).astype(np.float32)
    ref = oracle.box_iou_rotated_ref(b1, b2)
    assert ref is not None, "oracle/_ref/libbox_iou_rotated_ref.so is missing (needs /root/reference)"
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "box_iou_rotated.npz"), boxes1=b1, boxes2=b2, ious=ref, unit1=u1,
                        unit2=u2, unit_ious=oracle.box_iou_rotated_ref(u1, u2), rand_boxes=rb,
                        rand_ious=oracle.box_iou_rotated_ref(rb, rb[::-1].copy()))
    print("wrote box_iou_rotated.npz", ref.shape, float(ref.max()), float((ref > 0).mean()))


if __name__ == "__main__":
    main()
