"""Pins oracle/yolo_post.py -- the checker of tb200_graph_yolo_detect (SURVEY.md 8(f)-4) -- against the detection post-processing
of the UNMODIFIED reference example: (a) the committed fixture tests/golden/yolo_example_post.npz, produced by the example's own
functions (generator: tests/golden/make_golden_yolo_post.py); (b) the compiled example's boxes for the heads made from two more
seeds, tests/golden/yolo_example_post_seeded.npz (same generator).  Box for box, bit for bit: coordinates, scores, labels, the
quicksort's tie order, NMS."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle import yolo_post  # noqa: E402

ANCHORS = [10, 14, 23, 27, 37, 58, 81, 82, 135, 169, 344, 319]  # tm_yolov3_tiny_uint8.cpp:178
HEADS = [(0, 32, ANCHORS[6:12]), (1, 16, ANCHORS[0:6])]  # proposal order of main():487-490; anchors[(group - 1) * 6 + ...]


def _restatement(q32, s32, z32, q16, s16, z16):
    got = yolo_post.detect([q32, q16], [np.float32(s32), np.float32(s16)], [int(z32), int(z16)], HEADS, 80, 0.4, 0.25)[0]
    return np.array(got, np.float32).reshape(-1, 6)


def test_restatement_equals_the_committed_output_of_the_unmodified_example():
    d = np.load(os.path.join(ROOT, "tests", "golden", "yolo_example_post.npz"))
    assert np.array_equal(np.array([yolo_post._sigmoid(x) for x in d["sigmoid_x"]], np.float32), d["sigmoid_y"])
    for k in range(3):
        s32, z32, s16, z16 = d[f"qp_{k}"]
        want = d[f"boxes_{k}"]
        got = _restatement(d[f"q32_{k}"], s32, z32, d[f"q16_{k}"], s16, z16)
        assert len(want) > 100 and got.shape == want.shape
        assert np.array_equal(got, want), k


def test_restatement_equals_the_compiled_example_on_seeded_heads():
    import make_golden_yolo_post as gen

    d = np.load(os.path.join(ROOT, "tests", "golden", "yolo_example_post_seeded.npz"))
    for seed in (11, 12):
        heads = gen.random_heads(seed)
        want = d[f"boxes_seed{seed}"]
        got = _restatement(*heads)
        assert got.shape == want.shape and np.array_equal(got, want), seed


def test_device_table_arithmetic_equals_the_restatement():
    """The device looks sigmoid / exp up in 256-entry tables built on the host (engine.cu build_yolo_tables: float expf, the exp table
    held as doubles) and forms exp(dw) * anchor as a double product narrowed to float (yolo_detect.cu).  Emulated here in numpy for
    every byte, both data types and all YOLOv3-tiny anchors: identical to the float arithmetic of the example / restatement."""
    f32 = np.float32
    for is_u8, zero, scale in ((True, 137, 0.0831), (False, 0, 0.0517), (True, 0, 0.19), (True, 255, 0.004)):
        b = np.arange(256)
        q = b.astype(np.float32) if is_u8 else b.astype(np.uint8).view(np.int8).astype(np.float32)
        x = ((q - f32(zero)) * f32(scale)).astype(np.float32)
        sig = np.array([f32(1.0) / f32(f32(1.0) + yolo_post._expf(-v)) for v in x], np.float32)   # the device's table
        ex = np.array([np.float64(yolo_post._expf(v)) for v in x])                                  # (double)expf(x)
        assert np.array_equal(sig, np.array([yolo_post._sigmoid(v) for v in x], np.float32))
        for a in ANCHORS:
            dev = (ex * np.float64(f32(a))).astype(np.float32)        # (float)__dmul_rn(ex, (double)anchor)
            ref = np.array([f32(yolo_post._expf(v) * f32(a)) for v in x], np.float32)
            same = (dev == ref) | (np.isinf(dev) & np.isinf(ref))
            assert same.all(), (is_u8, zero, scale, a)
