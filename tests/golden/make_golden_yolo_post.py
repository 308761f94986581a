#!/usr/bin/env python3
"""Golden vectors for oracle/yolo_post.py: the detection post-processing of the UNMODIFIED examples/tm_yolov3_tiny_uint8.cpp
(compiled by oracle/build_ref.py into oracle/_ref/libyolo_example.so through oracle/yolo_example_shim.cpp), run on seeded
quantised head tensors.  Needs the reference tree at build time; the .npz files it writes are committed so that the pin holds
anywhere.
usage: make_golden_yolo_post.py [out.npz]"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(ROOT, "oracle", "_ref", "libyolo_example.so")


def example_lib():
    L = C.CDLL(LIB)
    L.yolo_example_postprocess.restype = C.c_int
    L.yolo_example_postprocess.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_int]
    L.yolo_example_sigmoid.restype = C.c_float
    L.yolo_example_sigmoid.argtypes = [C.c_float]
    return L


def random_heads(seed):
    """Quantised head tensors [1, 255, 13, 13] and [1, 255, 26, 26] with objectness shifted low (a few hundred proposals pass 0.4,
    plenty of overlaps for the NMS and equal scores for the sort's tie order)."""
    rng = np.random.default_rng(seed)
    s32, s16 = np.float32(rng.uniform(0.05, 0.2)), np.float32(rng.uniform(0.05, 0.2))
    z32, z16 = int(rng.integers(100, 180)), int(rng.integers(100, 180))
    q32 = rng.integers(0, 256, (1, 255, 13, 13)).astype(np.uint8)
    q16 = rng.integers(0, 256, (1, 255, 26, 26)).astype(np.uint8)
    for q, z in ((q32, z32), (q16, z16)):
        for a in range(3):
            q[0, a * 85 + 4] = np.clip(rng.normal(z - 40, 25, q[0, a * 85 + 4].shape), 0, 255).astype(np.uint8)
    return q32, s32, z32, q16, s16, z16


def run_example(L, q32, s32, z32, q16, s16, z16, prob=0.4, nms=0.25):
    p32 = ((q32[0].astype(np.float32) - np.float32(z32)) * s32).astype(np.float32)  # main():464-478
    p16 = ((q16[0].astype(np.float32) - np.float32(z16)) * s16).astype(np.float32)
    out = np.zeros((8192, 6), np.float32)
    n = L.yolo_example_postprocess(p32.ctypes.data, p16.ctypes.data, prob, nms, out.ctypes.data, len(out))
    assert 0 <= n <= len(out)
    return out[:n].copy()


def write_seeded(L, out=os.path.join(HERE, "yolo_example_post_seeded.npz")):
    """The example's boxes for the heads random_heads() makes from seeds 11 and 12 (tests/test_yolo_post_pinned.py rebuilds the heads)."""
    np.savez_compressed(out, **{f"boxes_seed{seed}": run_example(L, *random_heads(seed)) for seed in (11, 12)})
    print("wrote", out)


if __name__ == "__main__":
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "yolo_example_post.npz")
    L = example_lib()
    write_seeded(L)
    d = {}
    for k, seed in enumerate((5, 6, 7)):
        q32, s32, z32, q16, s16, z16 = random_heads(seed)
        d.update({f"q32_{k}": q32, f"q16_{k}": q16, f"qp_{k}": np.array([s32, z32, s16, z16], np.float64), f"boxes_{k}": run_example(L, q32, s32, z32, q16, s16, z16)})
    xs = ((np.arange(256) - 128.0) * 0.137).astype(np.float32)
    d["sigmoid_x"] = xs
    d["sigmoid_y"] = np.array([L.yolo_example_sigmoid(float(x)) for x in xs], np.float32)
    np.savez_compressed(out, **d)
    print("wrote", out, {k: v.shape for k, v in d.items() if k.startswith("boxes")})
