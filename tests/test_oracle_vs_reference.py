"""Pins oracle/tb200_oracle.c against the UNMODIFIED reference on seeded random layers -- including which float recipe (HCL /
REF) the reference's CPU device selects for which case.  The reference's outputs for every case below are committed in
tests/golden/reference_pins.npz; tests/golden/make_golden_reference_pins.py regenerates them from oracle/_ref (built by
oracle/build_ref.py where the reference tree exists).  CPU only."""
import numpy as np
import pytest

from tengine_b200 import abi, workloads
from tengine_b200.graphdef import GraphDef
from tests.helpers import Pin, layer_by_layer, layer_outputs


def _rand_conv(rng, dtype, n, c, h, w, oc, k, s, p, g, act, recipe):
    gd = GraphDef(dtype)
    u8 = dtype == abi.DT_UINT8
    x = gd.input(n, c, h, w, 0.02, 128 if u8 else 0)
    kk = (c // g) * k * k
    if u8:
        wq, ws, wz = rng.integers(0, 256, (oc, c // g, k, k)).astype(np.uint8), [0.004], 120
        so = 0.02 * 0.004 * np.sqrt(kk) * 74 * 74 / 100
    else:
        wq, ws, wz = rng.integers(-127, 128, (oc, c // g, k, k)).astype(np.int8), rng.uniform(0.001, 0.01, oc), 0
        so = 0.02 * 0.0055 * np.sqrt(kk) * 73 * 73 / 100
    b = rng.integers(-2000, 2000, oc).astype(np.int32)
    y = gd.conv(x, wq, b, ws, so, 110 if u8 else 0, stride=s, pad=p, group=g, activation=act, recipe=recipe, weight_zero=wz)
    gd.mark_output(y)
    xin = rng.integers(0, 256, (n, c, h, w)).astype(np.uint8) if u8 else rng.integers(-127, 128, (n, c, h, w)).astype(np.int8)
    return gd, xin


# (n, c, h, w, oc, k, stride, pad, group, act, recipe the reference CPU device is expected to follow)
INT8_CASES = [
    (1, 32, 14, 14, 64, 1, 1, 0, 1, 0, abi.RECIPE_HCL),    # conv_hcl_x86 (im2col + sgemm_i8)
    (2, 32, 8, 8, 48, 1, 1, 0, 1, 6, abi.RECIPE_HCL),      # batched 1x1: conv_hcl loops over n
    (1, 16, 15, 15, 24, 3, 1, 1, 1, 6, abi.RECIPE_HCL),    # conv_direct_hcl_int8 3x3 s1
    (1, 16, 15, 15, 24, 3, 2, 1, 1, -1, abi.RECIPE_HCL),   # conv_direct_hcl_int8 3x3 s2
    (1, 32, 16, 16, 32, 3, 1, 1, 32, 0, abi.RECIPE_HCL),   # conv_dw_hcl batch 1
    (1, 32, 16, 16, 32, 3, 2, 1, 32, 0, abi.RECIPE_HCL),
    (2, 32, 16, 16, 32, 3, 1, 1, 32, 0, abi.RECIPE_REF),   # batched depthwise -> conv_ref (conv_dw_hcl_x86.c:536)
    (2, 8, 9, 9, 16, 3, 1, 1, 2, 0, abi.RECIPE_REF),       # grouped, not depthwise -> conv_ref
    (1, 8, 12, 12, 16, 5, 1, 2, 1, 0, abi.RECIPE_HCL),     # 5x5 -> conv_hcl im2col
]

UINT8_CASES = [
    (1, 16, 12, 12, 24, 3, 1, 1, 1, 0, abi.RECIPE_HCL),
    (2, 32, 8, 8, 48, 1, 1, 0, 1, -1, abi.RECIPE_HCL),
    (1, 16, 12, 12, 16, 3, 1, 1, 16, 0, abi.RECIPE_REF),  # uint8 depthwise always conv_ref (conv_dw_hcl_x86.c:532)
    (2, 3, 17, 17, 16, 3, 2, 1, 1, 6, abi.RECIPE_HCL),
]


def _cid(c):
    return "n%d_c%d_%dx%d_oc%d_k%d_s%d_p%d_g%d_a%d_r%d" % c


def _conv_case(dtype, case):
    g, x = _rand_conv(np.random.default_rng(hash(case) & 0xffff), dtype, *case)
    return g, [x]


def _dw_pad_case(stride):
    g, x = _rand_conv(np.random.default_rng(77 + stride), abi.DT_INT8, 1, 32, 15, 17, 32, 3, stride, (1, 1, 0, 0), 32, 0, abi.RECIPE_HCL)
    return g, [x]


def _batched3x3_case(image=None):
    """The batch-2 3x3 convolution; image i: the same layer at batch 1 on image i alone."""
    g, x = _rand_conv(np.random.default_rng(5), abi.DT_INT8, 2, 16, 12, 12, 16, 3, 1, 1, 1, 0, abi.RECIPE_HCL)
    if image is None:
        return g, [x]
    g1, _ = _rand_conv(np.random.default_rng(5), abi.DT_INT8, 1, 16, 12, 12, 16, 3, 1, 1, 1, 0, abi.RECIPE_HCL)
    return g1, [x[image:image + 1]]


def _net_case(build, seed):
    g, b = build()
    return g, [b.random_input(seed)]


def _fc_bias_scale_case():
    rng = np.random.default_rng(3)
    g = GraphDef(abi.DT_UINT8)
    x = g.input(3, 64, 2, 2, 0.02, 128)
    w = rng.integers(0, 256, (40, 256)).astype(np.uint8)
    bias = rng.integers(-30000, 30000, 40).astype(np.int32)
    y = g.fc(x, w, bias, [0.004], 0.05, 120, weight_zero=119)
    g.layers[-1]["bias_scale"] = float(np.float32(0.02 * 0.004 * 1.37))
    g.mark_output(y)
    return g, [rng.integers(0, 256, (3, 64, 2, 2)).astype(np.uint8)]


def _every_layer(g):
    return layer_outputs(g)


def _outputs(g):
    return list(g.outputs)


DTYPES = {"int8": abi.DT_INT8, "uint8": abi.DT_UINT8}
# name -> (builder returning (graph, inputs), tensors the reference is asked for, how tests/helpers.Pin stores them)
CASES = {}
for _c in INT8_CASES:
    CASES["int8_conv_" + _cid(_c)] = (lambda c=_c: _conv_case(abi.DT_INT8, c), _outputs, "digest")
for _c in UINT8_CASES:
    CASES["uint8_conv_" + _cid(_c)] = (lambda c=_c: _conv_case(abi.DT_UINT8, c), _outputs, "values")
for _s in (1, 2):
    CASES[f"int8_dw_pad_s{_s}"] = (lambda s=_s: _dw_pad_case(s), _outputs, "values")
CASES["int8_batched3x3"] = (_batched3x3_case, _outputs, "values")
for _i in (0, 1):
    CASES[f"int8_batched3x3_image{_i}"] = (lambda i=_i: _batched3x3_case(i), _outputs, "digest")
CASES["mobilenet_v1_int8_b1"] = (lambda: _net_case(lambda: workloads.mobilenet_v1(abi.DT_INT8, batch=1), 1), _every_layer, "digest")
CASES["uint8_fc_bias_scale"] = (_fc_bias_scale_case, _outputs, "values")
for _t, _d in DTYPES.items():
    u8 = _d == abi.DT_UINT8
    CASES[f"tiny_net_{_t}"] = (lambda d=_d: _net_case(lambda: workloads.tiny_net(d, batch=2, seed=21), 9), _every_layer, "values" if u8 else "digest")
    CASES[f"tail_net_{_t}"] = (lambda d=_d: _net_case(lambda: workloads.tail_net(d, batch=2), 3), _every_layer, "digest")
    CASES[f"resnet50_{_t}"] = (lambda d=_d: _net_case(lambda: workloads.resnet50(d, batch=1, res=96, width=0.25, classes=40, seed=5), 3),
                               _every_layer, "delta" if u8 else "digest")
    CASES[f"yolov3_tiny_{_t}"] = (lambda d=_d: _net_case(lambda: workloads.yolov3_tiny(d, batch=1, res=96, width=0.25, head=27, seed=6), 3),
                                  _every_layer, "delta" if u8 else "digest")
    CASES[f"yolov5s_{_t}"] = (lambda d=_d: _net_case(lambda: workloads.yolov5s(d, batch=1, res=128, width=0.25, head=27, seed=3), 2),
                              _every_layer, "delta" if u8 else "digest")


def pinned(name):
    """(graph as the reference ran it, its inputs, the reference's outputs as a Pin)."""
    g, xs = CASES[name][0]()
    p = Pin(name, g)
    return p.graph, xs, p


@pytest.mark.parametrize("case", INT8_CASES, ids=_cid)
def test_int8_conv_bit_exact_and_recipe(oracle, case):
    gd, (xin,), ref = pinned("int8_conv_" + _cid(case))
    got = oracle.run(gd, [xin])[gd.outputs[0]]
    assert ref.matches(gd.outputs[0], got)
    assert (np.abs(got.astype(int)) >= 127).mean() < 0.2, "test vacuous: output saturated"


@pytest.mark.parametrize("stride", [1, 2])
def test_int8_depthwise_pad_h_differs_from_pad_w_uses_the_hcl_recipe(oracle, stride):
    """conv_dw_hcl_x86.c:539 only asks pad_h0 == pad_h1 and pad_w0 == pad_w1; pad_h may differ from pad_w (the kernel pads each
    axis with its own value, :131-132).  The device glue's conv_recipe() mirrors exactly this predicate."""
    gd, (xin,), pin = pinned(f"int8_dw_pad_s{stride}")
    ref = pin.values[gd.outputs[0]]
    assert np.array_equal(oracle.run(gd, [xin])[gd.outputs[0]], ref)
    gd.layers[0]["recipe"] = abi.RECIPE_REF  # the other recipe is NOT what the reference computes here (rare 1-LSB cases)
    other = oracle.run(gd, [xin])[gd.outputs[0]]
    assert np.abs(other.astype(int) - ref.astype(int)).max() <= 1


def test_int8_batched_3x3_reference_bug_is_known(oracle):
    """SURVEY fact 8: conv3x3s1_int8_sse ignores the batch dimension (conv_direct_hcl_int8_x86.c:95-200) but wins the
    selection for every int8 3x3 conv; images n>0 are therefore NOT computed by the reference's default path.  The
    oracle (and the device) compute every image; image 0 must agree."""
    gd, (xin,), want = pinned("int8_batched3x3")
    got = oracle.run(gd, [xin])[gd.outputs[0]]
    assert np.array_equal(got[0], want.values[gd.outputs[0]][0])
    # batch-1 runs of each image are the batch-correct reference
    for i in range(2):
        g1, _, w1 = pinned(f"int8_batched3x3_image{i}")
        assert w1.matches(g1.outputs[0], got[i:i + 1])


@pytest.mark.parametrize("case", UINT8_CASES, ids=_cid)
def test_uint8_conv_within_1lsb(oracle, case):
    gd, (xin,), pin = pinned("uint8_conv_" + _cid(case))
    ref = pin.values[gd.outputs[0]]
    assert ((ref == 0) | (ref == 255)).mean() < 0.3, "test vacuous: output saturated"
    for mode in (0, 1):
        got = oracle.run(gd, [xin], uint8_mode=mode)[gd.outputs[0]]
        d = np.abs(got.astype(int) - ref.astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 0.01, (mode, int(d.max()), float((d > 0).mean()))


@pytest.mark.parametrize("dtype", [abi.DT_INT8, abi.DT_UINT8])
def test_every_op_of_tiny_net(oracle, dtype):
    g, (x,), want = pinned("tiny_net_" + ("uint8" if dtype == abi.DT_UINT8 else "int8"))
    got = oracle.run(g, [x])
    for li, L in enumerate(g.layers):
        t = L["output"]
        if dtype == abi.DT_INT8:
            assert want.matches(t, got[t]), (li, abi.OP_NAMES[L["op"]])
        else:
            d = np.abs(got[t].astype(int) - want.values[t].astype(int))
            assert d.max() <= 1, (li, abi.OP_NAMES[L["op"]], int(d.max()))


def test_mobilenet_v1_int8_batch1_bit_exact(oracle):
    """C1 of BASELINE.json: tm_classification_int8 MobileNet-v1 224x224 batch 1 on the reference CPU backend."""
    g, (x,), want = pinned("mobilenet_v1_int8_b1")
    got = oracle.run(g, [x])
    for li, L in enumerate(g.layers):
        assert want.matches(L["output"], got[L["output"]]), f"layer {li}"
    assert len(np.unique(got[g.outputs[0]])) > 50, "test vacuous: classifier output collapsed"


@pytest.mark.parametrize("dtype", [abi.DT_INT8, abi.DT_UINT8], ids=["int8", "uint8"])
@pytest.mark.parametrize("net", ["resnet50", "yolov3_tiny"])
def test_benchmark_graphs_with_inplace_scales(oracle, net, dtype):
    """C3 / C4 of BASELINE.json at reduced width, quantised the way the reference's own tool does (max pooling and ReLU outputs
    share the input's scale, tools/quantize/quant_save_graph.cpp:136-200): every layer of the oracle against the UNMODIFIED
    reference.  This is what the device's byte-wise same-scale pooling / ReLU kernels and the gather-convolution kernels are
    ultimately compared with (tests/test_gpu_parity.py checks device == oracle on the same graphs)."""
    g, (x,), want = pinned(f"{net}_" + ("uint8" if dtype == abi.DT_UINT8 else "int8"))
    if dtype == abi.DT_INT8:
        got = oracle.run(g, [x])
        for li, L in enumerate(g.layers):
            assert want.matches(L["output"], got[L["output"]]), f"{net} layer {li} {abi.OP_NAMES[L['op']]}"
        return
    # uint8: layer by layer on the reference's own tensors (1 LSB per layer is the reference's fp32 noise; over 50+ layers it
    # propagates to ~10 LSB, which says nothing about any single layer)
    for li, got, ref in layer_by_layer(oracle, g, x, want):
        d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
        assert d.max() <= 1, f"{net} layer {li} {abi.OP_NAMES[g.layers[li]['op']]}: {int(d.max())} LSB"


@pytest.mark.parametrize("dtype", [abi.DT_INT8, abi.DT_UINT8], ids=["int8", "uint8"])
def test_tail_ops_sigmoid_mul_hardswish_flatten_softmax(oracle, dtype):
    """Glue ops around the classifier / detection heads (SURVEY.md 8(f)-1): Sigmoid, Eltwise-PROD (x * sigmoid(x): the int8
    spelling of YOLOv5s' activation), HardSwish (uint8 only in the reference), Flatten, FC, Softmax -- oracle == reference."""
    g, (x,), want = pinned("tail_net_" + ("uint8" if dtype == abi.DT_UINT8 else "int8"))
    got = oracle.run(g, [x])
    kinds = set()
    for li, L in enumerate(g.layers):
        t = L["output"]
        kinds.add(abi.OP_NAMES[L["op"]])
        assert want.matches(t, got[t]), (li, abi.OP_NAMES[L["op"]])
        assert len(np.unique(got[t])) > 8, "test vacuous"
    assert {"sigmoid", "softmax", "reshape", "eltwise"} <= kinds and (("hardswish" in kinds) == (dtype == abi.DT_UINT8))


def test_uint8_fc_uses_the_bias_tensors_own_scale(oracle):
    """fc_ref.c:141-146 multiplies the int32 bias by bias_tensor->scale, which a tmfile may set to something other than
    fl(s_in*s_w) (e.g. computed in double by the quantisation tool)."""
    g, (xin,), pin = pinned("uint8_fc_bias_scale")
    y = g.outputs[0]
    want = pin.values[y]
    got = oracle.run(g, [xin], uint8_mode=0)[y]
    d = np.abs(got.astype(int) - want.astype(int))
    assert d.max() <= 1 and len(np.unique(want)) > 20
    g.layers[-1]["bias_scale"] = float(np.float32(0.02) * np.float32(0.004))
    other = oracle.run(g, [xin], uint8_mode=0)[y]
    assert np.abs(other.astype(int) - want.astype(int)).max() > 1, "test vacuous: the bias scale does not matter here"


@pytest.mark.parametrize("dtype", [abi.DT_INT8, abi.DT_UINT8], ids=["int8", "uint8"])
def test_yolov5s_reduced_every_layer(oracle, dtype):
    """C5 of BASELINE.json (YOLOv5s; int8 keeps SiLU as Sigmoid + Eltwise-PROD, uint8 uses HardSwish as the reference's
    yolov5s-opt.py writes it) at reduced width / resolution: every layer of the oracle against the UNMODIFIED reference."""
    g, (x,), want = pinned("yolov5s_" + ("uint8" if dtype == abi.DT_UINT8 else "int8"))
    if dtype == abi.DT_INT8:
        got = oracle.run(g, [x])
        for li, L in enumerate(g.layers):
            assert want.matches(L["output"], got[L["output"]]), f"layer {li} {abi.OP_NAMES[L['op']]}"
        assert all(len(np.unique(got[t])) > 20 for t in g.outputs)
        return
    for li, got, ref in layer_by_layer(oracle, g, x, want):
        d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
        assert d.max() <= 1, f"layer {li} {abi.OP_NAMES[g.layers[li]['op']]}: {int(d.max())} LSB"
