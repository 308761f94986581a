import json
import os
import re

import numpy as np

from tengine_b200 import abi
from tengine_b200.graphdef import GraphDef

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    d = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    g = GraphDef.from_dict(d)
    ref = {int(k[5:]): v for k, v in d.items() if k.startswith("ref_t")}
    return g, d["input"], ref


def sha256(a):
    import hashlib

    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def seeded_arrays(g):
    """The arrays of g.to_dict() that the builders derive from numpy seeds alone: weights and weight scales."""
    return {k: v for k, v in g.to_dict().items() if k.endswith(("_weight", "_weight_scales"))}


def seeded_sha256(g):
    d = seeded_arrays(g)
    return sha256(np.concatenate([d[k].reshape(-1).view(np.uint8) for k in sorted(d)] or [np.zeros(0, np.uint8)]))


class Pin:
    """A graph pinned to what the reference was run on, plus the reference's outputs, from tests/golden/reference_pins.npz
    (generator: tests/golden/make_golden_reference_pins.py).  Weights and inputs are rebuilt from their numpy seeds (checked
    against a digest); scales, zero points and biases come from the file, because the workloads calibrate them with a torch fp32
    pass whose last bit depends on the host CPU.  A reference tensor is stored as its values, as its SHA-256 digest, or (deep
    uint8 graphs compared layer by layer) as its difference from the oracle's layer output on the reference's own inputs together
    with its digest -- rebuilt and checked by layer_by_layer()."""

    _file = None

    def __init__(self, name, g):
        if Pin._file is None:
            Pin._file = dict(np.load(os.path.join(GOLDEN, "reference_pins.npz")))
        d = {k[len(name) + 1:]: v for k, v in Pin._file.items() if k.startswith(name + ".")}
        assert d, f"{name}: not in reference_pins.npz (run tests/golden/make_golden_reference_pins.py)"
        assert np.array_equal(seeded_sha256(g), d["seeded_sha256"]), f"{name}: seeded weights differ from the pinned graph"
        self.graph = GraphDef.from_dict({**d, **seeded_arrays(g)})
        self.values = {int(k[1:]): v for k, v in d.items() if re.fullmatch(r"t\d+", k)}
        self.digests = dict(zip(d.get("sha256_ids", []), d.get("sha256", [])))
        ids = list(d.get("delta_ids", []))
        sizes = [int(np.prod(self.graph.dims(t))) for t in ids]
        self.deltas = {t: a.reshape(self.graph.dims(t)) for t, a in zip(ids, np.split(d["delta"], np.cumsum(sizes)[:-1]))} if ids else {}

    def matches(self, t, a):
        """a equals the reference's tensor t byte for byte."""
        return np.array_equal(a, self.values[t]) if t in self.values else np.array_equal(sha256(a), self.digests[t])


def layer_by_layer(oracle, g, x, pin):
    """Run every layer of g alone on the reference's tensors (the graph input x, then the reference's output of each earlier
    layer, rebuilt from `pin` and checked against its digest).  Yields (layer index, the oracle's output, the reference's output)."""
    ref = {g.inputs[0]: x}
    for li, L in enumerate(g.layers):
        h, src = single_layer_graph(g, li)
        got = oracle.run(h, [ref[t] for t in src])[h.outputs[0]]
        t = L["output"]
        ref[t] = (got.astype(np.int32) + pin.deltas[t]).astype(got.dtype)
        assert pin.matches(t, ref[t]), f"layer {li}: the reference's tensor does not rebuild (the oracle's output for it changed)"
        yield li, got, ref[t]


def quant_u8(x, scale, zp):
    # tests/op/test_timvx_op_convolution.cpp:120-132 get_uint8_data
    return np.clip(np.round(np.asarray(x, np.float64) / scale + zp), 0, 255).astype(np.uint8)


def kat_graphs():
    """Build (name, GraphDef, inputs, expected_real, tolerance) from tests/golden/reference_kats.json (`inputs`: one array per graph
    input)."""
    kats = json.load(open(os.path.join(GOLDEN, "reference_kats.json")))["kats"]
    out = []
    for k in kats:
        u8 = k["dtype"] == "uint8"
        g = GraphDef(abi.DT_UINT8 if u8 else abi.DT_INT8)
        n, c, h, w = k["input_dims"]
        x = g.input(n, c, h, w, k["input_scale"], k.get("input_zero", 0))
        if "input_q" in k:
            xin = np.array(k["input_q"], np.int8).reshape(n, c, h, w)
        elif "input_real" in k:  # int8: idata = round(real / scale) (test_opendla_op_relu.cpp:150-156)
            xin = np.clip(np.rint(np.array(k["input_real"], np.float64) / k["input_scale"]), -127, 127).astype(np.int8).reshape(n, c, h, w)
        elif "input_fill" in k:
            xin = quant_u8(np.full((n, c, h, w), k["input_fill"]), k["input_scale"], k["input_zero"])
        else:
            xin = quant_u8(k["input"], k["input_scale"], k["input_zero"]).reshape(n, c, h, w)
        inputs = [xin]
        oz = k.get("output_zero", 0)
        if k["op"] in ("conv", "fc"):
            if u8:
                wq = quant_u8(k["weight"], k["weight_scale"], k["weight_zero"]).reshape(k["weight_dims"])
                ws, wz = [k["weight_scale"]], k["weight_zero"]
            else:
                wq = np.array(k["weight_q"], np.int8).reshape(k["weight_dims"])
                ws, wz = k["weight_scales"], 0
            bq = np.array(k["bias_q"], np.int32) if "bias_q" in k else None
            if k["op"] == "conv":
                y = g.conv(x, wq, bq, ws, k["output_scale"], oz, stride=k["stride"], pad=k["pad"],
                           group=k["group"], activation=k["activation"], weight_zero=wz)
            else:
                y = g.fc(x, wq, bq, ws, k["output_scale"], oz, weight_zero=wz)
        elif k["op"] == "pool":
            y = g.pool(x, abi.POOL_MAX if k["method"] == "max" else abi.POOL_AVG, k["kernel"], k["stride"], k["pad"],
                       out_scale=k["output_scale"], out_zero=oz)
        elif k["op"] == "hardswish":
            y = g.hardswish(x, k["output_scale"], oz)
        elif k["op"] == "sigmoid":
            y = g.sigmoid(x, k["output_scale"], oz)
        elif k["op"] == "softmax":
            y = g.softmax(x, k["output_scale"], oz)
        elif k["op"] == "relu":
            y = g.relu(x, k["output_scale"], oz, negative_slope=k["negative_slope"])
        elif k["op"] == "relu2_sum":  # test_opendla_op_eltwise.cpp: two ReLU nodes on the same input, summed
            y = g.eltwise(g.relu(x, k["output_scale"], oz), g.relu(x, k["output_scale"], oz), k["output_scale"], oz, elt_type=abi.ELT_SUM)
        elif k["op"] in ("eltwise", "concat"):
            x1 = g.input(n, c, h, w, k["input1_scale"], k.get("input1_zero", 0))
            inputs.append(quant_u8(k["input1"], k["input1_scale"], k["input1_zero"]).reshape(n, c, h, w))
            if k["op"] == "eltwise":
                y = g.eltwise(x, x1, k["output_scale"], oz, elt_type=abi.ELT_SUM if k["elt"] == "sum" else abi.ELT_PROD)
            else:
                y = g.concat([x, x1], k["output_scale"], oz)
        else:
            raise ValueError(k["op"])
        g.mark_output(y)
        if "expected_fill" in k:
            exp = np.full(g.dims(y), k["expected_fill"], np.float64)
        else:
            exp = np.array(k["expected"], np.float64).reshape(g.dims(y))
        out.append((k["name"], g, inputs, exp, k.get("tolerance", 0.1)))
    return out


def dequant(g, t, q):
    ti = g.tensors[t]
    return (q.astype(np.float64) - ti["zero_point"]) * ti["scale"]


def layer_outputs(g):
    return [L["output"] for L in g.layers]


def diff_stats(a, b):
    d = np.abs(a.astype(np.int32) - b.astype(np.int32))
    return int(d.max()), int((d > 0).sum())


def single_layer_graph(g, li):
    """Layer `li` of GraphDef `g` as a graph of its own (its input tensors become graph inputs).  Returns the new graph and the
    ids (in `g`) of the tensors to feed.  Used to compare uint8 layers one at a time: the reference simulates uint8 in fp32, so
    each layer may differ by 1 LSB and over a deep network those differences propagate."""
    from tengine_b200.graphdef import GraphDef

    L = g.layers[li]
    h = GraphDef(g.data_type)
    ids = {}
    for t in L["inputs"]:
        if t not in ids:
            src = g.tensors[t]
            h.tensors.append(dict(dims=src["dims"], scale=src["scale"], zero_point=src["zero_point"]))
            ids[t] = len(h.tensors) - 1
            h.inputs.append(ids[t])
    src = g.tensors[L["output"]]
    h.tensors.append(dict(dims=src["dims"], scale=src["scale"], zero_point=src["zero_point"]))
    M = dict(L)
    M["inputs"] = [ids[t] for t in L["inputs"]]
    M["output"] = len(h.tensors) - 1
    h.layers.append(M)
    h.outputs = [M["output"]]
    return h, list(ids.keys())
