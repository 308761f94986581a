#!/usr/bin/env python3
"""Generate tests/golden/reference_pins.npz: the UNMODIFIED reference (oracle/_ref, built by oracle/build_ref.py where the
reference tree exists) run on every case of tests/test_oracle_vs_reference.py.  Per case the file holds the graph as the
reference ran it without its weights and weight scales (they are rebuilt from their seeds; a digest checks them), and the
reference's output tensors: values where a test compares within a tolerance, SHA-256 digests where it asks for equality, and for
the deep uint8 graphs that are compared layer by layer, digests plus each tensor's difference from the oracle's output for that
layer on the reference's own inputs (which is what lets tests/helpers.py layer_by_layer rebuild the tensor).  Needs
oracle/libtb200_oracle.so as well.

    python tests/golden/make_golden_reference_pins.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.pyoracle import Oracle, Reference  # noqa: E402
from tests.helpers import seeded_arrays, seeded_sha256, sha256, single_layer_graph  # noqa: E402
from tests.test_oracle_vs_reference import CASES  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_pins.npz")


def main():
    ref, oracle = Reference(), Oracle()
    d = {}
    for name, (build, tensors, mode) in CASES.items():
        g, xs = build()
        want, _ = ref.run(g, xs, want=tensors(g))
        seeded = seeded_arrays(g)
        d.update({f"{name}.{k}": v for k, v in g.to_dict().items() if k not in seeded})
        d[f"{name}.seeded_sha256"] = seeded_sha256(g)
        if mode == "values":
            d.update({f"{name}.t{t}": a for t, a in want.items()})
        else:
            d[f"{name}.sha256_ids"] = np.array(list(want), np.int32)
            d[f"{name}.sha256"] = np.stack([sha256(a) for a in want.values()])
        if mode == "delta":  # each layer alone on the reference's own input tensors (tests/helpers.py layer_by_layer)
            have, ids, deltas = {g.inputs[0]: xs[0], **want}, [], []
            for li, L in enumerate(g.layers):
                h, src = single_layer_graph(g, li)
                got = oracle.run(h, [have[t] for t in src])[h.outputs[0]]
                delta = want[L["output"]].astype(np.int32) - got.astype(np.int32)
                assert np.abs(delta).max() < 128, (name, li)
                ids.append(L["output"])
                deltas.append(delta.astype(np.int8).reshape(-1))
            d[f"{name}.delta_ids"] = np.array(ids, np.int32)
            d[f"{name}.delta"] = np.concatenate(deltas)
    np.savez_compressed(OUT, **d)
    print("wrote", OUT, f"({len(CASES)} cases, {os.path.getsize(OUT) / 1e3:.0f} kB)")


if __name__ == "__main__":
    main()
