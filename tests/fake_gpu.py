"""Stand-ins for the CUDA library (tengine_b200.runtime) and torch.cuda that follow the real interfaces, so that bench.py's control
flow can run without a GPU (tests/test_bench_flow.py, tests/bench_fake_gpu_main.py).  Test infrastructure only."""
import contextlib
import os
import sys
import types

import numpy as np


class FakeContext:
    def __init__(self, device=0, devices=None):
        self.devices = [int(device)] if devices is None else [int(d) for d in devices]
        self.device = self.devices[0]
        self.broadcast_kind = "nccl" if len(self.devices) > 1 else "none"

    def stream_of(self, i):
        return 1000 + i

    def probe_int8_tops(self):
        return 4500.0

    def close(self):
        pass


class FakeGraph:
    """Every output element of image i is a function of image i alone (like the real graphs: images are independent units)."""

    def __init__(self, ctx, gdef, flags=0):
        from tengine_b200 import runtime as real

        self.ctx, self.g = ctx, gdef
        n = gdef.dims(gdef.inputs[0])[0]
        r = len(ctx.devices)
        self._shards = [(ctx.devices[k],) + tuple(real.shard_range(n, r, k)) for k in range(r)]

    def shards(self):
        return list(self._shards)

    def run(self, inputs, outputs=None):
        if os.environ.get("FAKE_GPU_FAIL"):
            raise RuntimeError("injected failure in the middle of the run (FAKE_GPU_FAIL)")
        x = inputs[0]
        key = x.reshape(x.shape[0], -1).astype(np.int64).sum(axis=1)
        outs = outputs if outputs is not None else [np.empty(self.g.dims(o), self.g.np_dtype) for o in self.g.outputs]
        for o in outs:
            o[...] = (key % 251).astype(o.dtype).reshape((-1,) + (1,) * (o.ndim - 1))
        return outs

    def upload(self, i, x):
        pass

    def launch(self):
        pass

    def download(self, i, out):
        out[...] = (np.arange(out.size) % 251).astype(out.dtype).reshape(out.shape)

    def sync(self):
        pass

    def layer_kernels(self):
        names = ["conv_stem_nchw_tcgen05", "conv_dw3x3_tma_dp4a", "gemm_i8_tcgen05", "pool"]
        return [names[min(i, 3) if i < 2 else (1 + i % 2 if i < len(self.g.layers) - 2 else 3)] for i in range(len(self.g.layers))]

    def num_launches(self):
        return len(self.g.layers) + 1

    def profile(self):
        return [0.01 + 0.001 * i for i in range(len(self.g.layers))]

    def work(self):
        return 291.2e9, 2.612e9

    def arena_bytes(self):
        return 600 << 20, 1500 << 20, 4 << 20

    def close(self):
        pass


class FakeEvent:
    clock = [0.0]

    def __init__(self, enable_timing=False):
        self.t = None

    def record(self, stream=None):
        FakeEvent.clock[0] += 0.5
        self.t = FakeEvent.clock[0]

    def elapsed_time(self, other):
        return other.t - self.t



def install():
    """Replace tengine_b200.runtime and the torch.cuda entry points bench.py uses; returns a function that undoes it."""
    import torch

    import tengine_b200
    from tengine_b200 import runtime as real

    fake = types.SimpleNamespace(Context=FakeContext, Graph=FakeGraph, PinnedBuffer=None, shard_range=real.shard_range)
    saved = {"mod": sys.modules.get("tengine_b200.runtime"), "attr": getattr(tengine_b200, "runtime", None), "empty": torch.empty,
             "cuda": {k: getattr(torch.cuda, k) for k in ("set_device", "synchronize", "is_available", "ExternalStream", "Event", "device", "stream")}}
    sys.modules["tengine_b200.runtime"] = fake
    tengine_b200.runtime = fake
    torch.cuda.set_device = lambda d: None
    torch.cuda.synchronize = lambda d=None: None
    torch.cuda.is_available = lambda: False
    torch.cuda.ExternalStream = lambda ptr, device=None: object()
    torch.cuda.Event = FakeEvent
    torch.cuda.device = lambda d: contextlib.nullcontext()
    torch.cuda.stream = lambda s: contextlib.nullcontext()
    real_empty = torch.empty

    def fake_empty(*a, **k):
        # only the device buffers of bench.py (the 256 MB L2-flush buffers) are shrunk and moved to the CPU; everything else (e.g. the
        # buffers torch.distributed allocates) goes through untouched
        if str(k.get("device", "")).startswith("cuda"):
            return real_empty(16, dtype=k.get("dtype", torch.uint8))
        return real_empty(*a, **k)

    torch.empty = fake_empty

    def undo():
        sys.modules["tengine_b200.runtime"] = saved["mod"]
        tengine_b200.runtime = saved["attr"]
        torch.empty = saved["empty"]
        for k, v in saved["cuda"].items():
            setattr(torch.cuda, k, v)

    return undo
