#!/usr/bin/env python3
"""bench.py -- images/sec of the B200 int8 convolution + GEMM backend on BASELINE.json's headline workload.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload mobilenet_v1_int8] [--batch B] [--global-batch G]

One "step" = one pass of the hot path (the whole MobileNet-v1 int8 224x224 graph: 28 convolutions + global pool,
through tb200_graph_*) over one synthetic batch of 256 images per GPU.
  value   whole-job images/s with the batch already resident in HBM (device timing, CUDA events, max over ranks)
  e2e     the same through the reference-facing call tb200_graph_run() with HOST buffers (plain malloc'd arrays, as Tengine
          hands them over; the library page-locks them on first sight), H2D + D2H inside
  roofline  dominant kernel: algorithmic bytes / its event-timed duration vs the measured HBM peak
  cpu_baseline / --impl reference : the UNMODIFIED reference CPU backend (oracle/_ref) on this box's host cores
Multi-GPU: ONE process drives all N GPUs through the product (a tb200 context over N GPUs): every step hands ONE batch of
256 x N images (weak scaling) -- or --global-batch images (strong scaling, C4/C5) -- to tb200_graph_run, which shards dim 0
over the GPUs; the weights are packed once and reach the other GPUs by ONE ncclBroadcast at prerun; no collective
afterwards.  Under torchrun (one rank per GPU, as the driver launches it) rank 0 does this; the other ranks never touch a GPU:
they follow rank 0 through the barriers it announces over a gloo process group and leave when it says so.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec int8 CNN inference (MobileNet-v1 224x224)"
UNIT = "images/s"
# name -> (builder, data type, resolution, default images per GPU, metric label)
WORKLOADS = {
    "mobilenet_v1_int8": ("mobilenet_v1", "int8", 224, 256, "images/sec int8 CNN inference (MobileNet-v1 224x224)"),
    "mobilenet_v1_uint8": ("mobilenet_v1", "uint8", 224, 256, "images/sec uint8 CNN inference (MobileNet-v1 224x224)"),
    "resnet50_uint8": ("resnet50", "uint8", 224, 512, "images/sec uint8 CNN inference (ResNet-50 224x224)"),
    "resnet50_int8": ("resnet50", "int8", 224, 512, "images/sec int8 CNN inference (ResNet-50 224x224)"),
    "yolov3_tiny_uint8": ("yolov3_tiny", "uint8", 416, 16, "images/sec uint8 CNN inference (YOLOv3-tiny 416x416)"),
    "yolov3_tiny_int8": ("yolov3_tiny", "int8", 416, 16, "images/sec int8 CNN inference (YOLOv3-tiny 416x416)"),
    "yolov5s_int8": ("yolov5s", "int8", 640, 8, "images/sec int8 CNN inference (YOLOv5s 640x640)"),
    "yolov5s_uint8": ("yolov5s", "uint8", 640, 8, "images/sec uint8 CNN inference (YOLOv5s 640x640)"),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False

    def run(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.p.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        try:
            self.p.terminate()
        except Exception:
            pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(workload, batch, family):
    """dram__bytes_read.sum + dram__bytes_write.sum of the kernel family, summed over its launches of one step, from the
    committed `ncu --set full` capture (profiles/rNN_ncu_traffic.json, newest round first, made by tools/ncu_traffic_json.py; not
    measured live: ncu replays every kernel ~40x).  None when no capture is of this workload / batch."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        d = json.load(open(p))
        if d.get("workload") != workload or d.get("batch") != batch:
            continue
        f = d["families"].get(family)
        if f:
            return float(f["dram_bytes_per_step"])
    return None


def build_workload(name, batch):
    from tengine_b200 import abi, workloads

    if name not in WORKLOADS:
        raise SystemExit(f"unknown workload {name}; choose from {sorted(WORKLOADS)}")
    builder, dt, res, _, _ = WORKLOADS[name]
    return getattr(workloads, builder)(abi.DT_INT8 if dt == "int8" else abi.DT_UINT8, batch=batch, res=res)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, outs):
    """Write graph output i as <path>/output<i>.npy, its quantised values as float32 (exact).  When all outputs together exceed
    DUMP_LIMIT_BYTES, each is cut to its share of the limit: a sample of flat indices, seeded by i, in ascending order."""
    os.makedirs(path, exist_ok=True)
    total = 4 * sum(o.size for o in outs)
    for i, o in enumerate(outs):
        a = o.astype(np.float32)
        if total > DUMP_LIMIT_BYTES:
            keep = o.size * DUMP_LIMIT_BYTES // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(i).choice(o.size, keep, replace=False))]
        np.save(os.path.join(path, f"output{i}.npy"), a)


def usable_cpus():
    """CPUs this process may actually use: the affinity mask, capped by the cgroup CPU quota (cpu.max) when one is set."""
    cpus = sorted(os.sched_getaffinity(0))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    n = len(cpus)
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return cpus[:n], quota


def reference_cpu_rate(workload, window_s=12.0, threads_per_proc=int(os.environ.get("TB200_REF_THREADS", "1")), budget_s=170.0):
    """images/s of the UNMODIFIED reference CPU backend (oracle/_ref) using every host core this process may run on
    (affinity mask capped by the cgroup quota): P = cores/T independent processes x T OpenMP threads (T =
    TB200_REF_THREADS, default 1), each pinned to its own CPUs and looping batch-1 run_graph() -- the reference's best
    case for THROUGHPUT: its HCL kernels scale poorly with threads on these layer sizes (measured on 8 cores,
    MobileNet-v1 int8: 8x1 threads 60.7 img/s, 4x2 58.1, 2x4 42.1, 1x8 22.5), its batched int8 path is slower and, for
    3x3, wrong (SURVEY.md fact 8), and its cluster mask cannot describe more than 64 CPUs (source/system/cpu.c:120-121,269).
    Fleet measurement: all workers share ONE wall-clock window (REF_SHIM_WINDOW); each counts the images it completes inside
    it; throughput = sum of the counts / window length.  A starved worker lowers the figure by its own share only (round 1
    divided by the slowest worker's loop time and swung 6x between boxes).  Workers are plain subprocesses
    (python -m oracle.ref_worker) killed by PID if they overrun."""
    import subprocess
    import tempfile

    cpus, quota = usable_cpus()
    t = max(1, min(threads_per_proc, len(cpus)))
    procs = max(1, len(cpus) // t)
    g, b = build_workload(workload, 1)
    d = g.to_dict()
    d["input"] = b.random_input(1)
    tmp = tempfile.NamedTemporaryFile(suffix=".npz", delete=False)
    tmp.close()
    np.savez(tmp.name, **d)
    ps = []
    # start far enough ahead for every worker to have loaded the library, built the graph and done its warm-up run
    lead_s = 6.0 + 0.05 * procs + (6.0 if "resnet" in workload or "yolo" in workload else 0.0)
    t_start = time.time() + lead_s
    try:
        for i in range(procs):
            env = dict(os.environ)
            env["OMP_NUM_THREADS"] = str(t)
            env["REF_SHIM_CPUS"] = ",".join(str(c) for c in cpus[i * t:(i + 1) * t])
            env["REF_SHIM_WINDOW"] = f"{t_start * 1000.0:.3f} {(t_start + window_s) * 1000.0:.3f}"
            env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
            ps.append(subprocess.Popen([sys.executable, "-m", "oracle.ref_worker", tmp.name, "1", str(t)], cwd=ROOT,
                                       env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
        deadline = time.time() + budget_s
        res = []
        for p in ps:
            try:
                out, err = p.communicate(timeout=max(1.0, deadline - time.time()))
            except subprocess.TimeoutExpired:
                raise RuntimeError(f"reference worker pid {p.pid} did not finish within {budget_s:.0f} s")
            if p.returncode != 0:
                raise RuntimeError(f"reference worker failed rc={p.returncode}: {err[-500:]}")
            res.append(json.loads(out.strip().splitlines()[-1]))
    finally:
        for p in ps:
            if p.poll() is None:
                p.kill()
                p.wait()
        os.unlink(tmp.name)
    counts = sorted(r["images"] for r in res)
    total = sum(counts)
    rate = total / window_s
    lat = sorted(r["min_ms"] for r in res if r["images"] > 0)
    sample = (f"{procs} processes x {t} pinned threads looping batch-1 run_graph() of {workload} inside one common {window_s:.0f} s window: "
              f"{total} images (per worker min/median/max {counts[0]}/{counts[len(counts) // 2]}/{counts[-1]}), "
              f"best single-image latency {lat[0] if lat else float('nan'):.1f} ms, cgroup quota {quota if quota is not None else 'none'}")
    return rate, procs * t, sample


def run_reference_arm(args, rank):
    if rank != 0:
        return
    # one "step" = one common 10 s window of the whole worker fleet; warm-up windows are not measured separately (every worker
    # already performs an untimed warm-up run before the window opens) so that K steps finish within minutes
    rates = []
    t0 = time.time()
    steps = max(1, min(args.steps, 3))
    for s in range(steps):
        r, cores, sample = reference_cpu_rate(args.workload, window_s=10.0)
        rates.append(r)
        if time.time() - t0 > 150:
            break
    v = float(np.mean(rates))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(rates),
            "warmup": args.warmup, "ms_per_step": 10000.0, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": WORKLOADS[args.workload][1], "data": "synthetic",
            "config": {"workload": f"{args.workload}, reference CPU backend (oracle/_ref = unmodified source/device/cpu), batch-1 run_graph() loops on every host core; "
                                   f"a step = one 10 s fleet window ({v * 10.0:.0f} images)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def int8_tensor_peak(ctx=None):
    """(TOPS, source): the on-box tcgen05 kind::i8 peak measured live by the library's pure-MMA probe, else twice the measured
    dense bf16 rate of MEASURED_PEAKS.json (kind::i8 issues at twice the bf16 rate), else the nominal 4500."""
    if ctx is not None:
        try:
            t = ctx.probe_int8_tops()
            if t > 100:
                return t, "measured live: tcgen05.mma kind::i8 128x256x32 loop, one CTA per SM (tb200_probe_int8_tops)"
        except Exception:
            pass
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops" in d:
            return 2.0 * float(d["bf16_tflops"]), "2 x measured dense bf16 (MEASURED_PEAKS.json bf16_tflops)"
    return 4500.0, "nominal dense int8 (B200_PROFILING.md)"


# ---- rank protocol under torchrun (N > 1): a process group over gloo (CPU), so that the ranks which only wait never create a CUDA
#      context or an NCCL kernel on "their" GPU -- rank 0's library is the only user of all N GPUs.  The leader announces every
#      barrier before it enters it, so the followers do not need to know how many there are (a count mismatch between the two
#      roles is a dead-lock that only shows on a multi-GPU box). ----
def _gloo_on_loopback():
    """All ranks live on one node (the bench contract): bind gloo to the loopback interface instead of whatever the container's
    hostname resolves to (it may not resolve at all)."""
    os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")


class RankLead:
    def __init__(self, world, devices):
        self.world, self.devices = world, devices
        if world > 1:
            import datetime

            import torch.distributed as dist

            _gloo_on_loopback()
            dist.init_process_group("gloo", timeout=datetime.timedelta(minutes=60))

    def barrier(self):
        import torch

        if torch.cuda.is_available():
            for d in self.devices:
                torch.cuda.synchronize(d)
        if self.world > 1:
            import torch.distributed as dist

            dist.broadcast_object_list(["barrier"], src=0)
            dist.barrier()

    def finish(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.broadcast_object_list(["exit"], src=0)
            dist.destroy_process_group()


def rank_follow(world):
    """Every rank but 0: meet rank 0 at each barrier it announces, leave when it says so."""
    import datetime

    import torch.distributed as dist

    _gloo_on_loopback()
    dist.init_process_group("gloo", timeout=datetime.timedelta(minutes=60))
    n = 0
    while True:
        cmd = [None]
        dist.broadcast_object_list(cmd, src=0)
        if cmd[0] != "barrier":
            break
        dist.barrier()
        n += 1
    dist.destroy_process_group()
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="mobilenet_v1_int8")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (0: the workload's BASELINE.json batch)")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: total images per step, split over the GPUs")
    ap.add_argument("--no-tensorcore", action="store_true", help="route convs through the CUDA-core cross-check kernels")
    ap.add_argument("--cpu-window", type=float, default=12.0, help="cpu_baseline: length of the fleet window in seconds; 0 disables")
    ap.add_argument("--pinned", action="store_true", help="e2e with cudaHostAlloc'd caller buffers instead of pageable ones")
    ap.add_argument("--watchdog", type=float, default=780.0, help="seconds after which a stuck run dumps its Python stacks and exits (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the graph outputs of the last timed step to DIR/output<i>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.watchdog > 0 and int(os.environ.get("RANK", "0")) == 0:
        import faulthandler

        # a hung driver call must not hold the box forever (the followers of rank 0 are torn down by torchrun when it exits)
        faulthandler.dump_traceback_later(args.watchdog, exit=True)

    if args.workload not in WORKLOADS:
        raise SystemExit(f"unknown workload {args.workload}; choose from {sorted(WORKLOADS)}")
    if args.batch <= 0:
        args.batch = WORKLOADS[args.workload][3]
    global METRIC
    METRIC = WORKLOADS[args.workload][4]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    # The product shards the batch over the GPUs INSIDE one process (SURVEY.md 8(e): one tb200 context over N GPUs behind
    # tb200_graph_run).  Under torchrun the driver starts one rank per GPU: rank 0 drives all N GPUs through the library; the other
    # ranks never touch a GPU, they follow rank 0 through its barriers (rank_follow) and exit when it says so.
    ngpu = max(1, args.gpus)
    if rank != 0:
        rank_follow(world)
        return
    lead = RankLead(world, [0] if ngpu == 1 else list(range(ngpu)))
    try:
        import torch

        torch.cuda.set_device(0)
        run_product_arm(args, ngpu, world, lead.barrier)
    finally:
        lead.finish()  # also on an exception: the followers must not be left waiting


def run_product_arm(args, ngpu, world, barrier):
    import torch
    from tengine_b200 import abi
    from tengine_b200 import runtime as rt

    strong = args.global_batch > 0
    total_batch = args.global_batch if strong else args.batch * ngpu
    g, b = build_workload(args.workload, total_batch)
    devices = list(range(ngpu))
    ctx = rt.Context(devices=devices) if ngpu > 1 else rt.Context(0)
    flags = abi.PRERUN_DEFAULT | (abi.PRERUN_NO_TENSORCORE if args.no_tensorcore else 0)
    graph = rt.Graph(ctx, g, flags)  # packs once on GPU 0, ONE ncclBroadcast of the arena to the other GPUs
    shards = graph.shards()

    # caller buffers: plain numpy arrays (malloc'd, pageable) exactly like Tengine's ir_tensor->data; the library page-locks
    # them in place the first time it sees them
    if args.pinned:
        xb = rt.PinnedBuffer(g.dims(g.inputs[0]), g.np_dtype)
        yb = [rt.PinnedBuffer(g.dims(o), g.np_dtype) for o in g.outputs]
        x, ys = xb.array, [y.array for y in yb]
    else:
        x = np.empty(g.dims(g.inputs[0]), g.np_dtype)
        ys = [np.empty(g.dims(o), g.np_dtype) for o in g.outputs]
    rng = np.random.default_rng(42)
    if g.data_type == abi.DT_UINT8:
        x[...] = rng.integers(0, 256, x.shape, dtype=np.uint8)
    else:
        x[...] = rng.integers(-127, 128, x.shape, dtype=np.int8)

    # ---- correctness of every shard before anything is timed: the bytes each GPU produces for its slice must equal what a
    #      plain single-GPU context produces for the same images ----
    graph.run([x], ys)
    verified = "n/a"
    if ngpu > 1:
        sctx = rt.Context(devices[0])
        for (dev, first, count) in shards:
            gs, _ = build_workload(args.workload, count)
            sg = rt.Graph(sctx, gs, flags)
            want = sg.run([np.ascontiguousarray(x[first:first + count])])
            sg.close()
            for o, w in zip(ys, want):
                if not np.array_equal(o[first:first + count], w):
                    raise SystemExit(f"shard on cuda:{dev} (images {first}..{first + count - 1}) differs from the single-GPU result")
        sctx.close()
        verified = f"every shard's output bytes == a single-GPU context's result for the same images ({len(shards)} shards checked)"

    streams = [torch.cuda.ExternalStream(ctx.stream_of(i), device=devices[i]) for i in range(ngpu)]
    flush = [torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{d}") for d in devices]  # > 126 MB L2 each

    # ---------------- device-resident: `value` ----------------
    graph.upload(0, x)
    graph.sync()
    for _ in range(args.warmup):
        graph.launch()
    graph.sync()
    sampler = ClockSampler(devices[0])
    sampler.start()
    time.sleep(0.3)
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] for _ in devices]
    barrier()
    wall0 = time.time()
    for s in range(args.steps):
        for i, d in enumerate(devices):
            with torch.cuda.device(d), torch.cuda.stream(streams[i]):
                flush[i].zero_()  # L2 flush between timed iterations (outside the event pair)
                ev[i][s][0].record(streams[i])
        graph.launch()  # every GPU's shard, asynchronously
        for i, d in enumerate(devices):
            with torch.cuda.device(d):
                ev[i][s][1].record(streams[i])
    for d in devices:
        torch.cuda.synchronize(d)
    barrier()
    wall_dev = time.time() - wall0
    dev_ms = max(sum(a.elapsed_time(b_) for a, b_ in ev[i]) for i in range(ngpu))  # max over GPUs of the K-step device time
    clocks = sampler.finish()
    if args.dump_outputs:
        outs = [np.empty(g.dims(o), g.np_dtype) for o in g.outputs]
        for i, o in enumerate(outs):
            graph.download(i, o)
        graph.sync()
        dump_outputs(args.dump_outputs, outs)

    # ---------------- end to end through the reference-facing call with HOST buffers: `e2e` ----------------
    for _ in range(2):
        graph.run([x], ys)
    barrier()
    t0 = time.perf_counter()
    for s in range(args.steps):
        graph.run([x], ys)  # synchronous: H2D of every GPU's slice, kernels, D2H, join
    e2e_s = time.perf_counter() - t0
    barrier()

    # ---------------- per-kernel profile (events around every launch, GPU 0's shard) for the roofline ----------------
    torch.cuda.set_device(devices[0])
    prof = np.zeros(len(g.layers))
    nprof = min(args.steps, 5)
    for _ in range(nprof):
        prof += np.array(graph.profile())
    prof /= nprof
    kernels = graph.layer_kernels()
    shard0 = shards[0][2]

    images = total_batch * args.steps
    value = images / (dev_ms / 1000.0)
    e2e_value = images / e2e_s
    fam = {}
    for li, k in enumerate(kernels):
        fam.setdefault(k, []).append(li)
    dom = max(fam, key=lambda k: prof[fam[k]].sum())
    dom_ms = float(prof[fam[dom]].sum())
    dom_bytes, dom_ops = 0.0, 0.0
    frac_of_batch = shard0 / float(total_batch)
    for li in fam[dom]:
        L = g.layers[li]
        dom_bytes += (g.numel(L["inputs"][0]) + g.numel(L["output"])) * frac_of_batch
        if L["weight"] is not None:
            dom_bytes += L["weight"].size + (4 * g.dims(L["output"])[1] if L["bias"] is not None else 0)
            dom_ops += 2.0 * g.numel(L["output"]) * frac_of_batch * (L["weight"].size // g.dims(L["output"])[1])
    hbm_peak, hbm_src = measured_peaks()
    tops_peak, tops_src = int8_tensor_peak(ctx)
    ridge = tops_peak * 1e12 / (hbm_peak * 1e9)  # op/B
    intensity = dom_ops / dom_bytes if dom_bytes else 0.0
    if intensity > ridge:
        achieved = dom_ops / (dom_ms / 1000.0) / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": tops_peak, "unit": "TOP/s", "frac": achieved / tops_peak, "peak_source": tops_src}
    else:
        achieved = dom_bytes / (dom_ms / 1000.0) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "peak_source": hbm_src}
    roof.update({"kernel": dom, "launches_per_step": len(fam[dom]), "traffic": ncu_traffic(args.workload, shard0, dom),
                 "kernel_ms_per_step": dom_ms, "share_of_step": dom_ms / float(prof.sum()), "algorithmic_bytes_per_launch_set": dom_bytes,
                 "algorithmic_ops_per_launch_set": dom_ops, "arithmetic_intensity_op_per_byte": intensity, "ridge_op_per_byte": ridge,
                 "measured_on": f"cuda:{devices[0]} (its shard: {shard0} images)"})
    ops, byts = graph.work()
    step_ms = dev_ms / args.steps
    act_bytes, act_unshared, w_bytes = graph.arena_bytes()
    cpu = None
    if args.cpu_window > 0 and ngpu == 1:
        try:
            v, cores, sample = reference_cpu_rate(args.workload, window_s=args.cpu_window)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample}
        except Exception as e:  # oracle/_ref absent
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"unavailable: {e}"}
    res = WORKLOADS[args.workload][2]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ngpu, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": WORKLOADS[args.workload][1], "data": "synthetic",
        "config": {"workload": f"{args.workload} {res}x{res} " + (f"global batch {total_batch} split over {ngpu} GPU(s)" if strong else f"batch={args.batch} per GPU")
                               + (" (BASELINE.json configs[1])" if args.workload == "mobilenet_v1_int8" and not strong else ""),
                   "global_batch": total_batch,
                   "parallelism": (f"ONE process, one tb200 context over {ngpu} GPU(s): dim 0 sharded {[s[2] for s in shards]} inside tb200_graph_run; weights packed on GPU 0, "
                                   f"one {ctx.broadcast_kind} broadcast of the arena at prerun, no collective in the steady state" if ngpu > 1 else "single GPU"),
                   "l2": "256 MiB L2 flush per GPU between timed iterations; per-step activations >> 126 MB L2",
                   "layout": "NHWC int8 in HBM, channels padded to 16",
                   "verified": verified},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(x.nbytes), "d2h_bytes_per_step": int(sum(y.nbytes for y in ys)),
                "ms_per_step": e2e_s * 1000.0 / args.steps,
                "api": "tb200_graph_run(host NCHW in, host NCHW out) -- what the Tengine device's run() calls; caller buffers: "
                       + ("cudaHostAlloc'd" if args.pinned else "plain malloc'd numpy arrays, page-locked in place by the library on first sight")},
        "gpu_launches": graph.num_launches() * args.steps,
        "clocks": clocks,
        "roofline": roof,
        "whole_graph": {"algorithmic_gop_per_step": ops / 1e9, "algorithmic_gb_per_step": byts / 1e9,
                        "achieved_tops": ops / (step_ms / 1000.0) / 1e12, "achieved_gbs": byts / (step_ms / 1000.0) / 1e9,
                        "hbm_frac_per_gpu": byts / ngpu / (step_ms / 1000.0) / 1e9 / hbm_peak,
                        "kernel_ms_gpu0": {k: float(prof[v].sum()) for k, v in fam.items()},
                        "activation_arena_bytes_gpu0": act_bytes, "without_slot_reuse": act_unshared, "weight_arena_bytes": w_bytes},
        "cpu_baseline": cpu,
        "wall_s_device_region": wall_dev,
    }
    print(json.dumps(line), flush=True)
    graph.close()
    ctx.close()


if __name__ == "__main__":
    main()
