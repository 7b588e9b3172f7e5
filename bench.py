#!/usr/bin/env python3
"""bench.py -- the hot-path benchmark (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3|c4|c5] [--dump-outputs DIR]

One "step" = one pass of the workload's op list over one batch of synthetic frames.  Default workload = BASELINE.json
configs[1] ("c2"): the filter2D / sepFilter2D / GaussianBlur sweep 3x3..31x31 on 3840x2160 CV_8UC1 and CV_32FC1.
Prints ONE JSON line (rank 0):  metric = Mpix/s (destination pixels of every op, whole job), `value` = device-resident,
`e2e` = same ops through the host C ABI (pinned host buffers, H2D + D2H inside the timed region), `roofline` for the
kernel with the largest share of the step, `per_op` for every op, `cpu_baseline` = the reference's own CPU path
(oracle/_ref, or the C port when that is absent) on a bounded sample, `clocks` sampled during the timed region.
Multi-GPU (torchrun): frames shard across ranks (weak scaling); the only collective is an NCCL broadcast of the filter
taps / template per step.
--dump-outputs DIR: after the timed steps, rank 0 writes what every op of the workload returned in the last timed step as
DIR/<op>.npy (see dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared output by output.
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

K_SWEEP = (3, 5, 7, 9, 11, 13, 15, 21, 31)
W4K, H4K = 3840, 2160
W8K, H8K = 7680, 4320


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
# workload definitions: list of ops; each op = dict(name, make(ctx)->callable, px (dst pixels per frame), bytes (algorithmic
# bytes per frame, SURVEY 8d), frames)
# ------------------------------------------------------------------------------------------------------------------
def gauss_taps(k):
    import opencv_b200 as cvb
    return cvb.getGaussianKernel(k, 0).astype(np.float32)


def build_ops(workload, rng):
    """returns (ops, description).  Each op: name, kind, args, src spec (shape, dtype), dst spec, px, algo_bytes per frame"""
    ops = []
    if workload == "c1":
        nb = 64
        ops.append(dict(name="GaussianBlur_8UC3_1080p_k5", kind="gauss", k=5, src=((nb, 1080, 1920, 3), np.uint8), dst=((nb, 1080, 1920, 3), np.uint8),
                        px=1920 * 1080, abytes=1920 * 1080 * 6, frames=nb))
        desc = "C1: GaussianBlur 5x5 on 1920x1080 8UC3 (the reference's own CPU-runnable case), 64 frames per launch"
    elif workload == "c2":
        for depth, nb, es in (("u8", 16, 1), ("f32", 8, 4)):
            dt = np.uint8 if depth == "u8" else np.float32
            for k in K_SWEEP:
                ops.append(dict(name="GaussianBlur_%s_k%d" % (depth, k), kind="gauss", k=k, src=((nb, H4K, W4K, 1), dt), dst=((nb, H4K, W4K, 1), dt),
                                px=W4K * H4K, abytes=W4K * H4K * 2 * es, frames=nb))
            for k in K_SWEEP:
                ops.append(dict(name="sepFilter2D_%s_k%d" % (depth, k), kind="sep", k=k, src=((nb, H4K, W4K, 1), dt), dst=((nb, H4K, W4K, 1), dt),
                                px=W4K * H4K, abytes=W4K * H4K * 2 * es, frames=nb))
            for k in K_SWEEP:
                ops.append(dict(name="filter2D_%s_k%d" % (depth, k), kind="f2d", k=k, src=((nb, H4K, W4K, 1), dt), dst=((nb, H4K, W4K, 1), dt),
                                px=W4K * H4K, abytes=W4K * H4K * 2 * es, frames=nb))
        desc = "C2: GaussianBlur/sepFilter2D/filter2D k in %s on 3840x2160 8UC1 (16 frames/op) and 32FC1 (8 frames/op)" % (K_SWEEP,)
    elif workload == "c3":
        nb = 4
        s8 = ((nb, H8K, W8K, 3), np.uint8)
        for name, dsz, interp, ab in (("resize_8Kto4K_NEAREST", (3840, 2160), 0, 49.77e6), ("resize_8Kto4K_LINEAR", (3840, 2160), 1, 124.42e6),
                                      ("resize_8Kto5K_LINEAR", (5120, 2880), 1, 143.77e6), ("resize_8Kto5K_CUBIC", (5120, 2880), 2, 143.77e6)):
            ops.append(dict(name=name, kind="resize", interp=interp, src=s8, dst=((nb, dsz[1], dsz[0], 3), np.uint8), px=dsz[0] * dsz[1], abytes=ab, frames=nb))
        for i, nm in ((0, "NEAREST"), (1, "LINEAR"), (2, "CUBIC")):
            ops.append(dict(name="resize_4Kto8K_" + nm, kind="resize", interp=i, src=((nb, H4K, W4K, 3), np.uint8), dst=s8, px=W8K * H8K, abytes=124.42e6, frames=nb))
        for i, nm in ((0, "NEAREST"), (1, "LINEAR"), (2, "CUBIC")):
            ops.append(dict(name="warpAffine_8K_" + nm, kind="affine", interp=i, src=s8, dst=s8, px=W8K * H8K, abytes=199.07e6, frames=nb))
            ops.append(dict(name="warpPerspective_8K_" + nm, kind="persp", interp=i, src=s8, dst=s8, px=W8K * H8K, abytes=199.07e6, frames=nb))
        for nm, code, scn, dcn in (("BGR2GRAY", 6, 3, 1), ("GRAY2BGR", 8, 1, 3), ("BGR2YUV", 82, 3, 3), ("YUV2BGR", 84, 3, 3), ("BGR2HSV", 40, 3, 3), ("HSV2BGR", 54, 3, 3)):
            ops.append(dict(name="cvtColor_8K_" + nm, kind="cvt", code=code, src=((nb, H8K, W8K, scn), np.uint8), dst=((nb, H8K, W8K, dcn), np.uint8),
                            px=W8K * H8K, abytes=W8K * H8K * (scn + dcn), frames=nb))
        desc = "C3: resize / warpAffine / warpPerspective (NEAREST/LINEAR/CUBIC) + cvtColor on 7680x4320 8UC3, 4 frames/op"
    elif workload == "c4":
        nb = 16
        ops.append(dict(name="matchTemplate_CCORR_NORMED_4K_64x64", kind="mt", src=((nb, H4K, W4K, 1), np.uint8), dst=((nb, H4K - 63, W4K - 63, 1), np.float32),
                        px=(W4K - 63) * (H4K - 63), abytes=39.98e6, frames=nb, flops=6.488e10))
        ops.append(dict(name="cornerHarris_4K", kind="harris", src=((nb, H4K, W4K, 1), np.uint8), dst=((nb, H4K, W4K, 1), np.float32), px=W4K * H4K, abytes=41.47e6, frames=nb))
        ops.append(dict(name="goodFeaturesToTrack_4K", kind="gftt", src=((4, H4K, W4K, 1), np.uint8), dst=None, px=W4K * H4K, abytes=41.47e6, frames=4))
        desc = "C4: matchTemplate TM_CCORR_NORMED 4K vs 64x64, cornerHarris(2,3,0.04), goodFeaturesToTrack(1000,0.01,10) on 3840x2160 8UC1"
    elif workload == "c5":
        nb = 4
        ops.append(dict(name="SIFT_pyramid_DoG_4K", kind="sift", src=((nb, H4K, W4K, 1), np.uint8), dst=None, px=W4K * H4K, abytes=2883.7e6, frames=nb))
        ops.append(dict(name="cornerHarris_4K", kind="harris", src=((nb, H4K, W4K, 1), np.uint8), dst=((nb, H4K, W4K, 1), np.float32), px=W4K * H4K, abytes=41.47e6, frames=nb))
        desc = "C5: SIFT Gaussian pyramid + DoG (3 layers, sigma 1.6, upscaled base) + cornerHarris on 3840x2160 8UC1 frames, 4 frames/rank/step"
    else:
        raise SystemExit("unknown workload " + workload)
    return ops, desc


ROT = None
HPERSP = np.array([[0.95, 0.02, 50], [-0.015, 0.97, 30], [1e-6, 2e-6, 1]])


def rotation_matrix():
    # getRotationMatrix2D((3840,2160), 7 deg, 0.9)  (imgwarp.cpp:3468-3490)
    a = np.deg2rad(7.0); al = 0.9 * np.cos(a); be = 0.9 * np.sin(a); cx, cy = 3840.0, 2160.0
    return np.array([[al, be, (1 - al) * cx - be * cy], [-be, al, be * cx + (1 - al) * cy]])


def filter_kernel(k, rng):
    ker = rng.random((k, k)).astype(np.float32)
    return ker / ker.sum()


def run_op(api, op, src, dst, extra):
    """api: opencv_b200 (torch tensors) or opencv_b200.hal (numpy) -- same names and argument meaning"""
    kind = op["kind"]
    if kind == "gauss":
        return api.GaussianBlur(src, (op["k"], op["k"]), 0, dst=dst)
    if kind == "sep":
        t = extra["taps"][op["k"]]
        return api.sepFilter2D(src, -1, t, t, dst=dst)
    if kind == "f2d":
        return api.filter2D(src, -1, extra["kernels"][op["k"]], dst=dst)
    if kind == "resize":
        return api.resize(src, (dst.shape[2], dst.shape[1]), interpolation=op["interp"], dst=dst)
    if kind == "affine":
        return api.warpAffine(src, extra["rot"], (dst.shape[2], dst.shape[1]), flags=op["interp"], dst=dst)
    if kind == "persp":
        return api.warpPerspective(src, HPERSP, (dst.shape[2], dst.shape[1]), flags=op["interp"], dst=dst)
    if kind == "cvt":
        return api.cvtColor(src, op["code"], dst=dst)
    if kind == "mt":
        return api.matchTemplate(src, extra["templ"], 3, result=dst)
    if kind == "harris":
        return api.cornerHarris(src, 2, 3, 0.04, dst=dst)
    if kind == "gftt":
        return api.goodFeaturesToTrack(src, 1000, 0.01, 10, 3, 3, True, 0.04)
    if kind == "sift":
        return api.sift_pyramid(src, 3, 1.6, True)
    raise ValueError(kind)


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons, self.maxmhz = [], set(), None
        self.stop_flag = False

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.maxmhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception:
            self._run_smi()

    def _run_smi(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0])); self.maxmhz = float(f[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.15)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxmhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------------------------
def reference_oracle():
    from oracle.api import Oracle, available
    if available("ref"):
        return Oracle("ref"), "reference"
    from oracle import build_port
    build_port.build()
    return Oracle("port"), "port"


def cpu_run_op(orc, op, src, extra):
    kind = op["kind"]
    if kind == "gauss":
        return orc.GaussianBlur(src, (op["k"], op["k"]), 0)
    if kind == "sep":
        t = extra["taps"][op["k"]]
        return orc.sepFilter2D(src, -1, t, t)
    if kind == "f2d":
        return orc.filter2D(src, -1, extra["kernels"][op["k"]])
    if kind == "resize":
        return orc.resize(src, (op["dst"][0][2], op["dst"][0][1]), op["interp"])
    if kind == "affine":
        return orc.warpAffine(src, extra["rot"], (op["dst"][0][2], op["dst"][0][1]), op["interp"])
    if kind == "persp":
        return orc.warpPerspective(src, HPERSP, (op["dst"][0][2], op["dst"][0][1]), op["interp"])
    if kind == "cvt":
        return orc.cvtColor(src, op["code"], op["dst"][0][3])
    if kind == "mt":
        return orc.matchTemplate(src, extra["templ_np"], 3)
    if kind == "harris":
        return orc.cornerHarris(src, 2, 3, 0.04)
    if kind == "gftt":
        return orc.goodFeaturesToTrack(src, 1000, 0.01, 10, 3, 3, True, 0.04)
    if kind == "sift":
        return orc.sift_pyramid(src, 3, 1.6, True)
    raise ValueError(kind)


def cpu_frames(ops, rng):
    """one synthetic frame per distinct source spec"""
    cache = {}
    for op in ops:
        shp, dt = op["src"]
        key = (shp[1:], np.dtype(dt).str)
        if key not in cache:
            a = rng.integers(0, 256, shp[1:], dtype=np.uint8)
            a = a[:, :, 0] if shp[3] == 1 else a
            cache[key] = a.astype(dt)
        op["_cpu_src"] = cache[key]


def cpu_pass(orc, ops, extra):
    t0 = time.perf_counter()
    px = 0
    for op in ops:
        cpu_run_op(orc, op, op["_cpu_src"], extra)
        px += op["px"]
    return time.perf_counter() - t0, px


def make_extra(ops, rng, need_device):
    extra = {"taps": {k: None for k in K_SWEEP}, "kernels": {}, "rot": rotation_matrix()}
    for k in K_SWEEP:
        extra["kernels"][k] = filter_kernel(k, rng)
    return extra


DUMP_BYTES = 64_000_000


def dump_outputs(ops, out_dir, dev):
    """What each op returned in the last step, as DIR/<op name>[_<i>].npy (one file per array of the result, in the order the op returns
    them): float64 results stay float64, 8- and 16-bit results and float32 become float32, wider integers float64 -- all exact.  The files
    hold at most DUMP_BYTES together: an array larger than its share is written as a fixed sample of its elements (flattened, at sorted
    positions drawn from a generator seeded with the file name), the same positions in every run."""
    import zlib
    import torch
    arrays = []

    def leaves(name, x):
        if isinstance(x, (list, tuple)):
            items = [v for v in x if v is not None]
            for i, v in enumerate(items):
                leaves(name if len(items) == 1 else "%s_%d" % (name, i), v)
        elif x is not None:
            arrays.append((name, x))
    for op in ops:
        leaves(op["name"], op["_out"])
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays)) - 256          # 256: room for the .npy header
    for name, a in arrays:
        dt = np.float64 if str(a.dtype).endswith(("float64", "int32", "int64")) else np.float32
        n = int(a.numel()) if isinstance(a, torch.Tensor) else int(a.size)
        keep = share // np.dtype(dt).itemsize
        idx = None
        if n > keep:
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).integers(0, n, keep))
        if isinstance(a, torch.Tensor):
            t = a.reshape(-1)[torch.from_numpy(idx).to(dev)] if idx is not None else a
            v = t.cpu().numpy()
        else:
            v = np.asarray(a).reshape(-1)[idx] if idx is not None else np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), v.astype(dt))


def measure_device(workload, steps, W, use_graph, rank, world, local, rng, sample_clocks=True, dump_dir=None):
    """device-resident pass of one workload: returns (result dict, ops, extra, bufs).  value = Mpix/s over `steps` steps (CUDA events, max over ranks)"""
    import torch
    import torch.distributed as dist
    import opencv_b200 as cvb
    dev = torch.device("cuda", local)
    ops, desc = build_ops(workload, rng)
    extra = make_extra(ops, rng, True)

    # device-resident inputs / outputs: one buffer per distinct spec (every op's in+out working set > L2)
    bufs = {}

    def buf(spec, fill, owner=None):
        key = (spec[0], np.dtype(spec[1]).str, fill, owner)
        if key not in bufs:
            shp, dt = spec
            tdt = torch.uint8 if np.dtype(dt) == np.uint8 else torch.float32
            if fill:
                t = torch.randint(0, 256, shp, dtype=torch.uint8, device=dev, generator=torch.Generator(device=dev).manual_seed(1234 + rank))
                t = t if tdt == torch.uint8 else t.float()
            else:
                t = torch.empty(shp, dtype=tdt, device=dev)
            bufs[key] = t
        return bufs[key]

    for op in ops:
        op["_src"] = buf(op["src"], True)
        # ops of one shape share a destination, so a step leaves only the last one's result in it; to dump every op's result, each op
        # gets its own (before the graph is captured)
        op["_dst"] = buf(op["dst"], False, op["name"] if dump_dir else None) if op["dst"] is not None else None
    if workload == "c4":
        extra["templ"] = ops[0]["_src"][0, 700:764, 1000:1064, 0].contiguous()

    # The one collective of the path: rank 0's filter taps / kernels / template, NCCL broadcast once per step (= per batch).
    # It runs on a side stream one step ahead and lands in page-locked host memory (the C ABI takes these small operands as
    # host pointers), so the frame pipeline never drains for it.
    side = torch.cuda.Stream(device=dev)
    pin_taps = torch.empty((len(K_SWEEP), 31), dtype=torch.float32).pin_memory()
    pin_kern = torch.empty((len(K_SWEEP), 31 * 31), dtype=torch.float32).pin_memory()
    d_taps = torch.empty((len(K_SWEEP), 31), dtype=torch.float32, device=dev)
    d_kern = torch.empty((len(K_SWEEP), 31 * 31), dtype=torch.float32, device=dev)
    ev_ops = torch.cuda.Event()
    if rank == 0:
        tp0 = np.zeros((len(K_SWEEP), 31), np.float32); kn0 = np.zeros((len(K_SWEEP), 961), np.float32)
        for i, k in enumerate(K_SWEEP):
            tp0[i, :k] = gauss_taps(k); kn0[i, :k * k] = extra["kernels"][k].reshape(-1)
        h_taps0 = torch.from_numpy(tp0).pin_memory(); h_kern0 = torch.from_numpy(kn0).pin_memory()

    def prefetch_operands():
        with torch.cuda.stream(side):
            if rank == 0:
                d_taps.copy_(h_taps0, non_blocking=True); d_kern.copy_(h_kern0, non_blocking=True)
            if world > 1:
                dist.broadcast(d_taps, 0); dist.broadcast(d_kern, 0)
                if "templ" in extra:
                    dist.broadcast(extra["templ"], 0)
            pin_taps.copy_(d_taps, non_blocking=True); pin_kern.copy_(d_kern, non_blocking=True)
            ev_ops.record(side)

    def shared_operands():
        ev_ops.synchronize()                      # waits for the side stream only
        tp = pin_taps.numpy(); kn = pin_kern.numpy()
        for i, k in enumerate(K_SWEEP):
            extra["taps"][k] = tp[i, :k].copy(); extra["kernels"][k] = kn[i, :k * k].reshape(k, k).copy()
        prefetch_operands()                       # next step's broadcast overlaps this step's kernels

    prefetch_operands()

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in ops]

    def run_ops(record):
        if record:      # keep the GPU busy while the host enqueues, so the first op's event pair does not include launch latency
            big = ops[int(np.argmax([o["px"] * o["frames"] for o in ops]))]
            run_op(cvb, big, big["_src"], big["_dst"], extra)
        for i, op in enumerate(ops):
            if record:
                ev[i][0].record()
            op["_out"] = run_op(cvb, op, op["_src"], op["_dst"], extra)    # in a captured graph: its static outputs, rewritten by every replay
            if record:
                ev[i][1].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        shared_operands()
        run_ops(False)
    barrier()

    # The step's launches are captured ONCE into a CUDA graph and replayed: the step is ~50-190 short kernels and its wall time must
    # not depend on how fast this host thread can issue them (Python + driver contention with the NVML clock sampler doubled the
    # step time on some boxes).  Stream-ordered allocations inside the ops become graph memory nodes.  Ops that synchronise
    # (goodFeaturesToTrack returns host data) cannot be captured: those workloads run eagerly.
    graph, graph_note = None, "eager launches"
    n_before = cvb.launch_count()
    if not (not use_graph) and not any(op["kind"] in ("gftt",) for op in ops):
        try:
            shared_operands()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                run_ops(False)
            graph, graph_note = g, "one CUDA graph per step (captured once, replayed)"
        except Exception as exc:                      # noqa: BLE001 -- any capture failure falls back to eager launches
            print("graph capture failed, running eagerly: %r" % (exc,), file=sys.stderr)
            torch.cuda.synchronize()
            graph = None
    if graph is None:
        shared_operands()
        run_ops(False)
    launches_per_step = cvb.launch_count() - n_before          # the library counts launches as it issues (or captures) them
    barrier()

    def step():
        shared_operands()
        if graph is not None:
            graph.replay()
        else:
            run_ops(False)

    for _ in range(2):
        step()
    barrier()
    sampler = ClockSampler(local)
    if sample_clocks:
        sampler.start()
    per_op_ms = np.zeros(len(ops))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    t_host0 = time.perf_counter()
    for s in range(steps):
        step()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / steps
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    if dump_dir and rank == 0:
        dump_outputs(ops, dump_dir, dev)
    sampler.stop_flag = True
    if sample_clocks:
        sampler.join(timeout=2)
    # per-op times: eager steps with an event pair around every op (outside the timed region; the first pass re-warms the
    # stream-ordered allocator after the graph replays)
    shared_operands()
    run_ops(False)
    barrier()
    shared_operands()
    run_ops(True)
    barrier()
    for i in range(len(ops)):
        per_op_ms[i] = ev[i][0].elapsed_time(ev[i][1])
    launches = launches_per_step * steps
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    px_step_rank = sum(op["px"] * op["frames"] for op in ops)
    value = px_step_rank * world * steps / (total_ms * 1e-3) / 1e6
    peak, peak_src = peaks()
    per_op = {}
    for op, ms in zip(ops, per_op_ms):
        gbs = op["abytes"] * op["frames"] / (ms * 1e-3) / 1e9
        per_op[op["name"]] = {"ms": round(float(ms), 4), "mpix_s": round(op["px"] * op["frames"] / (ms * 1e-3) / 1e6, 1), "gbs": round(gbs, 1), "frac_hbm": round(gbs / peak, 4)}
    dom = int(np.argmax(per_op_ms))
    dgbs = ops[dom]["abytes"] * ops[dom]["frames"] / (per_op_ms[dom] * 1e-3) / 1e9
    # dram bytes per launch of the op's main kernel from `ncu --set full` (profiles/ncu_traffic.json, written from the committed captures)
    traffic = None
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as fh:
            traffic = json.load(fh).get(ops[dom]["name"])
    except (OSError, ValueError):
        traffic = None
    roofline = {"kernel": ops[dom]["name"], "bound": "hbm", "achieved": round(dgbs, 1), "peak": peak, "unit": "GB/s", "frac": round(dgbs / peak, 4), "traffic": traffic,
                "peak_source": peak_src, "share_of_step": round(float(per_op_ms[dom] / per_op_ms.sum()), 3),
                "note": "dominant = largest share of step time; per_op lists achieved GB/s and HBM fraction of every op (algorithmic bytes, SURVEY 8d)"}
    if ops[dom]["kind"] == "f2d":
        k = ops[dom]["k"]
        is_f32 = np.dtype(ops[dom]["src"][1]) == np.float32
        tfl = 2.0 * k * k * ops[dom]["px"] * ops[dom]["frames"] / (per_op_ms[dom] * 1e-3) / 1e12
        if k * k >= 130 and k >= 13:
            # from the reference's DFT switch on (130 taps) filter2D is a dense contraction on tcgen05: the tensor pipe bounds it, not HBM.
            # achieved = ALGORITHMIC flops (2 k^2 per pixel).  The MMAs issue more: the Toeplitz form pads every kernel row to K = k + 31 -> 48 / 64
            # columns, and float images run 3 x BF16 as two MMAs per K step (N = 64 + N = 32): 96 K MACs per 32 pixels per kernel row and K step.
            tpeak = 1681.6
            try:
                tpeak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
            except (OSError, ValueError, KeyError):
                pass
            K = 16 * ((k + 31 + 15) // 16) if is_f32 else 64
            issued_per_px = (2.0 * 3 * K * k) if is_f32 else (2.0 * 3 * K * k)          # f32: (64 + 32) / 32 = 3 MAC per K element and pixel; u8: three digit planes
            itfl = issued_per_px * ops[dom]["px"] * ops[dom]["frames"] / (per_op_ms[dom] * 1e-3) / 1e12
            ipeak = tpeak if is_f32 else 2 * tpeak
            roofline.update({"bound": "tensor", "achieved": round(tfl, 1), "peak": tpeak, "unit": "TFLOP/s", "frac": round(tfl / tpeak, 4),
                             "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, burst)",
                             "hbm": {"achieved": round(dgbs, 1), "peak": peak, "unit": "GB/s", "frac": round(dgbs / peak, 4)},
                             "issued": {"achieved": round(itfl, 1), "peak": ipeak, "unit": "TFLOP/s" if is_f32 else "TOP/s", "frac": round(itfl / ipeak, 3),
                                        "note": "MMA volume actually issued (Toeplitz zeros and the %s included) against the %s peak; the op time includes the border-extension / split kernel"
                                                % ("3 x BF16 split" if is_f32 else "three base-256 tap digits", "measured bf16" if is_f32 else "int8 = 2 x measured bf16")},
                             "note": "dominant = largest share of step time; a >= 130-tap filter2D is a tcgen05 contraction (kind::%s): tensor bound, achieved = algorithmic flops 2 k^2 per pixel; "
                                     "ncu: tensor pipe active ~50 %%, shared-memory operand wavefronts ~90 %% of peak (profiles/)" % ("f16, BF16 operands" if is_f32 else "i8")})
        else:
            # below that a k x k direct sum is k*k FMA per pixel: the FP32 pipe, not HBM, bounds it -- report that too
            fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
            roofline["fp32"] = {"achieved": round(tfl, 1), "peak": round(fp32_peak, 1), "unit": "TFLOP/s", "frac": round(tfl / fp32_peak, 3),
                                "note": "148 SM x 128 FMA lanes x 2 x 1.965 GHz; this op is FMA-issue bound (k*k MAC per pixel), its HBM fraction is not the limiter"}

    res = {"value": value, "total_ms": total_ms, "ms_per_step": total_ms / steps, "per_op": per_op, "roofline": roofline, "launches": int(launches),
           "launches_per_step": int(launches_per_step), "graph_note": graph_note, "host_enqueue_ms": host_enqueue_ms, "clocks": sampler.summary() if sample_clocks else None, "desc": desc}
    return res, ops, extra, bufs


def measure_e2e(workload, ops, extra, bufs, steps, rank, world, local):
    """the workload through the batch driver over HOST buffers (this rank's GPU): H2D + kernels + D2H inside the timed region (wall clock, max over ranks).
    The batch driver (include/b200cv_batch.h): its worker thread runs on the CPUs next to the GPU and first-touches the page-locked frame buffers
    there (NUMA-local staging); frames flow through the 3-stream upload / kernel / download pipeline."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    from opencv_b200.batch import BatchDriver
    drv = BatchDriver([local])
    hb = {}

    def hbuf(spec, fill, src_t=None):
        key = (spec[0], np.dtype(spec[1]).str, fill)
        if key not in hb:
            a = drv.pinned_frames(spec[0], spec[1])
            if fill:
                t = bufs[(spec[0], np.dtype(spec[1]).str, True, None)] if src_t is None else src_t
                a[...] = t.cpu().numpy()
            hb[key] = a
        return hb[key]
    hextra = dict(extra)
    if "templ" in extra:
        hextra["templ"] = extra["templ"].cpu().numpy()
    hsteps = max(1, min(steps, 3))
    if workload == "c5":
        # C5 end to end: host frames in, waves of pyramids + DoG kept on the device for the consumer of the wave (SURVEY 7.2: 1.9 GB per
        # frame cannot come back over PCIe), Harris responses downloaded.  32 frames per rank per step; 1024 frames = 4 steps on 8 ranks.
        nf = 32
        sspec = ((nf, H4K, W4K, 1), np.uint8)
        base = ops[0]["_src"]
        hsrc = hbuf(sspec, True, torch.cat([torch.roll(base, shifts=(17 * i, 31 * i), dims=(1, 2)) for i in range(nf // base.shape[0])]))
        hdst = hbuf(((nf, H4K, W4K, 1), np.float32), False)

        def hstep():
            drv.sift_harris(hsrc, hdst, 3, 1.6, 1, 2, 3, 0.04, wave=4)
        hpx = 2 * nf * W4K * H4K
        h2d, d2h, nops = hsrc.nbytes, hdst.nbytes, 2
        api = "b200cv_batch_sift_harris (include/b200cv_batch.h): %d host frames per rank per step in waves of 4, Harris responses downloaded, pyramids kept for the wave" % nf
    else:
        hops = [op for op in ops if op["kind"] not in ("gftt", "sift")]
        for op in hops:
            op["_hsrc"] = hbuf(op["src"], True); op["_hdst"] = hbuf(op["dst"], False)

        def hstep():
            for op in hops:
                run_op(drv, op, op["_hsrc"], op["_hdst"], hextra)
        hpx = sum(op["px"] * op["frames"] for op in hops)
        h2d = int(sum(op["_hsrc"].nbytes for op in hops)); d2h = int(sum(op["_hdst"].nbytes for op in hops)); nops = len(hops)
        api = "b200cv_batch_* (include/b200cv_batch.h) over page-locked cv::Mat-layout buffers: per-device worker thread, NUMA-local staging, 3-stream upload/kernel/download pipeline"
    hstep()
    barrier()
    t0 = time.perf_counter()
    for _ in range(hsteps):
        hstep()
    barrier()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e = {"value": hpx * world * hsteps / dt / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "h2d_gbs_per_rank": round(h2d * hsteps / dt / 1e9, 2), "d2h_gbs_per_rank": round(d2h * hsteps / dt / 1e9, 2),
           "steps": hsteps, "api": api, "ops": nops}
    hb.clear()
    drv.close()

    return e2e


def measure_hal_per_call():
    """synchronous single-frame calls through the host entry points on ordinary (pageable) numpy arrays: the shape of a cv_hal_* call"""
    from opencv_b200 import hal
    rng = np.random.default_rng(3)
    g4k = rng.integers(0, 256, (H4K, W4K), dtype=np.uint8)
    f4k = g4k.astype(np.float32)
    bgr8k = rng.integers(0, 256, (H8K, W8K, 3), dtype=np.uint8)
    cases = (("GaussianBlur_5x5_8UC1_4K", lambda: hal.GaussianBlur(g4k, (5, 5), 0), W4K * H4K),
             ("GaussianBlur_5x5_32FC1_4K", lambda: hal.GaussianBlur(f4k, (5, 5), 0), W4K * H4K),
             ("cvtColor_BGR2GRAY_8UC3_8K", lambda: hal.cvtColor(bgr8k, 6), W8K * H8K),
             ("resize_8Kto4K_LINEAR_8UC3", lambda: hal.resize(bgr8k, (W4K, H4K), interpolation=1), W4K * H4K))
    out = {"note": "one frame per call, pageable host memory, synchronous (upload + kernel + download + the destination's allocation): the cost of a cv:: call routed through the HAL seam"}
    for name, fn, px in cases:
        fn(); fn()
        t0 = time.perf_counter()
        n = 8
        for _ in range(n):
            fn()
        dt = (time.perf_counter() - t0) / n
        out[name] = {"ms_per_call": round(dt * 1e3, 3), "mpix_s": round(px / dt / 1e6, 1)}
    return out


def main():
    # keep stdout clean for the ONE JSON line: libraries (e.g. the NCCL version banner) write to fd 1 -> send that to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(json_fd, "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every launch from the host each step instead of replaying a captured CUDA graph")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short C3/C4/C5 passes that ride along with the default (C2) workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what each op of the workload returned in the last one "
                                                          "as DIR/<op>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    rng = np.random.default_rng(0x5EED0000 + 2 + rank)
    ops, desc = build_ops(args.workload, rng)
    W = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # ---------------- reference arm: the reference's own CPU implementation on the host cores ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        orc, kind = reference_oracle()
        extra = make_extra(ops, rng, False)
        if orc.has("gaussian_kernel"):
            for k in K_SWEEP:
                extra["taps"][k] = orc.getGaussianKernel(k, 0).astype(np.float32)
        cpu_frames(ops, rng)
        if args.workload == "c4":
            extra["templ_np"] = ops[0]["_cpu_src"][700:764, 1000:1064].copy()
        cores = orc.num_threads() if orc.has("get_num_threads") else 1
        for _ in range(args.warmup):
            cpu_pass(orc, ops, extra)
        t = 0.0; px = 0
        for _ in range(args.steps):
            dt, p = cpu_pass(orc, ops, extra)
            t += dt; px += p
        v = px / t / 1e6
        print(json.dumps({"impl": "reference", "metric": "Mpix/s", "value": v, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f32",
                          "data": "synthetic", "config": {"workload": desc, "sample": "1 frame per op per step (bounded sample of the same op list)"},
                          "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": cores, "kind": kind, "sample": "every op of the workload on one frame per step"},
                          "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ---------------- our arm -------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    import opencv_b200 as cvb
    from opencv_b200 import hal
    torch.cuda.set_device(local)
    cvb.init(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    res, ops, extra, bufs = measure_device(args.workload, args.steps, W, not args.no_graph, rank, world, local, rng, dump_dir=args.dump_outputs)
    value, total_ms, per_op, roofline, launches = res["value"], res["total_ms"], res["per_op"], res["roofline"], res["launches"]
    graph_note, host_enqueue_ms, desc = res["graph_note"], res["host_enqueue_ms"], res["desc"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- e2e: the same ops through the host C ABI (pinned host memory, H2D+D2H in the timed region) --------------
    e2e = None if args.no_e2e else measure_e2e(args.workload, ops, extra, bufs, args.steps, rank, world, local)

    # ---------------- the per-call HAL seam: what ONE cv:: call of a stock OpenCV built with the HAL header costs (pageable cv::Mat memory,
    # upload -> kernel -> download synchronously per frame, b200cv_hal_* = opencv_b200.hal over a single frame) -- rank 0 only, a handful of calls
    if e2e is not None and rank == 0 and args.workload == "c2":
        try:
            e2e["per_call_hal"] = measure_hal_per_call()
        except Exception as exc:                        # noqa: BLE001
            e2e["per_call_hal"] = {"error": repr(exc)[:200]}

    # ---------------- the other BASELINE configs (C3, C4, C5) measured in the same run: short device-resident passes with per-op tables --------
    extra_workloads = None
    if args.workload == "c2" and not args.no_extra:
        for op in ops:                                  # release the main workload's device and pinned buffers first
            for k in ("_src", "_dst", "_hsrc", "_hdst"):
                op.pop(k, None)
        bufs.clear()
        torch.cuda.empty_cache()
        extra_workloads = {}
        for w in ("c3", "c4", "c5"):
            try:
                r, o2, x2, b2 = measure_device(w, max(1, min(args.steps, 3)), 3, not args.no_graph, rank, world, local, np.random.default_rng(0x5EED0000 + ord(w[1]) + rank), sample_clocks=False)
                extra_workloads[w] = {"workload": r["desc"], "value": r["value"], "unit": "Mpix/s", "ms_per_step": r["ms_per_step"], "launch": r["graph_note"],
                                      "gpu_launches_per_step": r["launches_per_step"], "per_op": r["per_op"]}
                if not args.no_e2e:
                    extra_workloads[w]["e2e"] = measure_e2e(w, o2, x2, b2, 2, rank, world, local)
                for op in o2:
                    for k in ("_src", "_dst", "_hsrc", "_hdst"):
                        op.pop(k, None)
                b2.clear(); x2.clear(); del o2, b2, x2
                torch.cuda.empty_cache()
            except Exception as exc:                    # noqa: BLE001 -- an extra table must never take the headline line down with it
                extra_workloads[w] = {"error": repr(exc)[:300]}
                torch.cuda.synchronize()

    # ---------------- cpu baseline: the reference's own CPU path on this box's host cores (rank 0, N == 1) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        orc, kind = reference_oracle()
        cpu_frames(ops, rng)
        cextra = dict(extra)
        if args.workload == "c4":
            cextra["templ_np"] = ops[0]["_cpu_src"][700:764, 1000:1064].copy()
        cores = orc.num_threads() if orc.has("get_num_threads") else 1
        cpu_pass(orc, ops, cextra)
        t = 0.0; px = 0; n = 0
        while t < 10.0 and n < 20:
            dt, p = cpu_pass(orc, ops, cextra)
            t += dt; px += p; n += 1
        cpu = {"value": px / t / 1e6, "unit": "Mpix/s", "cores": cores, "kind": kind,
               "sample": "%d passes of the full op list on ONE frame per op (%.1f s of CPU work)" % (n, t)}

    if rank == 0:
        out = {"metric": "Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": W,
               "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f32",
               "data": "synthetic", "config": {"workload": desc, "l2": "every op streams a batch whose input+output exceed the 126 MB L2",
                                                "parallelism": "frames sharded across %d rank(s); NCCL broadcast of taps/kernels per step" % world,
                                                "launch": graph_note, "host_enqueue_ms_per_step": round(host_enqueue_ms, 3)},
               "gpu_launches": int(launches), "clocks": res["clocks"], "roofline": roofline, "per_op": per_op}
        if e2e:
            out["e2e"] = e2e
        if cpu:
            out["cpu_baseline"] = cpu
        if extra_workloads:
            out["config"]["extra_workloads"] = extra_workloads
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
