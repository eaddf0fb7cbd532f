#!/usr/bin/env python
"""bench.py -- ECO-Lite N=16 forward videos/s (BASELINE.json metric) on N GPUs of one node.

  python bench.py --gpus 1 --steps K --warmup W            # our arm (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --steps K --warmup W    # the reference arm: CPU implementation of the path

A step = one forward of the hot path over one batch of synthetic clips (uint8 frames, seed 1234,
minus the BGR mean; SURVEY.md 8(d)) per GPU.  Videos are independent in TEST phase, so the batch is
sharded across ranks with no data-path collective ("scaling": "weak").
  value   : videos/s with the batch already resident in HBM (fp32, caffe layout) when the timed region starts
  e2e     : the same through the reference-facing call with HOST buffers: the batch sits in the input blob's
            host memory (where caffe's data layer writes it), forward() uploads it, the fc8 logits are read
            back to the host -- all inside the timed region
  roofline: all launches of the implicit-GEMM conv kernel (the dominant kernel): algorithmic FLOPs
            (2*M*N*K per conv, SURVEY.md 8(d): 92.97 GFLOP/video) / their summed CUDA-event time
  cpu_baseline: the oracle (a port of caffe_3d's CPU algorithm: per-image im2col + SGEMM + separate
            BN/ReLU/pool passes) on this box's host cores, bounded sample; `strong` = the same clip through
            torch-CPU fp32 (oneDNN), SURVEY.md 8(d)'s "strong CPU" line
  parity  : the device logits of clip 0 of step 0 against the oracle run on that clip with the SAME weights
            (read back from the product), outside every timed region: oracle = checker, never the thing measured

The GPU arm generates its weights with tools/harness.py (numpy + the product's own surface); the oracle is only
imported by the CPU legs (cpu_baseline / parity on rank 0, --impl reference).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "eco-efficient-video-understanding_b200"),
          os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

_WORLD = int(os.environ.get("WORLD_SIZE", "1"))
_RANK = int(os.environ.get("RANK", "0"))
if _WORLD == 1 or (_RANK == 0 and "reference" in sys.argv):
    # CPU legs only (cpu_baseline at N=1, the reference arm on rank 0): one OpenMP thread per physical core, pinned.
    # Never in a multi-rank GPU run: with OMP_PLACES set, libgomp binds every rank's MAIN thread to place 0, and
    # eight kernel-launching threads then share one core.
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")

import numpy as np

GFLOP_PER_VIDEO = {("lite", 16): 92.97, ("full", 16): 128.83}
CLASSES = 101


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(tflops=d.get("bf16_tflops_sustained", d.get("bf16_tflops")), hbm=d.get("hbm_gbs"), src="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled through NVML
    every 5 ms (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []          # (t, sm_mhz, reasons bitmask)
        self.stop_flag = False
        self.max_mhz = None
        self.windows = []       # [(t0, t1)] timed regions

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML indexes physical GPUs; honour CUDA_VISIBLE_DEVICES if it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            while not self.stop_flag:
                try:
                    mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    try:
                        rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((time.perf_counter(), float(mhz), int(rs)))
                except Exception:
                    pass
                time.sleep(0.005)
        except Exception:
            pass

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def finish(self):
        self.stop_flag = True
        self.join(timeout=1.0)
        inside = [r for r in self.rows if any(a <= r[0] <= b for a, b in self.windows)] or self.rows
        sm = [r[1] for r in inside]
        reasons = set()
        for r in inside:
            for bit, name in self.REASONS.items():
                if r[2] & bit:
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=self.max_mhz, reasons=sorted(reasons),
                    samples=len(sm))


def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_forward(model, segments, steps, warmup, threads=None, params=None, x=None, classes=None):
    """The reference arm / cpu_baseline: oracle fp32 forward (caffe_3d's CPU algorithm), one clip per step.
    `params` (the product's weights) and `x` (one clip) make it the parity checker as well; returns
    (videos/s, ms/step, threads, logits fp32, logits bf16-mirror or None)."""
    import gen_eco_prototxt as gen
    from oracle import refnet
    threads = int(threads or physical_cores())  # one OpenMP thread per physical core (SMT siblings only add noise)
    refnet.lib().ref_set_num_threads(threads)
    cores = int(refnet.lib().ref_num_threads())
    kw = dict(segments=segments, batch=1)
    if classes:
        kw["classes"] = classes
    txt = (gen.eco_full_deploy if model == "full" else gen.eco_lite_deploy)(**kw)
    net = refnet.RefNet(txt)
    if params is not None:
        net.set_params(params)
    else:
        net.init_params(4321)
    if x is None:
        x = refnet.eco_input(1, segments)
    for _ in range(warmup):
        net.forward(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = net.forward(x)
    dt = time.perf_counter() - t0
    mirror = net.forward(x, bf16=True)["fc8"] if params is not None else None
    return steps / dt, dt / steps * 1e3, cores, out["fc8"], mirror


def cpu_strong_forward(params, x, segments, steps=3, warmup=1, threads=None):
    """torch-CPU fp32 (oneDNN / MKL) functional ECO-Lite on the same clip and weights: the strong CPU line."""
    import torch
    from oracle.torch_ref import torch_eco_lite, t
    threads = int(threads or physical_cores())
    torch.set_num_threads(threads)
    xt = t(x)
    with torch.no_grad():
        for _ in range(warmup):
            torch_eco_lite(params, xt, segments)
        t0 = time.perf_counter()
        for _ in range(steps):
            fc8, _ = torch_eco_lite(params, xt, segments)
    dt = time.perf_counter() - t0
    return steps / dt, dt / steps * 1e3, threads, fc8


DUMP_LIMIT_BYTES = 64 << 20
PARAM_SAMPLE = 1 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, one DIR/<name>.npy each, so that two
    builds run with the same arguments (hence the same seeded inputs and weights) can be compared output for output"""
    arrays = {k: np.ascontiguousarray(v, np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def param_sample(net):
    """a fixed, seeded sample of PARAM_SAMPLE elements of all parameter blobs (layer order, flattened)"""
    flat = np.concatenate([np.asarray(b.data, np.float32).ravel() for blobs in net.params.values() for b in blobs])
    idx = np.sort(np.random.default_rng(0).choice(flat.size, size=min(PARAM_SAMPLE, flat.size), replace=False))
    return flat[idx]


TRAIN_SOLVER = """base_lr: 0.001 lr_policy: "step" gamma: 0.1 stepsize: 24000 max_iter: 60000 iter_size: 1
momentum: 0.9 weight_decay: 0.0005 clip_gradients: 40 solver_type: NESTEROV"""   # models_ECO_Lite/kinetics/solver.prototxt (iter_size 1)


def train_main(a, rank, local_rank, world):
    """BASELINE config #4: ECO-Lite training, Kinetics-400 head, batch-sharded over the GPUs of one box, the ONLY collective
    being the gradient all-reduce (NCCL, bucketed, overlapped with backward).  One step = Solver::Step(1): clear diffs,
    forward, backward, exchange, clip + L2 + Nesterov update.  videos/s = world * batch * steps / time."""
    segments = a.segments if a.segments != 16 or "--segments" in sys.argv else 32
    batch = a.batch if "--batch" in sys.argv else 16
    classes = 400
    workload = "ECO-Lite N=%d training step (fwd+bwd+grad all-reduce+Nesterov), %d classes, batch %d videos/GPU, synthetic frames" % (
        segments, classes, batch)
    if a.impl == "reference":
        if rank != 0:
            return
        import gen_eco_prototxt as gen
        from oracle import refnet
        threads = physical_cores()
        refnet.lib().ref_set_num_threads(threads)
        net = refnet.RefNet(gen.eco_lite_train(segments=segments, classes=classes, batch=1), phase="TRAIN").init_params(4321)
        x = refnet.eco_input(1, segments).reshape(1, 3 * segments, 224, 224)
        lab = np.array([7], np.float32).reshape(1, 1, 1, 1)
        steps = max(1, min(a.steps, 2))
        t0 = time.perf_counter()
        for _ in range(steps):
            net.forward({"data": x, "label": lab})
            net.backward()
        dt = time.perf_counter() - t0
        vps = steps / dt
        print(json.dumps({"impl": "reference", "metric": "ECO-Lite-%d training videos/sec" % segments, "value": vps, "unit": "videos/s",
                          "n_gpus": a.gpus, "steps": steps, "warmup": 0, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": workload, "note": "oracle forward+backward (caffe_3d CPU algorithm), ONE clip per step, no update"},
                          "cpu_baseline": {"value": vps, "unit": "videos/s", "cores": threads, "kind": "port", "cpu_model": cpu_model(),
                                           "sample": "%d single-clip forward+backward passes" % steps},
                          "e2e": {"value": vps, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    import torch
    import caffe
    import gen_eco_prototxt as gen
    import harness
    from caffe.parallel import GradExchange
    from dist_util import Group
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path")
    torch.cuda.set_device(local_rank)
    caffe.set_device(local_rank)
    caffe.set_mode_gpu()
    grp = Group("nccl", torch.device("cuda", local_rank))
    solver = caffe.NesterovSolver(solver_text=TRAIN_SOLVER, net_text=gen.eco_lite_train(segments=segments, classes=classes, batch=batch))
    net = solver.net
    harness.init_params(net, 4321)
    ex = GradExchange(solver, nbuckets=a.buckets, overlap=bool(a.overlap))
    ex.broadcast_params(0)
    stream = ex.compute
    g = torch.Generator(device="cuda")
    g.manual_seed(1234 + rank)
    frames = torch.randint(0, 256, (batch, 3 * segments, 224, 224), generator=g, device="cuda", dtype=torch.uint8).float()
    frames -= torch.tensor([104.0, 117.0, 123.0], device="cuda").repeat(segments).view(1, 3 * segments, 1, 1)
    count = frames.numel()
    labels = np.random.default_rng(99 + rank).integers(0, classes, size=(batch, 1, 1, 1)).astype(np.float32)
    net.blobs["label"].data[...] = labels
    torch.cuda.synchronize()
    net.set_input_device("data", frames.data_ptr(), count)
    losses = []
    for _ in range(max(a.warmup, 3)):
        losses.append(solver.step(1))
    net.sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    grp.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(a.steps):
        losses.append(solver.step(1))
    e1.record(stream)
    grp.barrier()
    sampler.window(tw0, time.perf_counter())
    ms_total = grp.max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / a.steps
    value = world * batch * a.steps / (ms_total / 1e3)
    if a.dump_outputs and rank == 0:
        # the last timed step's loss and logits, and the parameters its update left behind
        dump_outputs(a.dump_outputs, {"loss": np.array([losses[-1]], np.float64),
                                      "fc8": np.array(net.blobs["fc8"].data, np.float32),
                                      "params_sample": param_sample(net)})
    # e2e: the batch comes from the input blob's pinned host mirror every step (what a data layer would fill), loss read back
    host_in = net.blobs["data"].data
    host_in[...] = frames.cpu().numpy()
    for _ in range(2):
        net.blobs["data"].data
        solver.step(1)
    grp.barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        net.blobs["data"].data
        net.blobs["label"].data
        losses.append(solver.step(1))
    torch.cuda.synchronize()
    grp.barrier()
    e2e_ms = grp.max_over_ranks((time.perf_counter() - t0) * 1e3)
    sampler.window(t0, time.perf_counter())
    clocks = sampler.finish()
    e2e_value = world * batch * a.steps / (e2e_ms / 1e3)
    # collective alone: the same buckets all-reduced back to back on an idle GPU (what is overlapped with backward above)
    coll_ms = None
    if world > 1:
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            torch.distributed.all_reduce(ex.grad)
        torch.cuda.synchronize()
        c0.record()
        for _ in range(5):
            torch.distributed.all_reduce(ex.grad)
        c1.record()
        torch.cuda.synchronize()
        coll_ms = grp.max_over_ranks(c0.elapsed_time(c1) / 5)
    gf_video = 3.0 * GFLOP_PER_VIDEO[("lite", 16)] * segments / 16.0   # forward + dgrad + wgrad implicit GEMMs (SURVEY 8(d): 557.8 at N=32)
    pk = peaks()
    achieved = batch * gf_video / ms_step   # GFLOP / ms = TFLOP/s
    _, _, arena = net.arenas()
    if rank != 0:
        grp.close()
        return
    line = {"metric": "ECO-Lite-%d training videos/sec (fwd+bwd+grad all-reduce+Nesterov update)" % segments, "value": value,
            "unit": "videos/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 activations / fp32 master weights and gradients",
            "data": "synthetic",
            "config": {"workload": workload, "global_batch": batch * world, "parallelism": "dp%d: batch-sharded replicas, NCCL SUM all-reduce of the gradient arena in %d buckets (%s), "
                       "1/world folded into the update" % (world, a.buckets, "launched from inside the backward pass" if a.overlap
                                                             else "launched when backward has been enqueued"),
                       "l2": "activations exceed the 126 MB L2", "solver": "models_ECO_Lite/kinetics/solver.prototxt values, iter_size 1"},
            "clocks": clocks, "gpu_launches": int(net.last_launch_count()) * a.steps,
            "e2e": {"value": e2e_value, "unit": "videos/s", "h2d_bytes_per_step": int(count * 4 + batch * 4), "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / a.steps},
            "collective": {"payload_bytes_per_iter": int(arena * 4), "buckets": a.buckets, "allreduce_alone_ms": coll_ms,
                           "overlap_with_backward": bool(a.overlap),
                           "note": "allreduce_alone_ms = the whole arena all-reduced on an idle GPU (after warm-up calls)"},
            "roofline": {"bound": "tensor", "kernel": "forward conv GEMMs + dgrad (same kernel) + wgrad_umma_kernel", "achieved": achieved,
                         "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "peak_source": pk["src"],
                         "traffic": None, "gflop_per_video": gf_video,
                         "note": "whole-step rate: algorithmic conv FLOPs (3 x forward) / ms_per_step, everything else included in the time"},
            "loss_first_last": [float(losses[0]), float(losses[-1])], "cpu_baseline": None}
    print(json.dumps(line))
    grp.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="lite", choices=["lite", "full"])
    ap.add_argument("--segments", type=int, default=16)
    ap.add_argument("--batch", type=int, default=32, help="videos per GPU per step")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer: BASELINE metric (forward videos/s); train: config #4 (fwd + bwd + NCCL grad all-reduce + Nesterov)")
    ap.add_argument("--buckets", type=int, default=3, help="train: gradient all-reduce buckets")
    ap.add_argument("--overlap", type=int, default=1, help="train: 1 = start each bucket's all-reduce from inside backward")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-calibrate", action="store_true", help="skip the BN calibration forwards of the weight harness (ncu captures)")
    ap.add_argument("--h2d-chunks", type=int, default=0, help="blocking forward: 0 auto (4 sub-batches), 1 unsplit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy: "
                         "infer: fc8 logits; train: loss, fc8 logits and a seeded sample of the updated parameters")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs records the GPU arm's outputs; the reference arm has none to record")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.mode == "train":
        return train_main(a, rank, local_rank, world)
    workload = "ECO-%s N=%d forward, %d classes, batch %d videos/GPU, synthetic 224x224x3 frames" % (
        "Lite" if a.model == "lite" else "Full", a.segments, CLASSES if a.model == "lite" else 400, a.batch)

    if a.impl == "reference":
        if rank != 0:
            return
        steps = max(1, min(a.steps, 10))
        vps, ms, cores, _, _ = cpu_reference_forward(a.model, a.segments, steps, min(a.warmup, 1))
        line = {"impl": "reference", "metric": "ECO-Lite-16 forward videos/sec", "value": vps, "unit": "videos/s",
                "n_gpus": a.gpus, "steps": steps, "warmup": min(a.warmup, 1), "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload,
                           "note": "reference CPU algorithm (oracle port of caffe_3d: per-image im2col + SGEMM), bounded sample: "
                                   "ONE clip per step and at most 10 steps, whatever --batch/--steps say (a CPU arm at batch 32 "
                                   "would take minutes per step); videos/s is per clip, so it compares with the GPU arm's videos/s"},
                "cpu_baseline": {"value": vps, "unit": "videos/s", "cores": cores, "kind": "port", "cpu_model": cpu_model(),
                                 "threads": "one OpenMP thread per physical core, OMP_PROC_BIND=close",
                                 "sample": "%d single-clip N=%d forwards" % (steps, a.segments)},
                "e2e": {"value": vps, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import caffe
    import gen_eco_prototxt as gen
    import harness

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    caffe.set_device(local_rank)
    caffe.set_mode_gpu()
    from dist_util import Group
    grp = Group("nccl", torch.device("cuda", local_rank))

    B, N = a.batch, a.segments
    classes = CLASSES if a.model == "lite" else 400
    txt = (gen.eco_full_deploy if a.model == "full" else gen.eco_lite_deploy)(segments=N, classes=classes, batch=B)
    net = caffe.Net.from_string(txt, caffe.TEST, keep_all_blobs=0, use_graph=0 if a.no_graph else 1, h2d_chunks=a.h2d_chunks)
    # harness weights: random init of the right architecture, BN statistics calibrated on the device with a small
    # every-blob net (N=4, one clip) so activations stay O(1) like a trained net's and the parity check below means something
    make = gen.eco_full_deploy if a.model == "full" else gen.eco_lite_deploy
    small = caffe.Net.from_string(make(segments=4, classes=classes, batch=1), caffe.TEST, keep_all_blobs=1)
    harness.init_params(small, 4321)
    if not a.no_calibrate:
        harness.calibrate_bn_on_device(small, harness.synthetic_frames(1, 4))
    harness.copy_params(net, small)
    del small
    stream = torch.cuda.Stream()          # a real (non-legacy) stream: the events below are recorded on it
    net.set_stream(stream.cuda_stream)

    # synthetic frames: uint8 U{0..255} seed 1234 (+rank), minus BGR mean, fp32 NCHW as the data layer hands over
    g = torch.Generator(device="cuda")
    g.manual_seed(1234 + rank)
    frames = torch.randint(0, 256, (B * N, 3, 224, 224), generator=g, device="cuda", dtype=torch.uint8).float()
    frames -= torch.tensor([104.0, 117.0, 123.0], device="cuda").view(1, 3, 1, 1)
    count = frames.numel()
    torch.cuda.synchronize()

    barrier = grp.barrier
    max_over_ranks = grp.max_over_ranks

    # ---------------- value: inputs resident in HBM ----------------
    net.set_input_device("data", frames.data_ptr(), count)
    for _ in range(max(a.warmup, 3)):
        net._forward(0, len(net.layers) - 1)
    net.sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(a.steps):
        net._forward(0, len(net.layers) - 1)
    e1.record(stream)
    barrier()
    sampler.window(tw0, time.perf_counter())
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    net.sync()
    launches = net.last_launch_count() * a.steps
    ms_step = ms_total / a.steps
    value = world * B * a.steps / (ms_total / 1e3)
    # logits of clip 0 from this plan (graph replay, production options), checked against the oracle further down
    dev_logits0 = np.array(net.blobs["fc8"].data[0:1], np.float32, copy=True)
    clip0 = frames[:N].cpu().numpy()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"fc8": net.blobs["fc8"].data})

    # ---------------- e2e: host buffers in, logits out, copies inside the timed region ----------------
    host_in = net.blobs["data"].data  # pinned host mirror of the input blob (what caffe's data layer fills)
    host_in[...] = frames.cpu().numpy()
    for _ in range(2):
        net.blobs["data"].data
        net._forward(0, len(net.layers) - 1)
        _ = net.blobs["fc8"].data
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(a.steps):
        net.blobs["data"].data            # mutable_cpu_data(): marks the host copy newer -> forward uploads it
        net._forward(0, len(net.layers) - 1)
        logits = net.blobs["fc8"].data    # device -> host read of the step's result (syncs)
    e1.record(stream)
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    wall_ms = (time.perf_counter() - t0) * 1e3
    sampler.window(t0, time.perf_counter())
    e2e_value = world * B * a.steps / (max(e2e_ms, wall_ms) / 1e3)
    assert np.isfinite(logits).all()

    # ---------------- e2e, pipelined serving variant (extension beyond caffe's blocking forward) ----------------
    # two pinned input buffers and two pinned logits buffers alternate; the H2D copy of step k+1 overlaps the
    # compute of step k; every step still moves the same bytes host->device and device->host.
    pin_in = [torch.empty(count, dtype=torch.float32).pin_memory() for _ in range(2)]
    pin_out = [torch.empty(B * classes, dtype=torch.float32).pin_memory() for _ in range(2)]
    src = frames.cpu().reshape(-1)
    for b_ in pin_in:
        b_.copy_(src)
    tickets = [None, None]
    for k in range(4):
        if tickets[k & 1] is not None:
            net.wait(tickets[k & 1])
        tickets[k & 1] = net.forward_pipelined(pin_in[k & 1].data_ptr(), count, pin_out[k & 1].data_ptr(), B * classes)
    for tk in tickets:
        net.wait(tk)
    barrier()
    t0 = time.perf_counter()
    tickets = [None, None]
    for k in range(a.steps):
        if tickets[k & 1] is not None:
            net.wait(tickets[k & 1])          # results of step k-2 are on the host; its buffers are free again
        tickets[k & 1] = net.forward_pipelined(pin_in[k & 1].data_ptr(), count, pin_out[k & 1].data_ptr(), B * classes)
    for tk in tickets:
        if tk is not None:
            net.wait(tk)
    pipe_ms = grp.max_over_ranks((time.perf_counter() - t0) * 1e3)
    sampler.window(t0, time.perf_counter())
    clocks = sampler.finish()
    e2e_pipe_value = world * B * a.steps / (pipe_ms / 1e3)
    assert torch.isfinite(pin_out[0]).all()

    # ---------------- e2e from raw uint8 frames (DataTransformer's mean subtraction done on the GPU) ----------------
    u8 = (frames + torch.tensor([104.0, 117.0, 123.0], device="cuda").view(1, 3, 1, 1)).clamp(0, 255).to(torch.uint8).cpu().reshape(-1)
    pin_u8 = [torch.empty(count, dtype=torch.uint8).pin_memory() for _ in range(2)]
    for b_ in pin_u8:
        b_.copy_(u8)
    net.reshape()  # drop the fp32 pipeline slots; the plan is rebuilt with uint8 slots
    load_ok = net._forward(0, len(net.layers) - 1)
    net.sync()
    tickets = [None, None]
    for k in range(4):
        if tickets[k & 1] is not None:
            net.wait(tickets[k & 1])
        tickets[k & 1] = net.forward_pipelined_u8(pin_u8[k & 1].data_ptr(), count, [104.0, 117.0, 123.0], pin_out[k & 1].data_ptr(), B * classes)
    for tk in tickets:
        net.wait(tk)
    barrier()
    t0 = time.perf_counter()
    tickets = [None, None]
    for k in range(a.steps):
        if tickets[k & 1] is not None:
            net.wait(tickets[k & 1])
        tickets[k & 1] = net.forward_pipelined_u8(pin_u8[k & 1].data_ptr(), count, [104.0, 117.0, 123.0], pin_out[k & 1].data_ptr(), B * classes)
    for tk in tickets:
        if tk is not None:
            net.wait(tk)
    u8_ms = grp.max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_u8_value = world * B * a.steps / (u8_ms / 1e3)
    net.set_stream(stream.cuda_stream)

    # ---------------- roofline: the conv kernel, CUDA events per launch on the launching stream ----------------
    net.set_input_device("data", frames.data_ptr(), count)
    conv_ms, conv_flops, conv_n, other_ms = 0.0, 0.0, 0, 0.0
    prof_iters = 3
    per_op = {}
    for _ in range(prof_iters):
        for op in net.profile_forward():
            t = per_op.setdefault(op["name"], [0.0, 0.0])
            t[0] += op["ms"] / prof_iters
            t[1] = op["flops"]
            if op["kind"] == 0:
                conv_ms += op["ms"]
                conv_flops += op["flops"]
                conv_n += 1
            else:
                other_ms += op["ms"]
    pk = peaks()
    # The per-launch CUDA-event profile runs eagerly (no graph) and carries event / launch gaps, so its sum exceeds the
    # graph-replayed step; the conv launches' SHARE of it is what carries over (it agrees with the ncu launch list in
    # profiles/).  conv time inside the timed step = share x ms_per_step; achieved = algorithmic conv FLOPs / that.
    eager_conv_ms, eager_other_ms = conv_ms / prof_iters, other_ms / prof_iters
    share = eager_conv_ms / max(eager_conv_ms + eager_other_ms, 1e-9)
    conv_ms_step = share * ms_step
    flops_step = conv_flops / prof_iters
    achieved = flops_step / (conv_ms_step * 1e-3) / 1e12 if conv_ms_step > 0 else 0.0
    burst = None
    try:
        burst = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops")
    except (OSError, ValueError):
        pass
    # dram bytes of the same launches from the committed ncu --set full capture (only valid for the captured workload)
    traffic, traffic_src = None, None
    for cand in ("r02_final_ncu_dram_bytes.json", "r01_final_ncu_dram_bytes.json"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", cand)))
            if tj["model"] == a.model and tj["batch"] == B and tj["segments"] == N:
                traffic, traffic_src = tj["conv_dram_bytes_per_step"], "profiles/" + cand
                break
        except (OSError, KeyError, ValueError):
            pass
    roofline = {"bound": "tensor",
                "kernel": "conv_umma_persistent_kernel / conv_umma_pair_kernel / stem_rows_kernel (all %d conv launches/step)" % (conv_n // prof_iters),
                "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"],
                "peak_source": pk["src"] + ": the step is timed as %d back-to-back replays, so the sustained figure applies" % a.steps,
                "frac_of_burst_peak": (achieved / burst) if burst else None,
                "whole_step_tflops": world and (B * GFLOP_PER_VIDEO.get((a.model, N), 0.0) / ms_step),
                "traffic": traffic, "traffic_unit": "bytes/step (dram read+write, all conv launches)",
                "traffic_source": traffic_src,
                "conv_ms_per_step": conv_ms_step, "other_ms_per_step": ms_step - conv_ms_step,
                "share_of_step": share,
                "top_ops_eager": [{"op": k, "ms": round(v[0], 4), "tflops": round(v[1] / (v[0] * 1e-3) / 1e12, 1) if v[0] > 0 and v[1] else None}
                                  for k, v in sorted(per_op.items(), key=lambda kv: -kv[1][0])[:8]],
                "method": "share of the conv launches in a per-launch CUDA-event profile (eager: %.3f + %.3f ms) applied to the "
                          "graph-timed ms_per_step" % (eager_conv_ms, eager_other_ms)}

    if rank != 0:
        grp.close()
        return
    cpu_baseline, parity = None, None
    if not a.no_cpu_baseline and world == 1:
        # CPU legs (the only place this arm touches oracle/): time the caffe-algorithm port and the torch-CPU graph on
        # clip 0 with the PRODUCT's weights, and use their logits to check the device's
        params = harness.params_dict(net)
        vps, ms, cores, ref_fc8, mirror_fc8 = cpu_reference_forward(a.model, N, steps=3, warmup=1, params=params, x=clip0,
                                                                  classes=classes)
        cpu_baseline = {"value": vps, "unit": "videos/s", "cores": cores, "kind": "port", "cpu_model": cpu_model(),
                        "logical_cpus": os.cpu_count(),
                        "threads": "one OpenMP thread per physical core, OMP_PROC_BIND=close",
                        "sample": "3 single-clip N=%d fp32 forwards of the oracle (caffe_3d CPU algorithm), clip 0 of the batch" % N}
        rel = lambda g, w: float(np.abs(g.astype(np.float64) - w).max() / max(np.abs(w).max(), 1e-30))
        parity = {"clip": 0, "blob": "fc8", "rel_max_vs_oracle_bf16_mirror": rel(dev_logits0, mirror_fc8),
                  "rel_max_vs_oracle_fp32": rel(dev_logits0, ref_fc8),
                  "oracle_bf16_mirror_vs_fp32": rel(mirror_fc8, ref_fc8),
                  "vs": "oracle (oracle/refnet.py) on clip 0 with the weights read back from the product; "
                        "tolerance of the tests: 2e-2 vs the bf16 mirror (tests/eco_testlib.py)"}
        if a.model == "lite":
            svps, sms, sthreads, s_fc8 = cpu_strong_forward(params, clip0, N)
            cpu_baseline["strong"] = {"value": svps, "unit": "videos/s", "threads": sthreads, "kind": "torch-cpu fp32 (oneDNN/MKL)",
                                      "sample": "3 single-clip N=%d forwards" % N,
                                      "agrees_with_port_rel_max": rel(s_fc8, ref_fc8)}
    line = {"metric": "ECO-Lite-16 forward videos/sec" if a.model == "lite" else "ECO-Full-16 forward videos/sec",
            "value": value, "unit": "videos/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload, "global_batch": B * world, "parallelism": "batch-sharded x%d, no collective" % world,
                       "l2": "inputs (%.0f MB/GPU) and activations exceed the 126 MB L2" % (count * 4 / 1e6),
                       "cuda_graph": not a.no_graph,
                       "batch_choice": "B=32 videos/GPU: best of the batch sweep B in {1, 8, 16, 32, 64} at the current kernels "
                                       "(profiles/r02_batch_sweep.md); res5 fills 147 of 148 SMs at exactly this batch"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "videos/s", "h2d_bytes_per_step": int(count * 4),
                    "d2h_bytes_per_step": int(B * classes * 4), "ms_per_step": max(e2e_ms, wall_ms) / a.steps,
                    "note": "caffe's blocking net.forward() on the fp32 input blob's (pinned) host mirror; inside the call the batch runs as "
                            "sub-batches on sub-nets so the copy of slice k+1 overlaps the compute of slice k (option h2d_chunks, "
                            "bit-identical logits)" if a.h2d_chunks != 1 else "caffe's blocking net.forward(), unsplit (h2d_chunks=1)",
                    "pipelined": {"value": e2e_pipe_value, "unit": "videos/s", "ms_per_step": pipe_ms / a.steps,
                                  "note": "eco_net_forward_pipelined: copy of step k+1 overlaps compute of step k; "
                                          "same bytes per step; wall clock"},
                    "pipelined_u8": {"value": e2e_u8_value, "unit": "videos/s", "ms_per_step": u8_ms / a.steps,
                                     "h2d_bytes_per_step": int(count),
                                     "note": "raw uint8 frames in, BGR mean subtracted on the GPU (the host half of the "
                                             "reference's DataTransformer), otherwise as pipelined"}},
            "e2e_u8": {"value": e2e_u8_value, "unit": "videos/s", "h2d_bytes_per_step": int(count), "d2h_bytes_per_step": int(B * classes * 4),
                       "note": "the declared serving entry point (eco_net_forward_pipelined_u8): raw uint8 frames from pinned host "
                               "memory, mean subtraction on the GPU, logits back to the host; wall clock over the same steps"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
            "gflop_per_video": GFLOP_PER_VIDEO.get((a.model, N))}
    print(json.dumps(line))
    grp.close()


if __name__ == "__main__":
    main()
