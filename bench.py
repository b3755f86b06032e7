#!/usr/bin/env python
"""bench.py -- hot-path throughput of the spatial-parallel conv engine on B200.

One "step" = one pass of the hot path over one synthetic image: forward and backward (dgrad +
wgrad) of every conv / pool layer of the reference's SPATIAL STAGE of AmoebaNet-D(18,416) at
8192x8192 (split_size=4: stem1-3 + cell1_normal1-3 = 62 convs + 13 pools; shapes extracted
from the reference's own model, tests/golden/layers_amoebanetd_sp4.json), each GPU working on
its tile (halo exchange between tiles + weight-grad allreduce at N>1), through the public
torchgems.spatial modules (which call libspconv.so through the C ABI).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference ...                     # the reference's CPU path (port)
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed

Prints ONE JSON line: metric/value/unit, ms_per_step, e2e, roofline, cpu_baseline, clocks,
gpu_launches.  Weights and inputs are seeded, so runs with the same arguments compute on identical
data and two builds can be compared output for output through --dump-outputs.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "amoebanet": ("layers_amoebanetd_sp4.json", "AmoebaNet-D(18,416) spatial stage (split_size=4) @ 8192x8192"),
    "resnet": ("layers_resnet101_sp2.json", "ResNet-v2-101 spatial stage (split_size=2) @ 4096x4096"),
}
METRIC = "images/sec (device-timed, max over ranks) AmoebaNet-D 8192^2 hot path (spatial-stage conv/pool fwd+bwd)"
DUMP_SAMPLE = 65536          # elements sampled per layer output / input gradient by --dump-outputs
DUMP_MAX_BYTES = 64 << 20


_T0 = time.time()


def _log(msg):
    """progress on stderr (stdout carries the ONE JSON line)"""
    sys.stderr.write("[bench %6.1fs] %s\n" % (time.time() - _T0, msg))
    sys.stderr.flush()


def load_layers(name):
    fn, desc = WORKLOADS[name]
    d = json.load(open(os.path.join(ROOT, "tests", "golden", fn)))
    return d, desc


def grid_for(n):
    """Tiling used for N GPUs: square when N is a perfect square, else vertical strips
    (reference train_spatial.py:241-290; square needs sqrt(P) integer)."""
    if n == 1:
        return "square", 1, 1
    q = int(round(n ** 0.5))
    if q * q == n:
        return "square", q, q
    return "vertical", 1, n


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:                                   # reap it: no sampler may outlive the benchmark
            self.proc.wait(timeout=10)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        self.t.join()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, l in self.lines:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def write_dump(out_dir, arrays):
    """--dump-outputs: save each tensor of `arrays` (name -> tensor) as out_dir/<name>.npy in float32."""
    import numpy as np

    host = {k: t.detach().float().cpu().numpy() for k, t in arrays.items()}
    nbytes = sum(a.nbytes for a in host.values())
    assert nbytes <= DUMP_MAX_BYTES, "--dump-outputs: %d bytes exceed the %d-byte limit" % (nbytes, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    _log("wrote %d arrays (%.1f MB) to %s" % (len(host), nbytes / 2**20, out_dir))


def conv_bytes_flops(l, tile_h, tile_w, esz):
    Ho = (tile_h + 2 * l["pad_h"] - l["R"]) // l["stride_h"] + 1
    Wo = (tile_w + 2 * l["pad_w"] - l["S"]) // l["stride_w"] + 1
    xin = l["C"] * tile_h * tile_w
    yout = l["K"] * Ho * Wo
    wn = l["K"] * l["C"] * l["R"] * l["S"]
    fl = 2.0 * wn * Ho * Wo
    return dict(fwd=((xin + yout + wn) * esz, fl), dgrad=((xin + yout + wn) * esz, fl),
                wgrad=((xin + yout) * esz + wn * 4, fl))


def pool_bytes(l, tile_h, tile_w, esz):
    Ho = (tile_h + 2 * l["pad"] - l["k"]) // l["stride"] + 1
    Wo = (tile_w + 2 * l["pad"] - l["k"]) // l["stride"] + 1
    xin, yout = l["C"] * tile_h * tile_w, l["C"] * Ho * Wo
    # backward: read dy, write dx; only max pooling also has to re-read x (to find the arg-max)
    return dict(fwd=((xin + yout) * esz, 0.0),
                bwd=((xin + yout + (xin if l["mode"] == "max" else 0)) * esz, 0.0))


# ------------------------------------------------------------------------------------------------
def usable_cpus():
    """Host threads this process can really use: scheduler affinity, capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def cpu_reference_setup(layers, base_scale, budget_s):
    """Thread count and sample size for the reference CPU path.  The reference gets its best
    configuration: the thread count is calibrated (oversubscribing a container whose quota is below
    the machine's core count makes the oneDNN path orders of magnitude slower, measured 68 s vs
    0.3 s per pass), and the sample (all layers at 1/scale linear size) is the largest whose pass
    fits `budget_s`.  Returns (threads, scale, seconds of one calibrated pass at base_scale)."""
    import torch

    from oracle import ref_port_torch as rp

    n = usable_cpus()
    cands = sorted({c for c in (n, n // 2, n // 4, 64, 32, 16, 8, 4) if 1 <= c <= n})
    best_t, best_c = None, cands[0]
    for c in cands:                                    # small to large; stop once it clearly gets worse
        torch.set_num_threads(c)
        rp.run_workload(layers, base_scale)            # per-shape warm-up at this thread count
        t = rp.run_workload(layers, base_scale, warm=False)
        if best_t is None or t < best_t:
            best_t, best_c = t, c
        elif t > 2.0 * best_t:
            break
    torch.set_num_threads(best_c)
    scale, t = base_scale, best_t
    # grow the sample while a pass is predicted to fit the budget; measured at every size because
    # the cost grows faster than the area once the working set leaves the caches (x5 per halving)
    while scale > 4 and 5.0 * t <= budget_s:
        scale //= 2
        rp.run_workload(layers, scale)
        t = rp.run_workload(layers, scale, warm=False)
    return best_c, scale, t


def run_reference(args):
    """--impl reference: the reference's own CPU path (restated with the PyTorch CPU ops it calls,
    oracle/ref_port_torch.py) on a bounded sample of the workload, all host threads."""
    import torch

    from oracle import ref_port_torch as rp

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    d, desc = load_layers(args.workload)
    steps = max(1, args.steps)
    # whole run (calibration + warm-up + K timed passes) bounded to ~2-3 minutes on a 16-CPU container
    budget = min(12.0, 120.0 / (steps + max(1, args.warmup)))
    if os.environ.get("SPCONV_BENCH_CPU_BUDGET_S"):          # tests: a smaller sample
        budget = float(os.environ["SPCONV_BENCH_CPU_BUDGET_S"])
    cores, scale, _ = cpu_reference_setup(d["layers"], args.cpu_scale, budget_s=budget)
    for _ in range(max(0, args.warmup - 1)):         # (cpu_reference_setup already ran one warm pass at this size)
        rp.run_workload(d["layers"], scale, warm=False)
    times = [rp.run_workload(d["layers"], scale, warm=False) for _ in range(steps)]
    t = statistics.median(times)
    # the sample is the same layer list at 1/scale linear size: work per image scales with scale^2
    val = 1.0 / (t * scale * scale)
    sample = ("all %d layers fwd+bwd at %dx%d (1/%d linear size), fp32, torch CPU ops, %d threads (calibrated; %d usable), "
              "%.2f s per pass, extrapolated x%d to %d^2" % (len(d["layers"]), d["image"] // scale, d["image"] // scale, scale,
                                                          cores, usable_cpus(), t, scale * scale, d["image"]))
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": len(times), "warmup": max(1, args.warmup), "ms_per_step": t * 1e3 * scale * scale, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "impl_note": "reference CPU path restated (pad + F.conv2d/F.*_pool2d + autograd)"},
        "cpu_baseline": {"value": val, "unit": "images/sec", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------
def cudnn_baseline(torch, layers_unique, order, dev, steps, warmup, full_size_cudnn=False):
    """The competitor BASELINE.md section 4 names: the identical layer list on STOCK PyTorch ops on the
    same B200 -- F.pad (the reference's ZeroPad2d copy, spatial.py:1020 / :1099, on every conv_spatial and
    every k>=3 Pool) + F.conv2d / F.*_pool2d (cuDNN / ATen) + autograd backward -- NCHW like the reference,
    cuDNN's default algorithm heuristics as the reference runs it (cudnn.benchmark's exhaustive search takes
    minutes at these sizes).  Two arms: bf16 storage, and fp32 storage with
    TF32 math (the reference's own dtype on tensor cores).  Same chain of independent layer fwd+bwd calls,
    same scratch tensors, CUDA events."""
    import torch.nn.functional as F

    out = {}
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        for arm, dt in (("bf16", torch.bfloat16), ("fp32_tf32", torch.float32)):
            _log("cudnn baseline arm %s" % arm)
            max_in = max(u["in_shape"][1] * u["in_shape"][2] * u["in_shape"][3] for u in layers_unique.values())
            max_out = max(u["out_shape"][1] * u["out_shape"][2] * u["out_shape"][3] for u in layers_unique.values())
            sx = torch.randn(max_in, dtype=dt, device=dev)
            sg = torch.randn(max_out, dtype=dt, device=dev) * 0.01
            ws = {}
            for key, u in layers_unique.items():
                l = u["layer"]
                if l["op"] == "conv":
                    ws[key] = (torch.randn(l["K"], l["C"], l["R"], l["S"], dtype=dt, device=dev) * 0.05).requires_grad_(True)

            def run_layer(key, split=1):
                u = layers_unique[key]
                l = u["layer"]
                ish = list(u["in_shape"])
                ish[2] //= split                      # `split` > 1: the top 1/split of the tile (see `splits` below)
                n = ish[1] * ish[2] * ish[3]
                x = sx[:n].view(ish).detach()
                if not u["first"]:
                    x.requires_grad_(True)
                if l["op"] == "conv":
                    xp = F.pad(x, (l["pad_w"], l["pad_w"], l["pad_h"], l["pad_h"])) if l.get("kind") == "conv_spatial" else x
                    y = F.conv2d(xp, ws[key], None, (l["stride_h"], l["stride_w"]), 0)
                else:
                    xp = F.pad(x, (l["pad"],) * 4) if l["k"] >= 3 else x
                    y = (F.max_pool2d if l["mode"] == "max" else F.avg_pool2d)(xp, l["k"], l["stride"], 0)
                gy = sg[:y.numel()].view(y.shape)
                if y.requires_grad:
                    y.backward(gy)
                x.grad = None
                if l["op"] == "conv":
                    ws[key].grad = None

            def ev(fn, reps):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / reps

            # per layer: one warm-up call, then 3 timed calls.  A convolution with a tensor of more than 2^31-1
            # elements makes cuDNN's default heuristics fall back to kernels that take SECONDS per call (measured
            # full-size on this B200: 3.9 s, 2.1 s, 11.3 s, 3.7 s for the four such layers, profiles/
            # r2a_bench_n1_with_cudnn.json -- a 29.4 s step, and minutes of bench time).  Those layers are timed
            # here on 1/split of the tile's rows and multiplied by split: cuDNN at its best, the comparison that
            # is hardest on libspconv.
            per, step_ms = [], 0.0
            for key, u in layers_unique.items():
                l = u["layer"]
                if l["op"] == "conv":
                    shape = "%d->%d %dx%d s%d @%dx%d" % (l["C"], l["K"], l["R"], l["S"], l["stride_h"], u["th"], u["tw"])
                else:
                    shape = "%s%d s%d C=%d @%dx%d" % (l["mode"], l["k"], l["stride"], l["C"], u["th"], u["tw"])
                big = max(u["in_shape"][1] * u["in_shape"][2] * u["in_shape"][3],
                          u["out_shape"][1] * u["out_shape"][2] * u["out_shape"][3])
                split = 1
                if l["op"] == "conv" and not full_size_cudnn:
                    while big // split > 2**31 - 1:
                        split *= 2
                run_layer(key, split)
                t1 = ev(lambda k=key, s_=split: run_layer(k, s_), 1)
                ms = (t1 if t1 > 50.0 else ev(lambda k=key, s_=split: run_layer(k, s_), 3)) * split
                e = dict(shape=shape, count=u["count"], fwd_bwd_ms=round(ms, 4))
                if split > 1:
                    e["timed_as"] = "%d x (1/%d of the rows)" % (split, split)
                per.append(e)
                step_ms += ms * u["count"]
            out[arm] = dict(ms_per_step=step_ms, images_per_sec=1000.0 / step_ms, per_layer=per)
            del sx, sg, ws
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out["what"] = ("stock F.pad + F.conv2d / F.*_pool2d + autograd (cuDNN/ATen, NCHW, default heuristics) over the same "
                   "layer list and tile, CUDA events; fwd_bwd_ms = pad + fprop + dgrad + wgrad of one layer; "
                   "ms_per_step = sum over the layer list of count * fwd_bwd_ms; convolutions holding a tensor of more than 2^31-1 "
                   "elements are timed on 1/split of the rows x split (entries with `timed_as`) because cuDNN takes "
                   "seconds per call on them at full size (29.4 s/step, profiles/r2a_bench_n1_with_cudnn.json; "
                   "--cudnn-full-size re-measures that)")
    return out


def model_stage_arm(torch, dev, dtype, image, steps, warmup):
    """The REAL spatial stage: the first six cells (stem1-3 + cell1_normal1-3, with their BatchNorm / ReLU /
    add / concat) of models.amoebanet.amoebanetd_spatial(18, 416) -- the module tree the reference's SP
    scripts train -- forward + backward on one tile of `image`^2, next to the same six cells of the stock
    (non-spatial) builder on cuDNN.  One GPU cannot hold the saved activations of the 8192^2 stage, so this arm
    runs the N=4 tile (4096^2)."""
    import torch.nn as nn

    from mpi4dl_b200.models import amoebanet

    def first6(m):
        return nn.Sequential(*list(m.children())[:6])

    res = {"image": image, "cells": "stem1, stem2, stem3, cell1_normal1..3", "dtype": str(dtype).replace("torch.", "")}
    builders = (("libspconv", lambda: first6(amoebanet.amoebanetd_spatial(0, 1, 1, mp_size=2, slice_method="square", num_classes=10,
                                                                         num_layers=18, num_filters=416))),
                ("stock_cudnn", lambda: first6(amoebanet.amoebanetd(num_classes=10, num_layers=18, num_filters=416))))
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = False
    try:
        for name, build in builders:
            _log("model stage arm %s" % name)
            torch.manual_seed(0)
            m = build().to(dev).to(dtype)
            if name == "libspconv":
                res["conv_modules"] = {}
                for x in m.modules():
                    if isinstance(x, nn.Conv2d):
                        res["conv_modules"][type(x).__name__] = res["conv_modules"].get(type(x).__name__, 0) + 1
            x = torch.randn(1, 3, image, image, device=dev, dtype=dtype)

            def step():
                y, _ = m(x)
                y.backward(torch.ones_like(y))
                for p_ in m.parameters():
                    p_.grad = None

            for _ in range(max(2, warmup)):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(max(2, steps)):
                step()
            e1.record()
            torch.cuda.synchronize()
            res[name + "_ms"] = e0.elapsed_time(e1) / max(2, steps)
            res[name + "_peak_GB"] = round(torch.cuda.max_memory_allocated(dev) / 1e9, 1)
            del m, x
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(dev)
    except Exception as e:  # noqa: BLE001 -- an auxiliary arm must never take the bench line down
        res["error"] = repr(e)[:300]
    finally:
        torch.backends.cudnn.benchmark = old
    return res


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="amoebanet", choices=list(WORKLOADS))
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--image", type=int, default=0, help="override the full image edge (debug)")
    ap.add_argument("--cpu-scale", type=int, default=32, help="linear down-scale of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--algo", default="auto", choices=["auto", "direct"])
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step from a CUDA graph (auto: when capture succeeds)")
    ap.add_argument("--no-cudnn-baseline", action="store_true")
    ap.add_argument("--cudnn-full-size", action="store_true",
                    help="time cuDNN on the whole tile even where a tensor exceeds 2^31-1 elements (adds minutes)")
    ap.add_argument("--no-model-stage", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy: "
                         "the flattened weight gradients, the step's result, and a fixed seeded sample of every distinct "
                         "layer's output and input gradient (the sampling adds one gather per sampled tensor to the step)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs saves the GPU path's outputs; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    # keep stdout clean for the ONE JSON line (NCCL / torchrun banners go to stderr)
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from mpi4dl_b200 import _lib
    from mpi4dl_b200.torchgems import spatial

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if world > 1:
        from mpi4dl_b200.torchgems import halo_transport
        halo_transport.negotiate(dev)            # collective: peer mailboxes unless some rank cannot
    L = _lib.lib()
    import ctypes as C
    sm, cc = C.c_int(), C.c_int()
    _lib.check(L.spc_device_info(local_rank, C.byref(sm), C.byref(cc)), "spc_device_info")

    d, desc = load_layers(args.workload)
    image = args.image or d["image"]
    shrink = d["image"] // image
    method, gr, gc = grid_for(world)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    esz = 2 if dtype == torch.bfloat16 else 4
    algo = _lib.SPC_ALGO_DIRECT if args.algo == "direct" else _lib.SPC_ALGO_AUTO

    # ---- build one module per distinct layer shape (weights shared by repeats) ------------------
    torch.manual_seed(0)          # the same weights (and host image) on every rank and in every run
    uniq = {}
    order = []
    for l in d["layers"]:
        l = dict(l)
        l["H"] //= shrink
        l["W"] //= shrink
        th, tw = l["H"] // gr, l["W"] // gc
        key = json.dumps({k: v for k, v in l.items() if k != "kind"}, sort_keys=True)
        if key not in uniq:
            if l["op"] == "conv":
                m = spatial.conv_spatial(rank, 1, world, l["C"], l["K"], (l["R"], l["S"]),
                                         stride=(l["stride_h"], l["stride_w"]), padding=(l["pad_h"], l["pad_w"]),
                                         bias=False, slice_method=method).to(dev).to(dtype)
                m.algo = algo
            else:
                m = spatial.Pool(rank, 1, world, l["k"], l["stride"], l["pad"], slice_method=method,
                                 operation="MaxPool2d" if l["mode"] == "max" else "AvgPool2d")
            uniq[key] = dict(layer=l, mod=m, th=th, tw=tw, count=0, first=(len(order) == 0))
        uniq[key]["count"] += 1
        order.append(key)

    # ---- scratch tensors (inputs larger than L2; reused across layers) --------------------------
    max_in = max(u["layer"]["C"] * u["th"] * u["tw"] for u in uniq.values())
    max_out = 0
    for u in uniq.values():
        l = u["layer"]
        if l["op"] == "conv":
            ho = (u["th"] + 2 * l["pad_h"] - l["R"]) // l["stride_h"] + 1
            wo = (u["tw"] + 2 * l["pad_w"] - l["S"]) // l["stride_w"] + 1
            u["out_shape"] = (1, l["K"], ho, wo)
        else:
            ho = (u["th"] + 2 * l["pad"] - l["k"]) // l["stride"] + 1
            wo = (u["tw"] + 2 * l["pad"] - l["k"]) // l["stride"] + 1
            u["out_shape"] = (1, l["C"], ho, wo)
        u["in_shape"] = (1, l["C"], u["th"], u["tw"])
        max_out = max(max_out, u["out_shape"][1] * ho * wo)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    scratch_x = torch.empty(max_in, dtype=dtype, device=dev).normal_(generator=g)
    scratch_gy = (torch.empty(max_out, dtype=dtype, device=dev).normal_(generator=g) * 0.01)
    total_params = sum(u["count"] * (u["mod"].weight.numel() if u["layer"]["op"] == "conv" else 0) for u in uniq.values())
    flat_grads = torch.zeros(total_params, dtype=dtype, device=dev)
    # host image tile for the e2e arm (the stem conv's input), pinned
    first = uniq[order[0]]
    host_img = torch.randn(first["in_shape"], dtype=dtype).pin_memory()
    dev_img = torch.empty(first["in_shape"], dtype=dtype, device=dev)
    host_out = torch.empty(1, dtype=torch.float32).pin_memory()

    def view(buf, shape):
        n = 1
        for s in shape:
            n *= s
        return buf[:n].view(shape)

    # --dump-outputs: layer outputs and input gradients are tens of GB per step and each is dropped after its layer,
    # so the step gathers a fixed seeded sample of them, once per distinct layer (repeats compute the same tensors)
    samples = {}
    if args.dump_outputs:
        gen = torch.Generator().manual_seed(4321)
        for i, key in enumerate(order):
            u = uniq[key]
            if order.index(key) != i:
                continue
            samples[i] = {}
            for name, shape in (("output", u["out_shape"]), ("input_grad", None if u["first"] else u["in_shape"])):
                if shape is not None:
                    n = math.prod(shape)
                    idx = torch.randint(n, (min(n, DUMP_SAMPLE),), generator=gen).sort().values.to(dev)
                    samples[i][name] = (idx, torch.empty(idx.numel(), dtype=dtype, device=dev))

    def take_sample(i, name, t):
        idx, buf = samples[i][name]
        with torch.no_grad():
            torch.index_select(t.reshape(-1), 0, idx, out=buf)

    def step_body(from_host_image):
        """One pass of the hot path: every layer fwd + bwd, gradient flatten, allreduce / P."""
        off = 0
        last = None
        for i, key in enumerate(order):
            u = uniq[key]
            x = dev_img if (from_host_image and i == 0) else view(scratch_x, u["in_shape"])
            x = x.detach()
            if not u["first"]:
                x.requires_grad_(True)
            y = u["mod"](x)
            sample = i in samples and not from_host_image
            if sample:
                take_sample(i, "output", y)
            y.backward(view(scratch_gy, u["out_shape"]))
            if sample and "input_grad" in samples[i]:
                take_sample(i, "input_grad", x.grad)
            x.grad = None
            if u["layer"]["op"] == "conv":
                w = u["mod"].weight
                flat_grads[off:off + w.numel()].copy_(w.grad.view(-1))   # SyncAllreduce flatten (comm.py:414-438)
                off += w.numel()
                w.grad = None
            last = y
        if world > 1:
            dist.all_reduce(flat_grads)                                   # comm.py:506-514
            flat_grads.div_(world)
        return last.detach().float().sum().view(1)

    graphs = {}
    last_result = {}

    def step(e2e=False):
        """e2e: the step's input image comes from pinned HOST memory and its result goes back to the host."""
        if e2e:
            dev_img.copy_(host_img, non_blocking=True)
        if graphs:
            graphs["e2e" if e2e else "dev"][0].replay()
            res = graphs["e2e" if e2e else "dev"][1]
        else:
            res = step_body(e2e)
        if e2e:
            host_out.copy_(res, non_blocking=True)
        last_result[e2e] = res

    def timed(nsteps, e2e):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(nsteps):
            step(e2e)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    _log("warm-up")
    for _ in range(max(args.warmup, 3)):
        step(False)
    step(True)
    torch.cuda.synchronize()
    _log("warm-up done")
    L.spc_launch_count(1)
    step(False)                                    # launches of ONE step, counted on the eager path
    torch.cuda.synchronize()
    launches_per_step = int(L.spc_launch_count(0))

    # ---- CUDA graph: the step is launch-bound on small tiles (N=8: ~1500 launches for ~24 ms of GPU work), so
    # the whole step -- halo post/collect included, their sequence numbers live in device memory -- is captured
    # once and replayed.  Same public-API calls, same kernels; only the CPU launch cost goes away.
    graph_note = "off"
    if args.graph != "off":
        ok = 1
        try:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            g_dev = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_dev):
                r_dev = step_body(False)
            g_e2e = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_e2e, pool=g_dev.pool()):
                r_e2e = step_body(True)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            ok = 0
            graph_note = "capture failed, eager launches: " + repr(e)[:200]
            sys.stderr.write("bench: CUDA graph capture failed: %r\n" % (e,))
            if args.graph == "on":
                raise
        if world > 1:
            flag = torch.tensor([ok], device=dev, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = int(flag.item())
        if ok:
            graphs["dev"] = (g_dev, r_dev)
            graphs["e2e"] = (g_e2e, r_e2e)
            graph_note = "whole step replayed from one CUDA graph (captured through the public torchgems.spatial API)"
            for _ in range(2):
                step(False)
                step(True)
        elif graph_note == "off":
            graph_note = "capture failed on a peer rank, eager launches"
    torch.cuda.synchronize()
    _log("launch mode: " + graph_note)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_wall0 = time.time()
    ms_total = timed(args.steps, False)
    launches = launches_per_step * args.steps
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        # saved before the e2e steps, which overwrite the weight gradients with those of the host image
        arrays = {"weight_grads": flat_grads, "step_result": last_result[False]}
        for i, s in samples.items():
            for name, (_, buf) in s.items():
                arrays["layer%02d_%s" % (i, name)] = buf
        write_dump(args.dump_outputs, arrays)
    ms_e2e = timed(args.steps, True)
    _log("timed: %.2f ms/step, e2e %.2f ms/step" % (ms_total / args.steps, ms_e2e / args.steps))

    # ---- per-kernel timing pass: every distinct layer-op through the C ABI, CUDA events ----------
    def ev_time(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    sp = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr())
    kinds = {}
    ops = []      # one record per (distinct layer, op)
    for key, u in uniq.items():
        l = u["layer"]
        x = view(scratch_x, u["in_shape"])
        gy = view(scratch_gy, u["out_shape"])
        y = torch.empty(u["out_shape"], dtype=dtype, device=dev)
        dx = torch.empty(u["in_shape"], dtype=dtype, device=dev)
        recs = []
        if l["op"] == "conv":
            w = u["mod"].weight.detach()
            dsc = _lib.ConvDesc(1, l["C"], u["th"], u["tw"], l["K"], l["R"], l["S"], l["stride_h"], l["stride_w"],
                                l["pad_h"], l["pad_w"], _lib.dtype_code(dtype), algo)
            nb = max(L.spc_conv_workspace_bytes(C.byref(dsc), i) for i in range(3))
            ws = torch.empty(nb + 16, dtype=torch.uint8, device=dev)
            dw = torch.zeros(w.shape, dtype=torch.float32, device=dev)
            bf = conv_bytes_flops(l, u["th"], u["tw"], esz)
            tc = [bool(L.spc_conv_uses_tcgen05(C.byref(dsc), i)) for i in range(3)]
            fns = [("fprop", lambda: _lib.check(L.spc_conv2d_fwd(C.byref(dsc), vp(x), None, vp(w), None, vp(y), vp(ws), nb, sp()), "fwd"), bf["fwd"], tc[0])]
            if not u["first"]:
                fns.append(("dgrad", lambda: _lib.check(L.spc_conv2d_dgrad(C.byref(dsc), vp(gy), vp(w), vp(dx), vp(ws), nb, sp()), "dgrad"), bf["dgrad"], tc[1]))
            fns.append(("wgrad", lambda: _lib.check(L.spc_conv2d_wgrad(C.byref(dsc), vp(x), None, vp(gy), vp(dw), None, 0, vp(ws), nb, sp()), "wgrad"), bf["wgrad"], tc[2]))
            def kernel_name(nm, is_tc):
                """which libspconv kernel serves this (layer, op) -- the dispatch rules of csrc/gemm_tc.cu"""
                if not is_tc:
                    return "wgrad_direct_kernel" if nm == "wgrad" else "conv_direct_kernel"
                taps, s1 = l["R"] * l["S"] > 1, l["stride_h"] == 1
                if taps and s1 and u["tw"] % 64 == 0:
                    if nm == "wgrad":
                        if l["S"] > 1 and l["K"] <= 128 and l["C"] <= 128:
                            return "wgrad_tap_kernel"
                    elif (l["K"] if nm == "fprop" else l["C"]) <= 128:
                        return "conv_tap_kernel"
                if nm == "wgrad":
                    return "pw_wgrad_pair_kernel" if (not taps and l["C"] >= 400 and l["K"] > 128) else "pw_wgrad_kernel"
                return "pw_gemm_kernel"

            for nm, fn, (by, fl), is_tc in fns:
                kern = kernel_name(nm, is_tc)
                recs.append((nm, kern, ev_time(fn), by, fl))
            shape = "%d->%d %dx%d s%d @%dx%d" % (l["C"], l["K"], l["R"], l["S"], l["stride_h"], u["th"], u["tw"])
        else:
            mode = _lib.SPC_POOL_MAX if l["mode"] == "max" else _lib.SPC_POOL_AVG
            dsc = _lib.PoolDesc(1, l["C"], u["th"], u["tw"], l["k"], l["stride"], l["pad"], mode, _lib.dtype_code(dtype))
            pb = pool_bytes(l, u["th"], u["tw"], esz)
            recs.append(("pool_fwd", "pool_fwd", ev_time(lambda: _lib.check(L.spc_pool2d_fwd(C.byref(dsc), vp(x), None, vp(y), sp()), "pool")), *pb["fwd"]))
            recs.append(("pool_bwd", "pool_bwd", ev_time(lambda: _lib.check(L.spc_pool2d_bwd(C.byref(dsc), vp(x), None, vp(gy), vp(dx), sp()), "poolb")), *pb["bwd"]))
            shape = "%s%d s%d C=%d @%dx%d" % (l["mode"], l["k"], l["stride"], l["C"], u["th"], u["tw"])
        for nm, kern, ms, by, fl in recs:
            ops.append(dict(shape=shape, op=nm, kernel=kern, count=u["count"], ms=ms, bytes=by, flops=fl))
            k = kinds.setdefault(kern, dict(ms=0.0, bytes=0.0, flops=0.0, launches=0))
            k["ms"] += ms * u["count"]
            k["bytes"] += by * u["count"]
            k["flops"] += fl * u["count"]
            k["launches"] += u["count"]
        del y, dx

    hbm, tfs, peak_src = peaks()
    # dominant kernel = the kernel with the largest share of the step; its roofline entry is the
    # launch-weighted aggregate over all its launches in one step (algorithmic bytes or flops of
    # those launches / their summed CUDA-event durations)
    dom_name, dk = max(kinds.items(), key=lambda kv: kv[1]["ms"])
    t_hbm = dk["bytes"] / (hbm * 1e9)
    t_tc = dk["flops"] / (tfs * 1e12)
    if t_hbm >= t_tc:
        roof = {"bound": "hbm", "achieved": dk["bytes"] / (dk["ms"] * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s"}
    else:
        roof = {"bound": "tensor", "achieved": dk["flops"] / (dk["ms"] * 1e-3) / 1e12, "peak": tfs, "unit": "TFLOP/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["kernel"] = dom_name
    roof["launches_per_step"] = dk["launches"]
    roof["peak_source"] = peak_src
    roof["share_of_step"] = dk["ms"] / sum(k["ms"] for k in kinds.values())
    # DRAM traffic of that kernel from the committed ncu --set full capture (profiles/), for the
    # heaviest single launch shape of the kernel, next to the same launch's algorithmic bytes
    roof["traffic"] = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        cand = sorted((o for o in ops if o["kernel"] == dom_name), key=lambda o: -o["ms"] * o["count"])
        for o in cand:
            kk = o["shape"] + " " + o["op"]
            if kk in tr:
                roof["traffic"] = tr[kk]["dram_bytes"]
                roof["traffic_launch"] = {"launch": kk, "algorithmic_bytes": o["bytes"], "event_ms": round(o["ms"], 4),
                                          "achieved_GBps": round(o["bytes"] / o["ms"] / 1e6, 1), "ncu": tr[kk].get("source")}
                break
        # every launch shape an ncu --set full capture exists for, good and bad alike (VERDICT r1 #11)
        roof["traffic_table"] = [
            {"launch": o["shape"] + " " + o["op"], "kernel": o["kernel"], "algorithmic_bytes": o["bytes"],
             "dram_bytes": tr[o["shape"] + " " + o["op"]]["dram_bytes"],
             "ratio": round(tr[o["shape"] + " " + o["op"]]["dram_bytes"] / o["bytes"], 2),
             "ncu": tr[o["shape"] + " " + o["op"]].get("source")}
            for o in ops if (o["shape"] + " " + o["op"]) in tr]
    except Exception:
        pass
    # whole-step roofline (BASELINE.md: sum over layer-ops of max(F/P, B/BW))
    t_roof = sum(o["count"] * max(o["bytes"] / (hbm * 1e9), o["flops"] / (tfs * 1e12)) for o in ops)
    roof["step_roofline_ms"] = t_roof * 1e3
    roof["step_frac"] = t_roof * 1e3 / (ms_total / args.steps)
    roof["kinds"] = {k: dict(ms=round(v["ms"], 3), launches=v["launches"], GBps=round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1),
                             TFLOPs=round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1)) for k, v in kinds.items()}
    per_layer = [dict(shape=o["shape"], op=o["op"], kernel=o["kernel"], count=o["count"], ms=round(o["ms"], 4),
                      GBps=round(o["bytes"] / o["ms"] / 1e6, 1), TFLOPs=round(o["flops"] / o["ms"] / 1e9, 1)) for o in ops]

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            _log("cpu baseline")
            from oracle import ref_port_torch as rp
            cores, cscale, _ = cpu_reference_setup(d["layers"], args.cpu_scale * shrink, budget_s=12.0)
            scale = cscale
            tcpu = rp.run_workload(d["layers"], scale, warm=False)
            cpu = {"value": 1.0 / (tcpu * (scale / shrink) ** 2), "unit": "images/sec", "cores": cores, "kind": "port",
                   "sample": "all %d layers fwd+bwd at 1/%d linear size (%dx%d image) in fp32 with the torch CPU ops the "
                             "reference calls (oracle/ref_port_torch.py; per-shape warm-up excluded), %.1f s timed, "
                             "extrapolated by area x%d; %d threads (calibrated, %d usable)" % (
                                 len(d["layers"]), scale // shrink, image * shrink // scale, image * shrink // scale, tcpu,
                                 (scale // shrink) ** 2, cores, usable_cpus())}
        ms_step = ms_total / args.steps
        cudnn = None
        if world == 1 and not args.no_cudnn_baseline:
            try:
                cudnn = cudnn_baseline(torch, uniq, order, dev, min(args.steps, 5), 2, args.cudnn_full_size)
                # where libspconv loses to stock cuDNN: our fprop+dgrad+wgrad (+ pool fwd+bwd) per layer vs its fwd_bwd
                ours = {}
                for o in ops:
                    ours[o["shape"]] = ours.get(o["shape"], 0.0) + o["ms"]
                for arm in ("bf16", "fp32_tf32"):
                    for r in cudnn[arm]["per_layer"]:
                        r["libspconv_ms"] = round(ours.get(r["shape"], float("nan")), 4)
                cudnn["loses_to_cudnn_bf16"] = [r["shape"] for r in cudnn["bf16"]["per_layer"]
                                                if r["libspconv_ms"] > r["fwd_bwd_ms"]]
                cudnn["speedup_vs_cudnn_bf16_step"] = round(cudnn["bf16"]["ms_per_step"] / ms_step, 3)
            except Exception as e:  # noqa: BLE001
                cudnn = {"error": repr(e)[:300]}
        stage = None
        if world == 1 and not args.no_model_stage and args.workload == "amoebanet" and not args.image:
            stage = model_stage_arm(torch, dev, dtype, 4096, 3, 2)
        out = {
            "metric": METRIC if args.workload == "amoebanet" else METRIC.replace("AmoebaNet-D 8192^2", "ResNet-v2-101 4096^2"),
            "value": 1000.0 / ms_step, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": args.dtype if args.dtype != "fp32" else "f32", "data": "synthetic",
            "config": {"workload": desc if not args.image else desc + " [debug image %d]" % image,
                       "global_batch": 1, "parallelism": "sp%d-%s" % (world, method), "tile": [image // gr, image // gc],
                       "layers": len(order), "l2_policy": "inputs larger than L2 (every layer tensor >> 126 MB)",
                       "note": "conv_spatial + Pool layers AND the 1x1 nn.Conv2d layers inside the spatial cells, "
                               "all through torchgems.spatial modules -> libspconv C ABI; BN/ReLU/concat excluded "
                               "(model_stage times the real cells with them)",
                       "algo": args.algo, "sm_count": sm.value, "launch_mode": graph_note},
            "e2e": {"value": 1000.0 / (ms_e2e / args.steps), "unit": "images/sec",
                    "h2d_bytes_per_step": host_img.numel() * host_img.element_size(), "d2h_bytes_per_step": 4},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "cudnn_baseline": cudnn,
            "model_stage": stage,
            "per_layer": per_layer,
        }
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        # tear down in order: captured graphs hold NCCL kernels; destroying the communicator under them hung the
        # process at exit (r2, N=2: JSON printed, exit only by timeout)
        dist.barrier()
        torch.cuda.synchronize()
        graphs.clear()
        import gc
        gc.collect()
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
