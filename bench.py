#!/usr/bin/env python
"""bench.py -- the measured line for the REHRSeg hot path on B200.

Workload (BASELINE.json `metric`: "patch fwd+bwd/sec & conv TFLOP/s vs bf16 peak"; north_star target "PlainConvUNet
3d_fullres 128^3 patch fwd+bwd"): one STEP = forward + backward of the nnU-Net PlainConvUNet (3d_fullres plan, 6 stages,
features 32..320, InstanceNorm + LeakyReLU) on a synthetic batch of 2 patches [2,1,128,128,128] per GPU, bf16 tensor-core
arithmetic with fp32 accumulation, fp32 master weights re-packed to bf16 every step (as after an optimiser update),
and -- for N > 1 -- the data-parallel gradient all-reduce over NCCL.  `value` = patches / s over all ranks.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a engine
    python bench.py --impl reference ...                            # the reference's CPU PyTorch path (oracle port)
    python bench.py --impl eager_gpu ...                            # informational: torch eager + cuDNN on the same GPU
    python bench.py --dump-outputs DIR ...                          # also write the last timed step's loss and gradients

Keys follow the driver contract: value (inputs resident in HBM), e2e (inputs copied from pinned host memory inside the
timed region through the public nn.Module API, loss read back), roofline (dominant kernel, measured live with CUDA
events), cpu_baseline (oracle on the host cores), clocks (nvidia-smi sampled during the timed region), gpu_launches.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line.  Native libraries print there too (NCCL's "NCCL version ..." banner when NCCL_DEBUG is
# set), so file descriptor 1 is pointed at stderr for the whole run and the JSON line is written to a saved copy of the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


import torch  # noqa: E402

PATCH = (128, 128, 128)
BATCH = 2
METRIC = "patch_fwd_bwd_per_s"
UNIT = "patches/s"
WORKLOAD = "nnUNet PlainConvUNet 3d_fullres fwd+bwd, synthetic 2x1x128x128x128 patch per GPU"


# ----------------------------------------------------------------------------------------------------------------
def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


def conv_flops(model: torch.nn.Module, in_shape) -> dict:
    """Algorithmic FLOPs (2*M*N*K) of every conv / transposed conv of `model` for one forward on `in_shape`
    ([B,C,D,H,W]) by shape propagation on the module tree (encoder stages -> decoder), and the fwd+bwd total:
    dgrad + wgrad = 2x fwd, except that the very first conv needs no input gradient."""
    b, c, d, h, w = in_shape
    fwd = 0.0
    first = None
    sp = [(d, h, w)]
    cur = (d, h, w)
    for stage in model.encoder.stages:
        for blk in stage[0].convs:
            cv = blk.conv
            cur = tuple((i + 2 * p - k) // s + 1 for i, k, s, p in zip(cur, cv.kernel_size, cv.stride, cv.padding))
            f = 2.0 * b * cur[0] * cur[1] * cur[2] * cv.out_channels * cv.in_channels * cv.kernel_size[0] * cv.kernel_size[1] * cv.kernel_size[2]
            if first is None:
                first = f
            fwd += f
        sp.append(cur)
    skips = sp[1:]
    cur = skips[-1]
    dec = model.decoder
    for s in range(len(dec.stages)):
        tc = dec.transpconvs[s]
        # kernel == stride transposed conv: every input voxel meets every weight once
        fwd += 2.0 * b * cur[0] * cur[1] * cur[2] * tc.in_channels * tc.out_channels * tc.kernel_size[0] * tc.kernel_size[1] * tc.kernel_size[2]
        cur = skips[-(s + 2)]
        for blk in dec.stages[s].convs:
            cv = blk.conv
            fwd += 2.0 * b * cur[0] * cur[1] * cur[2] * cv.out_channels * cv.in_channels * cv.kernel_size[0] * cv.kernel_size[1] * cv.kernel_size[2]
    seg = dec.seg_layers[-1]
    fwd += 2.0 * b * cur[0] * cur[1] * cur[2] * seg.in_channels * seg.out_channels
    return {"fwd": fwd, "fwd_bwd": 3.0 * fwd - first}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._pump, daemon=True)
        self.thr.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


DUMP_MAX_ELEMS = 1 << 18   # per gradient: the 3d_fullres UNet's 101 gradients come to ~20 MB in all


def dump_outputs(out_dir: str, loss: torch.Tensor, named_params) -> None:
    """Write what a training step hands its caller -- the loss and every parameter gradient -- as float32 `loss.npy` and
    `grad.<parameter name>.npy`, so that two builds can be compared output for output.  A gradient of more than
    DUMP_MAX_ELEMS elements is written flattened, as the same sorted sample of its elements on every run (a generator seeded
    by the parameter's name)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    for name, p in named_params:
        if p.grad is None:       # without deep supervision only the last seg layer reaches the loss
            continue
        g = p.grad.detach().float()
        if g.numel() > DUMP_MAX_ELEMS:
            idx = np.random.default_rng(zlib.crc32(name.encode())).choice(g.numel(), DUMP_MAX_ELEMS, replace=False)
            g = g.reshape(-1)[torch.from_numpy(np.sort(idx)).to(g.device)]
        np.save(os.path.join(out_dir, f"grad.{name}.npy"), g.cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's PlainConvUNet on the host cores
# ----------------------------------------------------------------------------------------------------------------
def _oracle_unet():
    from oracle import seg_model as ref_seg, third_party as tp
    kw = ref_seg.plan_kwargs("3d_fullres")
    kw.pop("upscale")
    torch.manual_seed(1234)
    return tp.PlainConvUNet(**kw)


def _cpu_step(model, x, g):
    for p in model.parameters():
        p.grad = None
    out = model(x)
    loss = (out * g).sum() / out.numel()
    loss.backward()
    return float(loss.detach())


def cpu_sample_inputs(ds: int, batch: int = 1):
    gen = torch.Generator().manual_seed(0)
    x = torch.randn((batch, 1, ds, PATCH[1], PATCH[2]), generator=gen)
    g = torch.randn((batch, 2, ds, PATCH[1], PATCH[2]), generator=torch.Generator().manual_seed(1))
    return x, g


def cpu_baseline(budget_s: float = 25.0) -> dict:
    """One bounded fwd+bwd of the oracle PlainConvUNet on the host cores: a depth slab [1,1,Ds,128,128] of one patch,
    Ds in {32,64,128} picked from a 32-slab calibration so that the timed sample is <= ~budget_s."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = _oracle_unet()
    x, g = cpu_sample_inputs(32)
    _cpu_step(model, x, g)  # oneDNN primitive warm-up + calibration
    t0 = time.perf_counter(); _cpu_step(model, x, g); t32 = time.perf_counter() - t0
    ds = 128 if t32 * 4 <= budget_s else (64 if t32 * 2 <= budget_s else 32)
    if ds != 32:
        x, g = cpu_sample_inputs(ds)
        t0 = time.perf_counter(); _cpu_step(model, x, g); t = time.perf_counter() - t0
    else:
        t = t32
    return {"value": (ds / PATCH[0]) / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"1 fwd+bwd of [1,1,{ds},128,128] ({ds}/128 of one patch), fp32 oracle PlainConvUNet, torch "
                      f"{torch.__version__} CPU, {t:.2f} s", "seconds": t}


def reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = _oracle_unet()
    x, g = cpu_sample_inputs(32)
    _cpu_step(model, x, g)
    t0 = time.perf_counter(); _cpu_step(model, x, g); t32 = time.perf_counter() - t0
    total = max(1, args.steps + args.warmup)
    budget = 150.0 / total
    ds = 128 if t32 * 4 <= budget else (64 if t32 * 2 <= budget else 32)
    x, g = cpu_sample_inputs(ds)
    for _ in range(args.warmup):
        _cpu_step(model, x, g)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _cpu_step(model, x, g)
    el = time.perf_counter() - t0
    val = args.steps * (ds / PATCH[0]) / el
    sample = f"each step = 1 fwd+bwd of [1,1,{ds},128,128] ({ds}/128 of one 128^3 patch), fp32, {cores} threads"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "device": "host CPU", "what": "oracle port of the reference PlainConvUNet "
                       "(dynamic_network_architectures 0.3.1 restated; /root/reference is absent on the GPU box)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------------------------
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the flagship workload (`value` and `e2e`); the extra configs time their own fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "eager_gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2-C5 / cuDNN-eager entries (bench_extras.py, each timed over its own fixed count)")
    ap.add_argument("--launch", default="graph", choices=["graph", "eager"],
                    help="b200 arm: replay the step from one CUDA graph (rehrseg_b200.graphs.GraphedTrainStep) or launch it from Python")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and parameter gradients of the last one to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU arms")
        return reference_arm(args)

    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path for the B200 arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from rehrseg_b200 import functional as Fn

    if args.impl == "b200":
        from rehrseg_b200 import seg_model as sm
        torch.manual_seed(1234)
        model = sm.plainconv_unet_3d_fullres().to(dev)
        dtype = "bf16"
    else:
        model = _oracle_unet().to(dev).to(memory_format=torch.channels_last_3d)
        dtype = "bf16 autocast (cuDNN)"
    params = [p for p in model.parameters()]
    flops = conv_flops(model, (BATCH, 1, *PATCH))

    gen = torch.Generator().manual_seed(100 + rank)
    x_host = torch.randn((BATCH, 1, *PATCH), generator=gen).pin_memory()
    g_host = torch.randn((BATCH, 2, *PATCH), generator=gen).pin_memory()
    x_dev, g_dev = x_host.to(dev), g_host.to(dev)
    dp = {"flat": None, "active": None}  # gradient bucket, sized after the first backward (unused seg layers get no grad)

    def loss_fn(out, g):
        return torch.dot(out.float().reshape(-1), g.reshape(-1)) / out.numel()  # <logits, g> / numel (SURVEY 8(d))

    use_graph = args.impl == "b200" and args.launch == "graph"
    gstep = None
    if use_graph:
        from rehrseg_b200.graphs import GraphedTrainStep
        # the whole step (weight re-pack, forward, loss, backward) captured once; replays re-read the live parameters
        # N > 1: the data-parallel gradient mean is captured too, in buckets that overlap the backward pass
        gstep = GraphedTrainStep(model, loss_fn, (x_dev, g_dev), dp_group=True if world > 1 else None)
        x_dev, g_dev = gstep.static_inputs       # "resident" steps run on the static inputs without any copy

    def fwd_bwd(x, g, eager=False):
        if use_graph and not eager:
            loss = gstep(x, g)                   # device->device copy into the static inputs unless x, g already are them
        else:
            for p in params:
                p.grad = None
            if args.impl == "b200":
                Fn.clear_weight_cache()  # bf16 operand copies are re-derived every step, as after an optimiser update
                out = model(x)
            else:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    out = model(x)
            loss = loss_fn(out, g)
            loss.backward()
        if world > 1 and not (use_graph and not eager):  # python-launched step: gradient mean over NVLink through one flat bucket
            if dp["active"] is None:
                dp["active"] = [p for p in params if p.grad is not None]
            grads = [p.grad for p in dp["active"]]
            flat = torch.cat([g.reshape(-1) for g in grads])      # one gather kernel into the bucket
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)            # NCCL ring / NVLS over NVLink
            off, views = 0, []
            for g in grads:
                views.append(flat[off:off + g.numel()].view_as(g))
                off += g.numel()
            torch._foreach_copy_(grads, views)                     # one batched scatter back into .grad
        return loss

    def step_resident():
        return fwd_bwd(x_dev, g_dev)

    # e2e: every step's inputs are copied from pinned host memory (image + cotangent, fp32, as train_all.py:524-529 moves its
    # batch) and the loss is read back.  The copy of step i+1 is issued on a side stream while step i computes (what a
    # DataLoader with pin_memory + non_blocking gives the reference), double-buffered; all copies are inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(x_dev), torch.empty_like(g_dev)) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"i": 0, "primed": False}

    def prefetch(slot):
        # the slot's previous consumer (two steps back) has completed: every step ends with a host read of its loss
        with torch.cuda.stream(copy_stream):
            bufs[slot][0].copy_(x_host, non_blocking=True)
            bufs[slot][1].copy_(g_host, non_blocking=True)
            ready[slot].record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        if not e2e_state["primed"]:
            prefetch(i % 2)
            e2e_state["primed"] = True
        torch.cuda.current_stream(dev).wait_event(ready[i % 2])
        x, g = bufs[i % 2]
        prefetch((i + 1) % 2)        # next step's inputs travel while this step's kernels run
        loss = fwd_bwd(x, g)
        e2e_state["i"] = i + 1
        return float(loss.detach())  # device -> host read of the step's result

    def timed(step_fn, steps, sampler=None):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = Fn.launches()
        e0.record()
        for _ in range(steps):
            out = step_fn()
        e1.record()
        torch.cuda.synchronize()
        launches = Fn.launches() - l0
        clocks = sampler.stop() if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), launches, clocks, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    phys = int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local]) if os.environ.get("CUDA_VISIBLE_DEVICES") else local
    ms, launches, clocks, loss = timed(step_resident, args.steps, ClockSampler(phys) if rank == 0 else None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model.named_parameters())
    step_e2e()
    ms_e2e, _, _, _ = timed(step_e2e, args.steps)

    # roofline of the dominant kernel: one instrumented step, CUDA events around every conv-engine launch
    roof = None
    kernels = {}
    if args.impl == "b200":
        torch.cuda.synchronize()
        l0 = Fn.launches()
        with Fn.kernel_timer() as kt:
            torch.cuda._sleep(200_000_000)  # let the host run ahead so launch latency stays out of the event pairs
            fwd_bwd(x_dev, g_dev, eager=True)   # launched from Python so that every conv-engine launch gets its event pair
        if use_graph:
            launches = gstep.engine_launches * args.steps   # engine kernels counted while the replayed step was captured
        summ = kt.summary()
        peaks = measured_peaks()
        for name, (n, tms, fl) in summ.items():
            kernels[name] = {"launches": n, "ms": round(tms, 4), "tflops": round(fl / tms / 1e9, 1) if tms > 0 else None}
        # dominant kernel = the (family, layer) INSTANTIATION with the largest time in the step -- a family mixes 1100 TFLOP/s
        # layers with 200 TFLOP/s parity-class launches, so a family average says little about either
        inst = {}
        for name, tag, tms, fl in kt.rows():
            n, t, f = inst.get((name, tag), (0, 0.0, 0.0))
            inst[(name, tag)] = (n + 1, t + tms, f + fl)
        if inst:
            (name, tag), (n, tms, fl) = max(inst.items(), key=lambda kv: kv[1][1])
            achieved = fl / tms / 1e9
            # the instrumented step is ONE eager step after an idle gap (clocks at their burst level): burst peak is the denominator
            peak = float(peaks["bf16_tflops"])
            fam_n, fam_ms, fam_fl = summ[name]
            # DRAM bytes (read + write) per launch of this instantiation from a committed `ncu --set full` capture, if one exists
            traffic, traffic_file = None, None
            tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
            if os.path.exists(tpath):
                with open(tpath) as f:
                    ent = json.load(f).get(f"{name}|{tag}")
                if ent:
                    traffic, traffic_file = ent.get("dram_bytes_per_launch"), ent.get("file")
            roof = {"kernel": name, "layer": tag, "bound": "tensor", "achieved": round(achieved, 1), "peak": peak, "unit": "TFLOP/s",
                    "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_file,
                    "launches_per_step": n, "avg_launch_ms": round(tms / n, 4), "flops_per_launch": fl / n,
                    "share_of_step": round(tms / (ms / args.steps), 4),
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops, burst ({peaks['_source']}): the kernel is timed in a single "
                                   "python-launched step after an idle gap (side-stream forks off while the event pairs are recorded)",
                    "frac_of_sustained": round(achieved / float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])), 4),
                    "family": {"launches_per_step": fam_n, "ms": round(fam_ms, 4), "tflops": round(fam_fl / fam_ms / 1e9, 1),
                               "share_of_step": round(fam_ms / (ms / args.steps), 4)}}

    # the other BASELINE configs, same run (C3 sharded over all ranks; the single-GPU ones only at N = 1)
    extras = {}
    if args.impl == "b200" and not args.no_extras:
        torch.cuda.empty_cache()
        import bench_extras
        extras = bench_extras.run_all(dev, measured_peaks(), rank, world, _oracle_unet, BATCH, PATCH)

    def teardown():
        """Captured NCCL kernels must be gone before the communicator is destroyed (GraphedTrainStep.close); a watchdog makes sure a
        stuck teardown can never hold the job: the JSON line is already out by then."""
        if world <= 1:
            return
        if gstep is not None:
            gstep.close()
        done = threading.Event()

        def watchdog():
            if not done.wait(20):
                os._exit(0)

        threading.Thread(target=watchdog, daemon=True).start()
        dist.barrier()
        dist.destroy_process_group()
        done.set()

    if rank != 0:
        teardown()
        return
    per_step = ms / args.steps
    value = world * BATCH * args.steps / (ms / 1e3)
    e2e_val = world * BATCH * args.steps / (ms_e2e / 1e3)
    peaks = measured_peaks()
    tfl = flops["fwd_bwd"] / (per_step * 1e-3) / 1e12
    line = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(per_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": world * BATCH, "patch": list(PATCH),
                       "parallelism": f"dp{world}" if world > 1 else "single", "cache": "per-step working set ~8 GB >> 126 MB L2",
                       "weights_repacked_each_step": True,
                       "launch": ("one CUDA graph per step (rehrseg_b200.graphs.GraphedTrainStep)" if use_graph else "python"), "algorithmic_tflop_per_step": round(flops["fwd_bwd"] / 1e12, 4)},
            "conv_tflops_per_gpu": round(tfl, 1), "frac_bf16_peak_burst": round(tfl / float(peaks["bf16_tflops"]), 4),
            "frac_bf16_peak_sustained": round(tfl / float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])), 4),
            "e2e": {"value": round(e2e_val, 3), "unit": UNIT, "h2d_bytes_per_step": world * (x_host.numel() + g_host.numel()) * 4,
                    "d2h_bytes_per_step": world * 4, "ms_per_step": round(ms_e2e / args.steps, 4)},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "kernels": kernels}
    if extras:
        line["configs"] = extras
        for key in ("sw_volumes_per_s",):    # BASELINE.json's metric names volumes/s explicitly: surface it at the top level
            v = extras.get("c3_sliding_window", {}).get(key)
            if v is not None:
                line[key] = v
    if args.impl != "b200":
        line["impl"] = args.impl
        line["gpu_launches"] = None
    if world == 1 and args.impl == "b200" and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    emit(line)
    teardown()


if __name__ == "__main__":
    main()
