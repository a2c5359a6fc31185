"""Development tool: the stage-2 intensity augmentation (rehrseg_b200/intensity.py) on the GPU next to the oracle chain on the host.
Writes one JSON file (default profiles/intensity_bench.json) with the GPU's name and power limit read in the same run:
  - CUDA-event time of `apply` with each transform forced on alone, for [2,1,16,256,256] and [8,1,16,256,256] patches, with the
    bytes its passes move and their share of 7.7 TB/s (HBM3e, B200 data sheet).  At these sizes the kernels are short and the call
    is bound by launches and host work, not by HBM: the share of peak says how far from the bandwidth bound it is, nothing more;
  - host time of `draw` with only the noise forced on (the noise field comes from np.random.normal on the host);
  - Stage2Sampler.batch samples/s, with IntensityAugment() (the reference's probabilities) and without intensity;
  - the oracle chain (numpy / scipy, one process) on the same batch shapes.
Usage: python tools/intensity_bench.py [out.json]"""
import json
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from oracle import intensity as oi
from rehrseg_b200 import augment
from rehrseg_b200.intensity import NAMES, IntensityAugment

HBM = 7.7e12
PAD = 12
FORCED = {"noise": {"p_per_sample": 1.0}, "blur": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "brightness": {"p_per_sample": 1.0}, "contrast": {"p_per_sample": 1.0}, "lowres": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "gamma_inv": {"p_per_sample": 1.0}, "gamma": {"p_per_sample": 1.0}}
OFF = {k: {"p_per_sample": 0.0} for k in NAMES}


def moved_bytes(name, plan):
    """Bytes the passes of one transform read and write (fp32), summed over its rows."""
    z, x, y = plan.shape
    v = z * x * y
    total = 0
    for r in plan.rows[name]:
        if name == "noise":
            total += 3 * v                       # read x and the noise field, write x
        elif name == "blur":
            total += 6 * v                       # three axis passes, each reads and writes a volume
        elif name == "brightness":
            total += 2 * v
        elif name == "contrast":
            total += 3 * v                       # moments, then read + write
        elif name == "lowres":
            p = z * (r[2] + 2 * PAD) * (r[3] + 2 * PAD)
            total += z * r[2] * r[3] + p + p + 4 * p + p + v   # gather, moments, two prefilter passes, upsample (pad read, x written)
        else:
            total += 4 * v                       # moments, powered moments, read + write
    return 4 * total


def time_apply(name, b, iters=20):
    aug = IntensityAugment(**{**OFF, name: FORCED[name]})
    src = torch.randn(b, 1, 16, 256, 256, device="cuda")
    x = src.clone()
    plan = aug.draw(b, 1, (16, 256, 256), random.Random(0), np.random.RandomState(0))
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for _ in range(3):
        x.copy_(src)
        aug.apply(x, plan)
    ms = []
    for e0, e1 in ev:
        x.copy_(src)
        e0.record()
        aug.apply(x, plan)
        e1.record()
    torch.cuda.synchronize()
    ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
    med = ms[len(ms) // 2]
    nbytes = moved_bytes(name, plan)
    return {"batch": [b, 1, 16, 256, 256], "rows": len(plan.rows[name]), "median_ms": round(med, 4), "min_ms": round(ms[0], 4),
            "bytes": nbytes, "GB_per_s": round(nbytes / (med * 1e-3) / 1e9, 1), "share_of_7.7TBps": round(nbytes / (med * 1e-3) / HBM, 4)}


def time_noise_draw(b, iters=5):
    aug = IntensityAugment(**{**OFF, "noise": FORCED["noise"]})
    rn, rp = np.random.RandomState(0), random.Random(0)
    t0 = time.perf_counter()
    for _ in range(iters):
        aug.draw(b, 1, (16, 256, 256), rp, rn)
    return round((time.perf_counter() - t0) / iters * 1e3, 2)


def time_sampler(intensity, b, iters=10):
    rng = np.random.RandomState(1)
    ds = augment.Stage2Sampler((256, 256, 16), 4, intensity=intensity)
    ds.add_subject((rng.rand(288, 288, 80) * 300).astype(np.float32), (rng.rand(288, 288, 80) > 0.6).astype(np.uint8),
                   (rng.rand(288, 288, 80) * 255).astype(np.uint8))
    random.seed(0)
    np.random.seed(0)
    for _ in range(2):
        ds.batch([0] * b)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        ds.batch([0] * b)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / iters
    return {"batch": b, "ms_per_batch": round(dt * 1e3, 2), "samples_per_s": round(b / dt, 1)}


def time_oracle(b, overrides, seeds=3):
    data = np.random.RandomState(2).randn(b, 1, 16, 256, 256).astype(np.float32)
    t0 = time.perf_counter()
    for s in range(seeds):
        oi.intensity_transform(data.copy(), np.random.RandomState(s), random.Random(s), **overrides)
    dt = (time.perf_counter() - t0) / seeds
    return {"batch": [b, 1, 16, 256, 256], "s_per_batch": round(dt, 3), "samples_per_s": round(b / dt, 2)}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                             "intensity_bench.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    res = {"gpu": gpu.strip().splitlines()[0] if gpu.strip() else None, "torch_device": torch.cuda.get_device_name(0),
           "note": "apply() time per call from CUDA events around the whole call (host table build + launches + kernels); at these "
                   "sizes launch- and host-bound, so share_of_7.7TBps is far below 1 by construction",
           "apply_forced_alone": {}, "noise_draw_host_ms": {}, "sampler_batch": {}, "oracle_chain_host": {}}
    for name in NAMES:
        res["apply_forced_alone"][name] = [time_apply(name, b) for b in (2, 8)]
        print(name, res["apply_forced_alone"][name], flush=True)
    for b in (2, 8):
        res["noise_draw_host_ms"][f"b{b}"] = time_noise_draw(b)
    for b in (2, 8):
        res["sampler_batch"][f"b{b}_intensity_defaults"] = time_sampler(IntensityAugment(), b)
        res["sampler_batch"][f"b{b}_no_intensity"] = time_sampler(None, b)
        res["oracle_chain_host"][f"b{b}_defaults"] = time_oracle(b, {}, seeds=5)
        res["oracle_chain_host"][f"b{b}_forced"] = time_oracle(b, FORCED, seeds=1)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
