"""Development tool: cost of the opt-in fp16 saturation check (rehrseg_b200.rangecheck) on the benchmarked C1 step -- forward +
backward of the PlainConvUNet 3d_fullres on a synthetic [2,1,128,128,128] batch, captured once with GraphedTrainStep
(range_check=False) and once with range_check=True on the same model, the same loss as bench.py and the same inputs.  The two
graphs are replayed in alternating rounds; each round times `--steps` replays with CUDA events.  Writes one JSON file (default
profiles/range_check_bench.json) with the GPU's name and power limit read in the same run: ms/step median, min and max over the
rounds for each variant, the relative cost of the check, both engine launch counts, and the (empty) report of the checked step.
Usage: python tools/range_check_bench.py [--out out.json] [--steps 20] [--rounds 7]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from rehrseg_b200 import seg_model as sm
from rehrseg_b200.graphs import GraphedTrainStep


def _time(step, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "range_check_bench.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("range_check_bench needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    torch.manual_seed(1234)
    model = sm.plainconv_unet_3d_fullres().cuda()
    gen = torch.Generator().manual_seed(100)
    x = torch.randn((2, 1, 128, 128, 128), generator=gen).cuda()
    g = torch.randn((2, 2, 128, 128, 128), generator=gen).cuda()

    def loss_fn(out, t):
        return torch.dot(out.float().reshape(-1), t.reshape(-1)) / out.numel()

    steps = {"off": GraphedTrainStep(model, loss_fn, (x, g)), "on": GraphedTrainStep(model, loss_fn, (x, g), range_check=True)}
    for s in steps.values():
        _time(s, 3)
    times = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, s in steps.items():
            times[k].append(_time(s, args.steps))
    med = {k: statistics.median(v) for k, v in times.items()}
    res = {
        "gpu": gpu[0] if gpu else "unknown",
        "workload": "C1: PlainConvUNet 3d_fullres fwd+bwd, 2x1x128^3, GraphedTrainStep replay",
        "steps_per_round": args.steps,
        "rounds": args.rounds,
        "ms_per_step": {k: {"median": round(med[k], 4), "min": round(min(v), 4), "max": round(max(v), 4),
                            "rounds": [round(t, 4) for t in v]} for k, v in times.items()},
        "check_cost_rel": round(med["on"] / med["off"] - 1.0, 5),
        "engine_launches": {k: s.engine_launches for k, s in steps.items()},
        "report_on_clean_input": [tuple(r) for r in steps["on"].range_report()],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
