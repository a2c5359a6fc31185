"""Development tool: the SR-stage training iteration (train_sr, train_all.py:118-139; BASELINE config C2's shape: patches_lr
[8,2,4,256,256], patches_hr [8,2,16,256,256]) with the plain loss statements and with loss_ops.FusedSRLoss, launched from Python
and replayed from one CUDA graph, for the plain and the UASR head.  Writes one JSON file (default profiles/sr_step_bench.json) with
the GPU's name and power limit read in the same run:
  - the loss alone, forward + backward on a fixed [8,2,4,256,256] prediction (and [8,1,4,256,256] uncertainty): CUDA-event time
    per iteration over >= 200 iterations after a warm-up, and the CUDA kernels one iteration launches (from a separate
    torch.profiler run); the fused and plain loss values on the same inputs, which must agree to 1e-5 relative;
  - the whole iteration (forward, loss, backward; no optimiser) in four variants: eager sr_train_step with the plain losses /
    with fused_loss, GraphedSRStep with the plain losses / with fused_loss.  The variants run in alternating rounds; each round
    times `--steps` iterations with CUDA events, and the JSON gives the median, min and max over the rounds.
Usage: python tools/sr_step_bench.py [--out out.json] [--steps 20] [--rounds 5]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from rehrseg_b200 import flavr, loss_ops, train_step as ts

B, S_LR, S_HR, H, W = 8, 4, 16, 256, 256
SEP, NS = 4, 4


def _batch(seed):
    g = torch.Generator().manual_seed(seed)
    lr = torch.rand((B, 2, S_LR, H, W), generator=g)
    lr[:, 1] = (lr[:, 1] > 0.8).float()
    hr = torch.rand((B, 2, S_HR, H, W), generator=g)
    hr[:, 1] = (hr[:, 1] > 0.8).float()
    return lr.cuda(), hr.cuda()


def _events(fn, iters, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _kernels(fn, iters=5):
    """CUDA kernels (and memsets / copies, counted apart) one call of fn launches, from a torch.profiler run of `iters` calls."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    mem = [e for e in ev if e.name.startswith(("Memset", "Memcpy"))]
    return {"kernels": round((len(ev) - len(mem)) / iters, 2), "memsets_copies": round(len(mem) / iters, 2)}


def loss_alone(unc, iters):
    g = torch.Generator(device="cuda").manual_seed(3)
    hat = torch.randn((B, 2, S_LR, H, W), generator=g, device="cuda") * 3
    hat[:, 0] = torch.rand((B, S_LR, H, W), generator=g, device="cuda")
    hat.requires_grad_(True)
    u = (torch.rand((B, 1, S_LR, H, W), generator=g, device="cuda") * 0.9 + 0.05).requires_grad_(True) if unc else None
    _, hr = _batch(4)
    l1, bd = torch.nn.L1Loss(), ts.BCEDiceLoss(1, 1)
    fused = loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc)
    out = (hat, u) if unc else hat

    def run(fused_loss):
        def f():
            hat.grad = None
            if u is not None:
                u.grad = None
            loss = ts._sr_loss(out, hr, l1, bd, SEP, NS, unc, fused_loss)
            loss.backward()
            return loss
        return f

    res = {}
    vals = {}
    for name, fl in (("plain", None), ("fused", fused)):
        vals[name] = float(run(fl)())
        res[name] = {"ms_fwd_bwd": round(_events(run(fl), iters, 20), 4), **_kernels(run(fl))}
    r = abs(vals["fused"] - vals["plain"]) / abs(vals["plain"])
    res["loss_plain"], res["loss_fused"], res["loss_rel_diff"] = vals["plain"], vals["fused"], r
    if r > 1e-5:
        raise SystemExit(f"fused and plain SR losses disagree: {vals} (rel {r:.3g})")
    return res


def whole_step(unc, steps, rounds):
    batch = _batch(5)
    lr_src, hr_src = batch

    def model():
        torch.manual_seed(0)
        return flavr.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc).cuda().train()

    l1, bd = torch.nn.L1Loss(), ts.BCEDiceLoss(1, 1)
    fused = loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc)
    m_eager = model()
    lr_dev = lr_src.clone()

    def eager(fused_loss):
        def f():
            lr_dev.copy_(lr_src)           # what GraphedSRStep's load does: the forward mutates its input in place
            return ts.sr_train_step(m_eager, (lr_dev, hr_src), l1, bd, None, None, SEP, NS, unc, fused_loss=fused_loss)["loss"]
        return f

    g_plain = ts.GraphedSRStep(model(), batch, l1, bd, SEP, NS, unc)
    g_fused = ts.GraphedSRStep(model(), batch, slice_separation=SEP, num_slices=NS, enable_uncertainty=unc, fused_loss=fused)
    variants = {"eager_plain": eager(None), "eager_fused": eager(fused),
                "graphed_plain": lambda: g_plain(batch)["loss"], "graphed_fused": lambda: g_fused(batch)["loss"]}
    losses = {k: float(f()) for k, f in variants.items()}
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, f in variants.items():
            times[k].append(_events(f, steps, 3))
    res = {}
    for k, t in times.items():
        med = statistics.median(t)
        res[k] = {"ms_per_step_median": round(med, 3), "ms_per_step_min": round(min(t), 3), "ms_per_step_max": round(max(t), 3),
                  "samples_per_s": round(B / med * 1e3, 1), "loss": losses[k]}
    res["graphed_engine_launches"] = {"plain": g_plain.step.engine_launches, "fused": g_fused.step.engine_launches}
    g_plain.close()
    g_fused.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sr_step_bench.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--loss-iters", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sr_step_bench needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    res = {"gpu": gpu.strip().splitlines()[0] if gpu.strip() else None, "torch_device": torch.cuda.get_device_name(0),
           "shape": {"patches_lr": [B, 2, S_LR, H, W], "patches_hr": [B, 2, S_HR, H, W], "slice_separation": SEP, "num_slices": NS},
           "note": "loss_alone: forward + backward of the loss on fixed inputs, CUDA events over loss_iters iterations; kernels per "
                   "iteration from a separate torch.profiler run.  whole_step: forward + loss + backward, no optimiser; CUDA events "
                   f"over {a.steps} steps per round, {a.rounds} rounds with the four variants alternating; median / min / max over "
                   "the rounds.  graphed_engine_launches counts the engine's own kernels per replay (ATen kernels not counted).",
           "loss_alone": {}, "whole_step": {}}
    for unc in (False, True):
        head = "uasr" if unc else "plain"
        res["loss_alone"][head] = loss_alone(unc, a.loss_iters)
        print(head, "loss_alone", res["loss_alone"][head], flush=True)
        res["whole_step"][head] = whole_step(unc, a.steps, a.rounds)
        print(head, "whole_step", res["whole_step"][head], flush=True)
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
