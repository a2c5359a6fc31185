"""Multi-GPU (NCCL over NVLink, one process per GPU) checks of the two places the hot path shards -- run by `torchrun` in a
sub-process on 2 GPUs, skipped on a single-GPU box:
  * data-parallel training: after `allreduce_gradients` every rank holds the SAME gradients, equal to the mean of the ranks'
    own gradients (each rank's own gradient is recomputed locally from every rank's batch);
  * sharded sliding window: (tile, mirror) units dealt over 2 ranks give the single-GPU blended logits within 2e-3 and the same
    result on both ranks."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["REHR_ROOT"])
import torch, torch.distributed as dist
from oracle import seg_model as ref_seg
from rehrseg_b200 import seg_model as sm, sliding_window as sw, train_step as ts, functional as Fn
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
kw = {k: v for k, v in ref_seg.plan_kwargs("tiny").items() if k != "upscale"}
torch.manual_seed(7)
model = sm.PlainConvUNet(**kw).to(dev)          # same seed on every rank -> identical replicas
params = [p for p in model.parameters()]

def batch(r):
    g = torch.Generator().manual_seed(100 + r)
    return torch.randn((2, 1, 16, 32, 32), generator=g).to(dev), torch.randn((2, 2, 16, 32, 32), generator=g).to(dev)

def grads_of(r):
    for p in params:
        p.grad = None
    x, t = batch(r)
    ((model(x).float() * t).sum() / t.numel()).backward()
    return [p.grad.clone() if p.grad is not None else None for p in params]

own = [grads_of(r) for r in range(world)]        # every rank recomputes every rank's gradient: the expected mean is local
for p, g in zip(params, own[rank]):
    p.grad = None if g is None else g.clone()
n = ts.allreduce_gradients(params)
assert n > 0
worst = 0.0
for i, p in enumerate(params):
    if p.grad is None:
        continue
    want = sum(o[i] for o in own) / world
    worst = max(worst, float((p.grad - want).abs().max() / (want.abs().max() + 1e-20)))
    gathered = [torch.empty_like(p.grad) for _ in range(world)]
    dist.all_gather(gathered, p.grad)
    assert all(torch.equal(gathered[0], q) for q in gathered), "ranks disagree after the all-reduce"
assert worst < 1e-5, worst

# the same mean from the CUDA-graph step with the bucketed all-reduce captured inside and overlapped with the backward pass
from rehrseg_b200.graphs import GraphedTrainStep
def loss_fn(out, t):
    return (out.float() * t).sum() / t.numel()
xb, tb = batch(rank)
step = GraphedTrainStep(model, loss_fn, (xb, tb), dp_group=True, dp_buckets=4)
for _ in range(2):
    step(xb, tb)
torch.cuda.synchronize()
worst_g = 0.0
for i, p in enumerate(params):
    if p.grad is None:
        continue
    want = sum(o[i] for o in own) / world
    worst_g = max(worst_g, float((p.grad - want).abs().max() / (want.abs().max() + 1e-20)))
    gathered = [torch.empty_like(p.grad) for _ in range(world)]
    dist.all_gather(gathered, p.grad)
    assert all(torch.equal(gathered[0], q) for q in gathered), "ranks disagree after the captured all-reduce"
assert worst_g < 1e-4, worst_g

# sharded sliding window vs the single-GPU driver
torch.manual_seed(3)
seg = sm.SegModel(**ref_seg.plan_kwargs("tiny")).to(dev).eval()
vol = torch.randn((1, 40, 64, 48), generator=torch.Generator().manual_seed(5)).to(dev)
patch = [16, 32, 32]
sl = sw._internal_get_sliding_window_slicers(vol.shape[1:], patch_size=patch)
with torch.no_grad():
    single = sw._internal_predict_sliding_window_return_logits(vol, sl, seg, True, 0, 1, patch, use_gaussian=True, deep_supervision=False)
    shard = sw.predict_sliding_window_sharded(vol, sl, seg, out_idx=0, patch_size=patch, use_gaussian=True, deep_supervision=False)
err = float((shard.float() - single.float()).norm() / single.float().norm())
assert err < 2e-3, err
both = [torch.empty_like(shard) for _ in range(world)]
dist.all_gather(both, shard)
assert torch.equal(both[0], both[1])
step.close()     # captured NCCL kernels must be released before the communicator is destroyed
if rank == 0:
    print(f"MULTIGPU_OK grads_max_rel {worst:.2e} graph_dp_max_rel {worst_g:.2e} sw_rel_l2 {err:.2e} tiles {len(sl)}", flush=True)
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_nccl_dp_gradients_and_sharded_sliding_window(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, REHR_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29617", str(script)]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MULTIGPU_OK" in res.stdout
