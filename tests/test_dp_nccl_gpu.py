"""Data-parallel exchange through the C-ABI (fdx_comm_*, NCCL) on 2 GPUs: the bucketed, overlapped
all-reduce captured inside the training graph must give every rank the same gradients / loss as (a) the
single un-overlapped call and (b) the mean of the two ranks' local gradients computed without any exchange.
Skipped with fewer than 2 visible GPUs (the CPU-side host logic is covered by tests/test_dp_gloo_cpu.py)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["FDX_ROOT"])
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
from flaxdiff_b200 import ops, utils
from flaxdiff_b200.inputs import DiffusionInputConfig
from flaxdiff_b200.models.simple_unet import Unet
from flaxdiff_b200.predictors import KarrasPredictionTransform
from flaxdiff_b200.schedulers import EDMNoiseScheduler
from flaxdiff_b200.trainer import GeneralDiffusionTrainer, adamw

def make(**kw):
    model = Unet(attention_configs=(None, None, None, {"heads": 8}), dtype=torch.bfloat16)
    return GeneralDiffusionTrainer(model, adamw(1e-3), EDMNoiseScheduler(1, sigma_max=80, rho=7, sigma_data=0.5),
                                   DiffusionInputConfig("image", (32, 32, 3), []), rngs=4,
                                   model_output_transform=KarrasPredictionTransform(0.5), device=dev, **kw)

def rel(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()

B = 4
g = torch.Generator().manual_seed(100 + rank)
img = torch.randint(0, 256, (B, 32, 32, 3), dtype=torch.uint8, generator=g).to(dev)
noise = torch.randn(B, 32, 32, 3, generator=g).to(dev)
t = torch.randn(B, generator=g).to(dev)

# (b) local gradients without any exchange, then an explicit mean through torch.distributed
tr0 = make(use_cuda_graph=False, distributed_training=False)
loss0 = tr0._fwd_bwd(img, noise, t).clone()
gl = tr0._grads.flat.clone()
dist.all_reduce(gl); gl /= world
dist.all_reduce(loss0); loss0 /= world

res = {}
for name, env, graph in (("overlap_graph", {"FDX_NO_DP_OVERLAP": "0"}, True), ("overlap_eager", {"FDX_NO_DP_OVERLAP": "0"}, False),
                         ("single_call", {"FDX_NO_DP_OVERLAP": "1"}, True), ("default", {}, True)):
    for k, v in env.items():
        os.environ[k] = v
    tr = make(use_cuda_graph=graph)
    assert tr._comm is not None and tr.world_size == world
    assert tr._overlap == (env.get("FDX_NO_DP_OVERLAP") == "0")   # unset: one exchange after the backward
    if graph:
        loss = tr._graphed_fwd_bwd(img, noise, t)
        loss = tr._graphed_fwd_bwd(img, noise, t)          # replay
    else:
        loss = tr._fwd_bwd(img, noise, t).clone()
    if not tr._overlap:
        tr._gbuf[-64:-63].copy_(loss)
        tr._comm.allreduce_avg_(tr._gbuf)
        loss = tr._gbuf[-64:-63].clone()
    torch.cuda.synchronize()
    e_g, e_l = rel(tr._grads.flat, gl), abs(loss.item() - loss0.item()) / abs(loss0.item())
    # every rank must hold the same bits
    chk = tr._grads.flat.double().sum().reshape(1).clone()
    both = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(both, chk)
    same = all(torch.equal(both[0], b) for b in both)
    res[name] = (e_g, e_l, same, len(tr._exchange.bounds))
    for k in env:
        os.environ.pop(k)
# a full train step through the public step function keeps the replicas identical
tr = make(use_cuda_graph=True)
step = tr._define_train_step(B)
for _ in range(3):
    tr.state, loss, tr.rngstate = step(tr.state, tr.rngstate, {"image": img}, rank)
chk = tr.state.params.flat.double().sum().reshape(1)
both = [torch.zeros_like(chk) for _ in range(world)]
dist.all_gather(both, chk)
res["replicas_identical"] = all(torch.equal(both[0], b) for b in both)
if rank == 0:
    print("RESULT", res, "nccl", ops.nccl_version(), flush=True)
    ok = all(v[0] < 2e-2 and v[1] < 1e-3 and v[2] for k, v in res.items() if k != "replicas_identical")
    ok = ok and res["replicas_identical"]
    print("OK" if ok else "FAIL", flush=True)
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_bucketed_overlapped_allreduce_two_gpus(tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "dp_worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, FDX_ROOT=root)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                       capture_output=True, text=True, env=env, timeout=600)
    sys.stderr.write(r.stdout[-3000:] + "\n" + r.stderr[-3000:])
    assert r.returncode == 0 and "\nOK" in ("\n" + r.stdout), r.stdout[-2000:]
