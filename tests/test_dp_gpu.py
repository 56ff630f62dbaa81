"""Data parallelism on real GPUs (SURVEY.md section 4, "distributed" row; 8e): two B200s, one process each, NCCL.

* N-GPU gradients after the bucketed all-reduce == 1-GPU gradients of the same GLOBAL batch (rank-strided shards);
* the CUDA-graph step (two graphs around inline bucket all-reduces) == the eager step with hook-issued, overlapped
  all-reduces, parameter for parameter, after several optimizer steps;
* a ragged global batch (unequal local batches, fno_b200.data.epoch_plan weights) still gives the global-mean gradient.
Skipped on a machine with fewer than two GPUs.
"""
import os
import socket
import sys
from pathlib import Path

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "sciml-pde_b200"))
CTOR = dict(num_channels=2, modes1=6, modes2=6, width=12, initial_step=4)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rel(a, b):
    a, b = (torch.view_as_real(t) if t.is_complex() else t for t in (a, b))
    return float(((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).detach())


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from fno_b200 import data
    from fno_b200.dp import BucketedGradAllReduce
    from fno_b200.fno import FNO2d
    from fno_b200.steptail import nrmse_loss
    from fno_b200.train import FusedTrainStep

    G = 8
    xx, yy, grid = (t.to(dev) for t in data.synthetic_batch(G, 32, CTOR["initial_step"], CTOR["num_channels"], seed=3))
    res = {}
    # (1) gradients: DP on rank-strided shards vs the whole global batch on one GPU
    torch.manual_seed(16)
    model = FNO2d(**CTOR).to(dev)
    ref = FNO2d(**CTOR).to(dev)
    ref.load_state_dict(model.state_dict())
    dp = BucketedGradAllReduce(model)
    dp.zero_grad()
    nrmse_loss(model(xx[rank::world], grid[rank::world]), yy[rank::world]).backward()
    dp.finish()
    nrmse_loss(ref(xx, grid), yy).backward()
    res["grad_err"] = max(_rel(p.grad, q.grad) for p, q in zip(model.parameters(), ref.parameters()))
    # (1b) ragged global batch of 5: local batches 3 and 2, weights 3*2/5 and 2*2/5
    dp.zero_grad()
    ref.zero_grad()
    sl = slice(0, 5)
    lx, ly, lg = xx[sl][rank::world], yy[sl][rank::world], grid[sl][rank::world]
    (nrmse_loss(model(lx, lg), ly) * (lx.shape[0] * world / 5.0)).backward()
    dp.finish()
    nrmse_loss(ref(xx[sl], grid[sl]), yy[sl]).backward()
    res["ragged_grad_err"] = max(_rel(p.grad, q.grad) for p, q in zip(model.parameters(), ref.parameters()))
    # (2) graph step with captured all-reduces vs eager step with hook-issued all-reduces
    outs = []
    for graph in (False, True):
        torch.manual_seed(16)
        m = FNO2d(**CTOR).to(dev)
        step = FusedTrainStep(m, lr=1e-3, weight_decay=1e-4, t_max=50, dp=BucketedGradAllReduce(m), graph=graph)
        losses = [float(step(xx[rank::world], yy[rank::world], grid[rank::world])) for _ in range(8)]
        torch.cuda.synchronize()
        outs.append((m, losses))
    res["graph_vs_eager_param_err"] = max(_rel(p, q) for p, q in zip(outs[1][0].parameters(), outs[0][0].parameters()))
    res["graph_vs_eager_loss_err"] = max(abs(a - b) / abs(b) for a, b in zip(outs[1][1], outs[0][1]))
    # every rank holds the same parameters
    flat = torch.cat([(torch.view_as_real(p) if p.is_complex() else p).detach().flatten() for p in outs[1][0].parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    res["rank_divergence"] = float(max((g - gathered[0]).abs().max() for g in gathered))
    if rank == 0:
        torch.save(res, os.path.join(out_dir, "dp_gpu.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(240)
def test_two_gpu_data_parallel_step(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    res = torch.load(tmp_path / "dp_gpu.pt")
    print(res)
    assert res["grad_err"] < 2e-5                      # fp32 summation order only (two half-batch means vs one mean)
    assert res["ragged_grad_err"] < 2e-5
    assert res["graph_vs_eager_param_err"] < 1e-5
    assert res["graph_vs_eager_loss_err"] < 1e-5
    assert res["rank_divergence"] == 0.0
