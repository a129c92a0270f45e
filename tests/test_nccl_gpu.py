"""Data parallel on real GPUs (VERDICT r1 weak #1g): two NCCL ranks, differently seeded, each on its own rays.  After
TrainStep's start-up broadcast and one backward, both ranks hold IDENTICAL .grad, equal to the mean of the two
single-rank gradients -- what the reference's DistributedDataParallel wrapper produces
(reflect_sampling_nerf_pipeline.py:73-77).  Needs >= 2 GPUs (skipped on a machine with one)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import synthetic_rays

pytestmark = pytest.mark.gpu
SIZES = dict(num_coarse_samples=32, num_importance_samples=32, num_reflect_coarse_samples=16, num_reflect_importance_samples=16)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from reflect_sampling_nerf_b200.model import ReflectSamplingNeRFModel, ReflectSamplingNeRFModelConfig
    from reflect_sampling_nerf_b200.rays import RayBundle
    from reflect_sampling_nerf_b200.train_path import TrainStep
    torch.manual_seed(100 + rank)                                # nerfstudio: machine.seed + global_rank
    model = ReflectSamplingNeRFModel(ReflectSamplingNeRFModelConfig(**SIZES)).cuda().train()
    stepper = TrainStep(model, world_size=world)                 # broadcasts rank 0's parameters
    n = 256
    batches = [[t.cuda() for t in synthetic_rays(n, 60 + r, pixel_area=3.2e-6)] for r in range(world)]
    g = torch.Generator().manual_seed(9)
    jit = {k: torch.rand(n, s, generator=g).cuda() for k, s in (("uniform", 33), ("pdf", 33), ("reciprocal", 17), ("reflect_pdf", 17))}
    model.set_jitter(**jit)

    def grads(batch, dp):
        model.field.dp_world_size = world if dp else 1
        for p in model.parameters():
            p.grad = None
        o, d, pa, img = batch
        out = model(RayBundle(origins=o, directions=d, pixel_area=pa))
        sum(model.get_loss_dict(out, {"image": img}).values()).backward()
        torch.cuda.synchronize()
        return torch.cat([p.grad.reshape(-1) for p in model.field.parameters() if p.grad is not None]).clone()
    singles = [grads(b, False) for b in batches]                  # every rank computes both single-rank gradients locally
    mean = sum(singles) / world
    mine = grads(batches[rank], True)                             # the data-parallel backward: one all-reduce of the blob
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine)
    res = {
        "identical_across_ranks": all(torch.equal(gathered[0], t) for t in gathered),
        "rel_err_vs_mean": float((mine - mean).norm() / mean.norm()),
        "params_identical": True,
    }
    flat = torch.cat([p.detach().reshape(-1) for p in model.field.parameters()])
    allp = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(allp, flat)
    res["params_identical"] = all(torch.equal(allp[0], t) for t in allp)
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_gradients_are_identical_and_the_mean(tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    res = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(2)]
    for r in res:
        assert r["params_identical"]
        assert r["identical_across_ranks"]
        assert r["rel_err_vs_mean"] < 2e-4, r          # fp32 atomics order in the wgrad flush differs run to run


def _worker_graph(rank, world, port, out_dir):
    """TrainStep(graph=True) at world_size 2: two CUDA graphs per step around the eager NCCL all-reduce."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from reflect_sampling_nerf_b200.model import ReflectSamplingNeRFModel, ReflectSamplingNeRFModelConfig
    from reflect_sampling_nerf_b200.rays import RayBundle
    from reflect_sampling_nerf_b200.train_path import TrainStep
    n, steps = 256, 8
    g = torch.Generator().manual_seed(9)
    jit = {k: torch.rand(n, s, generator=g).cuda() for k, s in (("uniform", 33), ("pdf", 33), ("reciprocal", 17), ("reflect_pdf", 17))}
    batches = [[t.cuda() for t in synthetic_rays(n, 200 + 10 * rank + i, pixel_area=3.2e-6)] for i in range(steps)]

    def train(graph):
        torch.manual_seed(100 + rank)
        model = ReflectSamplingNeRFModel(ReflectSamplingNeRFModelConfig(**SIZES)).cuda().train()
        model.set_jitter(**jit)
        stepper = TrainStep(model, world_size=world, graph=graph)
        p0 = torch.cat([p.detach().reshape(-1) for p in model.field.parameters()]).clone()
        losses = []
        for o, d, pa, img in batches:
            losses.append(stepper.step(RayBundle(origins=o, directions=d, pixel_area=pa), img).clone())
        torch.cuda.synchronize()
        assert (stepper.graph is not None) == graph
        if graph:
            assert "finish" in stepper.static              # the split form, not one graph with NCCL inside
        return p0, torch.cat([p.detach().reshape(-1) for p in model.field.parameters()]).clone(), torch.stack(losses)
    p0, p_eager, l_eager = train(False)
    p0g, p_graph, l_graph = train(True)
    allp = [torch.empty_like(p_graph) for _ in range(world)]
    dist.all_gather(allp, p_graph)
    res = {
        "same_start": bool(torch.equal(p0, p0g)),
        "params_identical": all(torch.equal(allp[0], t) for t in allp),
        "moved": float((p_eager - p0).norm()),
        "rel_err_update": float((p_graph - p_eager).norm() / (p_eager - p0).norm()),
        "loss_rel": float(((l_graph - l_eager).abs() / l_eager.abs()).max()),
    }
    torch.save(res, os.path.join(out_dir, f"g{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_split_graph_step_matches_the_eager_step(tmp_path):
    mp.spawn(_worker_graph, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    res = [torch.load(os.path.join(tmp_path, f"g{r}.pt")) for r in range(2)]
    for r in res:
        assert r["same_start"] and r["params_identical"], r
        assert r["moved"] > 0
        assert r["rel_err_update"] < 2e-2, r           # 8 RAdam steps; fp32 atomics order differs run to run
        assert r["loss_rel"] < 2e-2, r
