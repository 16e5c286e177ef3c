"""world_size-2 NCCL test (two GPUs of one node) of the ONE collective on the training path:
the flat gradient all-reduce (training/utils/distributed.py; reference: DDP over gloo,
warp_drive/training/trainers/trainer_a2c.py:137-146, utils/process_group_torch.py:6-20), and
of a two-rank Trainer iteration: after the update both ranks hold identical parameters.
Skipped on boxes with one GPU (run: gpurun --gpus 2 -- python -m pytest tests/test_gpu_nccl.py)."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist

    from warp_drive_b200.training.utils.distributed import flat_allreduce_mean_, init_process_group

    torch.cuda.set_device(rank)
    init_process_group("nccl", device_id=rank)
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(71, 256), torch.nn.ReLU(),
                                torch.nn.Linear(256, 43)).cuda()
    x = torch.randn(64, 71, device="cuda", generator=torch.Generator("cuda").manual_seed(100 + rank))
    model(x).square().mean().backward()
    local = [p.grad.clone() for p in model.parameters()]
    buf = flat_allreduce_mean_([p.grad for p in model.parameters()], world)
    gathered = [torch.zeros_like(buf) for _ in range(world)]
    flat_local = torch.cat([g.reshape(-1) for g in local])
    dist.all_gather(gathered, flat_local)
    mean = sum(gathered) / world
    got = torch.cat([p.grad.reshape(-1) for p in model.parameters()])
    ok = bool(torch.allclose(got, mean, atol=1e-6, rtol=1e-5))

    # ---- a two-rank Trainer iteration: different env seeds per rank, identical parameters
    import copy

    import yaml

    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_continuous import TagContinuous
    from warp_drive_b200.training.trainer import Trainer

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "warp_drive_b200", "training", "run_configs",
                           "tag_continuous.yaml"), encoding="utf8") as fp:
        cfg = yaml.safe_load(fp)
    cfg["env"].update(num_taggers=2, num_runners=8, episode_length=20)
    cfg["trainer"].update(num_envs=16, train_batch_size=16 * 5, num_episodes=4, seed=7)
    for p in cfg["policy"].values():
        p["model"]["fc_dims"] = [32, 32]
    cfg["saving"].update(basedir="/tmp", name="nccl_test", tag=f"rank{rank}",
                         metrics_log_freq=1000, model_params_save_freq=1000)
    env = TagContinuous(**cfg["env"])
    w = EnvWrapper(env, num_envs=16, env_backend="b200")
    pm = {"runner": sorted(env.runners), "tagger": sorted(env.taggers)}
    tr = Trainer(w, copy.deepcopy(cfg), pm, num_devices=world, device_id=rank, verbose=False)
    tr.train()
    flat = torch.cat([p.detach().reshape(-1) for pol in tr.policies
                      for p in tr.models[pol].parameters()])
    both = [torch.zeros_like(flat) for _ in range(world)]
    dist.all_gather(both, flat)
    same = bool(torch.equal(both[0], both[1]))
    finite = bool(torch.isfinite(flat).all())
    out.put((rank, ok, same, finite))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_flat_gradient_allreduce_and_two_rank_training_nccl():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(out.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert all(r[1] for r in res), "flat all-reduce (mean) differs from the gathered mean"
    assert all(r[2] for r in res), "ranks diverged after the update"
    assert all(r[3] for r in res)
