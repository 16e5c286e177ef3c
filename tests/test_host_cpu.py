"""CPU-only tests (run in the build container): host logic of the package, the C ABI
library's exports, and the rule that product code never touches oracle/."""
import ast
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from helpers import close


def test_library_exports_every_declared_symbol(wdb_lib):
    """Every function declared in include/wdb200.h is exported by libwdb200.so and typed
    in warp_drive_b200/lib.py (no compute call: there is no GPU here)."""
    from warp_drive_b200 import lib as wlib

    header = open(os.path.join(ROOT, "include", "wdb200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(wdb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(wlib.exported_symbols()), declared ^ set(wlib.exported_symbols())
    raw = ctypes.CDLL(wlib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert wdb_lib.wdb_abi_version() == 1
    assert wdb_lib.wdb_rng_state_bytes(10) == 16 + 80
    # only the C ABI is visible (kernels and helpers are hidden)
    out = subprocess.run(["nm", "-D", "--defined-only", wlib.LIB_PATH], capture_output=True,
                         text=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert {e for e in exported if e.startswith("wdb_")} == declared
    assert not [e for e in exported if "_kernel" in e]


def test_library_is_sm100a_only(wdb_lib):
    from warp_drive_b200 import lib as wlib

    out = subprocess.run(["cuobjdump", "--list-elf", wlib.LIB_PATH], capture_output=True,
                         text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_kernel_resource_usage_matches_the_residency_the_design_assumes(wdb_lib):
    """DESIGN.md 3.1 / 3.2 size the grids on: fused env kernel 96 registers x 320 threads ->
    two CTAs per SM (register file 65536); its 1024-thread instance (BASELINE config 4) must
    fit one CTA; the persistent MLP kernel 416 threads x 128 registers -> one CTA per SM.
    A compiler or source change that silently breaks this shows up here, without a GPU."""
    from warp_drive_b200 import lib as wlib

    out = subprocess.run(["cuobjdump", "--dump-resource-usage", wlib.LIB_PATH],
                         capture_output=True, text=True).stdout
    usage = {}
    name = None
    for line in out.splitlines():
        line = line.strip()
        if line.startswith("Function "):
            name = line[len("Function "):].rstrip(":")
        elif line.startswith("REG:") and name:
            usage[name] = {k: int(v) for k, v in re.findall(r"([A-Z]+):(\d+)", line)}
    def find(*parts):
        hits = [u for n, u in usage.items() if all(p in n for p in parts)]
        assert hits, (parts, list(usage)[:5])
        return hits

    for u in find("tag_continuous_kernel", "Li320E"):
        assert u["REG"] * 320 * 2 <= 65536 and u["STACK"] <= 128, u
    for u in find("tag_continuous_kernel", "Li1024E"):
        assert u["REG"] * 1024 <= 65536, u
    for u in find("mlp_forward_kernel"):
        assert u["REG"] * 416 <= 65536 and u["STACK"] <= 32, u
    for kernel in ("cartpole_step_kernel", "mountain_car_step_kernel", "pendulum_step_kernel",
                   "acrobot_step_kernel", "tag_gridworld_step_kernel", "sample_actions_kernel",
                   "reset_when_done_kernel"):
        for u in find(kernel):
            assert u["REG"] <= 80 and u["LOCAL"] == 0, (kernel, u)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "warp_drive_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            path = os.path.join(dirpath, fn)
            if fn.endswith(".py"):
                tree = ast.parse(open(path).read())
                for node in ast.walk(tree):
                    names = []
                    if isinstance(node, ast.Import):
                        names = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        names = [node.module or ""]
                    assert not any(n.split(".")[0] == "oracle" for n in names), path
            if fn.endswith((".cu", ".cuh", ".h", ".py")):
                text = open(path).read()
                assert "wd_oracle" not in text and "oracle/" not in text.replace(
                    "oracle/_ref", "").replace("oracle/)", ""), path


def test_kernel_path_rejects_cpu_tensors(wdb_lib):
    import torch

    from warp_drive_b200 import lib as wlib

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        wlib.ptr(torch.zeros(4))


# ------------------------------------------------------------------ data manager
def _dm(**kw):
    from warp_drive_b200.managers.data_manager import CUDADataManager

    return CUDADataManager(device="cpu", **kw)


def test_data_manager_registry_semantics():
    """Down-casts, *_at_reset twins, *_for_log buffers, scalars, reserved arrays
    (ref tests/warp_drive/pycuda_tests/test_data_manager.py:24-87)."""
    from warp_drive_b200.utils.data_feed import DataFeed

    dm = _dm(num_agents=5, num_envs=2, episode_length=3)
    assert dm.meta_info("n_agents") == 5 and dm.meta_info("n_agents").dtype == np.int32
    assert dm.get_shape("_done_") == (2,) and dm.get_shape("_log_mask_") == (4,)
    feed = DataFeed()
    feed.add_data(name="X", data=np.arange(10, dtype=np.float64).reshape(2, 5),
                  save_copy_and_apply_at_reset=True, log_data_across_episode=True)
    feed.add_data(name="Y", data=[[1, 2, 3, 4, 5], [6, 7, 8, 9, 10]])
    feed.add_data(name="a", data=100)
    feed.add_data(name="b", data=0.5)
    feed.add_data(name="flag", data=True)
    dm.push_data_to_device(feed)
    assert dm.get_dtype("X") == "float32" and dm.get_dtype("Y") == "int32"
    assert dm.pull_data_from_device("X").dtype == np.float32
    assert dm.device_data("a") == 100 and dm.device_data("a").dtype == np.int32
    assert dm.device_data("b").dtype == np.float32
    assert dm.device_data("flag") == 1 and dm.device_data("flag").dtype == np.int32
    assert dm.is_data_on_device("X_at_reset") and dm.reset_data_list == ["X"]
    assert dm.get_shape("X_for_log") == (4, 5) and dm.log_data_list == ["X"]
    # tensors are views of device memory, not of the host copy
    dm.data_on_device_via_torch("X")[:] = 7
    assert (dm.pull_data_from_device("X") == 7).all()
    assert (dm.pull_data_from_device("X_at_reset") == np.arange(10).reshape(2, 5)).all()
    dm.reset_device("X")
    assert (dm.pull_data_from_device("X") == np.arange(10).reshape(2, 5)).all()
    with pytest.raises(AssertionError):
        dm.push_data_to_device(feed)            # duplicate names are refused
    pool = DataFeed()
    pool.add_pool_for_reset(name="Y_pool", data=np.zeros((7, 5), np.int32), reset_target="Y")
    dm.push_data_to_device(pool)
    assert dm.get_reset_pool("Y") == "Y_pool" and "Y" not in dm.reset_data_list
    dm.add_shared_constants({"kIndexToActionArr": [[0, 0], [1, 0]]})
    assert dm.shared_constant("kIndexToActionArr").dtype == np.int32


def test_function_feed_and_kernel_lookup(wdb_lib):
    from warp_drive_b200.managers.function_manager import (
        CUDAFunctionFeed, CUDAFunctionManager)
    from warp_drive_b200.utils.data_feed import DataFeed

    dm = _dm(num_agents=5, num_envs=2, episode_length=3)
    feed = DataFeed()
    feed.add_data(name="X", data=np.zeros((2, 5), np.float32))
    feed.add_data(name="s", data=3)
    dm.push_data_to_device(feed)
    ff = CUDAFunctionFeed(dm)
    args = ff(["X", "s", ("episode_length", "meta"), ("X", "device")])
    assert args[0] is dm.device_data("X") and args[1] == 3 and args[2] == 3
    assert ff(["ignored once cached"]) is args
    fm = CUDAFunctionManager(num_agents=5, num_envs=2, device="cpu")
    assert fm.block == (5, 1, 1) and fm.grid == (2, 1)
    fm2 = CUDAFunctionManager(num_agents=5, num_envs=2, blocks_per_env=2, device="cpu")
    assert fm2.block == (3, 1, 1) and fm2.grid == (4, 1)        # function_manager.py:65-67
    fm.initialize_default_functions()
    fm.initialize_functions(["CudaTagContinuousStep", "CudaTagGridWorldStep", "testkernel"])
    f = fm.get_function("CudaTagGridWorldStep")
    assert callable(f) and callable(f[fm.grid, fm.block])
    with pytest.raises(KeyError):
        fm.initialize_functions(["NoSuchKernel"])
    with pytest.raises(RuntimeError):       # CPU tensors never reach a kernel
        fm.get_function("testkernel")(dm.device_data("X"), dm.device_data("X"),
                                      dm.device_data("_done_"), dm.device_data("X"), 2.0, 1, 1, 3)


# ------------------------------------------------------------------ CPU env backends
def _cfg(fx):
    out = {}
    for k in fx:
        if k.startswith("cfg__"):
            v = fx[k]
            out[k[5:]] = v.item() if v.shape == () else v
    return out


@pytest.mark.parametrize("name", ["test1", "test2", "config1"])
def test_cpu_gridworld_env_matches_reference_numpy(name):
    """BASELINE config 1: TagGridWorld via EnvWrapper(env_backend='cpu')."""
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_gridworld import TagGridWorld

    fx = load_golden(f"gridworld_numpy_{name}.npz")
    env = EnvWrapper(TagGridWorld(**_cfg(fx)), env_backend="cpu")
    obs = env.reset()
    N = env.n_agents
    assert close(np.stack([obs[a] for a in range(N)]), fx["obs0"], 1e-6).all()
    ep = 0
    for t in range(fx["actions"].shape[0]):
        if fx["episode"][t] != ep:
            env.reset()
            ep = fx["episode"][t]
        o, r, d, _ = env.step({a: int(fx["actions"][t][a]) for a in range(N)})
        assert close(np.stack([o[a] for a in range(N)]), fx["obs"][t], 1e-6).all(), t
        assert close(np.array([r[a] for a in range(N)]), fx["rewards"][t], 1e-6).all(), t
        assert bool(d["__all__"]) == bool(fx["done"][t])


@pytest.mark.parametrize("name", ["test1", "test2", "test3", "test4", "partial_mid"])
def test_cpu_tag_continuous_env_matches_reference_numpy(name):
    """Same seed -> same taggers / start state as the reference class; the vectorised CPU
    step tracks the reference NumPy step (2e-5)."""
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_continuous import TagContinuous

    fx = load_golden(f"tag_continuous_numpy_{name}.npz")
    env = EnvWrapper(TagContinuous(**_cfg(fx)), env_backend="cpu")
    obs = env.reset()
    N = env.n_agents
    dd = env.env.get_data_dictionary()
    assert (np.asarray(dd["agent_types"]["data"]) == fx["init__agent_types"]).all()
    for key in ("loc_x", "loc_y", "direction"):
        assert np.allclose(dd[key]["data"], fx[f"init__{key}"], atol=1e-6)
    assert np.allclose(dd["acceleration_actions"]["data"], fx["init__acceleration_actions"])
    assert np.allclose(dd["turn_actions"]["data"], fx["init__turn_actions"])
    assert close(np.stack([obs[a] for a in range(N)]), fx["obs0"], 2e-5).all()
    last = int(fx["episode_length"])
    for t in range(fx["actions"].shape[0]):
        o, r, d, _ = env.step({a: fx["actions"][t][a] for a in range(N)})
        assert (env.env.still_in_the_game == fx["still_in_the_game"][t]).all(), t
        ok = close(np.stack([o[a] for a in range(N)]), fx["obs"][t], 2e-5)
        assert ok.all(), (t, np.argwhere(~ok)[:4])
        if t + 1 != last:
            assert close(np.array([r[a] for a in range(N)]), fx["rewards"][t], 2e-5).all(), t
        assert bool(d["__all__"]) == bool(fx["done"][t])


def test_cpu_cartpole_env_runs():
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.single_agent.cartpole import ClassicControlCartPoleEnv

    env = EnvWrapper(ClassicControlCartPoleEnv(episode_length=50, seed=3), env_backend="cpu")
    o = env.reset()
    assert o[0].shape == (4,) and np.abs(o[0]).max() <= 0.05
    steps = 0
    while True:
        o, r, d, _ = env.step({0: steps % 2})
        steps += 1
        assert r[0] == 1.0
        if d["__all__"]:
            break
    assert 5 < steps <= 50


@pytest.mark.parametrize("module,cls,obs_dim,continuous", [
    ("mountain_car", "ClassicControlMountainCarEnv", 2, False),
    ("continuous_mountain_car", "ClassicControlContinuousMountainCarEnv", 2, True),
    ("acrobot", "ClassicControlAcrobotEnv", 6, False),
    ("pendulum", "ClassicControlPendulumEnv", 3, True)])
def test_cpu_classic_control_envs_run(module, cls, obs_dim, continuous):
    """Same module paths, class names, `name` attributes and step()/reset() contract as
    example_envs/single_agent/classic_control/* of the reference; the device twin declares
    the reference's data dictionary (state [+ constants] [+ reset pool])."""
    import importlib

    from warp_drive_b200.env_wrapper import EnvWrapper

    mod = importlib.import_module(f"warp_drive_b200.envs.single_agent.{module}")
    env_cls = getattr(mod, cls)
    assert env_cls.name == cls
    env = EnvWrapper(env_cls(episode_length=30, seed=5), env_backend="cpu")
    o = env.reset()
    assert o[0].shape == (obs_dim,) and o[0].dtype == np.float32
    again = env.reset()
    assert np.array_equal(o[0], again[0])          # fixed seed -> fixed initial state
    rs = np.random.RandomState(0)
    for steps in range(1, 31):
        a = rs.uniform(-2, 2, (1,)).astype(np.float32) if continuous else int(rs.randint(0, 3))
        o, r, d, _ = env.step({0: a})
        assert o[0].shape == (obs_dim,) and np.isfinite(o[0]).all() and np.isfinite(r[0])
        if d["__all__"]:
            break
    assert d["__all__"] and steps <= 30

    dev = getattr(mod, "CUDA" + cls)(episode_length=30, env_backend="b200", reset_pool_size=4,
                                     seed=5)
    data = dev.get_data_dictionary()
    assert "state" in data and not data["state"]["attributes"]["save_copy_and_apply_at_reset"]
    pool = dev.get_reset_pool_dictionary()
    assert pool["state_reset_pool"]["data"].shape[0] == 4
    assert pool["state_reset_pool"]["attributes"]["reset_target"] == "state"
    fixed = getattr(mod, "CUDA" + cls)(episode_length=30, env_backend="b200", seed=5)
    assert fixed.get_data_dictionary()["state"]["attributes"]["save_copy_and_apply_at_reset"]
    assert len(fixed.get_reset_pool_dictionary()) == 0


def test_spaces_and_registrar():
    from warp_drive_b200.utils import spaces
    from warp_drive_b200.utils.env_registrar import EnvironmentRegistrar
    from warp_drive_b200.envs.tag_gridworld import CUDATagGridWorld, TagGridWorld

    sp = spaces.obs_dict_to_spaces({0: np.zeros(3, np.float32), 1: {"a": [1, 2]}})
    assert sp[0].shape == (3,) and sp[1]["a"].shape == (2,)
    reg = EnvironmentRegistrar()
    reg.add(env_backend="cpu")(TagGridWorld)
    reg.add(env_backend="pycuda")(CUDATagGridWorld)
    assert reg.get("TagGridWorld", "cpu") is TagGridWorld
    assert reg.get("taggridworld", "numba") is CUDATagGridWorld
    assert reg.has_env("TagGridWorld", "pycuda") and not reg.has_env("Nope")


# ------------------------------------------------------------------ update-path math
def test_a2c_ppo_losses_follow_the_reference_formulas():
    """compute_loss_and_metrics on host tensors vs a literal transcription of the
    reference's formulas (a2c.py:80-130, ppo.py:127-136) for one small batch."""
    import torch
    from torch.distributions import Categorical

    from warp_drive_b200.training.algorithms.policygradient import A2C, PPO, discounted_returns

    g = torch.Generator().manual_seed(1)
    T, E, Np, A = 6, 3, 4, 5
    rewards = torch.randn(T, E, Np, generator=g)
    done = (torch.rand(T, E, generator=g) < 0.25).int()
    done[2, 1] = 1
    values = torch.randn(T, E, Np, generator=g, requires_grad=True)
    logits = [torch.randn(T, E, Np, A, generator=g, requires_grad=True) for _ in range(2)]
    probs = [torch.softmax(l, -1) for l in logits]
    actions = torch.randint(0, A, (T, E, Np, 2), generator=g)
    gamma = 0.9
    # literal reference recursion
    ret = torch.zeros_like(rewards)
    d = done.float()
    ret[-1] = d[-1][:, None] * rewards[-1] + (1 - d[-1][:, None]) * values.detach()[-1]
    for step in range(-2, -T - 1, -1):
        ret[step] = rewards[step] + (1 - d[step][:, None]) * gamma * ret[step + 1]
    assert torch.allclose(discounted_returns(rewards, done, values.detach(), gamma), ret)
    adv = ret - values.detach()
    logp = sum(Categorical(p).log_prob(actions[..., k]) for k, p in enumerate(probs))
    ent = sum(Categorical(p).entropy().mean() for p in probs)
    vf = torch.nn.MSELoss()(ret, values)
    want_a2c = (-logp * adv).mean() + 0.5 * vf - 0.05 * ent
    algo = A2C(discount_factor_gamma=gamma, vf_loss_coeff=0.5, entropy_coeff=0.05)
    loss, metrics = algo.compute_loss_and_metrics(10, actions, rewards, done, probs, values,
                                                  perform_logging=True)
    assert torch.allclose(loss, want_a2c, atol=1e-6)
    assert abs(metrics["Value function loss"] - vf.item()) < 1e-6
    loss.backward()
    assert values.grad is not None and logits[0].grad.abs().sum() > 0
    ratio = torch.exp(logp - logp.detach())
    surr = torch.minimum(ratio * adv, torch.clamp(ratio, 0.9, 1.1) * adv)
    want_ppo = -surr.mean() + 0.5 * vf - 0.05 * ent
    ppo = PPO(clip_param=0.1, discount_factor_gamma=gamma, vf_loss_coeff=0.5, entropy_coeff=0.05)
    loss2, _ = ppo.compute_loss_and_metrics(10, actions, rewards, done, probs, values)
    assert torch.allclose(loss2, want_ppo, atol=1e-6)
    # normalisation switches
    n = A2C(discount_factor_gamma=gamma, normalize_advantage=True, normalize_return=True)
    l3, _ = n.compute_loss_and_metrics(0, actions, rewards, done, probs, values)
    assert torch.isfinite(l3)


def test_param_scheduler_and_config_merge():
    from warp_drive_b200.training.trainer import load_run_config, recursive_merge_config_dicts
    from warp_drive_b200.training.utils.param_scheduler import ParamScheduler

    assert ParamScheduler(0.3).get_param_value(123) == 0.3
    s = ParamScheduler([[1000, 0.1], [2000, 0.05]])
    assert s.get_param_value(0) == 0.1 and s.get_param_value(5000) == 0.05
    assert abs(s.get_param_value(1500) - 0.075) < 1e-12
    cfg = load_run_config("tag_continuous")
    assert cfg["env"]["num_runners"] == 100 and cfg["policy"]["runner"]["lr"] == 0.005
    default = load_run_config("default_configs")
    merged = recursive_merge_config_dicts({"num_envs": 7}, default["trainer"])
    assert merged["num_envs"] == 7 and merged["train_batch_size"] == 10000
    for name in ("tag_gridworld", "single_cartpole"):
        assert load_run_config(name)["name"] == name


def test_all_nine_reference_run_configs_are_present():
    """Every run config of warp_drive/training/run_configs/ has a twin here with the same
    schema and the same values (saving.basedir, a path on the reference authors' machine,
    excepted), compared through the fingerprints in tests/golden/reference_run_configs.json."""
    import hashlib
    import json

    from warp_drive_b200.training.trainer import load_run_config

    with open(os.path.join(ROOT, "tests", "golden", "reference_run_configs.json")) as fp:
        theirs = json.load(fp)["sha256"]
    names = ["default_configs", "single_acrobot", "single_cartpole",
             "single_continuous_mountain_car", "single_mountain_car", "single_pendulum",
             "tag_continuous", "tag_gridworld", "tag_gridworld_with_reset_pool"]
    assert set(theirs) == set(names) - {"default_configs"}
    for name in names:
        ours = load_run_config(name)
        if name == "default_configs":
            continue
        assert {"name", "env", "trainer", "policy", "saving"} <= set(ours)
        for pol in ours["policy"].values():
            assert pol["algorithm"] in ("A2C", "PPO", "DDPG")
        ours["saving"].pop("basedir", None)
        text = json.dumps(ours, sort_keys=True).encode()
        assert hashlib.sha256(text).hexdigest() == theirs[name], name
    ddpg = load_run_config("single_pendulum")
    assert ddpg["trainer"]["n_step"] == 5 and ddpg["policy"]["shared"]["tau"] == 0.05
    assert ddpg["policy"]["shared"]["model"]["actor"]["output_w"] == 2.0
    assert load_run_config("single_mountain_car")["trainer"]["neg_pos_env_ratio"] == 10


def test_forward_sm_split_cost_model():
    """RolloutEngine._forward_side_by_side splits the SMs between two policies so that the
    slower launch is as short as possible (cost in tile-times: tiles per CTA, 1.3x for the
    small policy, +1.5 for the weight load).  Config 2: 1563 runner tiles vs 79 tagger tiles
    on 148 SMs -> the taggers get 9 SMs."""
    n_sm, tiles = 148, {"runner": 1563, "tagger": 79}
    best = None
    for k in range(1, n_sm // 2 + 1):
        cost = max(-(-tiles["runner"] // (n_sm - k)), 1.3 * -(-tiles["tagger"] // k)) + 1.5
        if best is None or cost < best[0]:
            best = (cost, k)
    assert best[1] == 9
    # and the engine source uses exactly this rule
    import inspect

    from warp_drive_b200.training import rollout

    src = inspect.getsource(rollout.RolloutEngine._forward_side_by_side)
    assert "1.3 * -(-tiles[order[1]] // k)" in src and "+ 1.5" in src
