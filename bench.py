#!/usr/bin/env python
"""bench.py -- rollout throughput of the B200-native engine on BASELINE.json config 2
(tag_continuous, 2000 envs x (5 taggers + 100 runners), discrete actions, K = 10 partial
observations), one process per GPU.

    python bench.py --gpus 1 --steps 200 --warmup 50
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference's NumPy CPU step (oracle port)
    python bench.py ... --dump-outputs DIR   # also save the last timed step's outputs (.npy)

One "step" = one rollout timestep of every env replica on this rank:
policy forward (2 policies) -> sample 2 action heads -> env.step -> bookkeeping ->
done-masked reset -> push to the training batch.  Rank 0 prints ONE JSON line.

  value     agent-steps/s (envs x agents x steps / s) of the whole device-resident
            rollout, all ranks, CUDA-event timed, max over ranks
  e2e       the same metric through the public EnvWrapper API with HOST buffers: every
            step copies the actions host->device from pinned memory and the step's
            observations/rewards/done device->host
  roofline  the dominant kernel (the fused sample+step+reset kernel) timed alone with
            CUDA events and an L2 flush between launches, against MEASURED_PEAKS.json
  cpu_baseline  oracle/numpy_ref.py (NumPy restatement of the reference CPU step) on the
            host cores, bounded sample
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json config 2 == warp_drive/training/run_configs/tag_continuous.yaml:10-34 of
# the reference with num_taggers = 5 (SURVEY.md section 8d)
ENV_CONFIG = dict(
    num_taggers=5, num_runners=100, grid_length=20.0, episode_length=500,
    max_acceleration=0.1, min_acceleration=-0.1, max_turn=2.356, min_turn=-2.356,
    num_acceleration_levels=20, num_turn_levels=20, skill_level_runner=1.0,
    skill_level_tagger=1.0, max_speed=1.0, seed=274880, use_full_observation=False,
    runner_exits_game_after_tagged=True, num_other_agents_observed=10,
    tag_reward_for_tagger=10.0, tag_penalty_for_runner=-10.0, step_penalty_for_tagger=0.0,
    step_reward_for_runner=0.0, edge_hit_penalty=0.0, end_of_game_reward_for_runner=1.0,
    tagging_distance=0.02)
MODEL_CONFIG = {"type": "fully_connected", "fc_dims": [256, 256], "model_ckpt_filepath": ""}
# BASELINE.json configs[3]: 2000 envs x 1024 agents, multi-block-per-env.  BASELINE.json does
# not fix the tagger / runner split or the arena: 24 taggers + 1000 runners on a 64 x 64 grid
# (config 2's agent density, SURVEY.md section 8d "Config 4"); everything else as config 2.
ENV_CONFIG_4 = dict(ENV_CONFIG, num_taggers=24, num_runners=1000, grid_length=64.0)
BENCH_CONFIGS = {
    2: {"env": ENV_CONFIG, "blocks_per_env": 1, "graph_cap": 50,
        "label": "BASELINE.json configs[1]"},
    4: {"env": ENV_CONFIG_4, "blocks_per_env": 2, "graph_cap": 4,
        "label": "BASELINE.json configs[3]"},
}
_ACTIVE = {"config": 2, "blocks_per_env": None}


def active_env_config():
    return BENCH_CONFIGS[_ACTIVE["config"]]["env"]


def active_blocks_per_env():
    return _ACTIVE["blocks_per_env"] or BENCH_CONFIGS[_ACTIVE["config"]]["blocks_per_env"]

# algorithmic bytes per agent-step (SURVEY.md section 8d / BASELINE.md section 3)
BYTES_FUSED = 516      # sample (2 x 21 probs) + step: reads 192, writes 324
BYTES_STEP_ONLY = 348  # step with actions in


def workload_config(n_envs, n_agents=None):
    """The `config` object of the JSON line -- identical for the b200 arm and the
    --impl reference arm (both measure the same BASELINE.json config)."""
    ec = active_env_config()
    n_agents = n_agents or ec["num_taggers"] + ec["num_runners"]
    out = {"workload": f"tag_continuous {n_envs} envs/GPU x ({ec['num_taggers']} taggers + "
                       f"{ec['num_runners']} runners), discrete 21x21 actions, K=10 partial obs, "
                       f"grid {ec['grid_length']:g} ({BENCH_CONFIGS[_ACTIVE['config']]['label']})",
           "envs_per_gpu": n_envs, "agents": n_agents}
    if _ACTIVE["config"] == 4:
        out["blocks_per_env"] = active_blocks_per_env()
    return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fp:
            return json.load(fp), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                     "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names)
                   if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(sm),
                "reasons": reasons}


def build_engine(n_envs, seed, graph_steps, use_graph=True, forward_dtype=None,
                 fused_forward=True, obs_tiles=False, pair_forward=False):
    import torch

    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_continuous import TagContinuous
    from warp_drive_b200.managers.function_manager import CUDASampler
    from warp_drive_b200.training.models.fully_connected import FullyConnected
    from warp_drive_b200.training.rollout import RolloutEngine
    from warp_drive_b200.training.utils.data_loader import create_and_push_data_placeholders

    env = TagContinuous(**active_env_config())
    wrapper = EnvWrapper(env, num_envs=n_envs, env_backend="b200",
                         blocks_per_env=active_blocks_per_env())
    wrapper.reset_all_envs()
    policy_map = {"runner": sorted(env.runners), "tagger": sorted(env.taggers)}
    sampler = CUDASampler(wrapper.cuda_function_manager)
    create_and_push_data_placeholders(
        env_wrapper=wrapper, action_sampler=sampler, policy_tag_to_agent_id_map=policy_map,
        training_batch_size_per_env=graph_steps)
    sampler.init_random(seed)
    torch.manual_seed(seed)
    models = {p: FullyConnected(wrapper, MODEL_CONFIG, p, policy_map).cuda().eval()
              for p in policy_map}
    wrapper.reset_all_envs()
    # the fused kernel hands observations straight to the per-policy forward buffers; the
    # [E, N, F] `observations` array is only materialised on demand
    stats = torch.zeros(64, dtype=torch.int32, device="cuda")
    engine = RolloutEngine(wrapper, models, policy_map, sampler, graph_steps,
                           use_cuda_graph=use_graph, forward_dtype=forward_dtype,
                           write_observations=False, stats=stats,
                           use_fused_forward=fused_forward, use_obs_tiles=obs_tiles,
                           use_pair_forward=pair_forward)
    engine.stats = stats
    return wrapper, engine, sampler, policy_map


def last_step_outputs(engine):
    """Host copies of what engine.rollout() hands its caller for the rollout's last timestep:
    per policy the actions sampled and the rewards received in that step and the
    observations it produced (the next step's policy input), and the done flags."""
    T = engine.T
    out = {"done_flags": engine._tensor("done_flags_batch")[T - 1]}
    for p in engine.policies:
        out[f"observations_{p}"] = engine.cur_obs[p]
        out[f"actions_{p}"] = engine._tensor(f"sampled_actions_batch_{p}")[T - 1]
        out[f"rewards_{p}"] = engine._tensor(f"rewards_batch_{p}")[T - 1]
    return {k: v.float().cpu().numpy() for k, v in out.items()}


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def write_outputs(outputs, out_dir):
    """One float32 .npy per array, DUMP_LIMIT_BYTES in all at most: beyond that, every
    array keeps the same fixed, seeded sample of env replicas (axis 0)."""
    n_envs = next(iter(outputs.values())).shape[0]
    keep = np.arange(n_envs)
    budget = DUMP_LIMIT_BYTES - 4096 * len(outputs)          # .npy headers
    total = sum(a.nbytes for a in outputs.values())
    if total > budget:
        n = max(1, n_envs * budget // total)
        keep = np.sort(np.random.RandomState(0).choice(n_envs, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a[keep], np.float32))


def issue_roofline(kernel, kernel_ms, E, N):
    """The fused step is instruction-issue-bound, not HBM-bound (DESIGN.md section 5): report
    the issue rate next to the HBM fraction.  warp-instructions per launch come from the
    committed ncu capture of the same configuration (profiles/ncu_traffic.json,
    smsp__inst_executed.sum); the time is this run's."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            tr = json.load(fh).get(kernel)
        if not tr or tr["envs"] != E or tr["agents"] != N or "warp_instructions" not in tr:
            return None
        peaks, _ = measured_peaks()
        sm_hz = float(peaks.get("sm_max_mhz", 1965.0)) * 1e6
        n_sm = 148
        ipc = tr["warp_instructions"] / (kernel_ms * 1e-3 * sm_hz * n_sm)
        return {"warp_instructions_per_launch": tr["warp_instructions"],
                "source": tr.get("source", "profiles/ncu_traffic.json"),
                "achieved_ipc_per_sm": ipc, "peak_ipc_per_sm": 4.0, "frac": ipc / 4.0,
                "floor_us_at_peak_issue": tr["warp_instructions"] / (4.0 * sm_hz * n_sm) * 1e6,
                "note": "IPC = ncu warp-instructions per launch / (this run's kernel time x "
                        "max SM clock x 148 SMs)"}
    except (OSError, ValueError, KeyError):
        return None


def flush_l2(buf):
    buf.add_(1)   # read+write 512 MiB > 126 MB L2


def time_dominant_kernel(wrapper, engine, iters=30):
    """CUDA-event time of the dominant kernel alone (the fused sample+step+reset+push
    launch), L2 flushed before every launch."""
    import torch

    flush = torch.zeros(128 * 1024 * 1024, dtype=torch.float32, device="cuda")
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(iters)]
    if engine.fused is None:
        probs = engine.evaluate_policies(-1)
        for i in range(iters + 3):
            engine.sample_actions(probs, -1)
            flush_l2(flush)
            if i >= 3:
                ev[i - 3][0].record()
            wrapper.step_all_envs()
            if i >= 3:
                ev[i - 3][1].record()
            wrapper.reset_only_done_envs()
        name, nbytes = "tag_continuous_kernel<false> (step only)", BYTES_STEP_ONLY
    else:
        dm = wrapper.cuda_data_manager
        with torch.no_grad():
            probs = {p: engine._forward(engine.models[p], engine.cur_obs[p])
                     for p in engine.policies}
        slots = {k: {p: dm.data_on_device_via_torch(f"{k}_batch_{p}")[0]
                     for p in engine.policies}
                 for k in ("sampled_actions", "rewards", "processed_observations")}
        done_b = dm.data_on_device_via_torch("done_flags_batch")[0]
        for i in range(iters + 3):
            flush_l2(flush)
            if i >= 3:
                ev[i - 3][0].record()
            engine.fused.launch(probs, actions_batch=slots["sampled_actions"],
                                rewards_batch=slots["rewards"],
                                obs_next=slots["processed_observations"], done_batch=done_b,
                                obs_next_tiles=engine.obs_tiles or None)
            if i >= 3:
                ev[i - 3][1].record()
        wide = active_blocks_per_env() > 1 or engine.env_wrapper.n_agents > 320
        name = ("tag_continuous_kernel<true> (fused sample+step+push+reset)"
                if not wide else
                f"tc_wide_kernel<true> (fused sample+step+push+reset, cluster of "
                f"{active_blocks_per_env()} CTA(s) per env)")
        nbytes = BYTES_FUSED
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return {"kernel": name, "ms_median": ms[len(ms) // 2], "ms_min": ms[0],
            "bytes_per_agent_step": nbytes}


def time_dominant_kernel_in_rollout(engine, n_steps=60):
    """CUDA-event time of the fused env launch INSIDE eager rollout timesteps (forwards +
    fused step, same stream): the cache state the kernel sees in the real loop (its
    probability inputs were just written by the forwards; the per-step working set of
    ~110 MB plus the moving batch slot exceeds what stays L2-resident, so no flush)."""
    import torch

    fused = engine.fused
    orig = fused.launch
    evs = []

    def timed(*a, **k):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        orig(*a, **k)
        e.record()
        evs.append((s, e))

    fused.launch = timed
    try:
        T = engine.T
        for i in range(n_steps + 5):
            engine.step(i % T)
    finally:
        fused.launch = orig
    torch.cuda.synchronize()
    ms = sorted(s.elapsed_time(e) for s, e in evs[5:])
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_mean": sum(ms) / len(ms)}


def time_e2e_host_buffers(wrapper, n_steps, warmup=3, n_copy_streams=4):
    """Public-API env.step() with host buffers (EnvWrapper.step_with_host_buffers): H2D
    actions, step, D2H obs/rewards/done, every step, the host waits for each result."""
    import torch

    dm = wrapper.cuda_data_manager
    actions_d = dm.data_on_device_via_torch("sampled_actions")
    names = ("observations", "rewards", "_done_")
    rs = np.random.RandomState(0)
    host_actions = [torch.from_numpy(rs.randint(0, 21, tuple(actions_d.shape)).astype(np.int32)
                                     ).pin_memory() for _ in range(4)]
    host_out = {}
    for k in names:
        dev = dm.data_on_device_via_torch(k)
        host_out[k] = torch.empty(dev.shape, dtype=dev.dtype).pin_memory()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(warmup + n_steps):
        if i == warmup:
            torch.cuda.synchronize()
            start.record()
        wrapper.step_with_host_buffers(host_actions[i % 4], host_out, n_copy_streams)
        wrapper.reset_only_done_envs()
    end.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(end) / n_steps
    h2d = actions_d.numel() * 4
    d2h = sum(t.numel() * t.element_size() for t in host_out.values())
    return ms, h2d, d2h


def cpu_baseline(sample_steps, n_procs=None, warmup=2):
    """oracle/numpy_ref.py on the host cores (bounded sample of config 2)."""
    from oracle.numpy_ref import timed_agent_steps_per_sec
    from warp_drive_b200.envs.tag_continuous import TagContinuous

    env = TagContinuous(**active_env_config())
    env.reset()
    dd = env.get_data_dictionary()
    cfg = {k: dd[k]["data"] for k in (
        "agent_types", "acceleration_actions", "turn_actions", "skill_levels", "step_rewards",
        "grid_length", "edge_hit_penalty", "max_speed", "distance_margin_for_reward",
        "tag_reward_for_tagger", "tag_penalty_for_runner", "end_of_game_reward_for_runner",
        "num_other_agents_observed", "use_full_observation", "runner_exits_game_after_tagged")}
    cfg["episode_length"] = env.episode_length
    init = {k: np.array(dd[k]["data"]) for k in
            ("loc_x", "loc_y", "speed", "direction", "acceleration")}
    return timed_agent_steps_per_sec(cfg, init, sample_steps, warmup=warmup, n_procs=n_procs)


def c_oracle_rate(n_envs=64, n_steps=10):
    """The C restatement of the CUDA kernel (OpenMP, all cores): extra context only."""
    import oracle
    from warp_drive_b200.envs.tag_continuous import TagContinuous

    env = TagContinuous(**active_env_config())
    env.reset()
    dd = env.get_data_dictionary()
    N, K = env.num_agents, env.num_other_agents_observed
    rep = lambda a, dt: np.ascontiguousarray(np.broadcast_to(np.asarray(a, dt), (n_envs, N))).copy()  # noqa: E731
    st = {k: rep(dd[k]["data"], np.float32) for k in
          ("loc_x", "loc_y", "speed", "direction", "acceleration", "edge_hit_reward_penalty")}
    st["still_in_the_game"] = rep(dd["still_in_the_game"]["data"], np.int32)
    st["num_runners"] = np.full(n_envs, env.num_runners, np.int32)
    st["nearest_neighbor_ids"] = np.zeros((n_envs, N, K), np.int32)
    st["_done_"] = np.zeros(n_envs, np.int32)
    st["_timestep_"] = np.zeros(n_envs, np.int32)
    cfg = {"agent_types": np.asarray(dd["agent_types"]["data"], np.int32)}
    for k in ("acceleration_actions", "turn_actions", "skill_levels", "step_rewards"):
        cfg[k] = np.asarray(dd[k]["data"], np.float32)
    for k in ("grid_length", "edge_hit_penalty", "max_speed", "distance_margin_for_reward",
              "tag_reward_for_tagger", "tag_penalty_for_runner",
              "end_of_game_reward_for_runner", "num_other_agents_observed",
              "use_full_observation", "runner_exits_game_after_tagged"):
        cfg[k] = dd[k]["data"]
    cfg["episode_length"] = env.episode_length
    rs = np.random.RandomState(0)
    acts = rs.randint(0, 21, (n_steps + 1, n_envs, N, 2)).astype(np.int32)
    obs = np.zeros((n_envs, N, 7 * K + 1), np.float32)
    rew = np.zeros((n_envs, N), np.float32)
    oracle.tag_continuous_step(st, cfg, acts[0], obs, rew)
    t0 = time.perf_counter()
    for t in range(n_steps):
        oracle.tag_continuous_step(st, cfg, acts[t + 1], obs, rew)
    dt = time.perf_counter() - t0
    return n_envs * N * n_steps / dt, oracle.lib().wd_oracle_num_threads()


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path = its NumPy
    step(), restated in oracle/numpy_ref.py, on all host cores.  Each 'step' is one env
    step of one replica per core (a bounded sample of the workload)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # config 4: one NumPy step of a 1024-agent env takes ~1 s, so the sample is shorter
    steps = max(1, min(args.steps, 400 if args.config == 2 else 8))
    warmup = max(3, min(args.warmup, 50)) if args.config == 2 else 3
    res = cpu_baseline(steps, n_procs=cores, warmup=warmup)
    value = res["agent_steps_per_sec"]
    line = {
        "impl": "reference", "metric": "agent_steps_per_sec", "value": value,
        "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": 1000.0 * cores * res["n_agents"] / value, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.envs),
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores,
                         "kind": "port",
                         "sample": f"bounded sample of the workload: {steps} env-steps x {cores} "
                                   f"env replicas (one per host core, all cores busy) x "
                                   f"{res['n_agents']} agents after {warmup} warm-up steps, "
                                   "oracle/numpy_ref.py = the reference's NumPy step() restated"},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- config 3
# BASELINE.json configs[2]: "Cartpole-v1 single_agent 10000 envs, PPO, 1xB200 (small-agent
# sampler-bound path)".  Env and policy from run_configs/single_cartpole.yaml (episode 500,
# fully_connected [32, 32]); SURVEY.md section 8d: reset_pool_size 1000.
CARTPOLE_CONSTS = [9.8, 0.1, 1.1, 0.5, 0.05, 10.0, 0.02, 12 * 2 * math.pi / 360, 2.4]
BYTES_CARTPOLE = 76     # state 16 R + 16 W, obs 16 W, reward 4, action 4, probs 8, done/timestep 12


def cartpole_c_oracle_rate(n_envs, n_steps, warmup=3):
    """CPU arm of config 3: the C restatement of the reference's CartPole step (oracle/
    wd_oracle.c, following cartpole_step_numba.py:6-83; the reference's own CPU physics live in
    the third-party gym package, which is not installed -> "port") on all host cores."""
    import oracle

    L = oracle.lib()
    rs = np.random.RandomState(0)
    st = rs.uniform(-0.05, 0.05, (n_envs, 1, 4)).astype(np.float32)
    done = np.zeros(n_envs, np.int32)
    rew = np.zeros((n_envs, 1), np.float32)
    obs = np.zeros((n_envs, 1, 4), np.float32)
    ts = np.zeros(n_envs, np.int32)
    acts = rs.randint(0, 2, (n_steps + warmup, n_envs, 1, 1)).astype(np.int32)
    t0 = 0.0
    for t in range(n_steps + warmup):
        if t == warmup:
            t0 = time.perf_counter()
        L.wd_oracle_cartpole_step(n_envs, st, acts[t], done, rew, obs, *CARTPOLE_CONSTS, ts, 500)
        d = done > 0
        if d.any():
            st[d] = rs.uniform(-0.05, 0.05, (int(d.sum()), 1, 4)).astype(np.float32)
            ts[d] = 0
            done[d] = 0
    dt = time.perf_counter() - t0
    return n_envs * n_steps / dt, L.wd_oracle_num_threads()


def config3_line_config(n_envs):
    return {"workload": f"CartPole-v1 single agent, {n_envs} envs/GPU, discrete(2), "
                        "fully_connected [32,32] policy, reset pool 1000 "
                        "(BASELINE.json configs[2])",
            "envs_per_gpu": n_envs, "agents": 1}


def run_reference_arm_config3(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    steps = max(1, min(args.steps, 2000))
    warmup = max(3, min(args.warmup, 50))
    rate, threads = cartpole_c_oracle_rate(args.envs3, steps, warmup)
    line = {
        "impl": "reference", "metric": "agent_steps_per_sec", "value": rate,
        "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": 1000.0 * args.envs3 / rate, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config3_line_config(args.envs3),
        "cpu_baseline": {"value": rate, "unit": "agent-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} env-steps x {args.envs3} envs, C restatement of the "
                                   "reference CartPole step (gym's CPU physics are third-party "
                                   "and absent), OpenMP over all cores, random actions"},
        "e2e": {"value": rate, "unit": "agent-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def run_config3(args):
    """One 'step' = one rollout timestep of every CartPole replica: forward -> sample -> step
    -> bookkeeping -> done-masked reset (from the pool) -> push to batch.  The whole T-step
    rollout is ONE launch (wdb_single_agent_rollout)."""
    import torch
    import torch.distributed as dist

    from warp_drive_b200 import lib as wlib
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.single_agent.cartpole import CUDAClassicControlCartPoleEnv
    from warp_drive_b200.managers.function_manager import CUDASampler
    from warp_drive_b200.training.models.fully_connected import FullyConnected
    from warp_drive_b200.training.rollout import RolloutEngine
    from warp_drive_b200.training.utils.data_loader import create_and_push_data_placeholders

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus
    E, K, W = args.envs3, args.steps, max(3, args.warmup)
    T = max(d for d in range(1, min(K, 100) + 1) if K % d == 0)
    env = CUDAClassicControlCartPoleEnv(episode_length=500, env_backend="b200",
                                        reset_pool_size=1000, seed=1234 + rank)
    w = EnvWrapper(env, num_envs=E, env_backend="b200")
    w.reset_all_envs()
    pm = {"shared": [0]}
    sampler = CUDASampler(w.cuda_function_manager)
    create_and_push_data_placeholders(env_wrapper=w, action_sampler=sampler,
                                      policy_tag_to_agent_id_map=pm,
                                      training_batch_size_per_env=T)
    sampler.init_random(1234 + rank)
    w.init_reset_pool(seed=99 + rank)
    torch.manual_seed(1234 + rank)
    mcfg = {"type": "fully_connected", "fc_dims": [32, 32], "model_ckpt_filepath": ""}
    models = {"shared": FullyConnected(w, mcfg, "shared", pm).cuda().eval()}
    eng = RolloutEngine(w, models, pm, sampler, T, use_cuda_graph=False)
    assert eng.sa is not None, "the whole-rollout kernel is not in use"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, math.ceil(W / T))):
        eng.rollout()
    reps = max(1, args.reps)
    rep_ms = []
    with ClockSampler(local_rank) as clocks:
        c0 = wlib.launch_count()
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a.record()
            for _ in range(K // T):
                eng.rollout()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b)], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            rep_ms.append(float(t.item()))
        launches = (wlib.launch_count() - c0) // reps
        t_hold = time.perf_counter()
        while time.perf_counter() - t_hold < 0.4:
            for _ in range(8):
                eng.rollout()
            torch.cuda.synchronize()
    elapsed_ms = sorted(rep_ms)[len(rep_ms) // 2]
    value = world * E * K / (elapsed_ms / 1000.0)

    # ---- e2e: public EnvWrapper API with host buffers, every step
    dm = w.cuda_data_manager
    actions_d = dm.data_on_device_via_torch("sampled_actions")
    rs = np.random.RandomState(0)
    host_actions = [torch.from_numpy(rs.randint(0, 2, tuple(actions_d.shape)).astype(np.int32)
                                     ).pin_memory() for _ in range(4)]
    host_out = {k: torch.empty(dm.data_on_device_via_torch(k).shape,
                               dtype=dm.data_on_device_via_torch(k).dtype).pin_memory()
                for k in ("observations", "rewards", "_done_")}
    n_e2e = min(K, 100)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(3 + n_e2e):
        if i == 3:
            torch.cuda.synchronize()
            a.record()
        w.step_with_host_buffers(host_actions[i % 4], host_out, 1)
        w.reset_only_done_envs()
    b.record()
    torch.cuda.synchronize()
    e2e_ms = a.elapsed_time(b) / n_e2e
    t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * E / (float(t.item()) / 1000.0)
    h2d = actions_d.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in host_out.values())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- the dominant (only) kernel alone: one T-step launch, L2 flushed before each
    peaks, peak_src = measured_peaks()
    flush = torch.zeros(128 * 1024 * 1024, dtype=torch.float32, device="cuda")
    ts = []
    for i in range(12):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); eng.rollout(); b.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(a.elapsed_time(b))
    kernel_ms = sorted(ts)[len(ts) // 2]
    per_step_us = kernel_ms * 1e3 / T
    achieved = BYTES_CARTPOLE * E * T / (kernel_ms * 1e-3) / 1e9
    flops = 2.0 * (4 * 32 + 32 * 32 + 32 * 2) * E * T
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
        "frac": achieved / peaks["hbm_gbs"], "traffic": None,
        "kernel": f"sa_rollout_kernel (ONE launch = {T} timesteps x {E} envs: fp32 forward + "
                  "sample + step + bookkeeping + pool reset + push)",
        "kernel_ms": kernel_ms, "kernel_us_per_timestep": per_step_us,
        "algorithmic_bytes_per_agent_step": BYTES_CARTPOLE,
        "peak_source": peak_src,
        "note": "10 000 single-agent envs move 0.76 MB per timestep: this path is bound by the "
                "dependent per-env chain (forward 1.2 K FMA -> softmax -> sample -> float64 "
                "physics), not by HBM; the figure of merit is launches and microseconds per "
                "timestep (the reference: ~50 launches and >= 5 host syncs per timestep)",
        "fp32_forward_gflops": flops / (kernel_ms * 1e-3) / 1e9,
    }
    line = {
        "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": elapsed_ms / K,
        "ms_per_step_reps": [m / K for m in rep_ms],
        "timing": f"median of {reps} repetitions of the K-step region (each: barrier + "
                  "synchronize, CUDA events, max over ranks)",
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config3_line_config(E),
        "config_detail": {"timesteps_per_launch": T, "cuda_graph": False,
                          "l2": "working set (state + batch slots of one rollout, "
                                f"{E * T * 28 / 1e6:.1f} MB) is L2-resident by nature; the "
                                "kernel is additionally timed with an explicit L2 flush"},
        "clocks": dict(clocks.summary(), window="timed region + 0.4 s of the same rollout"),
        "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                "path": "EnvWrapper.step_with_host_buffers + reset_only_done_envs, every step"},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if world == 1:
        # same-box GPU anchor: the reference's own numba step kernel (cubin built from the
        # reference sources by oracle/build_ref_numba.py), one launch = one env step only
        try:
            from oracle import ref_numba

            ref = ref_numba.RefNumbaKernel("cartpole")
            st = dm.data_on_device_via_torch("state").clone()
            act = torch.zeros((E, 1, 1), dtype=torch.int32, device="cuda")
            dn = torch.zeros(E, dtype=torch.int32, device="cuda")
            rw = torch.zeros((E, 1), device="cuda")
            ob = torch.zeros((E, 1, 4), device="cuda")
            tsr = torch.zeros(E, dtype=torch.int32, device="cuda")
            rt = []
            for i in range(22):
                st.copy_(dm.data_on_device_via_torch("state"))
                tsr.zero_()
                flush.add_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ref(E, st, act, dn, rw, ob, *CARTPOLE_CONSTS, tsr, 500)
                b.record()
                torch.cuda.synchronize()
                if i >= 2:
                    rt.append(a.elapsed_time(b) * 1e3)
            line["ref_gpu"] = {
                "kernel": "oracle/_ref/numba_cartpole.cubin = NumbaClassicControlCartPoleEnvStep "
                          "compiled by numba from the reference source, launched as the "
                          f"reference does (grid {E}, block 1)",
                "step_kernel_us": sorted(rt)[len(rt) // 2],
                "ours_us_per_timestep_whole_path": per_step_us,
                "note": "the reference kernel is the env step ALONE (no forward, sampler, "
                        "bookkeeping, reset or push); ours is the whole timestep"}
        except Exception as err:  # noqa: BLE001
            line["ref_gpu"] = {"unavailable": f"{type(err).__name__}: {err}"}
        if not args.skip_cpu_baseline:
            rate, threads = cartpole_c_oracle_rate(E, 300)
            line["cpu_baseline"] = {
                "value": rate, "unit": "agent-steps/s", "cores": threads, "kind": "port",
                "sample": f"300 env-steps x {E} envs, C restatement of the reference CartPole "
                          "step (oracle/wd_oracle.c), OpenMP over all cores"}
    else:
        line["cpu_baseline"] = {"value": None, "unit": "agent-steps/s", "cores": 0,
                                "kind": "port", "sample": "measured at N=1 only (rank 0)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------- --mode train
def train_iteration_stats(args, world, rank, local_rank, n_iters, reps, warm_iters=3):
    """Full training iterations on this rank's process group (already initialised): T-step
    rollout -> A2C/PPO update of both policies (fused loss kernel, cuBLAS forward/backward, flat
    Adam) -> ONE in-place NCCL all-reduce (mean) of the flat gradient arena.  Returns
    (elapsed_ms_per_rep list, phase medians, all-reduce us list, gradient elements, E, N, T)."""
    import copy

    import torch
    import torch.distributed as dist
    import yaml

    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_continuous import TagContinuous
    from warp_drive_b200.training.trainer import Trainer

    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    E, T = args.envs, args.train_steps
    with open(os.path.join(ROOT, "warp_drive_b200", "training", "run_configs",
                           "tag_continuous.yaml"), encoding="utf8") as fp:
        cfg = yaml.safe_load(fp)
    cfg["env"].update(ENV_CONFIG)
    cfg["trainer"].update(num_envs=E, train_batch_size=E * T, num_episodes=10 ** 6, seed=1234)
    for p in cfg["policy"].values():
        p["algorithm"] = args.algo
        if args.algo == "PPO":
            p["clip_param"] = 0.1
    cfg["saving"].update(metrics_log_freq=10 ** 9, model_params_save_freq=10 ** 9,
                         basedir="/tmp", name="bench_train", tag=f"rank{rank}")
    env = TagContinuous(**cfg["env"])
    wrapper = EnvWrapper(env, num_envs=E, env_backend="b200")
    pm = {"runner": sorted(env.runners), "tagger": sorted(env.taggers)}
    trainer = Trainer(wrapper, copy.deepcopy(cfg), pm, num_devices=world, device_id=rank,
                      verbose=False)
    wrapper.reset_all_envs()
    trainer.engine.resync_observations()
    N = wrapper.n_agents
    ar_events = []
    orig_ar = trainer._allreduce_gradients

    def timed_allreduce():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); orig_ar(); b.record()
        ar_events.append((a, b))

    trainer._allreduce_gradients = timed_allreduce

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def iteration(i, ev=None):
        if ev:
            ev[0].record()
        trainer._generate_rollout_batch()
        if ev:
            ev[1].record()
        trainer._update_model_params(i)
        if ev:
            ev[2].record()

    for i in range(warm_iters):
        iteration(i)
    torch.cuda.synchronize()
    ar_events.clear()
    rep_ms, phases = [], []
    for _ in range(reps):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_iters)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for i in range(n_iters):
            iteration(1000 + i, evs[i])
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rep_ms.append(float(t.item()))
        phases += [(e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])) for e in evs]
    ar_us = sorted(a.elapsed_time(b) * 1e3 for a, b in ar_events) if ar_events else []
    n_grad = sum(p.numel() for p in trainer._trained_params())
    roll = sorted(p[0] for p in phases)[len(phases) // 2]
    upd = sorted(p[1] for p in phases)[len(phases) // 2]
    del trainer, wrapper
    torch.cuda.empty_cache()
    return rep_ms, roll, upd, ar_us, n_grad, E, N, T


def train_summary(rep_ms, roll, upd, ar_us, n_grad, E, N, T, n_iters, world, algo):
    elapsed_ms = sorted(rep_ms)[len(rep_ms) // 2]
    it_ms = elapsed_ms / n_iters
    return {
        "algorithm": algo, "rollout_steps_per_iteration": T,
        "agent_steps_per_sec": world * E * N * T * n_iters / (elapsed_ms / 1000.0),
        "iteration_ms": it_ms, "rollout_ms": roll, "update_ms": upd,
        "allreduce_us_median": ar_us[len(ar_us) // 2] if ar_us else None,
        "allreduce_us_max": ar_us[-1] if ar_us else None,
        "allreduce_share_of_iteration": (ar_us[len(ar_us) // 2] / 1e3 / it_ms) if ar_us else 0.0,
        "gradient_elements": n_grad, "gradient_bytes": 4 * n_grad,
        "collective": "ONE in-place NCCL all-reduce (sum) of the flat gradient arena of all "
                      "policies + divide by world size, per iteration; no collective on the "
                      "rollout path (env replicas are independent)",
        "limiter": ("update: cuBLAS TF32 GEMMs with fused bias/ReLU/softmax/ReLU-backward "
                    f"kernels between them over the [{T}, {E}, Np, 71] batches (one autograd "
                    "node per policy) + fused loss kernel + flat Adam"
                    if upd > roll else "rollout"),
    }


def run_train_mode(args):
    """--mode train: one 'step' = one rollout timestep INSIDE full training iterations.  At
    --gpus 8 with 2000 envs per GPU this is BASELINE.json configs[4] (16000 envs sharded over
    8 x B200, PPO + NCCL gradient all-reduce)."""
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus
    T = args.train_steps
    n_iters = max(1, args.steps // T)
    K = n_iters * T
    reps = max(1, args.reps)
    with ClockSampler(local_rank) as clocks:
        stats = train_iteration_stats(args, world, rank, local_rank, n_iters, reps,
                                      warm_iters=max(3, math.ceil(args.warmup / T)))
    rep_ms, roll, upd, ar_us, n_grad, E, N, T = stats
    if rank == 0:
        tr = train_summary(*stats, n_iters, world, args.algo)
        elapsed_ms = sorted(rep_ms)[len(rep_ms) // 2]
        line = {
            "metric": "agent_steps_per_sec", "mode": "train", "value": tr["agent_steps_per_sec"],
            "unit": "agent-steps/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / K, "ms_per_step_reps": [m / K for m in rep_ms],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": dict(workload_config(E, N), mode="train",
                                                algorithm=args.algo, rollout_steps=T),
            "train": tr, "clocks": dict(clocks.summary(), window="timed region"),
            "gpu_launches": None,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=2000, help="env replicas per GPU")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json config: 2 = 2000 x 105 (the headline), 3 = CartPole x "
                         "10000 envs (whole rollout in one launch), 4 = 2000 x 1024 agents, one "
                         "env per thread-block cluster")
    ap.add_argument("--envs3", type=int, default=10000, help="config 3: env replicas per GPU")
    ap.add_argument("--mode", default="rollout", choices=["rollout", "train"],
                    help="train: full training iterations (rollout + A2C/PPO update + the flat "
                         "NCCL gradient all-reduce); config 2 env, 2000 envs per GPU = BASELINE "
                         "config 5 at --gpus 8")
    ap.add_argument("--train-steps", type=int, default=10,
                    help="--mode train: rollout timesteps per training iteration")
    ap.add_argument("--algo", default="PPO", choices=["A2C", "PPO"])
    ap.add_argument("--skip-train-probe", action="store_true",
                    help="config 2: do not append the short training-iteration measurement "
                         "(rollout + update + NCCL gradient all-reduce) to the line")
    ap.add_argument("--blocks-per-env", type=int, default=0,
                    help="config 4: CTAs per env (cluster size), default 2")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--forward-precision", default="tf32", choices=["fp32", "tf32", "bf16"],
                    help="precision of the torch policy forward when --torch-forward is given")
    ap.add_argument("--torch-forward", action="store_true",
                    help="run the policy forward through torch/cuBLAS instead of the fused "
                         "tcgen05 kernel (wdb_mlp_policy_forward)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--obs-tiles", action="store_true",
                    help="A/B switch: the env step also emits the bf16 MMA-ready copy of the "
                         "observations and the forward reads that (wdb_mlp_policy_forward_tiles)")
    ap.add_argument("--pair-forward", action="store_true",
                    help="A/B switch: both policies' forwards in ONE launch "
                         "(wdb_mlp_policy_forward_pair; add WDB_OPTIONS=pdl=1 for programmatic "
                         "dependent launches) instead of one launch per policy on two streams; "
                         "measured slower, see scripts/ab_forward_modes.py")
    ap.add_argument("--copy-streams", type=int, default=4,
                    help="streams the e2e observation D2H copy is split over")
    ap.add_argument("--reps", type=int, default=1,
                    help="repetitions of the K-step timed region (median reported)")
    ap.add_argument("--skip-ref-gpu", action="store_true",
                    help="do not time the reference's own CUDA kernels (oracle/_ref fatbin)")
    ap.add_argument("--cta-threads", type=int, default=0,
                    help="A/B switch: thread budget of one tag_continuous CTA (wdb_set_option)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the rollout's last timestep handed "
                         "to its caller to DIR/<name>.npy (float32; at most 64 MB, a fixed "
                         "seeded sample of env replicas beyond that)")
    args = ap.parse_args()
    if args.dump_outputs and (args.config == 3 or args.impl == "reference"
                              or args.mode == "train"):
        ap.error("--dump-outputs: only the b200 rollout of configs 2 and 4")
    if args.config == 3:
        return run_reference_arm_config3(args) if args.impl == "reference" else run_config3(args)
    _ACTIVE["config"] = args.config
    _ACTIVE["blocks_per_env"] = args.blocks_per_env or None
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.mode == "train":
        return run_train_mode(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    # host side of the e2e path: this rank's process (and the pinned buffers it first-touches)
    # on the NUMA node of its GPU
    from warp_drive_b200.utils.numa import bind_process_to_gpu

    bound_cores = bind_process_to_gpu(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    from warp_drive_b200 import lib as wlib

    if args.cta_threads:
        wlib.check(wlib.load().wdb_set_option(b"tc_cta_threads", args.cta_threads))
    K = args.steps
    W = max(3, args.warmup)
    # the rollout is captured as CUDA graphs of T timesteps; T divides K
    cap = BENCH_CONFIGS[args.config]["graph_cap"]       # batch slots held in HBM
    T = max(d for d in range(1, min(K, cap) + 1) if K % d == 0)
    if args.forward_precision == "tf32":
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
    wrapper, engine, sampler, policy_map = build_engine(
        args.envs, seed=1234 + rank, graph_steps=T, use_graph=not args.no_graph,
        forward_dtype=torch.bfloat16 if args.forward_precision == "bf16" else None,
        fused_forward=not args.torch_forward, obs_tiles=args.obs_tiles,
        pair_forward=args.pair_forward)
    E, N = wrapper.n_envs, wrapper.n_agents

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also captures the graph): the capture itself runs the rollout once; on top
    # of that AT LEAST 3 full replays, whatever --warmup says (a graph that has run once is
    # not warm: first-replay upload, cold TLB / L2, clock ramp)
    engine.rollout()
    torch.cuda.synchronize()
    launches_per_rollout = None
    for _ in range(max(3, math.ceil(W / T))):
        engine.rollout()
    # my kernels per T-step rollout (graph replays do not pass through the library, so
    # count one eager rollout)
    if not args.no_graph:
        c0 = wlib.launch_count()
        engine._rollout_eager()
        launches_per_rollout = wlib.launch_count() - c0
        engine.rollout()
    torch.cuda.synchronize()

    # ---- timed region: exactly K steps, CUDA events, barrier + synchronize on both sides.
    # A K-step region of a few milliseconds is at the mercy of one clock ramp or one slow
    # replay; --reps R repeats it R times back to back (each repetition is exactly K steps
    # with its own barrier / event pair / max over ranks) and reports the MEDIAN repetition;
    # all repetitions are listed in `ms_per_step_reps`.
    reps = max(1, args.reps)
    engine.stats.zero_()
    rep_ms = []
    with ClockSampler(local_rank) as clocks:
        c0 = wlib.launch_count()
        for _ in range(reps):
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            start.record()
            for _ in range(K // T):
                engine.rollout()
            end.record()
            barrier()
            t = torch.tensor([start.elapsed_time(end)], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            rep_ms.append(float(t.item()))
        stats_timed = engine.stats.cpu().numpy().tolist()
        c1 = wlib.launch_count()
        outputs = last_step_outputs(engine) if args.dump_outputs else None
        # the timed region lasts tens of milliseconds, one nvidia-smi poll at most: keep the
        # same rollout running (untimed) for ~0.4 s so that the clock samples are taken under
        # exactly this load
        t_hold = time.perf_counter()
        while time.perf_counter() - t_hold < 0.4:
            for _ in range(4):
                engine.rollout()
            torch.cuda.synchronize()
    elapsed_ms = sorted(rep_ms)[len(rep_ms) // 2]
    my_launches = ((c1 - c0) // reps) if args.no_graph else launches_per_rollout * (K // T)
    value = world * E * N * K / (elapsed_ms / 1000.0)

    # ---- e2e through the public API with host buffers (max over ranks)
    e2e_ms, h2d, d2h = time_e2e_host_buffers(wrapper, n_steps=min(K, 50),
                                             n_copy_streams=args.copy_streams)
    t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * E * N / (float(t.item()) / 1000.0)

    # ---- training-iteration probe (all ranks: it contains the one collective of the path,
    # the NCCL gradient all-reduce): a few full iterations, reported next to the rollout number
    train_probe = None
    if args.config == 2 and not args.skip_train_probe:
        try:
            stats = train_iteration_stats(args, world, rank, local_rank, n_iters=3, reps=3,
                                          warm_iters=2)
            train_probe = train_summary(*stats, 3, world, args.algo)
        except Exception as err:  # noqa: BLE001
            train_probe = {"error": f"{type(err).__name__}: {err}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (rank 0 only)
    peaks, peak_src = measured_peaks()
    dk = time_dominant_kernel(wrapper, engine)
    in_loop = time_dominant_kernel_in_rollout(engine) if engine.fused is not None else None
    # The roofline uses the stand-alone timing (L2 flushed, the launch is enqueued while the
    # flush kernel still runs, so no host launch latency can leak into the interval).  The
    # in-rollout timing is reported next to it: in eager mode the host sometimes falls behind
    # the GPU and the interval then includes the launch latency (median 90-107 us, min 82 us).
    kernel_ms = dk["ms_median"]
    achieved = dk["bytes_per_agent_step"] * E * N / (kernel_ms * 1e-3) / 1e9
    traffic = None      # DRAM bytes per launch from the committed ncu capture (same config only)
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles",
                               "ncu_traffic.json")) as fh:
            tr = json.load(fh).get(dk["kernel"])
        if tr and tr["envs"] == E and tr["agents"] == N:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                "traffic_note": "STATIC: ncu dram bytes per launch from the committed capture "
                                "of this configuration (profiles/ncu_traffic.json), not "
                                "measured in this run; "
                                "algorithmic bytes per launch = "
                                f"{dk['bytes_per_agent_step'] * E * N}",
                "kernel": dk["kernel"], "kernel_ms": kernel_ms,
                "kernel_ms_l2_flushed_standalone": dk["ms_median"],
                "kernel_ms_in_rollout": in_loop,
                "algorithmic_bytes_per_agent_step": dk["bytes_per_agent_step"],
                "peak_source": peak_src,
                "pair_evals": {"nominal_pairs_per_launch": E * N * (N - 1),
                               "nominal_pairs_per_s": E * N * (N - 1) / (kernel_ms * 1e-3),
                               "note": "the reference's O(N^2) neighbour sweep evaluates every "
                                       "ordered pair; config 4 is issue-bound on this sweep "
                                       "(SURVEY 8d), the cluster kernel scans only an x-window"},
                "issue": issue_roofline(dk["kernel"], kernel_ms, E, N),
                "l2": "kernel_ms = kernel_ms_l2_flushed_standalone: CUDA events around the "
                      "launch, L2 flushed before every launch; kernel_ms_in_rollout: events "
                      "around the launch inside eager rollout steps (may include host launch "
                      "latency)"}

    line = {
        "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": elapsed_ms / K,
        "ms_per_step_reps": [m / K for m in rep_ms],
        "timing": f"median of {reps} repetitions of the K-step region (each: barrier + "
                  "synchronize, CUDA events, max over ranks); >= 3 warm graph replays first",
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(E, N),
        "config_detail": {
            "rollout_step": "2 policies fully_connected [256,256]: forward + sample + step + "
                            "reset + push-to-batch",
            "policy_forward": ("wdb_mlp_policy_forward: fused tcgen05/TMEM MLP kernel, "
                               "bf16 operands, fp32 accumulate" if engine.fused_forward
                               else f"torch/cuBLAS {args.forward_precision} GEMMs (library)"),
            "graph_steps": T, "cuda_graph": not args.no_graph,
            "l2": "working set per step (~110 MB obs+probs+batch slots, batch slot "
                  "changes every step) exceeds what stays L2-resident; dominant "
                  "kernel additionally timed with an explicit L2 flush"},
        "clocks": dict(clocks.summary(), window="timed region + 0.4 s of the same rollout "
                                                  "replayed right after (untimed)"),
        "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                "host_cores_bound": (f"{len(bound_cores)} cores local to GPU {local_rank}"
                                     if bound_cores else "not bound"),
                "path": "EnvWrapper.step_with_host_buffers: pinned host actions in, "
                        "observations/rewards/done out to pinned host memory every step "
                        f"(obs copy split over {args.copy_streams} streams), host waits per step"},
        "gpu_launches": int(my_launches),
        "kernel_stats": {"exact_tie_path_agents": stats_timed[0], "tags": stats_timed[1],
                         "history_path_fallbacks": stats_timed[2],
                         "window_network_path_agents": stats_timed[3],
                         "agent_steps": E * N * K * reps,
                         "note": "device counters of the fused kernel over the timed region: "
                                 "agents that needed the exact tie-resolution path"},
        "roofline": roofline,
    }
    if train_probe is not None:
        line["train"] = train_probe
    # ---- same-box GPU anchor: the reference's own CUDA kernels on this GPU (N=1 only)
    if world == 1 and not args.skip_ref_gpu:
        try:
            from oracle.ref_gpu_bench import time_reference_tag_continuous

            if args.config == 2:
                ref_gpu = time_reference_tag_continuous(wrapper.env, E)
            else:
                # the reference's multi-block mode spins on global memory and dead-locks unless
                # every block of every env is co-resident (architecture_validate.py:53-99), and
                # needs 2 x [E, N, N-1] scratch (16.8 GB at E = 2000): time 64 envs x 2 blocks
                ref_gpu = time_reference_tag_continuous(wrapper.env, 64, bpe=2)
                if "step_kernel_us" in ref_gpu:
                    scale = E / 64.0
                    ref_gpu["scaled_to_envs"] = E
                    for k in ("step_kernel_us", "step_kernel_us_min", "sample_actions_kernel_us",
                              "reset_13_launches_us_none_done", "reset_13_launches_us_all_done",
                              "sequence_us_reset_only_when_done", "sequence_us_reset_every_step"):
                        ref_gpu[k + "_at_64_envs"] = ref_gpu[k]
                        ref_gpu[k] = ref_gpu[k] * scale
                    ref_gpu["scaling_note"] = (
                        "measured at 64 envs x 2 blocks (128 co-resident blocks), multiplied by "
                        f"{scale:g} to {E} envs: the reference kernel's time is linear in the "
                        "env count once the GPU is full (64 envs x 1024 threads fill 148 SMs "
                        "less than once, so this favours the reference)")
        except Exception as err:  # noqa: BLE001
            ref_gpu = {"unavailable": f"{type(err).__name__}: {err}"}
        if "step_kernel_us" in ref_gpu:
            ours_us = kernel_ms * 1e3
            ref_gpu["ours_fused_kernel_us"] = ours_us
            # like for like: OUR one launch does sample x2 + step + push + done-masked reset
            ref_gpu["speedup_env_path_kernels"] = (
                (ref_gpu["step_kernel_us"] + 2 * ref_gpu["sample_actions_kernel_us"]
                 + ref_gpu["reset_13_launches_us_none_done"]) / ours_us)
            ref_gpu["speedup_vs_reference_sequence"] = (
                ref_gpu["sequence_us_reset_only_when_done"] / ours_us)
            ref_gpu["note"] = ("speedup_env_path_kernels = (reference step + 2 x sample_actions "
                               "+ 13 masked reset launches, each timed alone with a flushed L2) "
                               "/ our ONE fused launch timed the same way; the reference side "
                               "has no policy forward, so compare with roofline.kernel_ms, not "
                               "with ms_per_step")
        line["ref_gpu"] = ref_gpu
    if any(stats_timed[8:32]):      # library built with -DWDB_PHASE_CLOCKS (profiling aid)
        line["phase_clocks_cta0"] = stats_timed[8:32]
        import ctypes
        raw = ctypes.CDLL(wlib.load()._name)
        if hasattr(raw, "wdb_debug_mlp_clocks"):
            buf = (ctypes.c_longlong * 96)()
            raw.wdb_debug_mlp_clocks(buf)
            line["mlp_clocks_cta0"] = list(buf)
    if world > 1:
        line["cpu_baseline"] = {"value": None, "unit": "agent-steps/s", "cores": 0, "kind": "port",
                                "sample": "measured at N=1 only (rank 0)"}
    elif not args.skip_cpu_baseline:
        cores = os.cpu_count() or 1
        n_sample = 150 if args.config == 2 else 6
        res = cpu_baseline(sample_steps=n_sample, n_procs=cores)
        line["cpu_baseline"] = {
            "value": res["agent_steps_per_sec"], "unit": "agent-steps/s", "cores": cores,
            "kind": "port",
            "sample": f"{n_sample} env-steps x {cores} processes x {N} agents of the same env "
                      "config (oracle/numpy_ref.py = reference NumPy step restated)"}
        try:
            rate, threads = c_oracle_rate()
            line["cpu_c_oracle"] = {"value": rate, "unit": "agent-steps/s", "threads": threads,
                                    "note": "C/OpenMP restatement of the CUDA kernel "
                                            "(oracle/wd_oracle.c), context only"}
        except Exception as err:  # noqa: BLE001
            line["cpu_c_oracle"] = {"error": str(err)}
    print(json.dumps(line))
    if outputs is not None:
        write_outputs(outputs, args.dump_outputs)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
