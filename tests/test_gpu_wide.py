"""GPU parity tests of the CLUSTER kernel (csrc/wdb_tc_wide.cu): blocks_per_env > 1 spreads
one TagContinuous env over a thread-block cluster (SURVEY.md section 8 config 4; reference
multi-block mode: warp_drive/cuda_includes/core/env_thread_sync.cu:31-62,
env_dim_mapper.h:22-31, tests/multiblocks_per_env/).

Three layers:
  * every parity test of tests/test_gpu_envs.py and the fused-step tests of
    tests/test_gpu_rollout.py re-run with blocks_per_env = 2 / 3 (the cluster kernel works at
    any env size), in all three k-nearest modes and with the x-window on and off;
  * 1024 agents per env against the C oracle AND against what the REFERENCE's own kernel
    computed with wkBlocksPerEnv = 2 and 4 (512 / 256 threads per block, which sm_100a can
    launch; fingerprints in tests/golden/ref_kernels.npz): state, observations, neighbour
    ids bit-identical, no tie escape;
  * the reference's own multi-block test shape (2 envs x 5 agents x 2 blocks).
"""
import numpy as np
import pytest
import torch

import test_gpu_envs as base
import test_gpu_rollout as roll
from helpers import RefTrace
from test_gpu_envs import tc_history  # noqa: F401  (fixture: history / network / exact)

pytestmark = pytest.mark.gpu


@pytest.fixture(params=[2, 3], ids=["bpe2", "bpe3"])
def bpe(request):
    base._BPE = request.param
    roll._BPE = request.param
    yield request.param
    base._BPE = 1
    roll._BPE = 1


@pytest.fixture(params=[1, 0], ids=["window", "nowindow"])
def window(request, wdb_lib):
    assert wdb_lib.wdb_set_option(b"tc_wide_window", request.param) == 0
    yield request.param
    wdb_lib.wdb_set_option(b"tc_wide_window", 1)


@pytest.mark.parametrize("name", base.TC_FIXTURES)
def test_wide_teacher_forced_vs_oracle(wdb_lib, name, tc_history, bpe, window):  # noqa: F811
    base.test_tag_continuous_teacher_forced_vs_oracle(wdb_lib, name, tc_history)


@pytest.mark.parametrize("shape", [(2, 5), (4, 23), (8, 105)])
@pytest.mark.parametrize("full_obs", [False, True])
def test_wide_bit_exact_vs_reference_cuda(wdb_lib, shape, full_obs, tc_history, bpe):  # noqa: F811
    """Our cluster kernel (bpe 2 / 3) against the reference kernel (its bpe = 1 build: the
    reference's result does not depend on the block split)."""
    base.test_tag_continuous_bit_exact_vs_reference_cuda(wdb_lib, shape, full_obs, tc_history)


def test_wide_tie_order(wdb_lib, tc_history, bpe, window):  # noqa: F811
    base.test_tag_continuous_tie_order_matches_reference_selection(wdb_lib, tc_history)


@pytest.mark.parametrize("bins", [0, 1, 4, 64])
def test_wide_bin_counts(wdb_lib, bins):
    """Any bin count must give the same result (0 = automatic)."""
    base._BPE = 2
    try:
        assert wdb_lib.wdb_set_option(b"tc_wide_bins", bins) == 0
        base.test_tag_continuous_teacher_forced_vs_oracle(wdb_lib, "config2_short", 1)
    finally:
        wdb_lib.wdb_set_option(b"tc_wide_bins", 0)
        base._BPE = 1


@pytest.mark.parametrize("blocks", [2, 4, 8])
def test_wide_1024_agents_vs_oracle(wdb_lib, blocks, tc_history, window):  # noqa: F811
    base._BPE = blocks
    try:
        base.test_tag_continuous_large_agent_counts_vs_oracle(wdb_lib, 1024, 24, 2, 64.0,
                                                              tc_history)
    finally:
        base._BPE = 1


@pytest.mark.parametrize("grid", [64.0, 20.0])
@pytest.mark.parametrize("blocks", [2, 4])
def test_wide_1024_agents_bit_exact_vs_reference_multiblock(wdb_lib, blocks, tc_history, grid):  # noqa: F811
    """BASELINE config 4 size against what the REFERENCE kernel computed in its own
    multi-block mode (wkBlocksPerEnv = 2 / 4; RefTrace): bit-equality of state,
    observations and neighbour ids over a free-running rollout -- no rank-wise tie escape.
    grid = 20: ten times config 4's agent density, so the candidate list of the threshold
    scan overflows all the time and the window-limited network path (stats[3]) carries the
    selection."""
    E, N, K, n_taggers = 2, 1024, 10, 24
    cfg, st0 = base._tc_synthetic(N, n_taggers, K, E, grid, seed=N)
    F = 7 * K + 1
    ref = RefTrace(f"tc_wide_N{N}_B{blocks}_grid{int(grid)}")
    a_st, dcfg = base._dev(st0), base._dev(cfg)
    a_obs = torch.zeros((E, N, F), device="cuda")
    a_rew = torch.zeros((E, N), device="cuda")
    rs = np.random.RandomState(1)
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    base._BPE = blocks
    try:
        tags = 0
        for t in range(12):
            actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
            alive_before = a_st["still_in_the_game"].clone()
            base.wdb_tc_step(wdb_lib, a_st, dcfg, actions, a_obs, a_rew, stats=stats)
            torch.cuda.synchronize()
            for k in base.STATE_F + ("still_in_the_game", "_timestep_"):
                assert ref.same(t, k, a_st[k]), (t, k)
            valid = torch.clamp(alive_before.sum(1, keepdim=True) - alive_before, max=K)
            mask = (torch.arange(K, device="cuda")[None, None] < valid[:, :, None]) & \
                   (alive_before[:, :, None] > 0)
            assert ref.same(t, "nearest_neighbor_ids", a_st["nearest_neighbor_ids"][mask]), t
            assert ref.same(t, "obs", a_obs), (t, "obs")
            # rewards: identical except where the reference's racy `rewards[tagger] += ...`
            # may lose a credit (taggers only)
            is_runner = dcfg["agent_types"] == 0
            assert ref.same(t, "runner_rewards", a_rew[:, is_runner]), (t, "runner rewards")
            tags += int((alive_before - a_st["still_in_the_game"]).sum())
        assert tags > 0
        if tc_history and grid < 64.0:
            assert int(stats[3]) > 0, "the window-limited network path never ran"
    finally:
        base._BPE = 1


def test_wide_reference_multiblock_shape(wdb_lib, tc_history):  # noqa: F811
    """The reference's own multi-block build shape (test_build_multiblocks.cu: 2 envs x 5
    agents x 2 blocks per env), both kernels in multi-block mode."""
    from conftest import load_golden
    from helpers import tc_cfg_from_fixture, tc_state_from_fixture

    E, N, blocks = 2, 5, 2
    fx = load_golden("tag_continuous_numpy_test1.npz")
    cfg = tc_cfg_from_fixture(fx)
    st0 = tc_state_from_fixture(fx, E)
    assert st0["loc_x"].shape[1] == N
    F = base._obs_dim(cfg, N)
    ref = RefTrace(f"tc_multiblock_E{E}_N{N}_B{blocks}")
    a_st, dcfg = base._dev(st0), base._dev(cfg)
    a_obs = torch.zeros((E, N, F), device="cuda")
    a_rew = torch.zeros((E, N), device="cuda")
    rs = np.random.RandomState(7)
    base._BPE = blocks
    try:
        steps = 0
        for t in range(int(cfg["episode_length"]) - 1):
            if bool(a_st["_done_"].any()):
                break
            actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
            base.wdb_tc_step(wdb_lib, a_st, dcfg, actions, a_obs, a_rew)
            torch.cuda.synchronize()
            for k in base.STATE_F + ("still_in_the_game", "_timestep_"):
                assert ref.same(t, k, a_st[k]), (t, k)
            assert ref.same(t, "obs", a_obs), (t, "obs")
            steps += 1
        assert steps == ref.steps("obs")    # the reference's episode ended at the same step
    finally:
        base._BPE = 1


# ---------------------------------------------------------------- fused rollout step, clusters
@pytest.mark.parametrize("full_obs", [False, True])
def test_wide_fused_step_equals_separate_calls(full_obs, bpe):
    roll.test_fused_step_equals_separate_calls(full_obs)


def test_wide_fused_step_without_reset_keeps_done_set(bpe):
    roll.test_fused_step_without_reset_keeps_done_set()


def test_wide_engine_cuda_graph_matches_eager(bpe):
    roll.test_engine_cuda_graph_matches_eager(True)


def test_wide_engine_batches(bpe):
    roll.test_engine_fused_matches_unfused_batches()


def test_wide_config4_through_wrapper_and_engine():
    """BASELINE config 4 shape through the public API: EnvWrapper(blocks_per_env=4) ->
    RolloutEngine with the FUSED cluster step (no [E, N, N-1] scratch is allocated), several
    episodes with resets; invariants + the batch equals the env arrays."""
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.tag_continuous import TagContinuous
    from warp_drive_b200.managers.function_manager import CUDASampler
    from warp_drive_b200.training.models.fully_connected import FullyConnected
    from warp_drive_b200.training.rollout import RolloutEngine
    from warp_drive_b200.training.utils.data_loader import create_and_push_data_placeholders

    kw = dict(roll.ENV_KW, num_taggers=24, num_runners=1000, grid_length=64.0,
              num_other_agents_observed=10, tagging_distance=0.3, episode_length=10)
    env = TagContinuous(**kw)
    E, T = 3, 4
    w = EnvWrapper(env, num_envs=E, env_backend="b200", blocks_per_env=4)
    w.reset_all_envs()
    assert not env.allocate_reference_scratch
    pm = {"runner": sorted(env.runners), "tagger": sorted(env.taggers)}
    s = CUDASampler(w.cuda_function_manager)
    create_and_push_data_placeholders(env_wrapper=w, action_sampler=s,
                                      policy_tag_to_agent_id_map=pm,
                                      training_batch_size_per_env=T)
    s.init_random(3)
    torch.manual_seed(0)
    cfg = {"type": "fully_connected", "fc_dims": [32, 32], "model_ckpt_filepath": ""}
    models = {p: FullyConnected(w, cfg, p, pm).cuda().eval() for p in pm}
    eng = RolloutEngine(w, models, pm, s, T, use_cuda_graph=True)
    assert eng.fused is not None, "the cluster kernel serves the fused step at 1024 agents"
    for _ in range(4):
        eng.rollout()
    torch.cuda.synchronize()
    dm = w.cuda_data_manager
    x, y = dm.pull_data_from_device("loc_x"), dm.pull_data_from_device("loc_y")
    assert ((x >= 0) & (x <= 64.0) & (y >= 0) & (y <= 64.0)).all()
    nn = dm.pull_data_from_device("nearest_neighbor_ids")
    assert nn.min() >= 0 and nn.max() < 1024
    assert int(eng.num_completed_episodes) >= E
    obs = dm.data_on_device_via_torch("observations")
    N = w.n_agents
    for p, ids in pm.items():
        i = torch.as_tensor(ids, device="cuda")
        assert torch.equal(eng.cur_obs[p], obs.view(E, N, -1)[:, i])
        assert torch.equal(dm.data_on_device_via_torch(f"rewards_batch_{p}")[T - 1],
                           dm.data_on_device_via_torch("rewards")[:, i])
