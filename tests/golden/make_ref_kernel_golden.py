"""Generate tests/golden/ref_kernels.npz: what the reference's own kernels compute in the
bit-exact parity cases of tests/test_gpu_envs.py, tests/test_gpu_wide.py and
tests/test_gpu_classic_control.py, stored as per-step fingerprints (tests/helpers.py).

Needs a GPU and the reference binaries that oracle/build_ref.py (CUDA-C kernels) and
oracle/build_ref_numba.py (numba kernels) compile into oracle/_ref/:

    python tests/golden/make_ref_kernel_golden.py [OUT.npz]

Each case runs our kernel and the reference kernel side by side on the same inputs, the
way the tests drove them before the fingerprints existed, and asserts that they agree
(torch.equal; bitwise for the classic-control steps); what is stored are the REFERENCE's
outputs.  Inputs are built exactly as in the tests, so the tests replay the same
trajectories.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_gpu_classic_control as cc  # noqa: E402
import test_gpu_envs as base  # noqa: E402
from conftest import load_golden  # noqa: E402
from helpers import (REF_KERNELS_GOLDEN, fingerprint, row_fingerprints,  # noqa: E402
                     tc_cfg_from_fixture, tc_state_from_fixture)
from oracle import ref_cuda, ref_numba  # noqa: E402
from warp_drive_b200 import lib as wlib  # noqa: E402

OUT = {}


def put(case, key, value):
    OUT.setdefault(f"{case}.{key}", []).append(value)


def nn_mask(alive_before, K):
    valid = torch.clamp(alive_before.sum(1, keepdim=True) - alive_before, max=K)
    return (torch.arange(K, device="cuda")[None, None] < valid[:, :, None]) & \
        (alive_before[:, :, None] > 0)


def tc_bit_exact(L, E, N, full_obs):
    """tests/test_gpu_envs.py::test_tag_continuous_bit_exact_vs_reference_cuda"""
    case = f"tc_E{E}_N{N}_full{int(full_obs)}"
    fxname = {5: "test3", 23: "partial_mid", 105: "config2_short"}[N]
    cfg = tc_cfg_from_fixture(load_golden(f"tag_continuous_numpy_{fxname}.npz"))
    cfg["use_full_observation"] = int(full_obs)
    if N == 5:
        cfg["num_other_agents_observed"] = 2
        cfg["distance_margin_for_reward"] = np.float32(1.5)
    cfg["episode_length"] = 60
    st0 = tc_state_from_fixture(load_golden(f"tag_continuous_numpy_{fxname}.npz"), E)
    K = int(cfg["num_other_agents_observed"])
    st0["nearest_neighbor_ids"] = np.zeros((E, N, K), np.int32)
    F = base._obs_dim(cfg, N)
    ref = ref_cuda.RefModule(E, N, 1)
    a_st, b_st, dcfg = base._dev(st0), base._dev(st0), base._dev(cfg)
    a_obs, b_obs = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N, F), device="cuda")
    a_rew, b_rew = torch.zeros((E, N), device="cuda"), torch.zeros((E, N), device="cuda")
    nd = torch.zeros((E, N, N - 1), device="cuda")
    nid = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda")
    init = base._dev(st0)
    rs = np.random.RandomState(7)
    for t in range(150):
        done = a_st["_done_"].cpu().numpy()
        for e in np.nonzero(done)[0]:
            for st in (a_st, b_st):
                for k in st:
                    st[k][e] = init[k][e]
        actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
        alive_before = a_st["still_in_the_game"].clone()
        base.wdb_tc_step(L, a_st, dcfg, actions, a_obs, a_rew)
        ref.tag_continuous_step(b_st, dcfg, actions, b_obs, b_rew, nd, nid)
        torch.cuda.synchronize()
        for k in base.STATE_F + base.STATE_I:
            if k != "num_runners":
                assert torch.equal(a_st[k], b_st[k]), (case, t, k)
            put(case, k, fingerprint(b_st[k]))
        assert torch.equal(a_obs, b_obs), (case, t, "obs")
        put(case, "obs", fingerprint(b_obs))
        if not full_obs:
            mask = nn_mask(alive_before, K)
            assert torch.equal(a_st["nearest_neighbor_ids"][mask],
                               b_st["nearest_neighbor_ids"][mask]), (case, t)
            put(case, "nearest_neighbor_ids", fingerprint(b_st["nearest_neighbor_ids"][mask]))
        put(case, "rewards", row_fingerprints(b_rew))
        b_st["num_runners"].copy_(a_st["num_runners"])
        b_st["_done_"].copy_(a_st["_done_"])


def tc_large(L, N, n_taggers, E, grid):
    """tests/test_gpu_envs.py::test_tag_continuous_large_agent_counts_vs_reference_cuda"""
    case = f"tc_large_E{E}_N{N}"
    K = 10
    cfg, st0 = base._tc_synthetic(N, n_taggers, K, E, grid, seed=N)
    F = 7 * K + 1
    ref = ref_cuda.RefModule(E, N, 1)
    a_st, b_st, dcfg = base._dev(st0), base._dev(st0), base._dev(cfg)
    a_obs, b_obs = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N, F), device="cuda")
    a_rew, b_rew = torch.zeros((E, N), device="cuda"), torch.zeros((E, N), device="cuda")
    nd = torch.zeros((E, N, N - 1), device="cuda")
    nid = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda")
    nd2, nid2 = torch.zeros_like(nd), torch.zeros_like(nid)
    rs = np.random.RandomState(1)
    for t in range(10):
        actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
        alive_before = a_st["still_in_the_game"].clone()
        base.wdb_tc_step(L, a_st, dcfg, actions, a_obs, a_rew, nd2, nid2)
        ref.tag_continuous_step(b_st, dcfg, actions, b_obs, b_rew, nd, nid)
        torch.cuda.synchronize()
        for k in base.STATE_F + ("still_in_the_game", "_timestep_"):
            assert torch.equal(a_st[k], b_st[k]), (case, t, k)
            put(case, k, fingerprint(b_st[k]))
        mask = nn_mask(alive_before, K)
        assert torch.equal(a_st["nearest_neighbor_ids"][mask], b_st["nearest_neighbor_ids"][mask])
        put(case, "nearest_neighbor_ids", fingerprint(b_st["nearest_neighbor_ids"][mask]))
        assert torch.equal(a_obs, b_obs), (case, t, "obs")
        put(case, "obs", fingerprint(b_obs))
        b_st["num_runners"].copy_(a_st["num_runners"])
        b_st["_done_"].copy_(a_st["_done_"])


def tc_wide_1024(L, blocks, grid):
    """tests/test_gpu_wide.py::test_wide_1024_agents_bit_exact_vs_reference_multiblock"""
    case = f"tc_wide_N1024_B{blocks}_grid{int(grid)}"
    E, N, K, n_taggers = 2, 1024, 10, 24
    cfg, st0 = base._tc_synthetic(N, n_taggers, K, E, grid, seed=N)
    F = 7 * K + 1
    ref = ref_cuda.RefModule(E, N, blocks)
    a_st, b_st, dcfg = base._dev(st0), base._dev(st0), base._dev(cfg)
    a_obs, b_obs = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N, F), device="cuda")
    a_rew, b_rew = torch.zeros((E, N), device="cuda"), torch.zeros((E, N), device="cuda")
    nd = torch.zeros((E, N, N - 1), device="cuda")
    nid = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda")
    rs = np.random.RandomState(1)
    is_runner = dcfg["agent_types"] == 0
    base._BPE = blocks
    try:
        for t in range(12):
            actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
            alive_before = a_st["still_in_the_game"].clone()
            base.wdb_tc_step(L, a_st, dcfg, actions, a_obs, a_rew)
            ref.tag_continuous_step(b_st, dcfg, actions, b_obs, b_rew, nd, nid)
            torch.cuda.synchronize()
            for k in base.STATE_F + ("still_in_the_game", "_timestep_"):
                assert torch.equal(a_st[k], b_st[k]), (case, t, k)
                put(case, k, fingerprint(b_st[k]))
            mask = nn_mask(alive_before, K)
            assert torch.equal(a_st["nearest_neighbor_ids"][mask],
                               b_st["nearest_neighbor_ids"][mask]), (case, t)
            put(case, "nearest_neighbor_ids", fingerprint(b_st["nearest_neighbor_ids"][mask]))
            assert torch.equal(a_obs, b_obs), (case, t, "obs")
            put(case, "obs", fingerprint(b_obs))
            assert torch.equal(a_rew[:, is_runner], b_rew[:, is_runner]), (case, t)
            put(case, "runner_rewards", fingerprint(b_rew[:, is_runner]))
            b_st["num_runners"].copy_(a_st["num_runners"])
            b_st["_done_"].copy_(a_st["_done_"])
    finally:
        base._BPE = 1


def tc_multiblock_shape(L):
    """tests/test_gpu_wide.py::test_wide_reference_multiblock_shape"""
    case = "tc_multiblock_E2_N5_B2"
    E, N, blocks = 2, 5, 2
    fx = load_golden("tag_continuous_numpy_test1.npz")
    cfg = tc_cfg_from_fixture(fx)
    st0 = tc_state_from_fixture(fx, E)
    F = base._obs_dim(cfg, N)
    ref = ref_cuda.RefModule(E, N, blocks)
    a_st, b_st, dcfg = base._dev(st0), base._dev(st0), base._dev(cfg)
    a_obs, b_obs = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N, F), device="cuda")
    a_rew, b_rew = torch.zeros((E, N), device="cuda"), torch.zeros((E, N), device="cuda")
    nd = torch.zeros((E, N, N - 1), device="cuda")
    nid = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda")
    rs = np.random.RandomState(7)
    base._BPE = blocks
    try:
        for t in range(int(cfg["episode_length"]) - 1):
            if bool(a_st["_done_"].any()):
                break
            actions = torch.from_numpy(base._random_actions(rs, E, N, cfg)).cuda()
            base.wdb_tc_step(L, a_st, dcfg, actions, a_obs, a_rew)
            ref.tag_continuous_step(b_st, dcfg, actions, b_obs, b_rew, nd, nid)
            torch.cuda.synchronize()
            for k in base.STATE_F + ("still_in_the_game", "_timestep_"):
                assert torch.equal(a_st[k], b_st[k]), (case, t, k)
                put(case, k, fingerprint(b_st[k]))
            assert torch.equal(a_obs, b_obs), (case, t, "obs")
            put(case, "obs", fingerprint(b_obs))
            b_st["num_runners"].copy_(a_st["num_runners"])
            b_st["_done_"].copy_(a_st["_done_"])
    finally:
        base._BPE = 1


def gridworld(L, full):
    """tests/test_gpu_envs.py::test_gridworld_bit_exact_vs_reference_cuda"""
    case = f"gw_full{int(full)}"
    E, N, B, T = 2, 5, 4, 20
    ref = ref_cuda.RefModule(E, N, 1)
    cfg = dict(wall_hit_penalty=0.1, tag_reward_for_tagger=10.0, tag_penalty_for_runner=2.0,
               step_cost_for_tagger=0.01, use_full_observation=full, world_boundary=B)
    F = 4 * N + 1 if full else 6
    rs = np.random.RandomState(5)
    x0 = torch.from_numpy(rs.randint(0, B + 1, (E, N)).astype(np.int32)).cuda()
    y0 = torch.from_numpy(rs.randint(0, B + 1, (E, N)).astype(np.int32)).cuda()
    moves = torch.from_numpy(base.MOVES).cuda()
    A = dict(x=x0.clone(), y=y0.clone(), done=torch.zeros(E, dtype=torch.int32, device="cuda"),
             ts=torch.zeros(E, dtype=torch.int32, device="cuda"),
             rew=torch.zeros((E, N), device="cuda"), obs=torch.zeros((E, N, F), device="cuda"))
    Bs = {k: v.clone() for k, v in A.items()}
    for t in range(100):
        for S in (A, Bs):
            d = S["done"] > 0
            S["x"][d], S["y"][d] = x0[d], y0[d]
            S["ts"][d], S["done"][d] = 0, 0
        actions = torch.from_numpy(rs.randint(0, 5, (E, N)).astype(np.int32)).cuda()
        base.wdb_gw_step(L, A["x"], A["y"], actions, A["done"], A["rew"], A["obs"], cfg,
                         full, B, A["ts"], T, moves)
        ref.tag_gridworld_step(Bs["x"], Bs["y"], actions, Bs["done"], Bs["rew"], Bs["obs"],
                               cfg, Bs["ts"], T, base.MOVES)
        torch.cuda.synchronize()
        for k in A:
            assert torch.equal(A[k], Bs[k]), (case, t, k)
            put(case, k, fingerprint(Bs[k]))


def classic_control(L, name):
    """tests/test_gpu_classic_control.py::test_step_vs_reference_numba_and_oracle"""
    case = f"cc_{name}"
    E = cc.E
    sdim, odim, adtype, consts, draw_state, draw_action = cc.ENVS[name]
    ours = getattr(L, f"wdb_{name}_step")
    ref = ref_numba.RefNumbaKernel(name)
    rs = np.random.RandomState(20260923 + len(name))
    p = wlib.ptr
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    for _ in range(cc.STEPS):
        s0 = draw_state(rs, E).astype(np.float32).reshape(E, 1, sdim)
        act = draw_action(rs, E).astype(adtype).reshape(E, 1, 1)
        ts0 = rs.randint(0, cc.EP_LEN, E).astype(np.int32)
        ts0[: E // 8] = cc.EP_LEN - 1
        d_s, d_a, d_ts = cuda(s0), cuda(act), cuda(ts0)
        d_done = torch.zeros(E, dtype=torch.int32, device="cuda")
        d_rew = torch.full((E, 1), 7.0, device="cuda")
        d_obs = torch.full((E, 1, odim), 7.0, device="cuda")
        wlib.check(ours(wlib.stream_ptr(), E, p(d_s), p(d_a), p(d_done), p(d_rew), p(d_obs),
                        *consts, p(d_ts), cc.EP_LEN))
        r_s, r_ts = cuda(s0), cuda(ts0)
        r_done = torch.zeros(E, dtype=torch.int32, device="cuda")
        r_rew = torch.full((E, 1), 7.0, device="cuda")
        r_obs = torch.full((E, 1, odim), 7.0, device="cuda")
        ref(E, r_s, d_a, r_done, r_rew, r_obs, *consts, r_ts, cc.EP_LEN)
        torch.cuda.synchronize()
        mine = torch.cat([d_s.reshape(E, -1), d_obs.reshape(E, -1), d_rew], 1)
        theirs = torch.cat([r_s.reshape(E, -1), r_obs.reshape(E, -1), r_rew], 1)
        assert torch.equal(mine.view(torch.int32), theirs.view(torch.int32)), case   # bitwise
        assert torch.equal(d_done, r_done) and torch.equal(d_ts, r_ts), case
        put(case, "outputs", fingerprint(theirs, bitwise=True))
        put(case, "done", fingerprint(r_done))
        put(case, "timestep", fingerprint(r_ts))


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else REF_KERNELS_GOLDEN
    L = wlib.load()
    for shape in ((2, 5), (4, 23), (8, 105)):
        for full_obs in (False, True):
            tc_bit_exact(L, *shape, full_obs)
    tc_large(L, 330, 20, 3, 30.0)
    for blocks in (2, 4):
        for grid in (64.0, 20.0):
            tc_wide_1024(L, blocks, grid)
    tc_multiblock_shape(L)
    for full in (True, False):
        gridworld(L, full)
    for name in cc.ENVS:
        classic_control(L, name)
    arrays = {k: np.asarray(v, np.uint32) for k, v in OUT.items()}
    np.savez_compressed(out, **arrays)
    print(f"{out}: {len(arrays)} entries, {sum(a.nbytes for a in arrays.values())} bytes")


if __name__ == "__main__":
    main()
