"""GPU parity tests of the env step kernels, called through the C ABI exactly like the
managers do, against (a) the CPU oracle and (b) what the reference's own CUDA kernels
computed from identical inputs (fingerprints in tests/golden/ref_kernels.npz).

Bars: integer / index / flag outputs bit-exact; float32 outputs within 1e-5 abs-or-rel
against the CPU oracle (libm vs libdevice sin/cos differ in the last bit) and BIT-EXACT
against the reference CUDA kernels (same compiler, same libdevice)."""
import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden
from helpers import RefTrace, close, copy_state, tc_cfg_from_fixture, tc_state_from_fixture

pytestmark = pytest.mark.gpu

TC_FIXTURES = ["test1", "test2", "test3", "test4", "partial_mid", "config2_short"]
STATE_F = ("loc_x", "loc_y", "speed", "direction", "acceleration", "edge_hit_reward_penalty")
STATE_I = ("still_in_the_game", "num_runners", "_done_", "_timestep_")


@pytest.fixture(params=[1, 0, 2], ids=["history", "network", "exact"])
def tc_history(request, wdb_lib):
    """Run the tag_continuous tests with every k-nearest strategy (temporal-coherence
    threshold, full sorting network, and the reference-literal exact path forced for every
    agent); results must be identical."""
    assert wdb_lib.wdb_set_option(b"tc_history", 1 if request.param else 0) == 0
    assert wdb_lib.wdb_set_option(b"tc_force_exact", 1 if request.param == 2 else 0) == 0
    yield request.param
    wdb_lib.wdb_set_option(b"tc_history", 1)
    wdb_lib.wdb_set_option(b"tc_force_exact", 0)


def _dev(d):
    return {k: (torch.from_numpy(np.ascontiguousarray(v)).cuda() if isinstance(v, np.ndarray) else v)
            for k, v in d.items()}


# blocks_per_env passed to wdb_tag_continuous_step: 1 = env replicas packed into CTAs; tests/
# test_gpu_wide.py re-runs the tests of this module with 2 / 4 (one env per cluster of CTAs)
_BPE = 1


def wdb_tc_step(L, st, cfg, actions, obs, rewards, nd=None, nid=None, stats=None):
    from warp_drive_b200 import lib as wlib

    E, N = st["loc_x"].shape
    p = wlib.ptr
    wlib.check(L.wdb_tag_continuous_step(
        wlib.stream_ptr(), E, N, _BPE, p(st["loc_x"]), p(st["loc_y"]), p(st["speed"]),
        p(st["direction"]), p(st["acceleration"]), p(cfg["agent_types"]),
        p(st["edge_hit_reward_penalty"]), float(cfg["edge_hit_penalty"]),
        float(cfg["grid_length"]), p(cfg["acceleration_actions"]), p(cfg["turn_actions"]),
        float(cfg["max_speed"]), int(cfg["num_other_agents_observed"]),
        p(cfg["skill_levels"]), int(cfg["runner_exits_game_after_tagged"]),
        p(st["still_in_the_game"]), int(cfg["use_full_observation"]), p(obs), p(actions),
        p(nd), p(nid), p(st["nearest_neighbor_ids"]), p(rewards), p(cfg["step_rewards"]),
        p(st["num_runners"]), float(cfg["distance_margin_for_reward"]),
        float(cfg["tag_reward_for_tagger"]), float(cfg["tag_penalty_for_runner"]),
        float(cfg["end_of_game_reward_for_runner"]), p(st["_done_"]), p(st["_timestep_"]),
        int(cfg["episode_length"]), p(stats)), "wdb_tag_continuous_step")


def _random_actions(rs, E, N, cfg):
    na, nt = len(cfg["acceleration_actions"]), len(cfg["turn_actions"])
    return np.stack([rs.randint(0, na, (E, N)), rs.randint(0, nt, (E, N))], -1).astype(np.int32)


def _obs_dim(cfg, N):
    K = int(cfg["num_other_agents_observed"])
    return 7 * (N - 1) + 1 if int(cfg["use_full_observation"]) else 7 * K + 1


@pytest.mark.parametrize("name", TC_FIXTURES)
def test_tag_continuous_teacher_forced_vs_oracle(wdb_lib, name, tc_history):
    """Every step starts the oracle from the GPU's current state, so differences cannot
    accumulate: a full multi-episode rollout with device-side resets."""
    fx = load_golden(f"tag_continuous_numpy_{name}.npz")
    cfg = tc_cfg_from_fixture(fx)
    E = 6
    st0 = tc_state_from_fixture(fx, E)
    N = st0["loc_x"].shape[1]
    F = _obs_dim(cfg, N)
    dst, dcfg = _dev(st0), _dev(cfg)
    obs = torch.zeros((E, N, F), device="cuda")
    rew = torch.zeros((E, N), device="cuda")
    rs = np.random.RandomState(42)
    n_steps = min(2 * int(cfg["episode_length"]) + 5, 230)
    worst = 0.0
    for t in range(n_steps):
        host = {k: v.cpu().numpy() for k, v in dst.items()}
        # device-side reset of done envs == restore initial state (checked separately)
        for e in np.nonzero(host["_done_"])[0]:
            for k in host:
                host[k][e] = st0[k][e]
        dst = _dev(host)
        actions = _random_actions(rs, E, N, cfg)
        ost = copy_state(host)
        o_obs, o_rew = oracle.tag_continuous_step(ost, cfg, actions)
        wdb_tc_step(wdb_lib, dst, dcfg, torch.from_numpy(actions).cuda(), obs, rew)
        got = {k: v.cpu().numpy() for k, v in dst.items()}
        for k in STATE_I:
            assert (got[k] == ost[k]).all(), (name, t, k)
        for k in STATE_F:
            ok = close(got[k], ost[k])
            assert ok.all(), (name, t, k)
        if not int(cfg["use_full_observation"]):
            K = int(cfg["num_other_agents_observed"])
            alive_before = host["still_in_the_game"]
            valid = np.minimum(alive_before.sum(1, keepdims=True) - alive_before, K)
            mask = (np.arange(K)[None, None, :] < valid[:, :, None]) & (alive_before[:, :, None] > 0)
            assert (got["nearest_neighbor_ids"][mask] == ost["nearest_neighbor_ids"][mask]).all(), (name, t)
        g_obs, g_rew = obs.cpu().numpy(), rew.cpu().numpy()
        ok = close(g_obs, o_obs)
        assert ok.all(), (name, t, np.argwhere(~ok)[:4])
        assert close(g_rew, o_rew).all(), (name, t)
        worst = max(worst, float(np.abs(g_obs - o_obs).max()))
    assert worst < 1e-5


@pytest.mark.parametrize("shape", [(2, 5), (4, 23), (8, 105)])
@pytest.mark.parametrize("full_obs", [False, True])
def test_tag_continuous_bit_exact_vs_reference_cuda(wdb_lib, shape, full_obs, tc_history):
    """Free-running rollout of OUR kernel against what the REFERENCE kernel computed from
    the same initial state with the same actions (RefTrace); every output array must be
    bit-identical.  (Steps where one tagger is credited for >= 2 tags are where the
    reference has a data race -- tag_continuous_step_pycuda.cu:324-329 -- and are excluded
    for rewards.)"""
    E, N = shape
    fxname = {5: "test3", 23: "partial_mid", 105: "config2_short"}[N]
    fx = load_golden(f"tag_continuous_numpy_{fxname}.npz")
    cfg = tc_cfg_from_fixture(fx)
    cfg["use_full_observation"] = int(full_obs)
    if N == 5:
        cfg["num_other_agents_observed"] = 2
        cfg["distance_margin_for_reward"] = np.float32(1.5)   # make tags frequent
    cfg["episode_length"] = 60
    st0 = tc_state_from_fixture(fx, E)
    K = int(cfg["num_other_agents_observed"])
    st0["nearest_neighbor_ids"] = np.zeros((E, N, K), np.int32)
    F = _obs_dim(cfg, N)
    ref = RefTrace(f"tc_E{E}_N{N}_full{int(full_obs)}")
    a_st, dcfg = _dev(st0), _dev(cfg)
    a_obs = torch.zeros((E, N, F), device="cuda")
    a_rew = torch.zeros((E, N), device="cuda")
    init = _dev(st0)
    rs = np.random.RandomState(7)
    racy_steps = 0
    for t in range(150):
        done = a_st["_done_"].cpu().numpy()
        for e in np.nonzero(done)[0]:
            for k in a_st:
                a_st[k][e] = init[k][e]
        actions = torch.from_numpy(_random_actions(rs, E, N, cfg)).cuda()
        alive_before = a_st["still_in_the_game"].clone()
        wdb_tc_step(wdb_lib, a_st, dcfg, actions, a_obs, a_rew)
        torch.cuda.synchronize()
        for k in STATE_F + STATE_I:
            if k == "num_runners":
                continue  # racy decrement in the reference; checked via alive flags
            assert ref.same(t, k, a_st[k]), (t, k)
        assert ref.same(t, "obs", a_obs), (t, "obs")
        if not full_obs:
            valid = torch.clamp(alive_before.sum(1, keepdim=True) - alive_before, max=K)
            mask = (torch.arange(K, device="cuda")[None, None] < valid[:, :, None]) & \
                   (alive_before[:, :, None] > 0)
            assert ref.same(t, "nearest_neighbor_ids", a_st["nearest_neighbor_ids"][mask]), t
        tagged = (alive_before - a_st["still_in_the_game"]).sum(1).cpu().numpy() if \
            int(cfg["runner_exits_game_after_tagged"]) else None
        same = ref.same_rows(t, "rewards", a_rew)
        if not same.all():
            # only envs with >= 2 simultaneous tags may differ (reference race)
            bad = np.nonzero(~same)[0]
            assert tagged is not None and bool((tagged[bad] >= 2).all()), (t, bad)
            racy_steps += 1
        else:
            assert ref.same(t, "num_runners", a_st["num_runners"]) or tagged is not None
    assert racy_steps < 40


def test_tag_continuous_tie_order_matches_reference_selection(wdb_lib, tc_history):
    """Agents pinned to the same corner produce exact distance ties; the reference's
    swap-based selection does NOT return them in id order (SURVEY.md section 7 'Hard
    parts').  Construct such states and compare ids with the oracle's literal algorithm."""
    fx = load_golden("tag_continuous_numpy_partial_mid.npz")
    cfg = tc_cfg_from_fixture(fx)
    E = 8
    st = tc_state_from_fixture(fx, E)
    N = st["loc_x"].shape[1]
    rs = np.random.RandomState(3)
    L = float(cfg["grid_length"])
    for e in range(E):
        # put random groups of agents on identical points / mirrored points
        pts = rs.rand(4, 2) * L
        grp = rs.randint(0, 4, N)
        st["loc_x"][e] = pts[grp, 0]
        st["loc_y"][e] = pts[grp, 1]
        st["still_in_the_game"][e, rs.rand(N) < 0.2] = 0
    st["speed"][:] = 0
    cfg["acceleration_actions"][:] = 0     # nobody moves: ties survive the kinematics
    actions = np.zeros((E, N, 2), np.int32)
    F = _obs_dim(cfg, N)
    dst, dcfg = _dev(st), _dev(cfg)
    obs, rew = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N), device="cuda")
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    ost = copy_state(st)
    o_obs, _ = oracle.tag_continuous_step(ost, cfg, actions)
    wdb_tc_step(wdb_lib, dst, dcfg, torch.from_numpy(actions).cuda(), obs, rew, stats=stats)
    K = int(cfg["num_other_agents_observed"])
    alive = st["still_in_the_game"]
    valid = np.minimum(alive.sum(1, keepdims=True) - alive, K)
    mask = (np.arange(K)[None, None, :] < valid[:, :, None]) & (alive[:, :, None] > 0)
    got = dst["nearest_neighbor_ids"].cpu().numpy()
    assert (got[mask] == ost["nearest_neighbor_ids"][mask]).all()
    assert close(obs.cpu().numpy(), o_obs).all()
    assert int(stats[0]) > 0       # the exact tie-resolution path really ran


def test_tag_continuous_full_size_properties(wdb_lib, tc_history):
    """BASELINE config 2 at full size (2000 x 105, K = 10): size-independent invariants
    over a whole 500-step episode with device-side resets."""
    fx = load_golden("tag_continuous_numpy_config2_short.npz")
    cfg = tc_cfg_from_fixture(fx)
    E = 2000
    st0 = tc_state_from_fixture(fx, E)
    N, K = st0["loc_x"].shape[1], int(cfg["num_other_agents_observed"])
    F = 7 * K + 1
    T = int(cfg["episode_length"])
    dst, dcfg = _dev(st0), _dev(cfg)
    init = _dev(st0)
    obs, rew = torch.zeros((E, N, F), device="cuda"), torch.zeros((E, N), device="cuda")
    is_runner = (dcfg["agent_types"] == 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    L = float(cfg["grid_length"])
    total_tags = 0
    for t in range(1, T + 1):
        actions = torch.randint(0, 21, (E, N, 2), generator=g, device="cuda", dtype=torch.int32)
        alive_before = dst["still_in_the_game"].clone()
        wdb_tc_step(wdb_lib, dst, dcfg, actions, obs, rew)
        if t % 25 and t != T:
            continue
        x, y, alive = dst["loc_x"], dst["loc_y"], dst["still_in_the_game"]
        assert bool(((x >= 0) & (x <= L) & (y >= 0) & (y <= L)).all())
        assert bool((alive <= alive_before).all())                      # nobody revives
        assert torch.equal(dst["num_runners"], (alive * is_runner).sum(1).int())
        assert bool((dst["_timestep_"] == t).all())
        assert bool((dst["_done_"] == int(t == T)).all() or (dst["num_runners"] == 0).any())
        o = obs.view(E, N, 7 * K + 1)
        assert bool((o[..., 7 * K][alive_before > 0] == np.float32(t) / np.float32(T)).all())
        assert bool((o[alive_before == 0] == 0).all())
        # nearest ids: distinct, alive, sorted by (float64) distance, truly the K nearest
        nn = dst["nearest_neighbor_ids"].long()
        for e in (0, E // 2, E - 1):
            xe, ye = x[e].double(), y[e].double()
            d = torch.sqrt((xe[:, None] - xe[None]) ** 2 + (ye[:, None] - ye[None]) ** 2)
            d = d + torch.where((alive_before[e] > 0)[None, :], 0.0, float("inf"))
            d.fill_diagonal_(float("inf"))
            for a in range(0, N, 13):
                if not alive_before[e, a]:
                    continue
                ids = nn[e, a]
                assert len(set(ids.tolist())) == K and bool((alive_before[e, ids] > 0).all())
                dd = d[a, ids]
                assert bool((dd[1:] >= dd[:-1] - 1e-6).all())
                kth = torch.sort(d[a]).values[K - 1]
                assert bool(dd[-1] <= kth + 1e-6)
        total_tags += int((alive_before - alive).sum())
    assert bool((dst["_done_"] == 1).all())
    # reset restores exactly the initial state for done envs
    from warp_drive_b200 import lib as wlib
    table = (wlib.ResetDesc * len(STATE_F + ("still_in_the_game", "num_runners")))()
    for i, k in enumerate(STATE_F + ("still_in_the_game", "num_runners")):
        table[i].dst, table[i].ref = dst[k].data_ptr(), init[k].data_ptr()
        table[i].bytes_per_env = dst[k][0].numel() * 4
        table[i].pool_rows = 0
    tdev = torch.from_numpy(np.frombuffer(table, dtype=np.uint8).copy()).cuda()
    wlib.check(wdb_lib.wdb_reset_when_done(wlib.stream_ptr(), tdev.data_ptr(), len(table),
                                           dst["_done_"].data_ptr(), dst["_timestep_"].data_ptr(),
                                           E, 0, 1, None))
    for k in STATE_F + ("still_in_the_game", "num_runners"):
        assert torch.equal(dst[k], init[k]), k
    assert int(dst["_done_"].sum()) == 0 and int(dst["_timestep_"].sum()) == 0


# ------------------------------------------------------------------ gridworld
def wdb_gw_step(L, x, y, actions, done, rew, obs, cfg, full, B, ts, T, moves):
    from warp_drive_b200 import lib as wlib

    p = wlib.ptr
    wlib.check(L.wdb_tag_gridworld_step(
        wlib.stream_ptr(), x.shape[0], x.shape[1], p(x), p(y), p(actions), p(done), p(rew),
        p(obs), float(cfg["wall_hit_penalty"]), float(cfg["tag_reward_for_tagger"]),
        float(cfg["tag_penalty_for_runner"]), float(cfg["step_cost_for_tagger"]), int(full),
        int(B), p(ts), int(T), p(moves)), "wdb_tag_gridworld_step")


MOVES = np.array([[0, 0], [1, 0], [-1, 0], [0, 1], [0, -1]], np.int32).reshape(-1)


@pytest.mark.parametrize("N,B,full", [(5, 4, True), (5, 4, False), (11, 10, True),
                                      (130, 30, False), (3, 2, True)])
def test_gridworld_bit_exact_vs_oracle(wdb_lib, oracle_lib, N, B, full):
    E, T = 301, 20
    cfg = dict(wall_hit_penalty=0.1, tag_reward_for_tagger=10.0, tag_penalty_for_runner=2.0,
               step_cost_for_tagger=0.01)
    rs = np.random.RandomState(N)
    x0 = rs.randint(0, B + 1, (E, N)).astype(np.int32)
    y0 = rs.randint(0, B + 1, (E, N)).astype(np.int32)
    F = 4 * N + 1 if full else 6
    hx, hy = x0.copy(), y0.copy()
    hdone, hts = np.zeros(E, np.int32), np.zeros(E, np.int32)
    hrew, hobs = np.zeros((E, N), np.float32), np.zeros((E, N, F), np.float32)
    dx, dy = torch.from_numpy(x0).cuda(), torch.from_numpy(y0).cuda()
    ddone, dts = torch.zeros(E, dtype=torch.int32, device="cuda"), torch.zeros(E, dtype=torch.int32, device="cuda")
    drew, dobs = torch.zeros((E, N), device="cuda"), torch.zeros((E, N, F), device="cuda")
    moves = torch.from_numpy(MOVES).cuda()
    for t in range(3 * T):
        # reset done envs on both sides
        d = hdone.astype(bool)
        hx[d], hy[d], hts[d], hdone[d] = x0[d], y0[d], 0, 0
        dd = torch.from_numpy(d).cuda()
        dx[dd], dy[dd] = torch.from_numpy(x0).cuda()[dd], torch.from_numpy(y0).cuda()[dd]
        dts[dd], ddone[dd] = 0, 0
        actions = rs.randint(0, 5, (E, N)).astype(np.int32)
        oracle_lib.wd_oracle_tag_gridworld_step(
            E, N, hx, hy, actions, hdone, hrew, hobs, 0.1, 10.0, 2.0, 0.01, int(full), B,
            hts, T, MOVES)
        wdb_gw_step(wdb_lib, dx, dy, torch.from_numpy(actions).cuda(), ddone, drew, dobs,
                    cfg, full, B, dts, T, moves)
        assert (dx.cpu().numpy() == hx).all() and (dy.cpu().numpy() == hy).all()
        assert (ddone.cpu().numpy() == hdone).all() and (dts.cpu().numpy() == hts).all()
        assert (drew.cpu().numpy() == hrew).all()          # bit-exact float32
        assert (dobs.cpu().numpy() == hobs).all()


@pytest.mark.parametrize("full", [True, False])
def test_gridworld_bit_exact_vs_reference_cuda(wdb_lib, full):
    E, N, B, T = 2, 5, 4, 20
    ref = RefTrace(f"gw_full{int(full)}")
    cfg = dict(wall_hit_penalty=0.1, tag_reward_for_tagger=10.0, tag_penalty_for_runner=2.0,
               step_cost_for_tagger=0.01, use_full_observation=full, world_boundary=B)
    F = 4 * N + 1 if full else 6
    rs = np.random.RandomState(5)
    x0 = torch.from_numpy(rs.randint(0, B + 1, (E, N)).astype(np.int32)).cuda()
    y0 = torch.from_numpy(rs.randint(0, B + 1, (E, N)).astype(np.int32)).cuda()
    moves = torch.from_numpy(MOVES).cuda()
    A = dict(x=x0.clone(), y=y0.clone(), done=torch.zeros(E, dtype=torch.int32, device="cuda"),
             ts=torch.zeros(E, dtype=torch.int32, device="cuda"),
             rew=torch.zeros((E, N), device="cuda"), obs=torch.zeros((E, N, F), device="cuda"))
    for t in range(100):
        d = A["done"] > 0
        A["x"][d], A["y"][d] = x0[d], y0[d]
        A["ts"][d], A["done"][d] = 0, 0
        actions = torch.from_numpy(rs.randint(0, 5, (E, N)).astype(np.int32)).cuda()
        wdb_gw_step(wdb_lib, A["x"], A["y"], actions, A["done"], A["rew"], A["obs"], cfg,
                    full, B, A["ts"], T, moves)
        torch.cuda.synchronize()
        for k in A:
            assert ref.same(t, k, A[k]), (t, k)


# ------------------------------------------------------------------ cartpole
def test_cartpole_vs_oracle(wdb_lib, oracle_lib):
    from warp_drive_b200 import lib as wlib

    E, T = 10000, 500
    rs = np.random.RandomState(0)
    s0 = rs.uniform(-0.05, 0.05, (E, 1, 4)).astype(np.float32)
    hs = s0.copy()
    hdone, hts = np.zeros(E, np.int32), np.zeros(E, np.int32)
    hrew, hobs = np.zeros((E, 1), np.float32), np.zeros((E, 1, 4), np.float32)
    ds = torch.from_numpy(s0).cuda()
    ddone = torch.zeros(E, dtype=torch.int32, device="cuda")
    dts = torch.zeros(E, dtype=torch.int32, device="cuda")
    drew, dobs = torch.zeros((E, 1), device="cuda"), torch.zeros((E, 1, 4), device="cuda")
    consts = [9.8, 0.1, 1.1, 0.5, 0.05, 10.0, 0.02, 12 * 2 * np.pi / 360, 2.4]
    p = wlib.ptr
    n_done = 0
    for t in range(120):
        # teacher forcing: both sides start from the GPU state; done envs restart
        hs = ds.cpu().numpy()
        d = ddone.cpu().numpy().astype(bool)
        hs[d] = s0[d]
        n_done += int(d.sum())
        ds.copy_(torch.from_numpy(hs))
        hts = dts.cpu().numpy()
        hts[d] = 0
        dts.copy_(torch.from_numpy(hts))
        ddone.zero_()
        hdone[:] = 0
        actions = rs.randint(0, 2, (E, 1, 1)).astype(np.int32)
        oracle_lib.wd_oracle_cartpole_step(E, hs, actions, hdone, hrew, hobs, *consts, hts, T)
        wlib.check(wdb_lib.wdb_cartpole_step(
            wlib.stream_ptr(), E, p(ds), p(torch.from_numpy(actions).cuda()), p(ddone),
            p(drew), p(dobs), *consts, p(dts), T))
        assert np.allclose(ds.cpu().numpy(), hs, rtol=1e-5, atol=1e-6)
        assert np.allclose(dobs.cpu().numpy(), hobs, rtol=1e-5, atol=1e-6)
        assert (ddone.cpu().numpy() == hdone).all()
        assert (drew.cpu().numpy() == 1.0).all()
        assert (dts.cpu().numpy() == hts).all()
    assert n_done > E // 2      # random policy: poles do fall, resets exercised


def _tc_synthetic(N, n_taggers, K, E, grid, seed):
    """A tag_continuous configuration that no fixture covers (large agent counts)."""
    rs = np.random.RandomState(seed)
    types = np.zeros(N, np.int32)
    types[rs.choice(N, n_taggers, replace=False)] = 1
    levels = 20
    cfg = {
        "agent_types": types,
        "acceleration_actions": np.concatenate([[0.0], np.linspace(-0.1, 0.1, levels)]).astype(np.float32),
        "turn_actions": np.concatenate([[0.0], np.linspace(-2.356, 2.356, levels)]).astype(np.float32),
        "skill_levels": np.where(types == 1, 1.0, 1.0).astype(np.float32),
        "step_rewards": np.where(types == 1, 0.0, 0.01).astype(np.float32),
        "episode_length": 50,
        "grid_length": np.float32(grid), "edge_hit_penalty": np.float32(-0.5),
        "max_speed": np.float32(1.0), "distance_margin_for_reward": np.float32(0.2),
        "tag_reward_for_tagger": np.float32(10.0), "tag_penalty_for_runner": np.float32(-10.0),
        "end_of_game_reward_for_runner": np.float32(1.0),
        "num_other_agents_observed": K, "use_full_observation": 0,
        "runner_exits_game_after_tagged": 1,
    }
    st = {
        "loc_x": (rs.rand(E, N) * grid).astype(np.float32),
        "loc_y": (rs.rand(E, N) * grid).astype(np.float32),
        "speed": (rs.rand(E, N) * 0.5).astype(np.float32),
        "direction": (rs.rand(E, N) * 2 * np.pi).astype(np.float32),
        "acceleration": np.zeros((E, N), np.float32),
        "edge_hit_reward_penalty": np.zeros((E, N), np.float32),
        "still_in_the_game": np.ones((E, N), np.int32),
        "num_runners": np.full(E, N - n_taggers, np.int32),
        "nearest_neighbor_ids": np.zeros((E, N, K), np.int32),
        "_done_": np.zeros(E, np.int32),
        "_timestep_": np.zeros(E, np.int32),
    }
    return cfg, st


@pytest.mark.parametrize("N,n_taggers,E,grid", [(150, 10, 5, 20.0), (330, 20, 3, 30.0),
                                                (1024, 24, 2, 64.0)])
def test_tag_continuous_large_agent_counts_vs_oracle(wdb_lib, N, n_taggers, E, grid, tc_history):
    """BASELINE config 4 territory (up to 1024 agents per env: one CTA per env, observations
    written straight to global memory, neighbour search without the history path) and the
    sizes in between (two envs per CTA without history; 330 agents = the 1024-thread
    variant).  Teacher-forced against the C oracle like the fixture-based test."""
    K = 10
    cfg, st0 = _tc_synthetic(N, n_taggers, K, E, grid, seed=N)
    F = 7 * K + 1
    dst, dcfg = _dev(st0), _dev(cfg)
    obs = torch.zeros((E, N, F), device="cuda")
    rew = torch.zeros((E, N), device="cuda")
    # the reference's per-agent global scratch (neighbor_distances / neighbor_ids_sorted_by_
    # distance, [E, N, N-1]): optional for small envs, required when the exact path's lists
    # do not fit shared memory
    nd = torch.zeros((E, N, N - 1), device="cuda") if N > 512 else None
    nid = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda") if N > 512 else None
    rs = np.random.RandomState(1)
    tags = 0
    for t in range(14):
        host = {k: v.cpu().numpy() for k, v in dst.items()}
        actions = _random_actions(rs, E, N, cfg)
        ost = copy_state(host)
        o_obs, o_rew = oracle.tag_continuous_step(ost, cfg, actions)
        wdb_tc_step(wdb_lib, dst, dcfg, torch.from_numpy(actions).cuda(), obs, rew, nd, nid)
        got = {k: v.cpu().numpy() for k, v in dst.items()}
        for k in STATE_I:
            assert (got[k] == ost[k]).all(), (N, t, k)
        for k in STATE_F:
            assert close(got[k], ost[k]).all(), (N, t, k)
        alive_before = host["still_in_the_game"]
        valid = np.minimum(alive_before.sum(1, keepdims=True) - alive_before, K)
        mask = (np.arange(K)[None, None, :] < valid[:, :, None]) & (alive_before[:, :, None] > 0)
        # The CPU oracle and the GPU agree on positions only to ~1 ulp (libm vs libdevice
        # sin/cos), so two neighbours whose float distances tie exactly on one side may be
        # ordered differently on the other (with 300+ agents this happens; the bit-level
        # arbiter is the reference-kernel test below).  Such rows must still hold
        # neighbours at the same distances, rank by rank, and are few.
        g_ids, o_ids = got["nearest_neighbor_ids"], ost["nearest_neighbor_ids"]
        bad_rows = np.unique(np.argwhere((g_ids != o_ids) & mask)[:, :2], axis=0)
        for e, a in bad_rows:
            px, py = ost["loc_x"][e].astype(np.float64), ost["loc_y"][e].astype(np.float64)
            dg = np.hypot(px[g_ids[e, a]] - px[a], py[g_ids[e, a]] - py[a])
            do = np.hypot(px[o_ids[e, a]] - px[a], py[o_ids[e, a]] - py[a])
            assert np.allclose(dg, do, rtol=1e-6, atol=1e-6), (N, t, e, a, g_ids[e, a], o_ids[e, a])
        assert len(bad_rows) <= max(1, E * N // 500), (N, t, len(bad_rows))
        ok = close(obs.cpu().numpy(), o_obs)
        for e, a in bad_rows:
            ok[e, a] = True
        assert ok.all(), (N, t, np.argwhere(~ok)[:4])
        assert close(rew.cpu().numpy(), o_rew).all(), (N, t)
        tags += int((alive_before - got["still_in_the_game"]).sum())
    assert tags > 0          # the margin is wide enough that runners really get tagged


@pytest.mark.parametrize("N,n_taggers,E,grid", [(330, 20, 3, 30.0)])
def test_tag_continuous_large_agent_counts_vs_reference_cuda(wdb_lib, N, n_taggers, E, grid,
                                                             tc_history):
    """The same large configurations against what the REFERENCE's own kernel computed
    (RefTrace): state, observations and neighbour ids bit-identical, including the order of
    neighbours whose float distances tie exactly.  (The reference kernel cannot be launched
    with 1024 threads per block on sm_100a -- CUDA_ERROR_LAUNCH_OUT_OF_RESOURCES, its
    register use -- so config-4 sizes are checked against the C oracle above and against
    the reference's multi-block mode in tests/test_gpu_wide.py.)"""
    K = 10
    cfg, st0 = _tc_synthetic(N, n_taggers, K, E, grid, seed=N)
    F = 7 * K + 1
    ref = RefTrace(f"tc_large_E{E}_N{N}")
    a_st, dcfg = _dev(st0), _dev(cfg)
    a_obs = torch.zeros((E, N, F), device="cuda")
    a_rew = torch.zeros((E, N), device="cuda")
    nd2 = torch.zeros((E, N, N - 1), device="cuda")
    nid2 = torch.zeros((E, N, N - 1), dtype=torch.int32, device="cuda")
    rs = np.random.RandomState(1)
    for t in range(10):
        actions = torch.from_numpy(_random_actions(rs, E, N, cfg)).cuda()
        alive_before = a_st["still_in_the_game"].clone()
        wdb_tc_step(wdb_lib, a_st, dcfg, actions, a_obs, a_rew, nd2, nid2)
        torch.cuda.synchronize()
        for k in STATE_F + ("still_in_the_game", "_timestep_"):
            assert ref.same(t, k, a_st[k]), (t, k)
        valid = torch.clamp(alive_before.sum(1, keepdim=True) - alive_before, max=K)
        mask = (torch.arange(K, device="cuda")[None, None] < valid[:, :, None]) & \
               (alive_before[:, :, None] > 0)
        assert ref.same(t, "nearest_neighbor_ids", a_st["nearest_neighbor_ids"][mask]), t
        assert ref.same(t, "obs", a_obs), (t, "obs")


@pytest.mark.parametrize("shape", [(4, 23), (8, 105)])
def test_tail_split_ctas_bit_exact_vs_reference_cuda(wdb_lib, shape, tc_history):
    """`tc_tail_split`: the envs of a partly filled last wave go out as ONE-env CTAs (config 2:
    592 three-env CTAs + 224 one-env CTAs).  Option value 2 forces half of the CTAs into that
    shape at any size: same bits as the reference kernel, step-only and through the fused
    rollout step."""
    import test_gpu_rollout as roll

    assert wdb_lib.wdb_set_option(b"tc_tail_split", 2) == 0
    try:
        test_tag_continuous_bit_exact_vs_reference_cuda(wdb_lib, shape, False, tc_history)
        roll.test_fused_step_equals_separate_calls(False)
        roll.test_engine_cuda_graph_matches_eager(True)
    finally:
        assert wdb_lib.wdb_set_option(b"tc_tail_split", 0) == 0
