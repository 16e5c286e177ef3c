"""GPU parity of the single-agent classic-control steps (CartPole + SURVEY 8 row f2:
MountainCar, ContinuousMountainCar, Pendulum, Acrobot), called through the C ABI, against

(a) what the REFERENCE's own numba kernels (compiled by numba, oracle/build_ref_numba.py)
    computed from identical inputs, stored as per-step fingerprints
    (tests/golden/ref_kernels.npz, tests/helpers.py RefTrace), and
(b) the C oracle (oracle/wd_oracle.c, glibc libm on the host).

Every step is an independent single-step comparison on freshly drawn states that cover the
clipping / wrapping / terminal branches (teacher forcing: the integrators are chaotic, a
free-running comparison would only measure that).

Bars (written here, cited in DESIGN.md):
  * vs the reference numba binaries: float32 state / obs / reward, done and timestep
    BIT-identical for every env-step, as measured on the B200
    (profiles/r3_classic_control_parity.json).
  * vs the C oracle: within 1e-5 abs-or-rel (Acrobot 2e-4; libm vs libdevice), flags equal except for at
    most MAX_BRANCH_FLIPS threshold flips.
A JSON summary goes to gpurun_out/classic_control_parity.json.
"""
import json
import os

import numpy as np
import pytest
import torch

from helpers import RefTrace

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E, STEPS, EP_LEN = 8192, 24, 200
# A last-bit difference (libm vs libdevice, or one fused multiply-add) in front of a branch --
# the angle wrap at +-pi, a clip bound, the terminal test -- changes the outcome by a finite
# jump.  That is a 1e-7-probability event per env-step; this many rows of the 196 608 compared
# per env may take the other branch before the test calls it a failure.
MAX_BRANCH_FLIPS = 3
# vs the C oracle (glibc sinf/cosf instead of libdevice's, 1-2 ulp apart): Acrobot integrates
# accelerations of several hundred rad/s^2 through four float32-rounded RK4 stages, which
# turns those ulps into 1e-5..1e-4 relative differences (the numba binary, same libdevice,
# stays bit-identical)
ORACLE_TOL = {"acrobot": 2e-4}
# ... and only in the regime the env visits from its start states (|dtheta1| <= pi, |dtheta2| <=
# 2 pi): near the velocity bounds (4 pi, 9 pi) the stage derivatives reach 1e4 rad/s^2 and the
# same ulps come out at 1e-3.  The reference numba binary is compared on ALL rows.
ORACLE_ROWS = {"acrobot": lambda s0: (np.abs(s0[:, 0, 2]) <= PI) & (np.abs(s0[:, 0, 3]) <= 2 * PI)}
PI = np.pi

_CARTPOLE_CONSTS = [9.8, 0.1, 1.1, 0.5, 0.05, 10.0, 0.02, 12 * 2 * np.pi / 360, 2.4]
_MC_CONSTS = [-1.2, 0.6, 0.07, 0.5, 0.0, 0.001, 0.0025]
_CMC_CONSTS = [-1.0, 1.0, -1.2, 0.6, 0.07, 0.45, 0.0, 0.0015]


def _mc_states(rs, n):
    s = np.stack([rs.uniform(-1.25, 0.65, n), rs.uniform(-0.08, 0.08, n)], -1)
    s = np.clip(s, [-1.2, -0.07], [0.6, 0.07])
    s[: n // 16, 0] = -1.2            # at the left wall (velocity zeroing branch)
    s[n // 16: n // 8, 0] = rs.uniform(0.44, 0.6, n // 8 - n // 16)   # around the goal
    return s


ENVS = {
    # name: (state dim, obs dim, action dtype, consts, state sampler, action sampler)
    "cartpole": (4, 4, np.int32, _CARTPOLE_CONSTS,
                 lambda rs, n: rs.uniform(-1, 1, (n, 4)) * [2.6, 3.0, 0.25, 3.0],
                 lambda rs, n: rs.randint(0, 2, n)),
    "mountain_car": (2, 2, np.int32, _MC_CONSTS, _mc_states,
                     lambda rs, n: rs.randint(0, 3, n)),
    "continuous_mountain_car": (2, 2, np.float32, _CMC_CONSTS, _mc_states,
                                lambda rs, n: rs.uniform(-1.5, 1.5, n)),
    "pendulum": (2, 3, np.float32, [],
                 lambda rs, n: rs.uniform(-1, 1, (n, 2)) * [12.0, 8.0],
                 lambda rs, n: rs.uniform(-3.0, 3.0, n)),
    "acrobot": (4, 6, np.int32, [],
                lambda rs, n: rs.uniform(-1, 1, (n, 4)) * np.where(
                    np.arange(n)[:, None] % 2 == 0, [PI, PI, 4 * PI, 9 * PI], [PI, PI, PI, 2 * PI]),
                lambda rs, n: rs.randint(0, 3, n)),
}


def _close(a, b, tol):
    return np.abs(a - b) <= tol + tol * np.abs(b)


def _report(name, entry):
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    path = os.path.join(out, "classic_control_parity.json")
    data = {}
    if os.path.exists(path):
        with open(path) as fp:
            data = json.load(fp)
    data[name] = entry
    with open(path, "w") as fp:
        json.dump(data, fp, indent=1, sort_keys=True)


@pytest.mark.parametrize("name", list(ENVS))
def test_step_vs_reference_numba_and_oracle(name, wdb_lib, oracle_lib):
    from warp_drive_b200 import lib as wlib

    sdim, odim, adtype, consts, draw_state, draw_action = ENVS[name]
    ours = getattr(wdb_lib, f"wdb_{name}_step")
    oracle_fn = getattr(oracle_lib, f"wd_oracle_{name}_step")
    ref = RefTrace(f"cc_{name}", bitwise=True)
    rs = np.random.RandomState(20260923 + len(name))
    p = wlib.ptr
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731

    n_samples = 0
    max_abs_oracle = 0.0
    flag_flips_oracle = 0
    bad_oracle = 0
    done_seen = set()
    for t in range(STEPS):
        s0 = draw_state(rs, E).astype(np.float32).reshape(E, 1, sdim)
        act = draw_action(rs, E).astype(adtype).reshape(E, 1, 1)
        ts0 = rs.randint(0, EP_LEN, E).astype(np.int32)
        ts0[: E // 8] = EP_LEN - 1            # the step that ends the episode
        # ours
        d_s, d_a, d_ts = cuda(s0), cuda(act), cuda(ts0)
        d_done = torch.zeros(E, dtype=torch.int32, device="cuda")
        d_rew = torch.full((E, 1), 7.0, device="cuda")
        d_obs = torch.full((E, 1, odim), 7.0, device="cuda")
        wlib.check(ours(wlib.stream_ptr(), E, p(d_s), p(d_a), p(d_done), p(d_rew), p(d_obs),
                        *consts, p(d_ts), EP_LEN))
        torch.cuda.synchronize()
        # C oracle
        h_s, h_ts = s0.copy(), ts0.copy()
        h_done = np.zeros(E, np.int32)
        h_rew = np.full((E, 1), 7.0, np.float32)
        h_obs = np.full((E, 1, odim), 7.0, np.float32)
        oracle_fn(E, h_s, act, h_done, h_rew, h_obs, *consts, h_ts, EP_LEN)

        mine = np.concatenate([d_s.cpu().numpy().reshape(E, -1), d_obs.cpu().numpy().reshape(E, -1),
                               d_rew.cpu().numpy()], 1)
        host = np.concatenate([h_s.reshape(E, -1), h_obs.reshape(E, -1), h_rew], 1)
        assert np.isfinite(mine).all()

        # ---- (a) vs the reference numba binary
        assert ref.same(t, "outputs", mine), (name, t, "state / obs / reward vs reference numba")
        m_done = d_done.cpu().numpy()
        assert ref.same(t, "done", m_done), (name, t, "done vs reference numba")
        assert ref.same(t, "timestep", d_ts), (name, t, "timestep vs reference numba")
        n_samples += E
        done_seen |= set(np.unique(m_done).tolist())

        # ---- (b) vs the C oracle
        ok = _close(mine, host, ORACLE_TOL.get(name, 1e-5)).all(1)
        compared = np.ones(E, bool)
        if name in ORACLE_ROWS:
            compared = ORACLE_ROWS[name](s0)
            assert _close(mine, host, 0.05).all(1).mean() > 0.99   # sanity outside that regime
        ok |= ~compared
        bad_oracle += int((~ok).sum())
        assert bad_oracle <= MAX_BRANCH_FLIPS, (name, "vs C oracle", mine[~ok][:3], host[~ok][:3])
        max_abs_oracle = max(max_abs_oracle, float(np.abs(mine - host)[ok & compared].max()))
        flag_flips_oracle += int(((m_done != h_done) & ok).sum())
        assert (d_ts.cpu().numpy() == h_ts).all()

    _report(name, {"env_steps": n_samples, "bit_identical_vs_reference_numba": 1.0,
                   "rows_on_other_branch_vs_c_oracle": bad_oracle,
                   "max_abs_diff_vs_c_oracle": max_abs_oracle,
                   "done_flag_flips_vs_c_oracle": flag_flips_oracle,
                   "done_values_seen": sorted(int(v) for v in done_seen)})
    print(f"[classic-control parity] {name}: all {n_samples} env-steps bit-identical to the "
          f"reference numba binary; vs C oracle max |diff| {max_abs_oracle:.3g}, "
          f"{flag_flips_oracle} done flips")
    assert flag_flips_oracle <= MAX_BRANCH_FLIPS, (name, flag_flips_oracle)
    assert 1 in done_seen                       # the episode-end branch ran
    if name == "mountain_car":
        assert 2 in done_seen                   # goal reached -> done = 2 (reference quirk)


@pytest.mark.parametrize("cls_name,pool", [
    ("MountainCar", 0), ("ContinuousMountainCar", 8), ("Pendulum", 0), ("Acrobot", 8)])
def test_env_classes_run_through_the_managers(cls_name, pool):
    """EnvWrapper -> CUDAFunctionManager name lookup -> kernel, with the reference's own
    positional argument lists, incl. reset pools and the done-masked reset."""
    from warp_drive_b200.env_wrapper import EnvWrapper
    from warp_drive_b200.envs.single_agent import classic_control as cc
    from warp_drive_b200.training.utils.data_loader import create_and_push_data_placeholders

    env = getattr(cc, f"CUDAClassicControl{cls_name}Env")(
        episode_length=25, env_backend="b200", reset_pool_size=pool, seed=11)
    n_envs = 64
    wrapper = EnvWrapper(env, num_envs=n_envs, env_backend="b200")
    wrapper.reset_all_envs()
    dm = wrapper.cuda_data_manager
    continuous = cls_name in ("ContinuousMountainCar", "Pendulum")
    create_and_push_data_placeholders(env_wrapper=wrapper, action_sampler=None,
                                      push_data_batch_placeholders=False)
    if pool >= 2:
        wrapper.init_reset_pool(seed=5)
        assert dm.get_reset_pool("state") == "state_reset_pool"
    actions = dm.data_on_device_via_torch("sampled_actions")
    rs = np.random.RandomState(3)
    saw_done = False
    for t in range(60):
        if continuous:
            actions[:] = torch.from_numpy(rs.uniform(-2, 2, (n_envs, 1, 1)).astype(np.float32)).cuda()
        else:
            actions[:] = torch.from_numpy(rs.randint(0, 3, (n_envs, 1, 1)).astype(np.int32)).cuda()
        wrapper.step_all_envs()
        done = dm.data_on_device_via_torch("_done_")
        saw_done |= bool(done.any().item())
        obs = dm.data_on_device_via_torch("observations")
        assert torch.isfinite(obs).all()
        wrapper.reset_only_done_envs()
        ts = dm.data_on_device_via_torch("_timestep_")
        assert int(ts.max().item()) <= 25
    assert saw_done
