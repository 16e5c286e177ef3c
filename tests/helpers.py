"""Shared helpers for the parity tests (state construction from golden fixtures)."""
import hashlib
import os

import numpy as np

REF_KERNELS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                  "ref_kernels.npz")


def fingerprint(a, bitwise=False):
    """32-bit fingerprint of an array's bytes in C order (torch tensors are copied to the
    host).  Equal arrays give equal fingerprints; a different array matches by chance with
    probability 2**-32.  Unless `bitwise`, -0.0 counts as +0.0, as in torch.equal."""
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f" and not bitwise:
        a = a + a.dtype.type(0)          # -0.0 + 0.0 == +0.0; every other value unchanged
    digest = hashlib.blake2b(a.tobytes(), digest_size=4).digest()
    return np.uint32(int.from_bytes(digest, "little"))


def row_fingerprints(a, bitwise=False):
    """fingerprint() of every row (leading index) of `a`."""
    return np.array([fingerprint(r, bitwise) for r in a], np.uint32)


class RefTrace:
    """What the reference's own kernels computed in one parity case, step by step, as
    fingerprints (tests/golden/ref_kernels.npz, written by
    tests/golden/make_ref_kernel_golden.py).  The full outputs are too large to store, and
    the comparisons against the reference are bit-exact, so a fingerprint is all they need.
    Entry `<case>.<key>` holds one fingerprint per step, or one per row and step.
    `bitwise`: as the case was recorded (see fingerprint())."""

    _data = None

    def __init__(self, case, bitwise=False):
        if RefTrace._data is None:
            RefTrace._data = dict(np.load(REF_KERNELS_GOLDEN, allow_pickle=False))
        self.case, self.bitwise = case, bitwise
        assert any(k.startswith(case + ".") for k in RefTrace._data), case

    def _entry(self, key):
        return RefTrace._data[f"{self.case}.{key}"]

    def steps(self, key):
        return len(self._entry(key))

    def same(self, t, key, ours):
        """`ours` equals the reference's `key` at step t."""
        return fingerprint(ours, self.bitwise) == self._entry(key)[t]

    def same_rows(self, t, key, ours):
        """Per row of `ours`: equal to that row of the reference's `key` at step t."""
        return row_fingerprints(ours, self.bitwise) == self._entry(key)[t]


def tc_cfg_from_fixture(fx):
    """Per-env constants of a tag_continuous fixture, typed like the device arrays."""
    cfg = {
        "agent_types": fx["init__agent_types"].astype(np.int32),
        "acceleration_actions": fx["init__acceleration_actions"].astype(np.float32),
        "turn_actions": fx["init__turn_actions"].astype(np.float32),
        "skill_levels": fx["init__skill_levels"].astype(np.float32),
        "step_rewards": fx["init__step_rewards"].astype(np.float32),
        "episode_length": int(fx["episode_length"]),
    }
    for key in ("grid_length", "edge_hit_penalty", "max_speed",
                "distance_margin_for_reward", "tag_reward_for_tagger",
                "tag_penalty_for_runner", "end_of_game_reward_for_runner"):
        cfg[key] = np.float32(fx[f"init__{key}"])
    for key in ("num_other_agents_observed", "use_full_observation",
                "runner_exits_game_after_tagged"):
        cfg[key] = int(fx[f"init__{key}"])
    return cfg


def tc_state_from_fixture(fx, n_envs):
    """Initial state replicated over n_envs (what EnvWrapper.reset_all_envs pushes)."""
    N = fx["init__loc_x"].shape[0]
    K = int(fx["init__num_other_agents_observed"])

    def rep(a, dtype):
        a = np.asarray(a).astype(dtype)
        return np.ascontiguousarray(np.broadcast_to(a, (n_envs,) + a.shape)).copy()

    st = {
        "loc_x": rep(fx["init__loc_x"], np.float32),
        "loc_y": rep(fx["init__loc_y"], np.float32),
        "speed": rep(fx["init__speed"], np.float32),
        "direction": rep(fx["init__direction"], np.float32),
        "acceleration": rep(fx["init__acceleration"], np.float32),
        "edge_hit_reward_penalty": rep(fx["init__edge_hit_reward_penalty"], np.float32),
        "still_in_the_game": rep(fx["init__still_in_the_game"], np.int32),
        "num_runners": np.full(n_envs, int(fx["init__num_runners"]), np.int32),
        "nearest_neighbor_ids": np.zeros((n_envs, N, K), np.int32),
        "_done_": np.zeros(n_envs, np.int32),
        "_timestep_": np.zeros(n_envs, np.int32),
    }
    return st


def copy_state(st):
    return {k: v.copy() for k, v in st.items()}


def close(a, b, tol=1e-5):
    """abs-or-rel closeness (the reference's own comparison rule, tightened from 1 %)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) <= tol * np.maximum(1.0, np.maximum(np.abs(a), np.abs(b)))
