"""The host layer (Environment / World object model / re-written scenarios) against the
UNMODIFIED reference, both on CPU: this package runs on the CPU oracle backend, so any
difference comes from the host code (action decoding, reset draws, obs/reward layout).

What the reference returned for the same seeds and actions is stored under
tests/golden/reference/ (recorded by tests/make_golden.py)."""
import pytest
import torch

from golden_util import load_reference_record
from oracle.backend import use_oracle

CASES = [
    ("balance", dict(n_agents=4)),
    ("transport", dict(n_agents=4)),
    ("navigation", dict(n_agents=8)),
    ("flocking", dict(n_agents=5)),
]


def rollout_record(name, continuous):
    return f"env_rollout_{name}_{'continuous' if continuous else 'discrete'}"


def _flatten(x):
    if isinstance(x, dict):
        return [v for k in sorted(x) for v in _flatten(x[k])]
    if isinstance(x, (list, tuple)):
        return [v for item in x for v in _flatten(item)]
    return [x]


def _assert_same(got, want, what, tol=0.0):
    g, w = _flatten(got), _flatten(want)
    assert len(g) == len(w), what
    for a, b in zip(g, w):
        assert a.shape == b.shape and a.dtype == b.dtype, f"{what}: {a.shape}/{a.dtype} vs {b.shape}/{b.dtype}"
        if a.dtype == torch.bool:
            assert torch.equal(a, b), what
        else:
            assert float((a - b).abs().max()) <= tol, f"{what}: {float((a - b).abs().max())}"


@pytest.mark.parametrize("name,kwargs", CASES)
@pytest.mark.parametrize("continuous", [True, False])
def test_rollout_matches_reference(name, kwargs, continuous):
    import vectorizedmultiagentsimulator_b200 as b200

    ref = load_reference_record(rollout_record(name, continuous))
    n_envs = ref["n_envs"]
    with use_oracle():
        mine = b200.make_env(name, num_envs=n_envs, device="cpu", seed=3, continuous_actions=continuous, **kwargs)
        _assert_same(mine.reset(seed=5), ref["reset"], f"{name} reset obs")
        for t, (actions, want) in enumerate(zip(ref["actions"], ref["steps"])):
            got = mine.step([a.clone() for a in actions])
            for part, label in zip(range(4), ("obs", "rews", "dones", "infos")):
                _assert_same(got[part], want[part], f"{name} step {t} {label}", tol=1e-6)
            if t == 5:  # partial reset mid-rollout (ref tests/test_vmas.py:249-262)
                _assert_same(mine.reset_at(2), ref["reset_at"], f"{name} reset_at obs", tol=1e-6)
    assert len(ref["steps"]) == 12


def test_stock_style_scenario_matches_reference():
    """tests/stock_style.py — per-agent is_overlapping / get_distance / Lidar.measure callbacks as the
    reference's scenario files write them — built from this package's modules, against the roll-out of
    the same scenario built from the reference's: identical (this is the CPU half of the pin;
    tests/test_env_gpu.py steps the same scenario on the CUDA backend against the oracle env)."""
    import stock_style
    import vectorizedmultiagentsimulator_b200 as b200

    ref = load_reference_record("env_stock_style")
    n_envs = ref["n_envs"]
    with use_oracle():
        mine = b200.make_env(stock_style.make_scenario(), num_envs=n_envs, device="cpu", seed=1, n_agents=3)
        for t, (actions, want) in enumerate(zip(ref["actions"], ref["steps"])):
            got = mine.step([a.clone() for a in actions])
            for part, label in zip(range(4), ("obs", "rews", "dones", "infos")):
                _assert_same(got[part], want[part], f"stock_style step {t} {label}", tol=0.0)
            if t == 4:
                _assert_same(mine.reset_at(3), ref["reset_at"], "stock_style reset_at obs", tol=0.0)
    assert len(ref["steps"]) == 10


def test_dynamics_zoo_matches_reference():
    """tests/crafted.py "dynamics_zoo": one agent per action model (differential drive RK4 / Euler,
    kinematic bicycle, drone, forward, rotation, holonomic with rotation, static) — the host-side torch
    formulation of this package against the reference's, bit for bit.  (The CUDA ingest kernel that fuses
    them is checked against this formulation in tests/test_env_gpu.py.)"""
    import crafted
    import vectorizedmultiagentsimulator_b200 as b200

    ref = load_reference_record("env_dynamics_zoo")
    n_envs = ref["n_envs"]
    with use_oracle():
        mine = b200.make_env(
            crafted.make_scenario("vectorizedmultiagentsimulator_b200", "dynamics_zoo"), num_envs=n_envs, device="cpu", seed=2
        )
        for t, actions in enumerate(ref["actions"]):
            got = mine.step([a.clone() for a in actions])
            _assert_same(got[0], ref["obs"][t], f"dynamics_zoo step {t} obs", tol=0.0)
            assert len(mine.agents) == len(ref["force"][t])
            for a_mine, force, torque in zip(mine.agents, ref["force"][t], ref["torque"][t]):
                assert torch.equal(a_mine.state.force, force), f"step {t}: force of {a_mine.name}"
                assert torch.equal(a_mine.state.torque, torque), f"step {t}: torque of {a_mine.name}"
    assert len(ref["actions"]) == 8


def test_spaces_and_random_actions_match_reference():
    import vectorizedmultiagentsimulator_b200 as b200

    ref = load_reference_record("env_spaces")
    with use_oracle():
        mine = b200.make_env("balance", num_envs=4, device="cpu", seed=0, n_agents=3)
    assert len(mine.action_space.spaces) == ref["n_action_spaces"] == 3
    assert tuple(mine.observation_space.spaces[0].shape) == ref["obs_shape"]
    mine.seed(1)
    _assert_same(mine.get_random_actions(), ref["random_actions"], "random actions")


def test_seed_isolation_from_global_rng():
    """Env draws must not disturb the user's global torch RNG (ref tests/test_vmas.py:308-323)."""
    import vectorizedmultiagentsimulator_b200 as b200

    torch.manual_seed(123)
    expected = torch.rand(3)
    torch.manual_seed(123)
    with use_oracle():
        env = b200.make_env("navigation", num_envs=4, device="cpu", seed=0, n_agents=3)
        env.step(env.get_random_actions())
    assert torch.equal(torch.rand(3), expected)
