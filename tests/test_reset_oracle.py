"""CPU checks of the episode-reset path (SURVEY §8(f)-4).

* the numpy oracle (``oracle/reset.py``): Philox4x32-10 against the published known-answer vectors,
  the sampler's invariants, and its distribution against the reference's own
  ``ScenarioUtils.spawn_entities_randomly`` (a different random stream, the same law);
* the host logic: ``Environment.reset_at`` with an int and with a bool mask on the CPU oracle backend;
* the ctypes mirror of ``VmasSpawn`` has the layout the C compiler gives the header's struct.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import reset as R
from oracle.backend import use_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# -- Philox ------------------------------------------------------------------------------------
# Random123 kat_vectors, philox4x32-10: (counter, key) -> output
PHILOX_KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    (
        (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344),
        (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1),
    ),
]


@pytest.mark.parametrize("counter,key,want", PHILOX_KAT)
def test_philox_known_answers(counter, key, want):
    got = R.philox4x32_10(counter, key)
    assert tuple(int(x) for x in got) == want


def test_philox_is_elementwise():
    c0 = np.arange(100, dtype=np.uint32)
    block = R.philox4x32_10((c0, 7, 9, 3), (11, 13))
    for i in (0, 17, 99):
        one = R.philox4x32_10((i, 7, 9, 3), (11, 13))
        assert [int(b[i]) for b in block] == [int(o) for o in one]


# -- sampler invariants --------------------------------------------------------------------------
def _spawn(B=256, E=7, **kw):
    pos = np.zeros((B, E, 2), np.float32)
    pos[:, 5] = (0.25, -0.25)
    pos[:, 6] = (-0.5, 0.5)
    args = dict(min_dist=0.3, x_bounds=(-1.0, 1.0), y_bounds=(-0.75, 0.75), seed=42, occupied_entities=(5, 6))
    args.update(kw)
    out, exhausted = R.spawn_entities(pos, [0, 1, 2, 3, -1], **args)
    return pos, out, exhausted


def test_spawn_respects_bounds_and_distances():
    extra = np.random.default_rng(0).uniform(-1, 1, (256, 2, 2)).astype(np.float32)
    pos, out, exhausted = _spawn(occupied=extra)
    assert exhausted == 0
    assert out[..., 0].min() >= -1 and out[..., 0].max() <= 1
    assert out[..., 1].min() >= -0.75 and out[..., 1].max() <= 0.75
    assert np.array_equal(pos[:, :4], out[:, :4])  # slab rows == returned draws
    pts = np.concatenate([out, pos[:, 5:7], extra], axis=1)
    d = np.linalg.norm(pts[:, :, None] - pts[:, None], axis=-1)
    for i in range(out.shape[1]):  # every drawn point against everything else
        for j in range(pts.shape[1]):
            if i != j:
                assert (d[:, i, j] >= 0.3 - 1e-6).all(), (i, j)


def test_spawn_is_deterministic_and_seed_sensitive():
    a = _spawn()[1]
    assert np.array_equal(a, _spawn()[1])
    assert not np.array_equal(a, _spawn(seed=43)[1])
    assert not np.array_equal(a, _spawn(stream_id=1)[1])
    rc = np.ones(256, np.int32)
    assert not np.array_equal(a, _spawn(reset_count=rc)[1])


def test_masked_spawn_equals_one_env_at_a_time():
    """The property the counter layout buys: an env's draws do not depend on which other envs are
    reset in the same call."""
    mask = np.zeros(256, bool)
    mask[[3, 77, 200]] = True
    pos_m, out_m, _ = _spawn(env_mask=mask)
    full = _spawn()[1]
    assert np.array_equal(out_m[mask], full[mask])
    assert not out_m[~mask].any() and not pos_m[~mask][:, :4].any()  # unselected envs untouched
    for i in (3, 77, 200):
        _, out_i, _ = _spawn(env_index=i)
        assert np.array_equal(out_i[i], full[i])


def test_env_offset_makes_shards_draw_what_the_whole_job_draws():
    full = _spawn()[1]
    lo = 100
    pos = np.zeros((56, 7, 2), np.float32)
    pos[:, 5] = (0.25, -0.25)
    pos[:, 6] = (-0.5, 0.5)
    out, _ = R.spawn_entities(
        pos, [0, 1, 2, 3, -1], min_dist=0.3, x_bounds=(-1.0, 1.0), y_bounds=(-0.75, 0.75), seed=42,
        occupied_entities=(5, 6), env_offset=lo,
    )
    assert np.array_equal(out, full[lo : lo + 56])


def test_exhaustion_is_reported():
    # 4 points that keep 1.5 apart cannot fit in a unit square
    pos = np.zeros((8, 4, 2), np.float32)
    _, exhausted = R.spawn_entities(
        pos, [0, 1, 2, 3], min_dist=1.5, x_bounds=(0, 1), y_bounds=(0, 1), seed=1, max_tries=64
    )
    assert exhausted == 8


def test_reset_state_zeroes_selected_rows():
    rng = np.random.default_rng(1)
    state = {k: rng.normal(size=(6, 3, 2)).astype(np.float32) for k in ("pos", "vel")}
    keep = {k: v.copy() for k, v in state.items()}
    count = np.zeros(6, np.int32)
    mask = np.array([0, 1, 0, 0, 1, 0], bool)
    R.reset_state(state, count, env_mask=mask)
    for k in state:
        assert not state[k][mask].any() and np.array_equal(state[k][~mask], keep[k][~mask])
    assert count.tolist() == [0, 1, 0, 0, 1, 0]
    R.reset_state(state, count, env_index=2)
    assert count.tolist() == [0, 1, 1, 0, 1, 0] and not state["pos"][2].any()


# -- same law as the reference's sampler ----------------------------------------------------------
def test_spawn_distribution_matches_reference_sampler():
    """4 spheres, min_dist 0.5 in [-1, 1]^2 around an occupied origin, 4000 envs: the reference's
    ``ScenarioUtils.spawn_entities_randomly`` (its draws stored by tests/make_golden.py) against this sampler."""
    from scipy.stats import ks_2samp

    from golden_util import load_reference_record

    ref = load_reference_record("spawn_sampler")["pos"].numpy()
    B, n = ref.shape[:2]
    assert (B, n) == (4000, 4)

    pos = np.zeros((B, n, 2), np.float32)
    R.spawn_entities(
        pos, list(range(n)), min_dist=0.5, x_bounds=(-1, 1), y_bounds=(-1, 1), seed=9,
        occupied=np.zeros((1, 1, 2), np.float32),
    )

    def features(p):
        d01 = np.linalg.norm(p[:, 0] - p[:, 1], axis=-1)
        d_last = np.linalg.norm(p[:, -1, None] - p[:, :-1], axis=-1).min(-1)
        r_last = np.linalg.norm(p[:, -1], axis=-1)
        return [p[:, 0, 0], p[:, -1, 1], d01, d_last, r_last]

    for f_ref, f_mine in zip(features(ref), features(pos)):
        assert ks_2samp(f_ref, f_mine).pvalue > 1e-3


# -- host logic: reset_at(int) and reset_at(mask) on the CPU oracle backend -------------------------
CASES = [
    ("balance", dict(n_agents=4)),
    ("transport", dict(n_agents=4)),
    ("navigation", dict(n_agents=4)),
    ("flocking", dict(n_agents=5)),
]


def _state(env):
    return {k: v.clone() for k, v in env.world.slab.state_dict().items()}


@pytest.mark.parametrize("name,kwargs", CASES)
def test_masked_reset_touches_only_flagged_envs(name, kwargs):
    import vectorizedmultiagentsimulator_b200 as b200

    n_envs = 16
    with use_oracle():
        env = b200.make_env(name, num_envs=n_envs, device="cpu", seed=0, **kwargs)
        gen = torch.Generator().manual_seed(0)
        for _ in range(3):
            env.step([torch.rand(n_envs, 2, generator=gen) * 2 - 1 for _ in env.agents])
        before = _state(env)
        steps_before = env.steps.clone()
        mask = torch.zeros(n_envs, dtype=torch.bool)
        mask[[1, 5, 6, 15]] = True
        obs = env.reset_at(mask)
        after = _state(env)
    assert len(obs) == len(env.agents) and all(torch.isfinite(o).all() for o in obs)
    for k in before:
        assert torch.equal(after[k][~mask], before[k][~mask]), f"{name}: {k} of an unflagged env changed"
    assert not torch.equal(after["pos"][mask], before["pos"][mask])
    assert float(after["vel"][mask].abs().max()) == 0.0
    assert torch.equal(env.steps[mask], torch.zeros(4)) and torch.equal(env.steps[~mask], steps_before[~mask])
    assert env.world.reset_count.tolist() == [1 + int(m) for m in mask.tolist()]


def test_masked_reset_is_refused_by_index_only_scenarios():
    import vectorizedmultiagentsimulator_b200 as b200
    from vectorizedmultiagentsimulator_b200.scenarios import balance

    class IndexOnly(balance.Scenario):
        supports_masked_reset = False

    with use_oracle():
        env = b200.make_env(IndexOnly(), num_envs=4, device="cpu", seed=0, n_agents=3)
        with pytest.raises(NotImplementedError):
            env.reset_at(torch.ones(4, dtype=torch.bool))
        with pytest.raises(ValueError):
            env.reset_at(torch.ones(3, dtype=torch.bool))
        env.reset_at(2)  # the reference's form still works


# -- struct layout ----------------------------------------------------------------------------------
def test_spawn_struct_layout_matches_the_header(tmp_path):
    from vectorizedmultiagentsimulator_b200 import _native

    fields = [name for name, *_ in _native.SpawnC._fields_]
    src = tmp_path / "layout.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vmas_b200.h"', "int main(void) {"]
    lines.append('  printf("%zu\\n", sizeof(VmasSpawn));')
    for f in fields:
        lines.append(f'  printf("%zu\\n", offsetof(VmasSpawn, {f}));')
    lines += ["  return 0;", "}"]
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[0] == ctypes.sizeof(_native.SpawnC)
    assert got[1:] == [getattr(_native.SpawnC, f).offset for f in fields]
