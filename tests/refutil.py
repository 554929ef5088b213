"""Test helpers to run the UNMODIFIED reference: the original VMAS project, from a checkout named by
``VMAS_REF`` or else as ``__graft_entry__.build`` compiled it into ``oracle/_ref`` (oracle/build_ref.py)."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE_DIR = os.environ.get("VMAS_REF") or os.path.join(os.path.dirname(HERE), "oracle", "_ref")


def have_reference():
    return os.path.isdir(os.path.join(REFERENCE_DIR, "vmas"))


def scenario_files():
    """{name: path} of every scenario file of the reference (``.py`` in a checkout, ``.pyc`` in oracle/_ref)."""
    out = {}
    for dirpath, _, files in os.walk(os.path.join(REFERENCE_DIR, "vmas", "scenarios")):
        for f in files:
            stem, ext = os.path.splitext(f)
            if ext in (".py", ".pyc") and stem != "__init__" and "__pycache__" not in dirpath:
                out.setdefault(stem, os.path.join(dirpath, f))
    return dict(sorted(out.items()))


def import_reference():
    """Imports the reference's ``vmas`` with the test-only ``gym`` stub on the path."""
    if not have_reference():
        raise RuntimeError("set VMAS_REF to a checkout of the original VMAS project, or build oracle/_ref")
    stubs = os.path.join(HERE, "_stubs")
    for p in (REFERENCE_DIR, stubs):
        if p not in sys.path:
            sys.path.insert(0, p)
    import vmas  # noqa: E402

    assert os.path.abspath(vmas.__file__).startswith(os.path.abspath(REFERENCE_DIR)), vmas.__file__
    return vmas


def world_state(world):
    """Reference (or this package's) world -> slab-layout tensors."""
    ents = world.entities
    agents = world.agents
    return dict(
        pos=torch.stack([e.state.pos for e in ents], 1).clone(),
        vel=torch.stack([e.state.vel for e in ents], 1).clone(),
        rot=torch.cat([e.state.rot for e in ents], 1).clone(),
        ang_vel=torch.cat([e.state.ang_vel for e in ents], 1).clone(),
        force=torch.stack([a.state.force for a in agents], 1).clone(),
        torque=torch.cat([a.state.torque for a in agents], 1).clone(),
    )


def per_env_fixed_rotations(world, desc):
    """item index -> [B,1] tensor for joints whose fixed rotation is a tensor."""
    idx = {id(e): i for i, e in enumerate(world.entities)}
    out = {}
    for c in world._joints.values():
        if isinstance(c.fixed_rotation, (int, float)):
            continue
        for k, it in enumerate(desc.items):
            if it["kind"] == 0 and it["a"] == idx[id(c.entity_a)] and it["b"] == idx[id(c.entity_b)]:
                out[k] = c.fixed_rotation.clone()
    return out


def pre_step(env, actions):
    """Everything ``Environment.step`` does before ``world.step()`` (ref environment.py:386-394)."""
    for i, agent in enumerate(env.agents):
        env._set_action(actions[i], agent)
    for agent in env.world.agents:
        env.scenario.env_process_action(agent)
    env.scenario.pre_step()


def post_step(env):
    env.scenario.post_step()
    env.steps += 1
    return env._get_from_scenario(get_observations=True, get_infos=True, get_rewards=True, get_dones=True)
