"""Generates the golden fixtures under tests/golden/ from the UNMODIFIED reference.

Run with ``VMAS_REF`` set to a checkout of the original VMAS project:

    VMAS_REF=/path/to/VectorizedMultiAgentSimulator python tests/make_golden.py

For every scenario below the reference is rolled out on CPU with seeded random actions and,
per step, the exact inputs of ``World.step`` (state slab incl. the processed action forces,
per-env joint rotations) and its outputs are recorded, together with the world description
(``plan.describe_world`` of the *reference* world), LIDAR measurements and a sample of
distance / overlap queries.  ``tests/golden/reference/`` holds, in addition, what the reference
returned in the comparisons of tests/test_env_vs_reference.py, tests/test_oracle_vs_reference.py and
tests/test_reset_oracle.py, so that those tests run without the reference.
"""
import itertools
import os
import random
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from refutil import import_reference, per_env_fixed_rotations, post_step, pre_step, world_state  # noqa: E402

from vectorizedmultiagentsimulator_b200.simulator import plan as P  # noqa: E402

# name, kwargs, num_envs, steps
CASES = [
    ("balance", dict(n_agents=4), 64, 100),  # BASELINE.json configs[0] (PR1 reference case)
    ("transport", dict(n_agents=4), 32, 25),
    ("navigation", dict(n_agents=8), 32, 25),
    ("flocking", dict(n_agents=5), 32, 25),
    ("pollock", dict(lidar=True), 8, 12),
    ("waterfall", dict(), 16, 20),
    ("reverse_transport", dict(), 16, 20),
    ("joint_passage", dict(), 16, 20),
    ("multi_give_way", dict(), 16, 20),
    ("give_way", dict(), 16, 20),
    ("wheel", dict(), 16, 20),
    ("dropout", dict(), 16, 15),
    ("wind_flocking", dict(), 16, 15),  # per-env gravity tensors (Entity.gravity as [B, 2])
    ("football", dict(), 8, 10),
    ("passage", dict(), 16, 15),
    # crafted worlds (tests/crafted.py) for the branches no reference scenario takes
    ("crafted_clamps", dict(), 33, 12),  # max_f / f_range / max_t / t_range, angular + linear friction
    ("crafted_joints_apart", dict(), 16, 4),  # joints with anchors clearly apart (strict-tolerance joint test)
    ("crafted_lonely", dict(), 1, 6),  # batch_dim = 1, no work item
    ("crafted_crowd", dict(), 4, 6),  # 70 entities
]


def record(vmas, name, kwargs, num_envs, steps):
    scenario = name
    if name.startswith("crafted_"):
        import crafted

        scenario = crafted.make_scenario("vmas", name[len("crafted_"):])
    env = vmas.make_env(scenario, num_envs=num_envs, device="cpu", seed=0, **kwargs)
    world = env.world
    desc = P.describe_world(world)
    fix = dict(name=name, kwargs=kwargs, desc=desc.to_json(), steps=[], lidar=[], queries=[])
    gen = torch.Generator().manual_seed(1)
    idx = {id(e): i for i, e in enumerate(world.entities)}
    prev_out = None
    for t in range(steps):
        actions = [
            (torch.rand(num_envs, a.action_size, generator=gen) * 2 - 1) * a.action.u_range_tensor
            for a in env.agents
        ]
        pre_step(env, actions)
        state_in = world_state(world)
        fixed = per_env_fixed_rotations(world, desc)
        gravity = {
            i: e.gravity.clone() for i, e in enumerate(world.entities) if desc.entities[i].get("gravity_per_env")
        }
        world.step()
        state_out = world_state(world)
        entry = dict(force=state_in["force"], torque=state_in["torque"], out=state_out)
        same = prev_out is not None and all(
            torch.equal(state_in[k], prev_out[k]) for k in ("pos", "vel", "rot", "ang_vel")
        )
        if not same:
            entry["state_in"] = {k: state_in[k] for k in ("pos", "vel", "rot", "ang_vel")}
        if fixed:
            entry["fixed_rot"] = fixed
        if gravity:
            entry["ent_gravity"] = gravity
        fix["steps"].append(entry)
        prev_out = state_out
        obs, rews, dones, infos = post_step(env)
        if t < 3 or t == steps - 1:
            entry["obs"] = [o.clone() for o in obs]
            entry["rews"] = [r.clone() for r in rews]
            entry["dones"] = dones.clone()
        # LIDAR: every sensor of every agent on the post-step state
        if t % 3 == 0:
            for a in world.agents:
                for s in a.sensors:
                    targets = [i for i, e in enumerate(world.entities) if e is not a and s.entity_filter(e)]
                    fix["lidar"].append(
                        dict(
                            step=t,
                            src=idx[id(a)],
                            targets=targets,
                            angles=s._angles.clone(),
                            max_range=float(s._max_range),
                            out=s.measure().clone(),
                        )
                    )
    # distance / overlap queries on the final state
    ents = world.entities
    rnd = random.Random(0)
    pairs = list(itertools.permutations(range(len(ents)), 2))
    rnd.shuffle(pairs)
    final = world_state(world)
    fix["final_state"] = final
    for a, b in pairs[:60]:
        pt = torch.randn(num_envs, 2, generator=gen)
        fix["queries"].append(
            dict(
                a=a,
                b=b,
                distance=world.get_distance(ents[a], ents[b]).clone(),
                overlap=world.is_overlapping(ents[a], ents[b]).clone(),
                point=pt,
                point_distance=world.get_distance_from_point(ents[a], pt).clone(),
            )
        )
    return fix


def _clone(x):
    """A step's results (tensors in lists / tuples / dicts), copied."""
    if isinstance(x, dict):
        return {k: _clone(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x)(_clone(v) for v in x)
    return x.clone()


# -- the reference's side of tests/test_env_vs_reference.py: same seeds, actions and call order --------------
def record_env_rollout(vmas, name, kwargs, continuous):
    n_envs, steps = 12, 12
    ref = vmas.make_env(name, num_envs=n_envs, device="cpu", seed=3, continuous_actions=continuous, **kwargs)
    rec = dict(n_envs=n_envs, reset=_clone(ref.reset(seed=5)), actions=[], steps=[])
    gen = torch.Generator().manual_seed(11)
    for t in range(steps):
        if continuous:
            actions = [
                (torch.rand(n_envs, a.action_size, generator=gen) * 2 - 1) * a.action.u_range_tensor for a in ref.agents
            ]
        else:
            actions = [torch.randint(0, 9, (n_envs, 1), generator=gen) for _ in ref.agents]
        rec["actions"].append([a.clone() for a in actions])
        rec["steps"].append(_clone(ref.step([a.clone() for a in actions])))
        if t == 5:  # partial reset mid-rollout (ref tests/test_vmas.py:249-262)
            rec["reset_at"] = _clone(ref.reset_at(2))
    return rec


def record_stock_style(vmas):
    import stock_style

    n_envs = 10
    ref = vmas.make_env(stock_style.make_scenario("vmas"), num_envs=n_envs, device="cpu", seed=1, n_agents=3)
    rec = dict(n_envs=n_envs, actions=[], steps=[])
    gen = torch.Generator().manual_seed(2)
    for t in range(10):
        actions = [(torch.rand(n_envs, a.action_size, generator=gen) * 2 - 1) for a in ref.agents]
        rec["actions"].append([a.clone() for a in actions])
        rec["steps"].append(_clone(ref.step([a.clone() for a in actions])))
        if t == 4:
            rec["reset_at"] = _clone(ref.reset_at(3))
    return rec


def record_dynamics_zoo(vmas):
    import crafted

    n_envs = 9
    ref = vmas.make_env(crafted.make_scenario("vmas", "dynamics_zoo"), num_envs=n_envs, device="cpu", seed=2)
    rec = dict(n_envs=n_envs, actions=[], obs=[], force=[], torque=[])
    gen = torch.Generator().manual_seed(3)
    for t in range(8):
        actions = [(torch.rand(n_envs, a.action_size, generator=gen) * 2 - 1) * a.action.u_range_tensor for a in ref.agents]
        rec["actions"].append([a.clone() for a in actions])
        rec["obs"].append(_clone(ref.step([a.clone() for a in actions])[0]))
        rec["force"].append([a.state.force.clone() for a in ref.agents])
        rec["torque"].append([a.state.torque.clone() for a in ref.agents])
    return rec


def record_spaces(vmas):
    ref = vmas.make_env("balance", num_envs=4, device="cpu", seed=0, n_agents=3)
    rec = dict(n_action_spaces=len(ref.action_space.spaces), obs_shape=tuple(ref.observation_space.spaces[0].shape))
    ref.seed(1)
    rec["random_actions"] = _clone(ref.get_random_actions())
    return rec


# -- the reference's side of tests/test_oracle_vs_reference.py: what its World.step received and returned ---
def record_oracle_case(vmas, name, kwargs, num_envs, steps, seed):
    scenario = name
    if name.startswith("crafted_"):
        import crafted

        scenario = crafted.make_scenario("vmas", name[len("crafted_"):], seed=1000 + seed)
    env = vmas.make_env(scenario, num_envs=num_envs, device="cpu", seed=seed, **kwargs)
    world = env.world
    desc = P.describe_world(world)  # the plan compiler reads the reference's own objects
    ents = world.entities
    # bit for bit only on the SIMD level of torch's CPU kernels it was recorded with
    rec = dict(desc=desc.to_json(), steps=[], queries=[], cpu_capability=torch.backends.cpu.get_cpu_capability())
    gen = torch.Generator().manual_seed(100 + seed)
    prev_out = None
    for t in range(steps):
        actions = [
            (torch.rand(num_envs, a.action_size, generator=gen) * 2 - 1) * a.action.u_range_tensor for a in env.agents
        ]
        pre_step(env, actions)
        state_in = world_state(world)
        entry = dict(force=state_in["force"], torque=state_in["torque"], lidar=[])
        # (the format of record(): the state is stored only where it is not the previous step's result)
        if prev_out is None or not all(torch.equal(state_in[k], prev_out[k]) for k in ("pos", "vel", "rot", "ang_vel")):
            entry["state_in"] = {k: state_in[k] for k in ("pos", "vel", "rot", "ang_vel")}
        fixed = per_env_fixed_rotations(world, desc)
        if fixed:
            entry["fixed_rot"] = fixed
        gravity = {i: e.gravity.clone() for i, e in enumerate(ents) if desc.entities[i].get("gravity_per_env")}
        if gravity:
            entry["ent_gravity"] = gravity
        world.step()
        entry["out"] = prev_out = world_state(world)
        post_step(env)
        if t % 4 == 0:  # LIDAR of every sensor on the post-step state
            for i, a in enumerate(ents):
                for s in getattr(a, "sensors", None) or []:
                    targets = [j for j, e in enumerate(ents) if e is not a and s.entity_filter(e)]
                    entry["lidar"].append(
                        dict(src=i, targets=targets, angles=s._angles.clone(), max_range=float(s._max_range),
                             out=s.measure().clone())
                    )
        rec["steps"].append(entry)
    # distance / overlap queries on the final state
    rec["final_state"] = world_state(world)
    for a, b in list(itertools.permutations(range(len(ents)), 2))[:40]:
        point = torch.randn(num_envs, 2, generator=gen)
        rec["queries"].append(
            dict(
                a=a, b=b, distance=world.get_distance(ents[a], ents[b]).clone(),
                overlap=world.is_overlapping(ents[a], ents[b]).clone(), point=point,
                point_distance=world.get_distance_from_point(ents[a], point).clone(),
            )
        )
    return rec


# -- the reference's side of tests/test_reset_oracle.py::test_spawn_distribution_matches_reference_sampler -
def record_spawn_sampler(vmas):
    from vmas.simulator.core import Landmark, Sphere, World
    from vmas.simulator.utils import ScenarioUtils

    B, n = 4000, 4
    torch.manual_seed(0)
    world = World(B, "cpu")
    ents = [Landmark(name=f"l{i}", shape=Sphere(0.05)) for i in range(n)]
    for e in ents:
        world.add_landmark(e)
    occ = torch.tensor([[[0.0, 0.0]]]).expand(B, 1, 2)
    ScenarioUtils.spawn_entities_randomly(ents, world, None, 0.5, (-1, 1), (-1, 1), occupied_positions=occ)
    return dict(pos=torch.stack([e.state.pos for e in ents], dim=1).clone())


def reference_records(vmas):
    """(file stem under tests/golden/reference, recorder) of every stored reference comparison."""
    import test_env_vs_reference as E
    import test_oracle_vs_reference as O

    out = []
    for name, kwargs in E.CASES:
        for continuous in (True, False):
            out.append((E.rollout_record(name, continuous), lambda v, a=(name, kwargs, continuous): record_env_rollout(v, *a)))
    out += [("env_stock_style", record_stock_style), ("env_dynamics_zoo", record_dynamics_zoo), ("env_spaces", record_spaces)]
    for i, case in enumerate(O.CASES):
        out.append((O.record_name(i, case), lambda v, c=case: record_oracle_case(v, *c)))
    out.append(("spawn_sampler", record_spawn_sampler))
    return out


def main():
    vmas = import_reference()
    out_dir = os.path.join(HERE, "golden")
    os.makedirs(out_dir, exist_ok=True)
    for name, kwargs, num_envs, steps in CASES:
        path = os.path.join(out_dir, f"{name}.pt")
        if os.path.exists(path) and "--all" not in sys.argv:
            continue  # fixtures are append-only; pass --all to regenerate everything
        fix = record(vmas, name, kwargs, num_envs, steps)
        torch.save(fix, path)
        print(f"{name:20s} B={num_envs:3d} T={steps:3d} lidar={len(fix['lidar']):3d} -> {os.path.getsize(path)/1e6:.2f} MB")
    ref_dir = os.path.join(out_dir, "reference")
    os.makedirs(ref_dir, exist_ok=True)
    for stem, recorder in reference_records(vmas):
        path = os.path.join(ref_dir, f"{stem}.pt")
        if os.path.exists(path) and "--all" not in sys.argv:
            continue
        torch.save(recorder(vmas), path)
        print(f"reference/{stem + '.pt':36s} -> {os.path.getsize(path)/1e6:.2f} MB")


if __name__ == "__main__":
    main()
