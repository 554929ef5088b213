"""The CPU oracle against the UNMODIFIED reference, bit for bit.

The reference was rolled out with seeded random actions — other seeds, batch sizes and scenario
arguments than tests/test_oracle_golden.py uses — and at every step what its ``World.step`` received
and returned was recorded (tests/make_golden.py -> tests/golden/reference/oracle_*.pt).  The oracle
receives exactly those inputs (teacher forcing) and must return what the reference returned: bit for
bit for the physics, the LIDAR readings and the distance / overlap queries.  This is the pin the
``oracle/`` docstrings refer to.
"""
import pytest
import torch

from golden_util import load_reference_record, teacher_forced_steps
from oracle import queries as Q
from oracle import world_step as WS
from vectorizedmultiagentsimulator_b200.simulator import plan as P

# name, kwargs, num_envs, steps, seed
CASES = [
    ("balance", dict(n_agents=3), 20, 30, 3),
    ("balance", dict(n_agents=5, package_mass=7), 9, 20, 4),
    ("transport", dict(n_agents=3, n_packages=2), 12, 20, 5),
    ("navigation", dict(n_agents=5), 12, 20, 6),
    ("flocking", dict(n_agents=4), 12, 15, 7),
    ("pollock", dict(lidar=True), 4, 6, 8),
    ("waterfall", dict(), 8, 12, 9),
    ("reverse_transport", dict(), 8, 12, 10),
    ("joint_passage", dict(), 6, 10, 11),
    ("wheel", dict(), 8, 12, 12),
    ("wind_flocking", dict(), 8, 10, 13),
    # crafted worlds (tests/crafted.py): action clamps, angular friction, joints with anchors apart,
    # a one-env batch without work items, 70 entities — branches no reference scenario takes
    ("crafted_clamps", dict(), 21, 15, 14),
    ("crafted_joints_apart", dict(), 10, 5, 15),
    ("crafted_lonely", dict(), 1, 5, 16),
    ("crafted_crowd", dict(), 3, 5, 17),
]
STATE = ("pos", "vel", "rot", "ang_vel")
TOL, RTOL = 2e-6, 1e-4


def record_name(i, case):
    return f"oracle_{case[0]}-{i}"


@pytest.mark.parametrize("name,kwargs,num_envs,steps,seed", CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(CASES)])
def test_oracle_equals_live_reference_bit_for_bit(name, kwargs, num_envs, steps, seed):
    i = CASES.index((name, kwargs, num_envs, steps, seed))
    ref = load_reference_record(record_name(i, CASES[i]))
    desc = P.WorldDescription.from_json(ref["desc"])
    tables = P.build_tables(desc)
    assert desc.batch_dim == num_envs and len(ref["steps"]) == steps
    # bit for bit where torch's CPU kernels run at the SIMD level the reference was recorded at; another level
    # rounds some vectorised ops differently in the last place, which the stiff joint forces amplify: there
    # the results have to agree to 1e-4 relative (2e-6 absolute near zero)
    exact = ref["cpu_capability"] == torch.backends.cpu.get_cpu_capability()

    def check(got, want, what):
        if exact or got.dtype == torch.bool:
            assert torch.equal(got, want), f"{what}: max |diff| {float((got.float() - want.float()).abs().max())}"
        else:
            bad = (got - want).abs() > TOL + RTOL * want.abs()
            assert not bad.any(), f"{what}: max |diff| {float((got - want).abs().max())}"

    for (t, state, fixed_rot, want), entry in zip(teacher_forced_steps(ref), ref["steps"]):
        WS.world_step(tables, state, fixed_rot=fixed_rot)  # the inputs of the reference's World.step
        for k in STATE:
            check(state[k], want[k], f"{name} step {t}: {k}")
        for ray in entry["lidar"]:  # LIDAR of every sensor on the post-step state (every 4th step)
            got = Q.cast_rays(
                tables, want["pos"], want["rot"], ray["src"], ray["targets"],
                ray["angles"] + want["rot"][:, ray["src"]].unsqueeze(-1), ray["max_range"],
            )
            check(got, ray["out"], f"{name} step {t}: lidar of entity {ray['src']}")
    # distance / overlap queries on the final state
    final = ref["final_state"]
    for q in ref["queries"]:
        a, b = q["a"], q["b"]
        check(Q.pair_distance(tables, final["pos"], final["rot"], a, b), q["distance"], f"{name} distance {a}-{b}")
        check(Q.pair_overlap(tables, final["pos"], final["rot"], a, b), q["overlap"], f"{name} overlap {a}-{b}")
        check(
            Q.distance_from_point(tables, final["pos"], final["rot"], a, q["point"]), q["point_distance"],
            f"{name} distance of {a} from a point",
        )
