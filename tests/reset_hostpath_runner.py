"""Resets every UNMODIFIED reference scenario file through the device-reset host path (the stand-in
of tests/test_reset_host_path.py) and prints one JSON report.  A process of its own: the scenario
files import ``vmas``, which has to be this package's alias, not the reference."""
import json
import os
import sys
import traceback

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import vectorizedmultiagentsimulator_b200 as b200  # noqa: E402
from dropin_runner import scenario_file  # noqa: E402
from refutil import scenario_files  # noqa: E402
from test_reset_host_path import HostPathBackend  # noqa: E402
from vectorizedmultiagentsimulator_b200 import scenarios  # noqa: E402
from vectorizedmultiagentsimulator_b200.simulator.core import World  # noqa: E402

World._backend_factory = staticmethod(lambda world: HostPathBackend(world))
World.uses_device_reset = property(lambda self: True)

report = {}
for name in scenario_files():
    try:
        env = b200.make_env(scenarios.load(scenario_file(name)).Scenario(), num_envs=5, device="cpu", seed=0)
        env.step(env.get_random_actions())
        env.reset_at(3)
        for agent in env.world.agents:  # what Agent._reset clears besides the slab rows
            if agent.action.u is not None:
                assert not agent.action.u[3].any(), "action.u of the reset env"
            state = getattr(agent.dynamics, "drone_state", None)
            if state is not None:
                assert not state[3].any() and state[0].any(), "dynamics state of the reset env"
        env.step(env.get_random_actions())
        env.reset()
        report[name] = dict(
            spawn_failures=env.world.spawn_failures(),
            reset_count=env.world.reset_count.tolist(),
            spawn_calls=len(env.world._get_backend()._native.calls),
        )
    except Exception as err:  # noqa: BLE001
        report[name] = dict(error="".join(traceback.format_exception_only(type(err), err)).strip()[:400])
print(json.dumps(report))
