"""Runs UNMODIFIED reference scenario files for a few steps and saves obs / rewards / dones.

    python dropin_runner.py ref  OUT.pt name [name ...]   # on the reference itself
    python dropin_runner.py b200 OUT.pt name [name ...]   # on this package (CPU oracle backend),
                                                          # scenario files loaded through the vmas alias
Two processes are needed because both expose a top-level module called ``vmas``.
"""
import os
import sys
import traceback

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import torch  # noqa: E402

from refutil import scenario_files  # noqa: E402

N_ENVS, STEPS = 6, 5


def scenario_file(name):
    """The reference's scenario file ``name`` (source in a checkout, bytecode in oracle/_ref)."""
    path = scenario_files().get(name)
    if path is None:
        raise FileNotFoundError(name)
    return path


def main():
    which, out, names = sys.argv[1], sys.argv[2], sys.argv[3:]
    ctx = None
    if which == "ref":
        from refutil import import_reference

        import importlib

        vmas = import_reference()
        ref_scenarios = importlib.import_module("vmas.scenarios")  # (``vmas.scenarios`` is a list of names)
        # (what the reference's make_env does with a scenario name, from the file itself)
        make = lambda n: vmas.make_env(  # noqa: E731
            ref_scenarios.load(scenario_file(n)).Scenario(), num_envs=N_ENVS, device="cpu", seed=0
        )
    else:
        import vectorizedmultiagentsimulator_b200 as b200
        from oracle.backend import use_oracle
        from vectorizedmultiagentsimulator_b200 import scenarios

        ctx = use_oracle()
        ctx.__enter__()
        # (what make_env does with a path to a scenario file, for source and bytecode files alike)
        make = lambda n: b200.make_env(  # noqa: E731
            scenarios.load(scenario_file(n)).Scenario(), num_envs=N_ENVS, device="cpu", seed=0
        )
    results = {}
    for name in names:
        try:
            env = make(name)
            env.seed(1)
            rollout = []
            for _ in range(STEPS):
                obs, rews, dones, _ = env.step(env.get_random_actions())
                leaves = []
                for o in obs:
                    leaves += list(o.values()) if isinstance(o, dict) else [o]
                rollout.append(
                    (torch.cat([x.reshape(N_ENVS, -1).float() for x in leaves], 1), torch.stack(rews, 1), dones.clone())
                )
            results[name] = rollout
        except Exception as err:  # noqa: BLE001
            results[name] = "ERR: " + "".join(traceback.format_exception_only(type(err), err)).strip()[:400]
    torch.save(results, out)


if __name__ == "__main__":
    main()
