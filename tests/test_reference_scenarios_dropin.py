"""Drop-in check: the reference's own, UNMODIFIED scenario files run on this package.

Every scenario file of the reference checkout is loaded through the ``vmas`` import alias
(``compat.install_vmas_alias``) into this package's ``make_env`` on the CPU oracle backend and
rolled out next to the reference itself (separate processes, same seed, ``get_random_actions``):
observations, rewards and dones must be identical.  This pins the host layer — object model,
``Environment`` action decoding for continuous / comm actions, dynamics models, velocity
controller, joints, sensors, reset protocol — against every client the reference ships.
"""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.reference

HERE = os.path.dirname(os.path.abspath(__file__))


def all_reference_scenarios():
    from refutil import scenario_files

    return list(scenario_files())


@pytest.mark.timeout(1500)
def test_every_reference_scenario_file_runs_unmodified_and_matches(tmp_path):
    names = all_reference_scenarios()
    assert len(names) >= 40
    outs = {}
    for which in ("ref", "b200"):
        out = os.path.join(str(tmp_path), which + ".pt")
        subprocess.run(
            [sys.executable, os.path.join(HERE, "dropin_runner.py"), which, out] + names,
            check=True,
            capture_output=True,
            timeout=1200,
        )
        outs[which] = torch.load(out)
    failures = []
    for name in names:
        ref, got = outs["ref"][name], outs["b200"][name]
        assert not isinstance(ref, str), f"the reference itself failed on {name}: {ref}"
        if isinstance(got, str):
            failures.append(f"{name}: {got}")
            continue
        for t, ((o1, r1, d1), (o2, r2, d2)) in enumerate(zip(ref, got)):
            if o1.shape != o2.shape or not torch.equal(d1, d2):
                failures.append(f"{name}: step {t} shape/done mismatch")
                break
            err = max(float((o1 - o2).abs().max()), float((r1 - r2).abs().max()))
            if err > 1e-6:
                failures.append(f"{name}: step {t} max |diff| {err:.2e}")
                break
    assert not failures, "\n".join(failures)
