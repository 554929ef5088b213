"""Loading the golden fixtures produced by tests/make_golden.py."""
import glob
import os

import torch

from vectorizedmultiagentsimulator_b200.simulator import plan as P

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
#: what the reference returned in the comparisons of tests/test_env_vs_reference.py,
#: tests/test_oracle_vs_reference.py and tests/test_reset_oracle.py (recorded by tests/make_golden.py)
REFERENCE_DIR = os.path.join(GOLDEN_DIR, "reference")


def load_reference_record(name):
    return torch.load(os.path.join(REFERENCE_DIR, f"{name}.pt"), weights_only=False)


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.pt")))


def load(name):
    fix = torch.load(os.path.join(GOLDEN_DIR, f"{name}.pt"), weights_only=False)
    desc = P.WorldDescription.from_json(fix["desc"])
    tables = P.build_tables(desc)
    return fix, desc, tables


def teacher_forced_steps(fix):
    """Yields (t, state_in, fixed_rot, state_out) with state_in as World.step received it."""
    prev = None
    for t, entry in enumerate(fix["steps"]):
        base = entry.get("state_in", prev)
        state_in = {k: base[k].clone() for k in ("pos", "vel", "rot", "ang_vel")}
        state_in["force"] = entry["force"].clone()
        state_in["torque"] = entry["torque"].clone()
        if "ent_gravity" in entry:  # per-env Entity.gravity tensors (wind_flocking)
            state_in["ent_gravity"] = {k: v.clone() for k, v in entry["ent_gravity"].items()}
        yield t, state_in, entry.get("fixed_rot", {}), entry["out"]
        prev = entry["out"]


STATE_KEYS = ("pos", "vel", "rot", "ang_vel", "force", "torque")


def max_abs_err(got, want, keys=STATE_KEYS):
    return max(float((got[k].cpu() - want[k]).abs().max()) for k in keys)


def max_rel_err(got, want, keys=STATE_KEYS, floor=1e-3):
    """max |got - want| / max(|want|, floor) — relative error with an absolute floor."""
    worst = 0.0
    for k in keys:
        g, w = got[k].cpu(), want[k]
        worst = max(worst, float(((g - w).abs() / w.abs().clamp_min(floor)).max()))
    return worst


def same_result(a, b, atol=1e-5, rtol=1e-4) -> bool:
    """Two different kernels (or launch decompositions) of the same arithmetic: identical bits in the
    exact build; in the opt-in fast-arithmetic build (VMAS_B200_ARITH=fast) the compiler fuses and
    approximates per kernel, so there they only have to agree to the parity tolerance."""
    from vectorizedmultiagentsimulator_b200 import _native

    if _native.ARITH == "exact" or a.dtype == torch.bool:
        return torch.equal(a, b)
    a, b = a.float(), b.float()
    return bool(((a - b).abs() <= atol + rtol * b.abs()).all())
