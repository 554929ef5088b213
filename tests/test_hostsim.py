"""The specialised substep kernels' device code, run on the CPU (tests/hostsim).

The warp-tile kernel (``csrc/spec_tile_kernel.cuh``: a warp owns 32 envs; far tests per env, then the
narrow phase of the near (item, env) pairs compacted over the lanes, results summed per entity in
item order) must produce the same bits as the thread-per-env formulation (``spec_env_step``): same
statements, same accumulation order.  ``tests/hostsim`` compiles
both from the very headers ``nvcc`` compiles — with g++ and a small ``cuda_runtime.h`` stand-in — and
runs the tile kernel's phases as loops over the lanes with the shared-memory tile poisoned
with NaN first, so a row read before its owner wrote it, a wrong owner, a wrong row index or a wrong
summation order all show up here, without a GPU.  (On the GPU the same equality is asserted in
``tests/test_cabi_gpu.py``.)  libm's sincosf / expf / log1pf differ from CUDA's in the last bit, so
against the reference's golden vectors the CPU run is compared to a tolerance only.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from golden_util import STATE_KEYS, golden_names, load, teacher_forced_steps
from vectorizedmultiagentsimulator_b200 import _native, codegen

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_DIR = os.path.join(HERE, "hostsim")
SIM_LIB = os.path.join(SIM_DIR, "_hostsim.so")
CSRC = _native.CSRC


def _build():
    sources = [os.path.join(SIM_DIR, "hostsim.cpp"), os.path.join(SIM_DIR, "shim", "cuda_runtime.h")] + _native.HEADERS
    codegen.generate(_native.GENERATED)
    if os.path.exists(SIM_LIB) and all(os.path.getmtime(f) <= os.path.getmtime(SIM_LIB) for f in sources):
        return
    subprocess.run(
        ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-DVMAS_HOSTSIM",
         "-I", os.path.join(SIM_DIR, "shim"), "-I", CSRC, "-I", _native.INCLUDE,
         os.path.join(SIM_DIR, "hostsim.cpp"), "-o", SIM_LIB],
        check=True,
    )


@pytest.fixture(scope="module")
def sim():
    _build()
    lib = C.CDLL(SIM_LIB)
    lib.hostsim_step.argtypes = [C.c_uint64, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int] * 3
    lib.hostsim_step.restype = C.c_int
    return lib


def _run(lib, world_hash, variant, state, mask_words=None, first=0, n=None, substeps=1):
    """One World.step (or a range of substeps) on a copy of ``state``; returns the new state."""
    arr = {k: np.ascontiguousarray(state[k].numpy().astype(np.float32)).copy() for k in STATE_KEYS}
    arr["rot"] = arr["rot"].reshape(arr["rot"].shape[0], -1)
    B = arr["pos"].shape[0]
    mask = None if mask_words is None else np.asarray(mask_words, dtype=np.uint32)
    rc = lib.hostsim_step(
        world_hash, variant, B, *(arr[k].ctypes.data for k in STATE_KEYS),
        None if mask is None else mask.ctypes.data, int(mask is not None), first, substeps if n is None else n,
    )
    if rc == -2:
        pytest.skip("this world has no tile kernel")
    assert rc == 0
    return arr


def specialised_goldens():
    lib = _native.load()
    out = []
    for name in golden_names():
        _, desc, _ = load(name)
        if lib.vmas_b200_find_specialization(codegen.world_hash(desc)) >= 0:
            out.append(name)
    return out


def test_hostsim_covers_every_specialised_world(sim):
    from vectorizedmultiagentsimulator_b200 import jit

    # worlds compiled at run time (jit.py) by earlier tests of this process are registered after the library's own
    for job in list(jit._jobs.values()):
        assert job.done.wait(timeout=300)
    at_run_time = sum(job.index >= 0 for job in jit._jobs.values())
    assert sim.hostsim_num_worlds() == _native.load().vmas_b200_num_specializations() - at_run_time >= 4
    assert set(specialised_goldens()) >= {"balance", "transport", "navigation", "flocking"}


@pytest.mark.parametrize("name", specialised_goldens())
def test_tile_equals_thread_per_env_bitwise(sim, name):
    fix, desc, tables = load(name)
    h = codegen.world_hash(desc)
    words = (tables.n_masked + 31) // 32
    rng = np.random.default_rng(0)
    checked = 0
    for t, state_in, _, want in teacher_forced_steps(fix):
        if t % 3:
            continue
        # without the broad-phase mask (every candidate pair evaluated), and with random masks
        masks = [None] + ([rng.integers(0, 2**32, words, dtype=np.uint64).astype(np.uint32) for _ in range(2)] if words else [])
        for mask in masks:
            if mask is None or desc.substeps == 1:
                a = _run(sim, h, 0, state_in, mask, substeps=desc.substeps)
                b = _run(sim, h, 1, state_in, mask, substeps=desc.substeps)
            else:  # masked worlds are launched one substep at a time
                a = _run(sim, h, 0, state_in, mask, first=1, n=1)
                b = _run(sim, h, 1, state_in, mask, first=1, n=1)
            for k in STATE_KEYS:
                assert np.array_equal(a[k], b[k]), f"{name} step {t} field {k} (mask {mask})"
            assert all(np.isfinite(b[k]).all() for k in STATE_KEYS)
            checked += 1
        # a tile that is not full: the last lanes shadow the last env and store nothing
        part = {k: v[:37] for k, v in state_in.items() if k in STATE_KEYS}
        a, b = _run(sim, h, 0, part, substeps=desc.substeps), _run(sim, h, 1, part, substeps=desc.substeps)
        assert all(np.array_equal(a[k], b[k]) for k in STATE_KEYS)
    assert checked >= 3


@pytest.mark.parametrize("name", ["navigation", "flocking"])  # sphere-only: no batch-wide mask involved
def test_cpu_run_is_close_to_the_reference_golden_vectors(sim, name):
    """Sanity of the stand-in itself: the CPU run of the device code lands on the reference's result
    (tolerance: libm vs CUDA transcendentals, amplified by the stiff contact forces)."""
    fix, desc, _ = load(name)
    h = codegen.world_hash(desc)
    for t, state_in, _, want in teacher_forced_steps(fix):
        if t > 8:
            break
        got = _run(sim, h, 1, state_in, substeps=desc.substeps)
        for k in ("pos", "vel", "rot", "ang_vel"):
            w = want[k].numpy().reshape(got[k].shape)
            assert np.all(np.abs(got[k] - w) <= 1e-5 + 1e-4 * np.abs(w)), f"{name} step {t} {k}"
