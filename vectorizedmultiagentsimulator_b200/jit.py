"""Run-time specialisation of the substep kernel for ANY world (ref core.py:1091-1177: arbitrary worlds
are the reference's contract).

``codegen.py`` pre-builds specialised kernels for a handful of preset worlds; every other world used
to run on the generic table-driven kernels at 2-15x the time.  Here the same template
(``csrc/spec_kernel.cuh``) is compiled for the world at hand when its plan is first uploaded: the
world's constexpr tables are emitted (``codegen.emit_world``), ``nvcc`` builds a small shared object
for sm_100a (a few seconds, in a background thread; cached on disk by world hash and arithmetic
flags), and its launch functions are registered with the main library
(``vmas_b200_register_specialization``).  Until the object is ready the world steps on the generic
kernels; both produce identical bits (tests/test_cabi_gpu.py), so the switch is invisible.

``VMAS_B200_JIT``: ``async`` (default) | ``block`` (wait for the compiler) | ``off``.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading
from typing import Dict, Optional

from . import _native, codegen
from .simulator import plan as P

MODE = os.environ.get("VMAS_B200_JIT", "async")
assert MODE in ("async", "block", "off"), MODE
CACHE_DIR = os.environ.get("VMAS_B200_JIT_DIR") or os.path.join(_native.CSRC, "generated", "jit")


def _cached_or_new(filename: str) -> str:
    """Path of a compiled object: the one in ``CACHE_DIR`` (what ``__graft_entry__.build`` compiled ahead of
    time) if it is there, else where a new one goes: ``CACHE_DIR`` when it can be written to, else a per-user
    temporary directory (an installed or read-only source tree)."""
    path = os.path.join(CACHE_DIR, filename)
    if os.path.exists(path):
        return path
    try:
        os.makedirs(CACHE_DIR, exist_ok=True)
    except OSError:
        pass
    if not os.access(CACHE_DIR, os.W_OK):
        fallback = os.path.join(tempfile.gettempdir(), f"vmas_b200_jit_{os.getuid()}")
        os.makedirs(fallback, mode=0o700, exist_ok=True)
        if os.stat(fallback).st_uid != os.getuid():  # objects are loaded from here: only from a directory of ours
            fallback = tempfile.mkdtemp(prefix="vmas_b200_jit_")
        path = os.path.join(fallback, filename)
    return path


_TEMPLATE = """// GENERATED at run time by vectorizedmultiagentsimulator_b200/jit.py — one world's specialised kernels.
#include "spec_kernel.cuh"
#include "spec_tile_kernel.cuh"

namespace vmas {{

{world}

}}  // namespace vmas

using W = vmas::{name};
extern "C" {{
cudaError_t vmas_jit_launch(const vmas::SpecArgs& a, cudaStream_t stream) {{ return vmas::launch_spec<W>(a, stream); }}
cudaError_t vmas_jit_launch_tile(const vmas::SpecArgs& a, cudaStream_t stream) {{ return vmas::launch_tile<W>(a, stream); }}
int vmas_jit_has_tile(void) {{ return vmas::TileLayout<W>::SUPPORTED ? 1 : 0; }}
int vmas_jit_spec_args_bytes(void) {{ return (int)sizeof(vmas::SpecArgs); }}
}}
"""

_STEP_TEMPLATE = """// GENERATED at run time by vectorizedmultiagentsimulator_b200/jit.py — one whole-step kernel:
// the world's specialised substep kernel with a scenario's step program + observation rows as its epilogue.
#include "spec_kernel.cuh"

namespace vmas {{

{world}

{post}

}}  // namespace vmas

using W = vmas::{name};
using P = vmas::{post_name};
extern "C" {{
cudaError_t vmas_jit_launch_fused(const vmas::SpecArgs& a, const vmas::EpiArgs& e, cudaStream_t stream) {{
  return vmas::launch_fused<W, P>(a, e, stream);
}}
cudaError_t vmas_jit_launch_env(const vmas::SpecArgs& a, const vmas::EpiArgs& e, const vmas::ActArgs& act, cudaStream_t stream) {{
  return vmas::launch_env<W, P>(a, e, act, stream);
}}
int vmas_jit_has_ingest(void) {{ return P::N_ACT > 0 ? 1 : 0; }}
int vmas_jit_spec_args_bytes(void) {{ return (int)sizeof(vmas::SpecArgs); }}
int vmas_jit_epi_args_bytes(void) {{ return (int)sizeof(vmas::EpiArgs); }}
int vmas_jit_act_args_bytes(void) {{ return (int)sizeof(vmas::ActArgs); }}
}}
"""

_lock = threading.Lock()
_jobs: Dict[int, "Job"] = {}
_keepalive = []  # loaded objects must outlive the registry entries that point into them


def _source_stamp() -> str:
    """Hash of the headers the object is compiled from: a header edit invalidates the cache."""
    h = hashlib.sha1()
    for name in ("geometry.cuh", "query.cuh", "spec_kernel.cuh", "spec_tile_kernel.cuh"):
        h.update(open(os.path.join(_native.CSRC, name), "rb").read())
    h.update(open(os.path.join(_native.INCLUDE, "vmas_b200.h"), "rb").read())
    return h.hexdigest()[:12]


class Job:
    """One world's compilation: ``index`` is the registered specialisation once ``done`` is set."""

    def __init__(self, desc: P.WorldDescription):
        self.hash = codegen.world_hash(desc)
        self.desc = desc
        self.done = threading.Event()
        self.index = -1
        self.error: Optional[str] = None
        self.seconds = 0.0

    def run(self):
        import time

        t0 = time.perf_counter()
        try:
            self.index = self._compile_and_register()
        except Exception as err:  # noqa: BLE001  (stay on the generic kernels)
            self.error = f"{type(err).__name__}: {err}"
        self.seconds = time.perf_counter() - t0
        self.done.set()

    def _compile_and_register(self) -> int:
        desc = self.desc
        name, text, h = codegen.emit_world(desc, "run-time specialisation")
        so = _cached_or_new(f"{h:016x}_{_native.ARITH}_{_source_stamp()}.so")
        stem = so[: -len(".so")]
        if not os.path.exists(so):
            with open(stem + ".cu", "w") as fh:
                fh.write(_TEMPLATE.format(world=text, name=name))
            flags = _native.NVCC_FLAGS + _native.ARITH_FLAGS[_native.ARITH]
            tmp = f"{so}.{os.getpid()}.tmp"
            cmd = [_native._nvcc()] + flags + ["-I", _native.INCLUDE, "-I", _native.CSRC, "-o", tmp, stem + ".cu"]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            if proc.returncode != 0:
                raise RuntimeError(f"nvcc failed: {proc.stderr[-600:]}")
            os.replace(tmp, so)  # atomic: concurrent processes (one per GPU) may race on the same world
        obj = C.CDLL(so)
        lib = _native.load()
        launch = C.cast(obj.vmas_jit_launch, C.c_void_p)
        tile = C.cast(obj.vmas_jit_launch_tile, C.c_void_p) if obj.vmas_jit_has_tile() else None
        with _lock:
            index = lib.vmas_b200_register_specialization(
                C.c_uint64(h), desc.n_entities, len(desc.items), launch, tile, obj.vmas_jit_spec_args_bytes()
            )
            if index < 0:
                raise RuntimeError(lib.vmas_b200_last_error().decode())
            _keepalive.append(obj)
        return index


def available() -> bool:
    if MODE == "off":
        return False
    try:
        _native._nvcc()
        return True
    except RuntimeError:
        return False


def request(desc: P.WorldDescription) -> Optional[Job]:
    """Starts (or finds) the compilation of ``desc``'s specialisation; None if the world cannot be
    specialised (too large, per-env gravity tensors) or the JIT is off / has no compiler."""
    if not available() or not codegen.specializable(desc):
        return None
    h = codegen.world_hash(desc)
    with _lock:
        job = _jobs.get(h)
        if job is None:
            job = _jobs[h] = Job(desc)
            if MODE == "block":
                start = job.run
            else:
                thread = threading.Thread(target=job.run, name=f"vmas-b200-jit-{h:016x}", daemon=True)
                start = thread.start
        else:
            start = None
    if start is not None:
        start()
    return job


class StepKernelJob(Job):
    """The whole-step kernel of one (world, observation columns, step program): ``index`` is the handle for
    ``VmasEnvStep.fused_kernel`` once ``done`` is set."""

    def __init__(self, desc: P.WorldDescription, cols, instrs, acts=()):
        super().__init__(desc)
        self.cols, self.instrs, self.acts = cols, instrs, tuple(acts)
        self.post_hash = codegen.post_hash(cols, instrs, self.acts)
        self.key = (self.hash ^ ((self.post_hash << 1) | (self.post_hash >> 63))) & 0xFFFFFFFFFFFFFFFF

    def _compile_and_register(self) -> int:
        desc = self.desc
        name, text, h = codegen.emit_world(desc, "whole-step kernel")
        post_name, post_text, _ = codegen.emit_post(self.cols, self.instrs, self.acts)
        so = _cached_or_new(f"step_{self.key:016x}_{_native.ARITH}_{_source_stamp()}.so")
        stem = so[: -len(".so")]
        if not os.path.exists(so):
            with open(stem + ".cu", "w") as fh:
                fh.write(_STEP_TEMPLATE.format(world=text, post=post_text, name=name, post_name=post_name))
            flags = _native.NVCC_FLAGS + _native.ARITH_FLAGS[_native.ARITH]
            tmp = f"{so}.{os.getpid()}.tmp"
            cmd = [_native._nvcc()] + flags + ["-I", _native.INCLUDE, "-I", _native.CSRC, "-o", tmp, stem + ".cu"]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            if proc.returncode != 0:
                raise RuntimeError(f"nvcc failed: {proc.stderr[-600:]}")
            os.replace(tmp, so)
        obj = C.CDLL(so)
        lib = _native.load()
        with _lock:
            handle = lib.vmas_b200_register_step_kernel(
                C.c_uint64(self.key), desc.n_entities, len(desc.items), C.cast(obj.vmas_jit_launch_fused, C.c_void_p),
                C.cast(obj.vmas_jit_launch_env, C.c_void_p) if obj.vmas_jit_has_ingest() else None,
                obj.vmas_jit_spec_args_bytes(), obj.vmas_jit_epi_args_bytes(), obj.vmas_jit_act_args_bytes(),
            )
            if handle <= 0:
                raise RuntimeError(lib.vmas_b200_last_error().decode())
            _keepalive.append(obj)
        return handle


_step_jobs: Dict[int, StepKernelJob] = {}


def request_step_kernel(desc: P.WorldDescription, cols, instrs, acts=(), block: bool = False) -> Optional[StepKernelJob]:
    """Starts (or finds) the compilation of the whole-step kernel; None if the world cannot be specialised.
    ``acts``: [(agent row, u_range x 2, u_multiplier x 2)] of the policy agents if the kernel is to ingest
    their (continuous, holonomic) actions itself."""
    if not available() or not codegen.specializable(desc):
        return None
    job = StepKernelJob(desc, cols, instrs, acts)
    with _lock:
        have = _step_jobs.get(job.key)
        if have is None:
            _step_jobs[job.key] = job
            if MODE == "block" or block:
                start = job.run
            else:
                start = threading.Thread(target=job.run, name=f"vmas-b200-jit-step-{job.key:016x}", daemon=True).start
        else:
            job, start = have, None
    if start is not None:
        start()
    return job


def prebuild_step_kernels(verbose: bool = False):
    """Compiles the whole-step kernels of the preset worlds (``codegen.PRESETS``) whose scenario is written
    on a step program, so that they are in the on-disk cache before the first capture (``__graft_entry__.build``).
    Returns ``[(label, key)]``."""
    import torch

    from . import scenarios

    built = []
    stamp = f"_{_source_stamp()}."
    if os.path.isdir(CACHE_DIR):  # objects compiled from older headers can never be loaded again
        for name in os.listdir(CACHE_DIR):
            if stamp not in name:
                os.remove(os.path.join(CACHE_DIR, name))
    for scenario, kwargs, *_ in codegen.PRESETS:
        sc = scenarios.load(scenario + ".py").Scenario()
        if not (hasattr(sc, "_step_program") and hasattr(sc, "_observation_plan")):
            continue
        world = sc.env_make_world(1, torch.device("cpu"), **dict(kwargs))
        prog, plan = sc._step_program(), sc._observation_plan()
        cols, lidars = plan.compile(world)
        if lidars:
            continue
        index = {id(e): i for i, e in enumerate(world.entities)}
        desc = P.describe_world(world)
        if not codegen.specializable(desc):
            continue
        label = scenario + "(" + ", ".join(f"{k}={v}" for k, v in kwargs.items()) + ")"
        instrs = prog.instructions(lambda e: index[id(e)])
        columns = codegen.fuse_value_columns(cols, plan.buffer_sources, instrs) if (cols[..., 0] != 0).any() else None
        # with and without the action ingest as the kernel's prologue (step_env_kernel / step_fused_kernel); an
        # environment adds one STORE per result leaf to the program when it captures its step, so its own
        # variant is compiled then (seconds) — these two make sure the templates build, and serve
        # VMAS_B200_RESULTS_IN_PLACE=0
        from .simulator.dynamics.basic import Holonomic

        agents = world.policy_agents
        holonomic = all(type(a.dynamics) is Holonomic and a.action_size == 2 for a in agents)
        row = {id(a): j for j, a in enumerate(world.agents)}
        acts = tuple(
            (row[id(a)], *(float(v) for v in a.action.u_range_tensor.tolist()), *(float(v) for v in a.action.u_multiplier_tensor.tolist()))
            for a in agents
        ) if holonomic else ()
        for variant in ((), acts) if acts else ((),):
            job = StepKernelJob(desc, columns, instrs, variant)
            job.run()
            if job.error:
                raise RuntimeError(f"whole-step kernel of {label}: {job.error}")
            if verbose:
                print(f"whole-step kernel {job.key:016x}  {label}  ({job.seconds:.1f} s)")
            built.append((label, job.key))
    return built
