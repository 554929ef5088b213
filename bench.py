#!/usr/bin/env python
"""bench.py — env-steps/s of the VMAS physics hot path behind ``Environment.step`` on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (default): BASELINE.json configs[1] — scenario ``balance``, 32768 envs per GPU, 4 agents,
continuous random actions pre-generated before the timed region (weak scaling: every rank
steps its own independent shard of envs; no data-path collective).  ``--config`` selects the
other BASELINE configs (transport3, navigation, flocking = 262144 envs strong-scaled).

One JSON line is printed by rank 0:
  value        whole-job env-steps/s, actions already resident in HBM
  e2e          same metric through the public API with HOST buffers: per step the actions are
               copied from pinned host memory and obs/rewards/dones are copied back to it
  roofline     the fused substep kernel: algorithmic bytes per launch / CUDA-event duration
  cpu_baseline the CPU oracle port of the same env on this box's host cores (bounded sample)
Timing: per-iteration CUDA events on the launching stream, summed; L2 is flushed (512 MiB
memset) between iterations outside the brackets; max over ranks.

``--dump-outputs DIR`` writes what the timed ``Environment.step`` returned in its last timed step
(rank 0's envs) as ``DIR/<name>.npy``: the inputs are seeded, so two builds run with the same
arguments can be compared output for output.

``--impl reference`` times the oracle port of the path (the reference is pure Python and does not
travel to the GPU box; the port issues the same eager torch op chain and is bit-identical to it,
see tests/) through the same Environment API: on the host cores (default), or with
``--ref-device cuda`` on the GPU — the reference's own PyTorch-CUDA path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "env-steps/sec"

#: BASELINE.json configs[1..4].  ``envs``: per GPU (weak scaling) or of the whole job (strong scaling).
CONFIGS = {
    "balance": dict(scenario="balance", kwargs=dict(n_agents=4), envs=32768, scaling="weak", ref="BASELINE.json configs[1]"),
    "transport3": dict(
        scenario="transport", kwargs=dict(n_agents=4, n_lines=2, substeps=3), envs=16384, scaling="weak",
        ref="BASELINE.json configs[2]: box + 2 line landmarks, 3 substeps",
    ),
    "navigation": dict(
        scenario="navigation", kwargs=dict(n_agents=8), envs=8192, scaling="weak",
        ref="BASELINE.json configs[3]: LIDAR, 12 rays per agent",
    ),
    "flocking": dict(
        scenario="flocking", kwargs=dict(n_agents=5), envs=262144, scaling="strong",
        ref="BASELINE.json configs[4]: 262144 envs sharded over the GPUs",
    ),
}


def resolve_config(args, world):
    """(cfg, envs of this rank's shard, envs of the whole job, scaling)."""
    cfg = CONFIGS[args.config]
    scaling = args.scaling or cfg["scaling"]
    if scaling == "strong":
        total = args.total_envs or (cfg["envs"] if cfg["scaling"] == "strong" else cfg["envs"] * 8)
        assert total % world == 0, f"--total-envs {total} is not a multiple of {world} ranks"
        return cfg, total // world, total, scaling
    per_gpu = args.envs_per_gpu or (cfg["envs"] if cfg["scaling"] == "weak" else cfg["envs"] // 8)
    return cfg, per_gpu, per_gpu * world, scaling


def workload_string(cfg, per_gpu, total, world, scaling):
    """The one description of the workload both arms print (the driver compares the strings)."""
    kw = ", ".join(f"{k}={v}" for k, v in cfg["kwargs"].items())
    return (
        f"{cfg['scenario']}({kw}), {total} envs = {per_gpu} per GPU x {world} GPU(s) ({scaling} scaling), "
        f"random continuous actions ({cfg['ref']})"
    )


# --------------------------------------------------------------------------------------------
def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--config", default="balance", choices=sorted(CONFIGS), help="BASELINE.json config (default: configs[1])")
    p.add_argument("--envs-per-gpu", type=int, default=None, help="weak scaling: envs of every rank")
    p.add_argument("--scaling", default=None, choices=["weak", "strong"], help="default: the config's own")
    p.add_argument("--total-envs", type=int, default=None, help="strong scaling: envs of the whole job")
    p.add_argument(
        "--ref-device", default="cpu", choices=["cpu", "cuda"],
        help="--impl reference: run the reference's eager torch op chain on the host cores (the reference arm) "
        "or on the GPU (the north star's PyTorch-CUDA denominator)",
    )
    p.add_argument("--cpu-steps", type=int, default=None, help="steps of the CPU baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-flush", action="store_true", help="keep L2 warm between iterations (not a bench value)")
    p.add_argument("--no-graph", action="store_true", help="step eagerly instead of replaying a CUDA graph")
    p.add_argument(
        "--dump-outputs", metavar="DIR", default=None,
        help="write the observations, rewards, dones and infos of the last timed step as DIR/<name>.npy",
    )
    return p.parse_args()


def dist_info():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    QUERY = (
        "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
        "clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL,
                text=True,
            )
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first_sample(self, timeout_s: float = 8.0):
        """nvidia-smi takes a while to attach (and slows launches while it does): the timed
        region must not start before its first line has arrived."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.02)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for name, flag in zip(names, parts[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": mx,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def pregenerate_actions(env, steps, seed, device, pin=False):
    """[steps][n_agents] tensors of shape [B, action_size], U(-u_range, u_range), from a CPU generator."""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    out = []
    for _ in range(steps):
        per_agent = []
        for a in env.agents:
            u = (torch.rand(env.num_envs, a.action_size, generator=gen, device="cpu") * 2 - 1) * a.action.u_range_tensor.cpu()
            if pin:
                u = u.pin_memory()
            else:
                u = u.to(device)
            per_agent.append(u)
        out.append(per_agent)
    return out


# --------------------------------------------------------------------------------------------
def usable_cpus() -> int:
    """Host cores this process may actually use (affinity mask and cgroup quota, not os.cpu_count)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:  # noqa: BLE001
        pass
    return n


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def pin_to_gpu_numa(local: int):
    """Restricts this rank to the host cores next to its GPU (the PCI device's ``local_cpulist``):
    the per-step launch path is host work, and a rank scheduled on the far socket pays for it in
    every CUDA-event bracket.  Returns a short description (for the JSON line) or None."""
    try:
        out = subprocess.run(
            ["nvidia-smi", f"--id={local}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
            capture_output=True, text=True, timeout=20,
        ).stdout.strip().lower()
        if not out:
            return None
        bus = out[-12:] if len(out) > 12 else out  # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
        near = _parse_cpulist(open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read())
        allowed = os.sched_getaffinity(0)
        cpus = sorted(near & allowed)
        if not cpus or len(cpus) == len(allowed):
            return None
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cores local to GPU {local} ({bus})"
    except Exception:  # noqa: BLE001
        return None


def run_reference_env(cfg, n_envs, device, warmup, max_steps, time_budget_s):
    """Times the oracle port — the reference's eager torch op chain behind the same Environment
    API — on the host cores (``device="cpu"``: the reference arm) or on the GPU (``"cuda"``: the
    reference's PyTorch-CUDA path, the north star's "10x" denominator).

    CPU: the intra-op thread count is calibrated first (eager torch on many tiny ops gets *slower*
    with too many threads; the sweep is returned).  Returns a dict.
    """
    import contextlib

    import vectorizedmultiagentsimulator_b200 as b200
    from oracle.backend import use_oracle

    on_gpu = device != "cpu"
    cores = usable_cpus()
    sweep = {}
    # tensors the op chain creates from python scalars land on the device, as in the reference
    # (it passes device=self.device everywhere)
    scope = torch.device(device) if on_gpu else contextlib.nullcontext()
    sync = (lambda: torch.cuda.synchronize()) if on_gpu else (lambda: None)
    with use_oracle(allow_cuda=on_gpu), scope:
        # action_checks="sync": the reference's asserts (two host syncs per agent and step)
        env = b200.make_env(
            cfg["scenario"], num_envs=n_envs, device=device, seed=0, action_checks="sync", **cfg["kwargs"]
        )
        actions = pregenerate_actions(env, 4, seed=1, device=device)
        env.step(actions[0])  # allocator, plan compile
        best = 1
        if not on_gpu:
            candidates = sorted({c for c in (cores, 64, 32, 16, 8, 4) if c <= cores}) or [1]
            best, best_t = candidates[0], float("inf")
            for c in candidates:  # small thread counts first; stop when it gets clearly worse
                torch.set_num_threads(c)
                env.step(actions[1])
                t0 = time.perf_counter()
                env.step(actions[2])
                dt = time.perf_counter() - t0
                sweep[c] = round(dt * 1e3, 2)
                if dt < best_t:
                    best, best_t = c, dt
                elif dt > 1.5 * best_t:
                    break
            torch.set_num_threads(best)
        for t in range(warmup):
            env.step(actions[t % 4])
        sync()
        steps, t0 = 0, time.perf_counter()
        while steps < max_steps:
            env.step(actions[steps % 4])
            steps += 1
            if time.perf_counter() - t0 > time_budget_s and steps >= 2:
                break
        sync()
        dt = time.perf_counter() - t0
    return dict(value=n_envs * steps / dt, seconds=dt, steps=steps, threads=best, sweep_ms_per_step=sweep, cores=cores)


def main_reference(args):
    rank, world, local = dist_info()
    if rank != 0:
        return
    world = max(world, args.gpus) if world == 1 else world
    cfg, per_gpu, total, scaling = resolve_config(args, world)
    on_gpu = args.ref_device == "cuda"
    device = f"cuda:{local}" if on_gpu else "cpu"
    W = max(args.warmup, 3)
    try:
        # bounded sample: every step is the per-GPU share of the workload; at most --steps of them
        r = run_reference_env(cfg, per_gpu, device, W, max(1, args.steps), time_budget_s=90.0)
    except Exception as err:  # noqa: BLE001
        print(json.dumps({"impl": "reference", "unavailable": f"{type(err).__name__}: {err}"[:300]}), flush=True)
        return
    value, seconds, steps = r["value"], r["seconds"], r["steps"]
    where = (
        f"eager torch op chain on {torch.cuda.get_device_name(local)} (the reference's PyTorch-CUDA path)"
        if on_gpu
        else f"{r['threads']} intra-op threads (calibrated; ms per step by thread count: {r['sweep_ms_per_step']}) "
        f"of {r['cores']} usable cores"
    )
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": "env-steps/s",
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * seconds / steps,
        "higher_is_better": True,
        "scaling": scaling,
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": workload_string(cfg, per_gpu, total, world, scaling),
            "reference_device": args.ref_device,
            "note": "oracle port of the reference path (the same eager torch op chain, bit-identical to the "
            "reference on CPU, tests/test_oracle_vs_reference.py); the pure-Python reference does not travel "
            "to the GPU box.  Each step is one GPU's share of the workload (env-steps/s does not depend on it)",
        },
        "cpu_baseline": {
            "value": value,
            "unit": "env-steps/s",
            "cores": 0 if on_gpu else r["threads"],
            "kind": "port",
            "sample": f"{steps} env steps of {per_gpu} envs ({seconds:.1f} s), {where}",
        },
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def step_outputs(result):
    """{name: float32 / float64 host array} of what ``Environment.step`` returned: observations and rewards
    ``[n_agents, envs, ...]``, dones ``[envs]``, every info leaf ``[n_agents, envs, ...]``."""
    import numpy as np

    import vectorizedmultiagentsimulator_b200 as b200

    obs, rews, dones, infos = result
    out = {"observations": b200.stack_views(obs), "rewards": b200.stack_views(rews), "dones": dones}
    if infos and isinstance(infos[0], dict):
        for key in sorted(infos[0]):
            out[f"info_{key}"] = torch.stack([info[key] for info in infos])
    host = {}
    for name, t in out.items():
        t = t.detach().cpu()
        host[name] = t.numpy().astype(np.float64 if t.dtype in (torch.float64, torch.int64) else np.float32)
    return host


def dump_outputs(directory, arrays, env_dim):
    """Writes ``arrays`` as ``directory/<name>.npy``.  Above 64 MiB in all, a fixed, seeded sample of the envs
    (``env_dim``: the env axis of each array) is written instead, with their indices as ``env_index.npy``."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    n_envs = arrays["dones"].shape[0]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = max(1, n_envs * DUMP_LIMIT_BYTES // (total + 8 * n_envs))
        index = np.sort(np.random.default_rng(0).choice(n_envs, size=keep, replace=False))
        arrays = {name: np.take(a, index, axis=env_dim[name]) for name, a in arrays.items()}
        arrays["env_index"] = index.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.ascontiguousarray(a))


# --------------------------------------------------------------------------------------------
def main_b200(args):
    rank, world, local = dist_info()
    import torch.distributed as dist

    pinned = pin_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        # NCCL_DEBUG=VERSION makes NCCL print a banner on stdout, in front of the one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)

    import vectorizedmultiagentsimulator_b200 as b200
    from vectorizedmultiagentsimulator_b200 import _native as nat
    from vectorizedmultiagentsimulator_b200 import shard

    if os.environ.get("VMAS_B200_L2_FETCH"):
        nat.load().vmas_b200_set_l2_fetch_granularity(int(os.environ["VMAS_B200_L2_FETCH"]))
    from vectorizedmultiagentsimulator_b200.simulator import plan as P

    cfg, B, total, scaling = resolve_config(args, world)
    K, W = args.steps, max(args.warmup, 3)
    if scaling == "strong":
        env = shard.make_shard_env(
            cfg["scenario"], total, rank, world, device, seed=0, cuda_graph=not args.no_graph, **cfg["kwargs"]
        )
    else:
        env = b200.make_env(
            cfg["scenario"], num_envs=B, device=device, seed=rank, cuda_graph=not args.no_graph, **cfg["kwargs"]
        )
    backend = env.world._get_backend()
    backend.refresh()
    desc = backend.tables.desc
    bytes_per_env_substep = P.algorithmic_bytes_per_env_substep(desc)
    launches_per_step = desc.substeps if backend.tables.n_masked else 1  # substep-kernel launches per world.step

    flush = None if args.no_flush else torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=device)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            # a rank that slept in the barrier runs its first step's host work slowly (first bracket 0.1-0.17 ms
            # against a median of 0.03, profiles/r2_4gpu_bench.json): spin the core awake, outside every bracket
            t0 = time.perf_counter()
            while time.perf_counter() - t0 < 2e-3:
                pass
        torch.cuda.synchronize()

    def timed_loop(step_fn, n):
        """Σ over iterations of the CUDA-event time of step_fn(i); L2 flushed outside the brackets."""
        pairs = []
        for i in range(n):
            if flush is not None:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step_fn(i)
            e1.record()
            pairs.append((e0, e1))
        torch.cuda.synchronize()
        times = [a.elapsed_time(b) for a, b in pairs]
        timed_loop.last = times
        return sum(times)  # ms

    remeasured = []
    counted = {"before": 0}  # backend.launches at the start of the pass that counts

    def measured(step_fn, n, label):
        """timed_loop, once more if a bracket shows a transient stall of the box: > 4x the median and at least
        0.05 ms above it.  Seen as one ~50 ms bracket in the middle of a loop (about one run in 15 on an otherwise
        idle GPU) and as a 0.17 ms first bracket behind the multi-rank barrier (profiles/r2_4gpu_bench.json); the
        brackets of an undisturbed loop stay within 1.4x of their median.  Reported in the line."""
        ms = timed_loop(step_fn, n)
        times = sorted(timed_loop.last)
        if n >= 5 and times[-1] > 4 * times[len(times) // 2] and times[-1] > times[len(times) // 2] + 0.05:
            remeasured.append(
                f"{label}: the first pass had a bracket of {times[-1]:.1f} ms ({times[-1] / times[len(times) // 2]:.0f}x "
                f"the median, {ms / n * 1e3:.1f} us per step overall): transient stall, the {n} steps were timed again"
            )
            counted["before"] = backend.launches
            ms = timed_loop(step_fn, n)
        return ms

    # ---- arm 1: actions resident in HBM --------------------------------------------------
    dev_actions = pregenerate_actions(env, W + K, seed=1 + rank, device=device)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # samples every timed region below (Environment.step, kernel-only, e2e)
    for t in range(W):
        env.step(dev_actions[t])
    if rank == 0:
        sampler.wait_first_sample()
    barrier()
    counted["before"] = backend.launches
    # the results of the last step of the first timed pass (a re-measurement steps on from a state that depends
    # on whether it happened): what --dump-outputs writes
    last_step, keep_last = [], bool(args.dump_outputs) and rank == 0

    def value_step(i):
        result = env.step(dev_actions[W + i])
        if keep_last and i == K - 1 and not last_step:
            last_step.append(result)

    wall0 = time.perf_counter()
    ms_total = measured(value_step, K, "value")
    wall = time.perf_counter() - wall0
    dumped = step_outputs(last_step[0]) if keep_last else None
    del last_step[:]
    brackets = sorted(timed_loop.last)
    bracket_us = {
        "min": round(1e3 * brackets[0], 1), "median": round(1e3 * brackets[len(brackets) // 2], 1),
        "p90": round(1e3 * brackets[min(len(brackets) - 1, (9 * len(brackets)) // 10)], 1), "max": round(1e3 * brackets[-1], 1),
        "largest": [[i, round(1e3 * x, 1)] for x, i in sorted(((x, i) for i, x in enumerate(timed_loop.last)), reverse=True)[:3]],
    }
    launches = backend.launches - counted["before"]
    barrier()

    # ---- the substep kernel inside Environment.step: the same env stepped eagerly once more (a
    # graph replay has no per-kernel events), L2 flushed before each step; the kernel then runs
    # behind the ingest / broad-phase kernels of its own step, i.e. with the slab L2-warm
    graph_mode = env.cuda_graph
    env.cuda_graph = False
    backend.kernel_events = []
    n_inside = min(K, 50)
    for i in range(n_inside):
        if flush is not None:
            flush.zero_()
        env.step(dev_actions[W + i])
    torch.cuda.synchronize()
    pairs = backend.kernel_events
    backend.kernel_events = None
    env.cuda_graph = graph_mode
    kernel_in_step_ms = sum(a.elapsed_time(b) for a, b in pairs) / len(pairs) if pairs else 0.0

    # ---- the substep kernel alone: world.step() back to back, L2 flushed before every launch.
    # The flush (~100 us on the GPU) lets the host queue the next launch ahead, so the event
    # bracket around the kernel holds no host latency (inside Environment.step it does).
    backend.kernel_events = []
    for _ in range(K):
        if flush is not None:
            flush.zero_()
        env.world.step()
    torch.cuda.synchronize()
    kernel_ms = sum(a.elapsed_time(b) for a, b in backend.kernel_events) / max(1, len(backend.kernel_events))
    backend.kernel_events = None

    # ---- arm 2: end to end with host buffers --------------------------------------------------
    # Software-pipelined like a training loop would: the results of step t-1 travel to pinned host
    # memory on a copy stream while step t (action upload + kernels) runs.  Every bracket holds one
    # action upload, one step and one complete result download (of the previous step; a final
    # bracket drains the last one), so K steps' worth of each are inside the timed region.
    host_actions = pregenerate_actions(env, W + K, seed=101 + rank, device=device, pin=True)
    # one pinned block per step ([A, B, action_size] when the agents' actions have one size): one upload
    same_size = len({tuple(a.shape) for a in host_actions[0]}) == 1
    # Environment.step is handed the pinned host tensors themselves: the step's kernel reads them over PCIe where
    # they lie (no staging copy).  Measured against an explicit upload in front of the step: 187 vs 208 us per
    # step (profiles/r2z_bench_pinned.json, r2z_bench.json).  VMAS_BENCH_PINNED_ACTIONS=0: the explicit upload.
    pinned_actions = os.environ.get("VMAS_BENCH_PINNED_ACTIONS", "1") == "1" and env.continuous_actions
    # one pinned block per step ([A, B, action_size] when the agents' actions have one size): one upload
    same_size = len({tuple(a.shape) for a in host_actions[0]}) == 1
    if same_size:
        host_blocks = [torch.stack(step_actions).pin_memory() for step_actions in host_actions]
        dev_block = torch.empty_like(host_blocks[0], device=device)
    obs0, rew0, done0, _ = env.step(dev_actions[0])
    # pinned host buffers for a step's results (observations and rewards of all agents as one tensor each,
    # dones), two sets: every separate download costs ~8 us of the bracket (measured: one copy per result
    # tensor 231 us per step, three copies 205 us; profiles/r2y_bench_per_tensor_downloads.json)
    host_sets = [
        (
            torch.empty((len(obs0),) + tuple(obs0[0].shape), dtype=obs0[0].dtype).pin_memory(),
            torch.empty((len(rew0),) + tuple(rew0[0].shape), dtype=rew0[0].dtype).pin_memory(),
            torch.empty(done0.shape, dtype=done0.dtype).pin_memory(),
        )
        for _ in range(2)
    ]
    h2d_bytes = sum(a.numel() * a.element_size() for a in host_actions[0])
    d2h_bytes = sum(t.numel() * t.element_size() for t in host_sets[0])
    copy_stream = torch.cuda.Stream(device=device)
    pending = [None]

    def download(slot):
        main = torch.cuda.current_stream()
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            for dst, src in zip(host_sets[slot], pending[0]):
                dst.copy_(src, non_blocking=True)

    def e2e_step(i):
        main = torch.cuda.current_stream()
        # this step's actions first (an explicit host->device copy issued while the 8 MB download is in flight
        # crawls at ~5 GB/s and holds the step's first kernel back; profiles/r2f_e2e_timeline.txt), then the
        # previous step's results start travelling while this step's kernels run
        if pinned_actions:
            actions = host_actions[(W + i) % len(host_actions)]  # (read by the step's kernel where they lie)
        elif same_size:
            dev_block.copy_(host_blocks[(W + i) % len(host_blocks)], non_blocking=True)
            actions = list(dev_block.unbind(0))
        else:
            actions = [a.to(device, non_blocking=True) for a in host_actions[(W + i) % len(host_actions)]]
        if pending[0] is not None:
            download(i & 1)
        obs, rews, dones, _ = env.step(actions)
        # (the per-agent results of a step sit back to back in one block: one view each, no stacking copy)
        fresh = (b200.stack_views(obs), b200.stack_views(rews), dones)
        main.wait_stream(copy_stream)  # the bracket closes after the download it overlapped
        pending[0] = fresh

    def e2e_drain(_):
        download(0)
        torch.cuda.current_stream().wait_stream(copy_stream)

    # untimed warm-up of the pipelined loop: the first dozens of transfers after an idle link are slower
    # (measured: 285 us per step over the first 20 steps, 205 us in steady state)
    for t in range(max(40, W)):
        e2e_step(t - W)
    barrier()
    ms_e2e = measured(e2e_step, K, "e2e")
    e2e_brackets = list(timed_loop.last)
    ms_e2e += timed_loop(e2e_drain, 1)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    env.check_actions_now()

    # ---- reduce over ranks ---------------------------------------------------------------------
    stats = torch.tensor([ms_total, ms_e2e, kernel_ms, kernel_in_step_ms], dtype=torch.float64, device=device)
    per_rank = [stats.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, stats)
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, kernel_ms, kernel_in_step_ms = (float(x) for x in stats.tolist())
    value = total * K / (ms_total * 1e-3)
    e2e_value = total * K / (ms_e2e * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the fused substep kernel -----------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # one launch advances B envs by one substep (worlds with line / box pairs) or by all S substeps
    # (sphere-only worlds: the state stays in registers); bytes per launch = bytes x B either way
    alg_bytes = bytes_per_env_substep * B
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic = traffic_src = None
    tj = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = tj["%s_%s" % (cfg["scenario"], "_".join(f"{k}={v}" for k, v in cfg["kwargs"].items()))][str(B)]
        traffic = ent["dram_bytes_read"] + ent["dram_bytes_write"]
        traffic_src = ent["source"]
    except Exception:  # noqa: BLE001
        pass
    roofline = {
        "bound": "hbm",
        "kernel": "substep kernel, mapping=%s, arithmetic=%s" % (backend._dev_tables.mapping, nat.ARITH),
        "achieved": achieved,
        "peak": peak,
        "unit": "GB/s",
        "frac": achieved / peak,
        "traffic": traffic,
        "traffic_source": traffic_src,
        "peak_source": peak_src,
        "bytes_per_launch": alg_bytes,
        "bytes_per_env_substep": bytes_per_env_substep,
        "substep_launches_per_step": launches_per_step,
        "kernel_us": kernel_ms * 1e3,
        "kernel_us_inside_env_step": kernel_in_step_ms * 1e3 if kernel_in_step_ms else None,
        "frac_inside_env_step": (alg_bytes / (kernel_in_step_ms * 1e-3) / 1e9 / peak) if kernel_in_step_ms else None,
        "how": "CUDA events recorded by the library around the substep kernel; kernel_us: standalone world.step() "
        "loop, L2 flushed before each launch; kernel_us_inside_env_step: the benched env stepped eagerly "
        "(Environment.step, L2 flushed before each step), the kernel running behind its step's ingest / broad-phase kernels",
    }
    substep_roofline = roofline
    # the whole Environment.step against the same peak: compulsory bytes of one step (slab traffic of
    # every substep, the actions read, the observations / rewards / dones written) / ms_per_step
    out_bytes = sum(t.numel() * t.element_size() for t in list(obs0) + list(rew0) + [done0])
    step_bytes = bytes_per_env_substep * B * desc.substeps + h2d_bytes + out_bytes
    roofline_step = {
        "bytes_per_step": step_bytes,
        "achieved": step_bytes / (ms_total / K * 1e-3) / 1e9,
        "unit": "GB/s",
        "frac": step_bytes / (ms_total / K * 1e-3) / 1e9 / peak,
        "note": "Environment.step as a whole (graph replay): slab traffic of all substeps + actions in + "
        "observations, rewards, dones out, over ms_per_step",
    }

    if launches == K and graph_mode:
        # Every timed step was ONE launch (step_env_kernel: action ingest + broad phase + substeps + step program
        # + observation rows): that kernel is the timed region, and the bracket around Environment.step is its
        # duration (plus the two event records).  The substep kernel on its own is kept below.
        traffic = traffic_src = None
        try:
            ent = tj["%s_%s" % (cfg["scenario"], "_".join(f"{k}={v}" for k, v in cfg["kwargs"].items()))]["step_env_kernel"][str(B)]
            traffic = ent["dram_bytes_read"] + ent["dram_bytes_write"]
            traffic_src = ent["source"]
        except Exception:  # noqa: BLE001
            pass
        step_us = ms_total / K * 1e3
        roofline = {
            "bound": "hbm",
            "kernel": "step_env_kernel: the whole Environment.step in one launch (action ingest, batch-wide broad phase "
            "with a grid barrier, substeps, step program, observation rows), arithmetic=%s" % nat.ARITH,
            "achieved": step_bytes / (step_us * 1e-6) / 1e9,
            "peak": peak,
            "unit": "GB/s",
            "frac": step_bytes / (step_us * 1e-6) / 1e9 / peak,
            "traffic": traffic,
            "traffic_source": traffic_src,
            "peak_source": peak_src,
            "bytes_per_launch": step_bytes,
            "bytes_per_env_substep": bytes_per_env_substep,
            "kernel_us": step_us,
            "launches_per_step": 1,
            "how": "the only kernel of a timed step: duration = the CUDA-event bracket around Environment.step "
            "(value's own brackets, L2 flushed before each); algorithmic bytes = slab rows of the substep + actions "
            "read + agent.action.u, observations, rewards, dones written",
            "substep_kernel": substep_roofline,
        }

    # ---- same kernel at a batch that is not launch/latency-bound: 1 Mi envs (state tiled) -----------------
    try:
        big_B = 1 << 20
        reps = max(1, big_B // B)
        big_B = reps * B

        class _BigSlab:
            def __init__(self, slab):
                self.t = tuple(t.repeat(reps, *([1] * (t.dim() - 1))).contiguous() for t in slab.tensors())

            def tensors(self):
                return self.t

        big = _BigSlab(env.world.slab)
        old = backend.tables.desc.batch_dim
        backend.tables.desc.batch_dim = big_B
        big_dt = nat.DeviceTables(backend.tables, None, device)
        backend.tables.desc.batch_dim = old
        def time_big():
            times = []
            for _ in range(12):
                if flush is not None:
                    flush.zero_()
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                nat.world_step(backend.lib, big_dt, big, events=ev)
                torch.cuda.synchronize()
                times.append(ev[0].elapsed_time(ev[1]))
            times = sorted(times[2:])
            return times[len(times) // 2]

        big_ms = time_big()
        big_ms_identity = None
        if big_dt.env_order is not None:
            # env scheduling: first the identity order (above), then the order built from the signatures
            big_ms_identity = big_ms
            nat.build_env_order(backend.lib, big_dt)
            big_ms = time_big()
        big_achieved = bytes_per_env_substep * big_B * launches_per_step / (big_ms * 1e-3) / 1e9
        substep_roofline["at_1Mi_envs"] = {
            "kernel_us": big_ms * 1e3 / launches_per_step,
            "kernel_us_identity_order": None if big_ms_identity is None else big_ms_identity * 1e3 / launches_per_step,
            "achieved": big_achieved,
            "frac": big_achieved / peak,
            "note": f"the substep kernel and state tiled to {big_B} envs (slab > L2); at {B} envs the slab is "
            f"{alg_bytes / 1e6:.1f} MB = {alg_bytes / peak / 1e3:.1f} us of HBM time, below launch latency",
        }
        del big, big_dt
    except Exception as err:  # noqa: BLE001
        substep_roofline["at_1Mi_envs"] = {"error": str(err)}

    # ---- CPU baseline (bounded sample, rank 0, N=1 only) ---------------------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r = run_reference_env(cfg, B, "cpu", 2, args.cpu_steps or 200, time_budget_s=20.0)
        cpu_baseline = {
            "value": r["value"],
            "unit": "env-steps/s",
            "cores": r["threads"],
            "kind": "port",
            "sample": f"{r['steps']} env steps of {B} envs ({r['seconds']:.1f} s), CPU oracle port behind the same "
            f"Environment API, {r['threads']} intra-op threads (calibrated; ms per step by thread count: "
            f"{r['sweep_ms_per_step']}) of {r['cores']} usable cores",
        }

    line = {
        "metric": METRIC,
        "value": value,
        "unit": "env-steps/s",
        "n_gpus": world,
        "steps": K,
        "warmup": args.warmup,
        "ms_per_step": ms_total / K,
        "higher_is_better": True,
        "scaling": scaling,
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": workload_string(cfg, B, total, world, scaling),
            "substeps": desc.substeps,
            "arithmetic": nat.ARITH,
            "timing": "sum of per-iteration CUDA-event brackets around Environment.step; max over ranks",
            "l2": "flushed between iterations (512 MiB memset outside the brackets)" if flush is not None else "NOT flushed",
            "api": "make_env(..., cuda_graph=%s); Environment.step" % (not args.no_graph),
            "warmup_steps_run": W,
            "wall_ms_per_step_incl_flush": 1e3 * wall / K,
            "bracket_us": bracket_us,
            "remeasured": remeasured or None,
            "host_affinity": pinned,
        },
        "clocks": clocks,
        "e2e": {
            "value": e2e_value,
            "unit": "env-steps/s",
            "h2d_bytes_per_step": h2d_bytes,
            "d2h_bytes_per_step": d2h_bytes,
            "ms_per_step": ms_e2e / K,
            "how": ("per step: Environment.step is handed the actions as pinned HOST tensors (its kernel reads them "
                    "over PCIe), " if pinned_actions else "per step: the actions are uploaded from a pinned host block, "
                    "Environment.step runs, ") + "and the observations, rewards, dones travel to pinned host buffers; "
            "the download of step t-1 overlaps the kernels of step t on a copy stream, inside the brackets",
            "bracket_ms_first5_last5": [round(x, 4) for x in e2e_brackets[:5] + e2e_brackets[-5:]],
            "bracket_us": {
                "min": round(1e3 * min(e2e_brackets), 1), "median": round(1e3 * sorted(e2e_brackets)[len(e2e_brackets) // 2], 1),
                "p90": round(1e3 * sorted(e2e_brackets)[min(len(e2e_brackets) - 1, (9 * len(e2e_brackets)) // 10)], 1),
                "max": round(1e3 * max(e2e_brackets), 1),
                "largest": [[i, round(1e3 * x, 1)] for x, i in sorted(((x, i) for i, x in enumerate(e2e_brackets)), reverse=True)[:3]],
            },
            "pcie_roofline": "the download alone (8.4 MB at the measured 56 GB/s, profiles/r2b_pcie.txt) is 160 us per "
            "step of 32768 balance envs = 2.05e8 env-steps/s",
        },
        "gpu_launches": launches,
        "roofline": roofline,
        "roofline_step": roofline_step,
        "per_rank_ms_per_step": [float(r[0]) / K for r in per_rank],
        "per_rank_e2e_ms_per_step": [float(r[1]) / K for r in per_rank],
        "cpu_baseline": cpu_baseline,
    }
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped, {name: 0 if name == "dones" else 1 for name in dumped})
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse_args()
    if args.impl == "reference":
        main_reference(args)
    else:
        main_b200(args)
