"""Execution backends behind ``World.step`` / ``cast_rays`` / the distance queries.

``PlanRuntime`` holds the host logic every backend shares: compiling the world into
:class:`~.simulator.plan.PlanTables` when its static structure changed, resolving LIDAR
target lists from ``entity_filter`` callables, and tracking per-env joint rotations.

``CudaBackend`` is the product: it uploads the tables once and turns each API call into one
call of the C-ABI library (``include/vmas_b200.h``) on torch's current CUDA stream.  It
refuses to run anywhere else — there is deliberately no CPU or torch-eager fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Tuple

import torch
from torch import Tensor

from .simulator import plan as P


class PlanRuntime:
    def __init__(self, world):
        self.world = world
        self.tables: Optional[P.PlanTables] = None
        self._plan_version = -1
        self._targets_cache: Dict[Tuple[int, Callable], List[int]] = {}
        self._entity_index: Dict[int, int] = {}
        self._joint_constraints = []  # (item index, JointConstraint) for per-env fixed rotations

    # -- plan ----------------------------------------------------------------------------
    def refresh(self) -> bool:
        """Recompile if the world's static structure changed.  Returns True if it did."""
        w = self.world
        w._ensure_slab()
        if self.tables is not None and self._plan_version == w._plan_version:
            return False
        desc = P.describe_world(w)
        self.tables = P.build_tables(desc)
        self._plan_version = w._plan_version
        self._targets_cache.clear()
        ents = w.entities
        self._entity_index = {id(e): i for i, e in enumerate(ents)}
        # joint constraints in item order (items 0..J-1 are the joints)
        by_pair = {}
        for c in w._joints.values():
            by_pair[(self._entity_index[id(c.entity_a)], self._entity_index[id(c.entity_b)])] = c
        self._joint_constraints = []
        for k, it in enumerate(desc.items):
            if it["kind"] != P.K_JOINT:
                break
            self._joint_constraints.append((k, by_pair[(it["a"], it["b"])]))
        self.on_new_tables()
        return True

    def on_new_tables(self):
        pass

    def index_of(self, entity) -> int:
        self.refresh()
        try:
            return self._entity_index[id(entity)]
        except KeyError:
            raise RuntimeError(f"Entity '{entity.name}' does not belong to this world") from None

    def per_env_fixed_rotations(self) -> Dict[int, Tensor]:
        """item index → ``[B, 1]`` fixed rotation, for the joints whose value is a tensor."""
        out = {}
        for k, c in self._joint_constraints:
            if not c.rotate and not isinstance(c.fixed_rotation, (int, float)):
                out[k] = c.fixed_rotation
        return out

    # -- LIDAR target lists ----------------------------------------------------------------
    def ray_targets(self, entity, entity_filter: Callable) -> List[int]:
        """Entities a ray from ``entity`` can hit (ref core.py:1678-1691)."""
        self.refresh()
        key = (id(entity), entity_filter)  # holding the callable keeps its identity unique
        cached = self._targets_cache.get(key)
        if cached is not None:
            return cached
        if len(self._targets_cache) > 512:
            self._targets_cache.clear()
        targets = []
        for i, e in enumerate(self.world.entities):
            if entity is e or not entity_filter(e):
                continue
            assert e.collides(entity) and entity.collides(e), "Rays are only casted among collidables"
            P._shape_kind(e.shape)  # raises for unsupported shapes
            targets.append(i)
        self._targets_cache[key] = targets
        return targets


def _require_cuda(world):
    dev = torch.device(world.device)
    if dev.type != "cuda":
        raise RuntimeError(
            f"vectorizedmultiagentsimulator_b200 runs its physics only on CUDA (sm_100a); world device is "
            f"'{dev}'. There is no CPU fallback."
        )
    if dev.index is None:  # "cuda" -> the concrete device its tensors live on
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


class CudaBackend(PlanRuntime):
    """One process-local driver of the sm_100a kernels for one world (one GPU)."""

    def __init__(self, world):
        super().__init__(world)
        self.device = _require_cuda(world)
        from . import _native

        self.lib = _native.load()  # raises if the extension is not built
        self._native = _native
        self._dev_tables = None
        self._fixed_rot_versions = {}
        self._ray_cache: Dict[Tuple[int, Callable], Tensor] = {}
        self.launches = 0
        #: when set to a list, every step() appends a (begin, end) event pair bracketing the
        #: substep kernel(s) (bench.py's roofline measurement)
        self.kernel_events = None
        #: while a list: the library launches of a step being captured, in order (Environment._capture)
        self.trace = None

    # -- tables ----------------------------------------------------------------------------
    def on_new_tables(self):
        self._ingest_arr = None
        self._dev_tables = self._native.DeviceTables(self.tables, self.world, self.device)
        self._fixed_rot_versions = {}
        self._ray_cache.clear()
        # a world without an ahead-of-time specialisation gets one compiled at run time (jit.py); it
        # steps on the generic kernels until the compiler is done (identical bits either way)
        self._jit_job = None
        if self._dev_tables.specialization < 0:
            from . import jit

            self._jit_job = jit.request(self.tables.desc)
            self._adopt_jit()

    def _adopt_jit(self, wait: bool = False):
        """Switches to the run-time specialised kernels once their compilation has finished."""
        job = self._jit_job
        if job is None:
            return
        if wait:
            job.done.wait()
        if not job.done.is_set():
            return
        self._jit_job = None
        if job.index >= 0:
            self._dev_tables = self._native.DeviceTables(self.tables, self.world, self.device)
            self._fixed_rot_versions = {}
        elif job.error:
            import warnings

            warnings.warn(f"vmas_b200: run-time specialisation failed, staying on the generic kernels ({job.error})")

    def wait_for_jit(self):
        """Blocks until a pending run-time specialisation is in use (a CUDA-graph capture calls this: the
        captured step must already contain the kernel it will keep replaying)."""
        self.refresh()
        self._adopt_jit(wait=True)

    def _sync_fixed_rotations(self):
        dt = self._dev_tables
        if dt.joint_rot is None:
            return
        for k, c in self._joint_constraints:
            if c.rotate:
                continue
            ver = c._fixed_rotation_version
            if self._fixed_rot_versions.get(k) == ver:
                continue
            value = c.fixed_rotation
            if isinstance(value, (int, float)):
                dt.joint_rot[:, k].fill_(float(value))
            else:
                dt.joint_rot[:, k].copy_(value.reshape(-1))
            self._fixed_rot_versions[k] = ver

    # -- hot path ---------------------------------------------------------------------------
    def _sync_entity_gravity(self):
        dt = self._dev_tables
        if dt.ent_gravity is None:
            return
        ents = self.world.entities
        for i in dt.gravity_entities:
            dt.ent_gravity[:, i].copy_(ents[i].gravity)

    def step(self):
        tables = self._dev_tables
        self.refresh()
        if self._jit_job is not None:
            self._adopt_jit()
        if self._dev_tables is not tables:
            # the ingest launch built the broad-phase mask into the tables just replaced: build it anew
            self._mask_ready = False
        self._sync_fixed_rotations()
        self._sync_entity_gravity()
        slab = self.world.slab
        events = None
        if self.kernel_events is not None:
            events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            self.kernel_events.append(events)
        # 2: the fused ingest launch of this step already built the first substep's broad-phase mask
        mode = 2 if (getattr(self, "_mask_ready", False) and self.world.exact_broad_phase) else self.world.exact_broad_phase
        self._mask_ready = False
        n = self._native.world_step(self.lib, self._dev_tables, slab, exact_broad_phase=mode, events=events)
        self.launches += n
        if self.trace is not None:
            self.trace.append(("step", n, int(mode)))
        if not torch.cuda.is_current_stream_capturing():
            self.after_step()  # (a graph replay calls it itself: Environment._step_graphed)

    def after_step(self):
        """Host-side bookkeeping after a World.step ran (eagerly or as part of a graph replay): every
        ``ENV_REORDER_EVERY`` steps the envs are re-sorted by the contact signature the substep kernel
        recorded, so that the threads of a warp step envs that take the same branches."""
        dt = self._dev_tables
        if dt is None or dt.env_order is None:
            return
        self._steps_since_reorder = getattr(self, "_steps_since_reorder", 0) + 1
        if self._steps_since_reorder >= self._native.ENV_REORDER_EVERY:
            self._steps_since_reorder = 0
            self.launches += self._native.build_env_order(self.lib, dt)

    def _targets_tensor(self, entity, entity_filter) -> Tuple[int, Tensor]:
        src = self.index_of(entity)
        key = (id(entity), entity_filter)
        t = self._ray_cache.get(key)
        if t is None:
            if len(self._ray_cache) > 512:
                self._ray_cache.clear()
            idx = self.ray_targets(entity, entity_filter)
            t = torch.tensor(idx if idx else [0], dtype=torch.int32, device=self.device)
            t._n_valid = len(idx)
            self._ray_cache[key] = t
        return src, t

    def cast_rays(self, entity, angles: Tensor, max_range: float, entity_filter) -> Tensor:
        src, targets = self._targets_tensor(entity, entity_filter)
        slab = self.world.slab
        angles = angles.to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty_like(angles)
        self._native.cast_rays(
            self.lib, self._dev_tables, slab, src, targets, targets._n_valid, angles, None, float(max_range), out
        )
        self.launches += 1
        return out

    def lidar_measure(self, sensor) -> Tensor:
        """``sensor._angles + agent.rot`` is folded into the kernel (ref sensors.py:116-121)."""
        src, targets = self._targets_tensor(sensor.agent, sensor.entity_filter)
        slab = self.world.slab
        out = torch.empty_like(sensor._angles)
        self._native.cast_rays(
            self.lib,
            self._dev_tables,
            slab,
            src,
            targets,
            targets._n_valid,
            sensor._angles,
            src,
            float(sensor._max_range),
            out,
        )
        self.launches += 1
        return out

    # -- batched sensors / queries (one launch for many sensors or pairs) ---------------------------
    def _all_spheres(self, entity_indices) -> bool:
        shapes = self.tables.ent_i32[:, 0]
        return all(int(shapes[i]) == P.SHAPE_SPHERE for i in entity_indices)

    def lidar_measure_many(self, sensors) -> Tensor:
        """``[Q, B, R]`` ranges of ``Q`` LIDARs with the same number of rays, in one launch."""
        self.refresh()
        key = ("lidars",) + tuple(id(s) for s in sensors)
        pack = self._ray_cache.get(key)
        if pack is None:
            n_rays = {s._angles.shape[1] for s in sensors}
            assert len(n_rays) == 1, "sensors measured together must have the same number of rays"
            src, off, flat = [], [0], []
            for s in sensors:
                src.append(self.index_of(s.agent))
                flat += self.ray_targets(s.agent, s.entity_filter)
                off.append(len(flat))
            i32 = lambda v: torch.tensor(v if v else [0], dtype=torch.int32, device=self.device)  # noqa: E731
            pack = (
                i32(src),
                i32(off),
                i32(flat),
                torch.stack([s._angles[0] for s in sensors]).to(self.device, torch.float32).contiguous(),
                torch.tensor([float(s._max_range) for s in sensors], dtype=torch.float32, device=self.device),
                n_rays.pop(),
                self._native.RAYS_SPHERE_TARGETS if self._all_spheres(flat) else 0,
            )
            self._ray_cache[key] = pack
        src, off, flat, angles, ranges, n_rays, flags = pack
        out = torch.empty(len(sensors), self.world.batch_dim, n_rays, dtype=torch.float32, device=self.device)
        self._native.cast_rays_batched(
            self.lib, self._dev_tables, self.world.slab, src, off, flat, angles, ranges, n_rays, out, flags=flags
        )
        self.launches += 1
        return out

    def run_program(self, prog, observe=None) -> Optional[Tensor]:
        """A ``program.StepProgram`` (the scenario's reward / done glue) in one launch, together with the
        state-slab columns of the observation plan ``observe`` if one is given."""
        self.refresh()
        cached = prog.device_cache.get(id(self))
        if cached is None or cached[0] != self._plan_version:
            N = self._native
            c = N.StepProgramC()
            c.n_instr = len(prog.instr)
            for k, (op, dst, a, b, arg, imm, entities) in enumerate(prog.instr):
                if entities is not None:
                    arg = self.index_of(entities[0]) | (self.index_of(entities[1]) << 16)
                ins = c.instr[k]
                ins.op, ins.dst, ins.a, ins.b, ins.arg, ins.imm = op, dst, a, b, arg, imm
            cached = (self._plan_version, c)
            prog.device_cache[id(self)] = cached
        c = cached[1]
        B = self.world.batch_dim
        for slot, buf in enumerate(prog.buffers):
            t = prog.resolve(buf)
            assert t.device == self.device and t.is_contiguous() and t.shape == (B,), "program buffers are contiguous [B] tensors on the world's device"
            assert t.dtype in (torch.float32, torch.bool, torch.uint8), "program buffers are fp32 or bool"
            c.buffers[slot] = t.data_ptr()
        if observe is not None:
            before = self.launches
            out = self.observe(observe, program=c)
            if self.trace is not None:
                self.trace.append(("post", self.launches - before, prog, observe, c, out))
            return out
        self._native.post_step(self.lib, self._dev_tables, self.world.slab, c, None, 0, 0, None)
        self.launches += 1
        if self.trace is not None:
            self.trace.append(("post", 1, prog, None, c, None))
        return None

    def observe(self, plan, program=None) -> Tensor:
        """``[rows, B, width]`` observation block of an ``observe.ObservationPlan``: one launch
        for the state-slab columns, one for all LIDAR columns."""
        self.refresh()
        cols, lidars = plan.compile(self.world)
        dev = plan.device_cache.get(id(self))
        B, F = self.world.batch_dim, plan.width
        if dev is None:
            dev = {"cols": torch.from_numpy(cols).to(self.device).contiguous(), "rays": None}
            dev["any_state"] = bool((cols[..., 0] != 0).any())
            if lidars:
                sensors = [s for _, _, s, _ in lidars]
                n_rays = {s._angles.shape[1] for s in sensors}
                assert len(n_rays) == 1, "LIDARs of one observation plan must have the same number of rays"
                src, off, flat = [], [0], []
                for s in sensors:
                    src.append(self.index_of(s.agent))
                    flat += self.ray_targets(s.agent, s.entity_filter)
                    off.append(len(flat))
                i32 = lambda v: torch.tensor(v if v else [0], dtype=torch.int32, device=self.device)  # noqa: E731
                dev["rays"] = (
                    i32(src),
                    i32(off),
                    i32(flat),
                    torch.stack([s._angles[0] for s in sensors]).to(self.device, torch.float32).contiguous(),
                    torch.tensor([float(s._max_range) for s in sensors], dtype=torch.float32, device=self.device),
                    n_rays.pop(),
                    torch.tensor([r * B * F + c for r, c, _, _ in lidars], dtype=torch.int64, device=self.device),
                    (self._native.RAYS_RANGE_MINUS_DISTANCE if lidars[0][3] else 0)
                    | (self._native.RAYS_SPHERE_TARGETS if self._all_spheres(flat) else 0),
                )
            plan.device_cache[id(self)] = dev
        out = torch.empty(plan.n_rows, B, F, dtype=torch.float32, device=self.device)
        buffers = plan.resolve_buffers()
        for t in buffers:
            assert t.device == self.device and t.dtype == torch.float32 and t.is_contiguous() and t.shape == (B,), \
                "observation value columns read contiguous fp32 [B] tensors on the world's device"
        if program is not None and buffers:
            # value columns read what the program stores: the program first, then the gather (in a captured
            # step both run in the whole-step kernel's epilogue, in this order, in the thread of the env)
            self._native.post_step(self.lib, self._dev_tables, self.world.slab, program, None, 0, 0, None)
            self._native.gather_observations(
                self.lib, self._dev_tables, self.world.slab, dev["cols"], plan.n_rows, F, out, buffers
            )
            self.launches += 2
        elif program is not None:
            # the scenario's reward / done program rides in the same launch as the state-slab columns
            self._native.post_step(
                self.lib, self._dev_tables, self.world.slab, program, dev["cols"] if dev["any_state"] else None,
                plan.n_rows, F, out,
            )
            self.launches += 1
        elif dev["any_state"]:
            self._native.gather_observations(
                self.lib, self._dev_tables, self.world.slab, dev["cols"], plan.n_rows, F, out, buffers
            )
            self.launches += 1
        if dev["rays"] is not None:
            src, off, flat, angles, ranges, n_rays, out_off, flags = dev["rays"]
            self._native.cast_rays_batched(
                self.lib, self._dev_tables, self.world.slab, src, off, flat, angles, ranges, n_rays, out, out_off, F,
                flags,
            )
            self.launches += 1
            for r, c, sensor, flipped in lidars:
                sensor._last_measurement = None if flipped else out[r, :, c : c + n_rays]
        return out

    def distance_shaping(self, pairs, factor: float, prev: Tensor):
        """``(dist, rew)`` of shape ``[K, B]`` with ``rew = prev - dist * factor``; ``prev`` (fp32
        ``[K, B]``, contiguous) is overwritten with ``dist * factor``.  One launch."""
        self.refresh()
        key = ("pairs",) + tuple((id(a), id(b)) for a, b in pairs)
        idx = self._ray_cache.get(key)
        if idx is None:
            idx = torch.tensor(
                [[self.index_of(a), self.index_of(b)] for a, b in pairs], dtype=torch.int32, device=self.device
            )
            self._ray_cache[key] = idx
        K, B = len(pairs), self.world.batch_dim
        assert prev.shape == (K, B) and prev.dtype == torch.float32 and prev.is_contiguous()
        out = torch.empty(2, K, B, dtype=torch.float32, device=self.device)
        self._native.distance_shaping(self.lib, self._dev_tables, self.world.slab, idx, factor, prev, out[0], out[1])
        self.launches += 1
        return out[0], out[1]

    def pair_query_many(self, pairs, mode: int) -> Tensor:
        """``[K, B]``: mode 0 distances, 1 overlaps (bool), 2 centre distances, one launch."""
        self.refresh()
        key = ("pairs+hint",) + tuple((id(a), id(b)) for a, b in pairs)
        cached = self._ray_cache.get(key)
        if cached is None:
            from .simulator.core import Sphere

            idx = torch.tensor(
                [[self.index_of(a), self.index_of(b)] for a, b in pairs], dtype=torch.int32, device=self.device
            )
            spheres = all(isinstance(e.shape, Sphere) for pair in pairs for e in pair)
            cached = self._ray_cache[key] = (idx, self._native.QUERY_SPHERES if spheres else 0)
        idx, hint = cached
        dtype = torch.bool if mode == 1 else torch.float32
        out = torch.empty(len(pairs), self.world.batch_dim, dtype=dtype, device=self.device)
        self._native.pair_query_batched(self.lib, self._dev_tables, self.world.slab, idx, mode | hint, out)
        self.launches += 1
        return out

    # -- action ingestion ----------------------------------------------------------------------
    def ingest_actions(self, actions, specs, clamp: bool, bad_flag, action_kind=None, steps=None, broad_phase=False) -> None:
        """One launch: validate + scale the policy actions and write ``agent.action.u`` and the
        force / torque rows of the slab.  ``specs``: [(agent, dynamics code, u buffer)].
        ``broad_phase``: the caller guarantees that nothing moves an entity before the coming
        ``world.step()``; the launch then also builds that step's first broad-phase mask."""
        self.refresh()
        broad_phase = bool(broad_phase and self.tables.n_masked > 0 and self.world.exact_broad_phase)
        n = len(specs)
        arr = getattr(self, "_ingest_arr", None)
        if arr is None or len(arr) != n or getattr(self, "_ingest_kind", None) != action_kind:
            self._ingest_kind = action_kind
            arr = (self._native.AgentActionsC * n)()
            agent_row = {id(a): j for j, a in enumerate(self.world.agents)}
            self._ingest_drones = []
            for c, (agent, dyn, u) in zip(arr, specs):
                c.u = u.data_ptr()
                c.action_size = agent.action_size
                c.agent_index = agent_row[id(agent)]
                c.dynamics = dyn
                c.entity_index = self.index_of(agent)
                c.action_kind = self._native.ACT_CONTINUOUS
                if action_kind is not None and action_kind != self._native.ACT_CONTINUOUS:
                    c.action_kind = action_kind
                    for j, choices in enumerate(agent.discrete_action_nvec):
                        c.nvec[j] = int(choices)
                if dyn >= self._native.DYN_DIFF_DRIVE:  # the kinematic models' parameters
                    model = agent.dynamics
                    params = [float(model.dt), float(agent.mass), float(agent.moment_of_inertia),
                              1.0 if model.integration == "rk4" else 0.0, 0.0, 0.0, 0.0, 0.0]
                    if dyn == self._native.DYN_BICYCLE:
                        params[4:7] = [float(model.l_f), float(model.l_r), float(model.max_steering_angle)]
                    elif dyn == self._native.DYN_DRONE:
                        params[4:8] = [float(model.I_xx), float(model.I_yy), float(model.I_zz), float(model.g)]
                        self._ingest_drones.append((c, model))
                    for j, v in enumerate(params):
                        c.dyn_params[j] = v
                rng = agent.action.u_range_tensor.tolist()
                mul = agent.action.u_multiplier_tensor.tolist()
                for j in range(agent.action_size):
                    c.u_range[j] = rng[j]
                    c.u_multiplier[j] = mul[j]
            self._ingest_arr = arr
        for c, a in zip(arr, actions):
            c.actions = a.data_ptr()
        for c, model in self._ingest_drones:  # a reset re-binds the drone's 12-state tensor
            c.dyn_state = model.drone_state.data_ptr()
        for lo in range(0, n, self._native.MAX_INGEST_AGENTS):
            hi = min(n, lo + self._native.MAX_INGEST_AGENTS)
            chunk = (self._native.AgentActionsC * (hi - lo)).from_address(
                C.addressof(arr) + lo * C.sizeof(self._native.AgentActionsC)
            )
            self._native.ingest_actions(
                self.lib, self._dev_tables, self.world.slab, chunk, hi - lo, clamp, bad_flag,
                steps=steps if lo == 0 else None,  # the step counter and the broad phase ride in the first launch
                broad_phase=broad_phase and lo == 0,
            )
            self.launches += 1
        self._mask_ready = broad_phase

    # -- episode reset (device side, SURVEY 8(f)-4) ------------------------------------------------
    @staticmethod
    def _selection(env_index):
        """``None`` / int / bool tensor ``[B]``  ->  (env_index or None, uint8 mask view or None)."""
        if env_index is None:
            return None, None
        if isinstance(env_index, Tensor):
            if env_index.dtype != torch.bool or env_index.dim() != 1:
                raise TypeError("a tensor env selection must be a 1-D bool mask over the envs")
            return None, env_index.contiguous().view(torch.uint8)
        return int(env_index), None

    def _slab_handle(self):
        """Sizes + slab pointers for the reset entry points; they do not need the compiled plan (a
        scenario's collision filters may depend on state that only its first reset creates)."""
        slab = self.world.slab
        cached = getattr(self, "_slab_handle_cache", None)
        if cached is None or cached[0] is not slab:
            index = {id(e): i for i, e in enumerate(self.world.entities)}
            cached = self._slab_handle_cache = (slab, self._native.SlabHandle(slab), index)
        return cached[1]

    def _slab_index_of(self, entity) -> int:
        self._slab_handle()
        try:
            return self._slab_handle_cache[2][id(entity)]
        except KeyError:
            raise RuntimeError(f"Entity '{entity.name}' does not belong to this world") from None

    def reset_state(self, env_index, reset_count: Optional[Tensor]) -> None:
        """``World.reset(env_index)`` in one launch: zero the state rows of the selected envs and bump
        their episode counters (ref core.py:1179-1181, 286-296)."""
        index, mask = self._selection(env_index)
        if mask is not None:
            assert mask.shape[0] == self.world.batch_dim and mask.device == self.device
        self._native.reset_state(self.lib, self._slab_handle(), index, mask, reset_count)
        self.launches += 1

    def spawn(
        self,
        entities,
        env_index,
        min_dist: float,
        x_bounds,
        y_bounds,
        seed: int,
        stream_id: int,
        reset_count: Optional[Tensor],
        status: Optional[Tensor],
        occupied: Optional[Tensor] = None,
        occupied_entities=(),
        want_positions: bool = False,
        max_tries: int = 1 << 16,
    ) -> Optional[Tensor]:
        """Rejection-sampled respawn (ref utils.py:241-319) of up to ``MAX_SPAWN`` positions per
        selected env in one launch.  ``entities``: ``Entity`` objects (their slab rows are written)
        or ``None`` entries (position only returned).  ``occupied``: fp32 ``[B or 1, K, 2]``.
        Returns the drawn positions ``[B, n, 2]`` when ``want_positions`` (rows of unselected envs
        are zero), else ``None``."""
        n = len(entities)
        assert 0 < n <= self._native.MAX_SPAWN and len(occupied_entities) <= self._native.MAX_SPAWN
        index, mask = self._selection(env_index)
        sp = self._native.SpawnC()
        sp.n_spawn = n
        for i, e in enumerate(entities):
            sp.entity[i] = -1 if e is None else self._slab_index_of(e)
        sp.n_occupied_entities = len(occupied_entities)
        for i, e in enumerate(occupied_entities):
            sp.occupied_entity[i] = self._slab_index_of(e)
        B = self.world.batch_dim
        if occupied is not None and occupied.shape[1] > 0:
            occupied = occupied.to(device=self.device, dtype=torch.float32).contiguous()
            assert occupied.dim() == 3 and occupied.shape[2] == 2 and occupied.shape[0] in (1, B)
            sp.occupied = occupied.data_ptr()
            sp.n_occupied = occupied.shape[1]
            # a [1, K, 2] block is shared by all envs (for a single env index it is that env's rows)
            sp.occupied_env_stride = occupied.shape[1] * 2 if (occupied.shape[0] == B and index is None) else 0
            if index is not None and occupied.shape[0] == B and B > 1:
                sp.occupied = occupied[index].data_ptr()
        out = None
        if want_positions:
            out = torch.zeros(B, n, 2, dtype=torch.float32, device=self.device)
            sp.out = out.data_ptr()
        sp.min_dist = float(min_dist)
        sp.x_lo, sp.x_hi = float(x_bounds[0]), float(x_bounds[1])
        sp.y_lo, sp.y_hi = float(y_bounds[0]), float(y_bounds[1])
        sp.env_index = -1 if index is None else index
        sp.env_mask = None if mask is None else mask.data_ptr()
        sp.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        sp.stream_id = int(stream_id) & 0xFFFFFFFF
        sp.env_offset = int(getattr(self.world, "env_offset", 0)) & 0xFFFFFFFF
        sp.reset_count = None if reset_count is None else reset_count.data_ptr()
        sp.status = None if status is None else status.data_ptr()
        sp.max_tries = int(max_tries)
        self._native.spawn_entities(self.lib, self._slab_handle(), sp)
        self.launches += 1
        return out

    # -- queries -----------------------------------------------------------------------------
    def pair_distance(self, a, b) -> Tensor:
        ia, ib = self.index_of(a), self.index_of(b)
        out = torch.empty(self.world.batch_dim, dtype=torch.float32, device=self.device)
        self._native.pair_query(self.lib, self._dev_tables, self.world.slab, ia, ib, 0, out)
        self.launches += 1
        return out

    def pair_overlap(self, a, b) -> Tensor:
        ia, ib = self.index_of(a), self.index_of(b)
        out = torch.empty(self.world.batch_dim, dtype=torch.bool, device=self.device)
        self._native.pair_query(self.lib, self._dev_tables, self.world.slab, ia, ib, 1, out)
        self.launches += 1
        return out

    def distance_from_point(self, entity, point: Tensor) -> Tensor:
        ie = self.index_of(entity)
        point = point.to(device=self.device, dtype=torch.float32)
        if point.dim() == 1:
            point = point.unsqueeze(0)
        point = point.expand(self.world.batch_dim, 2).contiguous()
        out = torch.empty(self.world.batch_dim, dtype=torch.float32, device=self.device)
        self._native.point_query(self.lib, self._dev_tables, self.world.slab, ie, point, out)
        self.launches += 1
        return out
