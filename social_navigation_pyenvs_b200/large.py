"""One very large crowd (tens of thousands of humans in ONE environment), optionally sharded by agent across GPUs.

Every rank owns a contiguous slice of agents and evaluates their forces against ALL agents (ordered pairs: the reference's
symmetric accumulation, forces.py:148, is not carried across ranks).  The only exchange per sub-step is an all-gather of the
entity view (x, y, vx, vy, r+safety) over NCCL / NVLink; it is double buffered so the step kernel writes the next view's own
slice while reading the current one.  Reference semantics: motion_model_manager.py:354-373 for a single env.

With a robot (`robot=`), `step` is SocialNavGym.step (social_nav_gym.py:227-250) for the one env: the swept collision / goal / reward
check, then n_substeps x (robot.step; update_humans), then optionally the actual check; `scan` is the robot's laser.  The robot is
fixed, holonomic or unicycle (no motion model), visible to the humans or not.  Every rank keeps the robot and recomputes it
identically, so the flags and the robot are the same on every rank.

The checks read the humans from the entity view: positions, radii and the velocity the humans exert force with -- R(yaw) bv for
headed models.  That is the stored velocity for every state the engine produces and after every reset; it can differ only for rows
the engine did not produce, until their first step -- including rows whose velocity was computed as R(yaw) bv on the host (a host
cos / sin can differ from the device's in the last bit).
"""
import ctypes

import numpy as np
import torch

from . import _lib as L
from .engine import CrowdEngine, SFMS
from .parallel import all_gather_columns, all_gather_columns_packed, agent_shard

# unit_capacity="auto" starts with this many partial-sum slots per 128-agent block (DESIGN 4.3: what the bench crowd lists)
AUTO_UNITS_PER_BLOCK = 32


class _UnitSlots:
    """The scratch of the tiled path, with the partial sums of a culled step sized for `unit_capacity` (agent block, entity chunk)
    units in reach (SNP_OPT_UNIT_SCRATCH) instead of one per chunk and agent.  None: the default size.  An int: that many slots.
    "auto": min(all units, AUTO_UNITS_PER_BLOCK per agent block) to start with; after a call that listed more units than that, the
    next call gets ceil(1.25 x the most listed) -- which costs one device synchronisation per call to read the count.  Units without
    a slot are evaluated by the finish kernel: the results are the same bits whatever the capacity, only slower."""

    def _setup_units(self, unit_capacity, blocks, J, size_of, device):
        self._units_all, self._size_of, self._units_device = blocks * J, size_of, device
        self._auto = isinstance(unit_capacity, str)
        if unit_capacity is None:
            cap = None
        elif self._auto:
            if unit_capacity != "auto":
                raise ValueError(f"unit_capacity must be None, an int >= 0 or 'auto' (got {unit_capacity!r})")
            cap = min(self._units_all, AUTO_UNITS_PER_BLOCK * blocks)
        else:
            cap = int(unit_capacity)
            if cap < 0 or cap != unit_capacity or isinstance(unit_capacity, bool):
                raise ValueError(f"unit_capacity must be None, an int >= 0 or 'auto' (got {unit_capacity!r})")
        self._stats = torch.zeros((2,), dtype=torch.int32, device=device)  # the last call's (most units listed, units without a slot)
        self._stats_valid, self._last_capacity = False, cap
        self._alloc_units(cap)

    def _alloc_units(self, cap):
        self.unit_capacity = cap
        self.scratch = None  # release the old scratch before the new one is allocated
        self.scratch = torch.empty(int(self._size_of(cap)), dtype=torch.uint8, device=self._units_device)

    def _unit_bits(self):
        return 0 if self.unit_capacity is None else L.SNP_OPT_UNIT_SCRATCH

    def _collect_units(self, first):
        """After a C call with a capacity: its unit counts (int32 words 1 and 2 of the scratch) into the step's, on the stream."""
        if self.unit_capacity is None:  # the default size keeps no counts
            return
        w = self.scratch[:12].view(torch.int32)[1:3]
        if first:
            self._stats.copy_(w)
        else:
            torch.maximum(self._stats[0:1], w[0:1], out=self._stats[0:1])
            self._stats[1:2] += w[1:2]

    def _end_units(self):
        """After a step: the counts exist when it had a capacity (a step with one that does not take the work list is refused
        before any launch).  "auto" grows for the next step."""
        listed = self.unit_capacity is not None
        self._stats_valid, self._last_capacity = listed, self.unit_capacity
        if self._auto and listed:
            most = int(self._stats[0].item())  # the synchronisation "auto" costs
            if most > self.unit_capacity:
                self._alloc_units(min(self._units_all, -(-5 * most // 4)))

    def unit_stats(self):
        """The last step's {capacity, max_listed, fallback_units}: the partial-sum slots it had (None: the default size), the most
        (agent block, entity chunk) units listed in one of its sub-steps and the units the finish kernel evaluated for want of a slot.
        The counts are kept only with a capacity: None at the default size."""
        most, fallback = (int(v) for v in self._stats.tolist()) if self._stats_valid else (None, None)
        return {"capacity": self._last_capacity, "max_listed": most, "fallback_units": fallback}


def device_spatial_order(px, py, world=1):
    """scenarios.spatial_order of every env's positions on the device (snp_spatial_order): px, py device tensors [E, N] (or [N]) of
    float32 / float64 -> int64 device tensor of the same shape, perm[e][k] = the index the human going to place k has now.  world > 1
    also deals the 128-human tiles to `world` ranks (scenarios.deal_tiles; N a whole number of tiles).  Non-finite positions raise
    ValueError (reading that flag synchronises the stream)."""
    lib = L.lib()
    x, y = px.contiguous(), py.contiguous()
    E, N = (1, x.numel()) if x.dim() == 1 else tuple(x.shape)
    perm = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    flag = torch.empty((1,), dtype=torch.int32, device=x.device)
    scratch = torch.empty((L.check_size(lib.snp_spatial_order_scratch_bytes(E, N)),), dtype=torch.uint8, device=x.device)
    dt = L.SNP_F64 if x.dtype == torch.float64 else L.SNP_F32
    L.check(lib.snp_spatial_order(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), E, N, dt, int(world),
                                  ctypes.c_void_p(perm.data_ptr()), ctypes.c_void_p(flag.data_ptr()), ctypes.c_void_p(scratch.data_ptr()),
                                  scratch.numel(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    if int(flag.item()):
        raise ValueError("spatial order: a position is NaN or infinite")
    return perm


def _gather_crowd(eng, perm, offset, src):
    """eng's per-agent arrays (its slice [offset, offset + eng.N) of every env) := those of `src` re-numbered by perm [E, M] (device
    int64); src = (dyn [10, E, M], stat [4, E, M], goals [G, 2, E, M], goal_idx [E, M], goal_cnt [E, M]) not overlapping eng's."""
    dyn, stat, goals, gi, gc = src
    c = eng._crowd()  # the source crowd: eng's E, G, dtype and parameters, its own N and arrays
    c.N = gi.shape[-1]
    c.dyn, c.stat, c.goals, c.goal_idx, c.goal_cnt = dyn.data_ptr(), stat.data_ptr(), goals.data_ptr(), gi.data_ptr(), gc.data_ptr()
    err = torch.zeros((1,), dtype=torch.int32, device=eng.device)
    L.check(eng.lib.snp_gather_crowd(ctypes.byref(eng._crowd()), ctypes.byref(c), ctypes.c_void_p(perm.data_ptr()), int(offset),
                                     ctypes.c_void_p(err.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    if int(err.item()):
        raise ValueError("renumber: a permutation entry is out of range")


def _own_arrays(eng):
    """Copies of eng's per-agent arrays: the source of a re-numbering of the crowd itself."""
    return eng.dyn.clone(), eng.stat.clone(), eng.goals.clone(), eng.goal_idx.clone(), eng.goal_cnt.clone()


class LargeCrowd(_UnitSlots):
    def __init__(self, model, states, goals, walls=None, dtype=torch.float64, device="cuda", symmetric=True, numba_compat=False,
                 rank=0, world=1, group=None, safety=None, exchange="auto", shard=None, robot=None, robot_safety=None, consider_robot=False,
                 unit_capacity=None):
        """states [N_total,13], goals [N_total,G,2] (the WHOLE crowd on every rank; each rank keeps its slice).
        shard=(offset, n_local) with world=1 steps only that slice against a frozen rest of the crowd (profiling what ONE rank of
        a sharded run executes, on one GPU).
        robot: the robot's 13-wide reference row (robot.get_safe_state(), as CrowdEngine.set_robot_rows), robot_safety its safety
        space (default 0); consider_robot: the humans feel its force (motion_model_manager.py:35).
        unit_capacity: None, an int or "auto" -- the partial-sum slots of the scratch (_UnitSlots; unit_stats()).  The default size
        holds n_local * n_total / 16 bytes of partial sums in fp64; a capacity near what a step lists lets crowds of millions of
        humans fit on one GPU.  With a capacity, Moussaid models, culling = False and a slice that does not start on a 128-human
        tile raise NotImplementedError at the step."""
        states = np.asarray(states, np.float64)
        goals = np.asarray(goals, np.float64)
        self.n_total = states.shape[0]
        self.rank, self.world, self.group = rank, world, group
        self.offset, self.n_local = agent_shard(self.n_total, rank, world) if shard is None else shard
        sl = slice(self.offset, self.offset + self.n_local)
        saf = None if safety is None else np.asarray(safety, np.float64)[None, sl]
        if consider_robot and robot is None:
            raise ValueError("consider_robot needs a robot row")
        self.eng = CrowdEngine.from_reference_arrays(model, states[None, sl], goals[None, sl], walls=walls, safety=saf, consider_robot=False,
                                                     all_params_equal=symmetric, numba_compat=numba_compat, dtype=dtype, device=device)
        self.has_robot = robot is not None
        if self.has_robot:
            self.eng.robot = torch.zeros((L.ROBOT_FIELDS, 1), dtype=dtype, device=self.eng.device)
            self.eng.set_robot_rows(np.asarray(robot, np.float64).reshape(1, 13), safety=[0.0 if robot_safety is None else float(robot_safety)])
            self.eng.consider_robot = bool(consider_robot)  # the robot is not a row of `states`: only the step options carry it
            # the radii of the WHOLE crowd (the checks and the laser see every human)
            self.radius = torch.as_tensor(states[:, 8], dtype=dtype, device=self.eng.device)
        self.type = SFMS.index(model)
        # exchange of the entity view between ranks: "p2p" = the producer kernel stores into every rank's next view through
        # peer-mapped (torch symmetric memory, NVLink) pointers and only a barrier separates sub-steps; "nccl" = all-gather
        # after every sub-step.  "auto" tries p2p on multi-GPU runs and falls back to nccl.
        self.exchange, self._symm = "nccl", None
        # a view buffer = the [5, N] entity view followed by the [N/128, 5] bounding boxes of its 128-entity tiles (see
        # snp_large_run_p2p)
        self._n_tiles = (self.n_total + 127) // 128
        vlen = 5 * self.n_total + 5 * self._n_tiles
        fused_ok = self.n_local % 128 == 0
        if world > 1 and exchange in ("auto", "p2p") and fused_ok:
            try:
                import torch.distributed as dist
                import torch.distributed._symmetric_memory as symm_mem
                grp = group if group is not None else dist.group.WORLD
                self._vbuf = [symm_mem.empty((vlen,), dtype=dtype, device=self.eng.device) for _ in range(2)]
                self._flags = symm_mem.empty((16,), dtype=torch.int64, device=self.eng.device)
                for v in self._vbuf + [self._flags]:
                    v.zero_()
                self._symm = [symm_mem.rendezvous(v, grp) for v in self._vbuf]
                self._symm_flags = symm_mem.rendezvous(self._flags, grp)
                self._peer_ptrs = [(ctypes.c_void_p * world)(*[int(p) for p in h.buffer_ptrs]) for h in self._symm]
                self._peer_flags = (ctypes.c_void_p * world)(*[int(p) for p in self._symm_flags.buffer_ptrs])
                torch.cuda.synchronize()
                self._symm[0].barrier()
                self.exchange = "p2p"
            except Exception as exc:  # no peer access / symmetric memory unavailable
                if exchange == "p2p":
                    raise
                self._p2p_error = repr(exc)
        elif world == 1 and fused_ok and exchange != "nccl":
            self.exchange = "fused"  # one GPU: the sub-step loop inside one C call, no barrier
        if self.exchange != "p2p":  # this rank's own two view buffers
            self._vbuf = [torch.zeros((vlen,), dtype=dtype, device=self.eng.device) for _ in range(2)]
            self._flags = torch.zeros((16,), dtype=torch.int64, device=self.eng.device)
            self._peer_ptrs = [(ctypes.c_void_p * 1)(v.data_ptr()) for v in self._vbuf]
            self._peer_flags = (ctypes.c_void_p * 1)(self._flags.data_ptr())
        self.view = [v[:5 * self.n_total].view(5, self.n_total) for v in self._vbuf]
        self._epoch = 0
        self._err = torch.zeros((1,), dtype=torch.int32, device=self.eng.device)
        dt, lib = (L.SNP_F64 if dtype == torch.float64 else L.SNP_F32), self.eng.lib
        size_of = lambda units: (lib.snp_large_scratch_bytes(self.n_local, self.n_total, dt) if units is None else
                                 L.check_size(lib.snp_large_scratch_bytes_units(self.n_local, self.n_total, dt, units)))
        self._setup_units(unit_capacity, -(-self.n_local // 128), -(-self.n_total // 128), size_of, self.eng.device)
        self.culling = True
        self.cur = 0
        self._sharded_slice = shard is not None
        if shard is not None:  # the frozen rest of the crowd: both view buffers start from the whole crowd's entries
            whole = CrowdEngine.from_reference_arrays(model, states[None], goals[None], consider_robot=False, all_params_equal=symmetric, dtype=dtype, device=device)
            for v in self.view:
                L.check(whole.lib.snp_large_publish(ctypes.byref(whole._crowd()), self.type, ctypes.c_void_p(v.data_ptr()), self.n_total, 0, self._stream()))
        self._publish()

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _gather(self, buf):
        all_gather_columns(buf, self.offset, self.n_local, self.world, self.group)
        if self.exchange == "p2p":
            self._symm[0].barrier()

    def check_peers(self):
        """Raises if a rank never reached a sub-step barrier (the barrier kernel timed out instead of hanging the GPU)."""
        if int(self._err.item()):
            raise RuntimeError("LargeCrowd: a peer rank did not reach the sub-step barrier")

    def _publish(self):
        v = self.view[self.cur]
        L.check(self.eng.lib.snp_large_publish(ctypes.byref(self.eng._crowd()), self.type, ctypes.c_void_p(v.data_ptr()), self.n_total,
                                               self.offset, self._stream()))
        self._gather(v)

    def renumber(self):
        """Re-numbers the whole crowd patch by patch (scenarios.spatial_order of the current positions, then deal_tiles over the ranks
        when world > 1 and the crowd is a whole number of 128-human tiles) and returns perm (int64 [n_total], host): perm[k] is the
        index the human now at k had before, new_rows = old_rows[perm]; np.argsort(perm) undoes it.  Every per-agent array moves with
        its human -- state, carried desired force, safety, goal list and the index of the current goal -- and so do the radii the
        checks and the laser read; the view and its tile boxes are republished.  Every index reported afterwards (rows, laser hits)
        is in the new numbering.  The steps that follow compute what a crowd built from the re-numbered rows computes, bit for bit,
        and their far-tile culling skips as much as on a freshly ordered crowd.  Every rank computes the same permutation from the
        view it holds; with world > 1 the other ranks' agents arrive in one all-gather.  Slice sizes and offsets, the robot and the
        unit capacity do not change."""
        if self._sharded_slice:
            raise ValueError("renumber: a crowd built with shard= steps a slice against a frozen rest and cannot be re-numbered")
        e, M, v = self.eng, self.n_total, self.view[self.cur]
        deal = self.world if self.world > 1 and M % 128 == 0 else 1
        perm = device_spatial_order(v[0], v[1], world=deal)
        if self.world == 1:
            src = _own_arrays(e)
        else:  # the whole crowd in the old numbering, from every rank's slice
            d = e.dtype
            dyn, stat = torch.empty((L.DYN_FIELDS, 1, M), dtype=d, device=e.device), torch.empty((L.STAT_FIELDS, 1, M), dtype=d, device=e.device)
            goals = torch.empty((e.G, 2, 1, M), dtype=d, device=e.device)
            ints = torch.empty((2, M), dtype=torch.int32, device=e.device)
            sl = slice(self.offset, self.offset + self.n_local)
            dyn[..., sl], stat[..., sl], goals[..., sl] = e.dyn, e.stat, e.goals
            ints[0, sl], ints[1, sl] = e.goal_idx[0], e.goal_cnt[0]
            all_gather_columns_packed([dyn.view(-1, M), stat.view(-1, M), goals.view(-1, M), ints], self.offset, self.n_local, self.world,
                                      self.group)
            src = (dyn, stat, goals, ints[0:1], ints[1:2])
        _gather_crowd(e, perm.view(1, M), self.offset, src)
        if self.has_robot:
            self.radius = self.radius[perm]
        self._publish()
        L.check(e.lib.snp_large_tile_boxes(ctypes.c_void_p(self.view[self.cur].data_ptr()), M,
                                           L.SNP_F64 if e.dtype == torch.float64 else L.SNP_F32, self._stream()))
        return perm.cpu().numpy()

    def step(self, dt=0.0125, n_substeps=1, action=None, kinematics="holonomic", pre_checks=False, post_checks=False):
        """n_substeps updates of the crowd.  With a robot: SocialNavGym.step -- the swept check on the current state (pre_checks),
        n_substeps x (robot.step(action, dt); update_humans(dt)), the actual check on the end state (post_checks); the clock
        (eng.time_now) advances by dt per sub-step.  action (vx, vy), or (v, r) with kinematics="unicycle"; None keeps the robot
        where it is (and the swept check sweeps a robot at rest).  Results: decode_flags(), robot_rows()."""
        if kinematics not in ("holonomic", "unicycle"):
            raise ValueError("kinematics must be 'holonomic' or 'unicycle'")
        mode = 0
        if self.has_robot:
            if action is None:
                self.eng.action.zero_()
            else:
                self.eng.action.copy_(torch.as_tensor(np.asarray(action, np.float64).reshape(2, 1), dtype=self.eng.dtype))
                mode = 1 if kinematics == "holonomic" else 3
            self.eng.flags.zero_()
            self.eng.checks.zero_()
        elif action is not None or pre_checks or post_checks:
            raise ValueError("this crowd has no robot: build it with robot=")
        if pre_checks:
            self._checks(dt, mode, pre=True)
        c = self.eng._crowd()
        o = self.eng._opts(dt, 1, robot_mode=mode, advance_time=self.has_robot)
        o.reserved = (0 if self.culling else L.SNP_OPT_NO_CULLING) | self._unit_bits()
        # p2p / fused: the whole sub-step loop in ONE C call, nothing returns to Python in between; nccl: one sub-step per call on
        # this rank's own buffers, then the all-gather of the next view
        nccl = self.exchange == "nccl"
        world, rank, calls, k = (1, 0, n_substeps, 1) if nccl else (self.world, self.rank, 1, int(n_substeps))
        for call in range(calls):
            L.check(self.eng.lib.snp_large_run_p2p(ctypes.byref(c), ctypes.byref(o), self._peer_ptrs[0], self._peer_ptrs[1], self.cur, self.n_total,
                                                   self.offset, world, rank, self._peer_flags, self._epoch, k,
                                                   ctypes.c_void_p(self._err.data_ptr()), ctypes.c_void_p(self.scratch.data_ptr()),
                                                   self.scratch.numel(), self._stream()))
            self._collect_units(first=call == 0)
            self._epoch += k
            self.cur ^= k & 1
            if nccl:
                self._gather(self.view[self.cur])
        if n_substeps > 0:
            self._end_units()
        if post_checks:
            self._checks(dt, mode, pre=False)

    def _checks(self, dt, mode, pre):
        o = self.eng._opts(dt, 0, robot_mode=mode, pre_checks=pre, post_checks=not pre)
        L.check(self.eng.lib.snp_large_checks(ctypes.byref(self.eng._crowd()), ctypes.byref(o), ctypes.c_void_p(self.view[self.cur].data_ptr()),
                                              ctypes.c_void_p(self.radius.data_ptr()), self.n_total, self._stream()))

    def decode_flags(self):
        """The checks of the last step (CrowdEngine.decode_flags for the one env: arrays of length 1)."""
        return self.eng.decode_flags()

    def robot_rows(self):
        """The robot as a 13-wide reference row."""
        return self.eng.robot_rows()[0][0]

    def scan(self, range_, samples, max_distance, robot_radius=0.0):
        """The robot's laser (LaserSensor.get_laser_measurements, robot_agent.py:77-82) over the whole crowd and the walls: one
        snp_laser launch.  Returns device tensors (ranges [samples] in the crowd's dtype, hits [samples] int32: the global human
        index, M + the wall segment's ordinal, or -1)."""
        if not self.has_robot:
            raise ValueError("this crowd has no robot: build it with robot=")
        if max_distance > 10:
            raise ValueError("Maxium distance for laser is 10 meters")  # sensors.py:13
        e = self.eng
        pose = e.robot[[L.ROBOT_PX, L.ROBOT_PY, L.ROBOT_TH]].contiguous()
        ranges = torch.empty((int(samples),), dtype=e.dtype, device=e.device)
        hits = torch.empty((int(samples),), dtype=torch.int32, device=e.device)
        v = self.view[self.cur]
        a = L.SnpLaserArgs()
        a.E, a.N, a.samples = 1, self.n_total, int(samples)
        a.dtype = L.SNP_F64 if e.dtype == torch.float64 else L.SNP_F32
        a.px, a.py, a.radius = v[0].data_ptr(), v[1].data_ptr(), self.radius.data_ptr()
        a.walls = None if e.walls is None else e.walls.data_ptr()
        a.W, a.S, a.walls_per_env = e.W, e.S, 0
        a.pose, a.range, a.max_distance, a.robot_radius = pose.data_ptr(), float(range_), float(max_distance), float(robot_radius)
        a.ranges, a.hits = ranges.data_ptr(), hits.data_ptr()
        L.check(e.lib.snp_laser(ctypes.byref(a), self._stream()))
        return ranges, hits

    def local_rows(self, template):
        """This rank's agents as reference rows; `template` [n_local,13] supplies the static columns."""
        return self.eng.rows(np.asarray(template, np.float64)[None])[0]


class TiledCrowdEngine(_UnitSlots, CrowdEngine):
    """CrowdEngine for E environments of any number of humans each, N > 512 included: `update_humans` and `step` run
    snp_large_batch_step (the tiled kernels of LargeCrowd with an environment axis) in one call per step.  Environment e steps
    bit for bit as a LargeCrowd built from environment e alone.  Loading and reading are CrowdEngine's (from_reference_arrays,
    rows, robot_rows, set_robot_rows, decode_flags, set_safety_space, walls shared or per env), and so is the policies' lookahead
    without a query of the env: lookahead(query_env=False) (the constant-velocity propagation, snp_constant_velocity) and
    lookahead_from(next) work at any N (snp_lookahead splits an env's humans over several CTAs when one cannot hold them), and so do
    predict(query_env=False) and predict_from(next), CADRL's action choice with its value network on the device (snp_value_lookahead).  The
    checks without a step (run_checks, check_actual_collisions_and_goal, collision_detection_and_reaching_goal) work at any N.
    Per-agent parameter rows, respawn and the snp_step features the tiled path does not have (peek and the lookahead through it,
    lookahead(query_env=True), imitation_learning_step, sim_update, step_host) raise.  `scratch` is the call's workspace (view buffers, tile boxes, partial sums, work lists); nothing in it is
    carried from one step to the next.  culling=False evaluates every pair (the same result).  unit_capacity (a constructor and
    from_reference_arrays keyword): None, an int or "auto", as for LargeCrowd (_UnitSlots; unit_stats())."""

    def __init__(self, *args, unit_capacity=None, **kwargs):
        super().__init__(*args, **kwargs)
        dt, lib, E, N = (L.SNP_F64 if self.dtype == torch.float64 else L.SNP_F32), self.lib, self.E, self.N
        size_of = lambda units: (lib.snp_large_batch_scratch_bytes(E, N, dt) if units is None else
                                 L.check_size(lib.snp_large_batch_scratch_bytes_units(E, N, dt, units)))
        self._setup_units(unit_capacity, E * -(-N // 128), -(-N // 128), size_of, self.device)
        self.culling = True

    def _run(self, o):
        o.reserved = (0 if self.culling else L.SNP_OPT_NO_CULLING) | self._unit_bits()
        L.check(self.lib.snp_large_batch_step(ctypes.byref(self._crowd()), ctypes.byref(o), ctypes.c_void_p(self.scratch.data_ptr()),
                                              self.scratch.numel(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        if o.n_substeps > 0:
            self._collect_units(first=True)
            self._end_units()

    def update_humans(self, t=0.0, dt=0.0125, post_update=True, n_substeps=1):
        """MotionModelManager.update_humans (motion_model_manager.py:354) for every env: `n_substeps` Euler updates in one call."""
        self._run(self._opts(dt, n_substeps, post_update=post_update))

    def step(self, action=None, dt=0.0125, n_substeps=20, pre_checks=True, post_checks=False, kinematics="holonomic"):
        """SocialNavGym.step for every env (social_nav_gym.py:227-250), as CrowdEngine.step: the swept check on the current state,
        `n_substeps` x (robot.step(action, dt); update_humans(dt)), the actual check on the end state (post_checks).  `action` [E,2]
        (vx, vy), or (v, r) with kinematics="unicycle"; None reuses self.action.  Results in self.flags / checks / time_now."""
        if kinematics not in ("holonomic", "unicycle"):
            raise ValueError("kinematics must be 'holonomic' or 'unicycle'")
        if action is not None:
            a = torch.as_tensor(action, dtype=self.dtype, device=self.device)
            self.action.copy_(a.t() if a.shape == (self.E, 2) else a)
        self._run(self._opts(dt, n_substeps, robot_mode=1 if kinematics == "holonomic" else 3, pre_checks=pre_checks,
                             post_checks=post_checks, advance_time=True))

    def run_checks(self, action=None, pre=True, post=True, kinematics="holonomic"):
        """CrowdEngine.run_checks at any N, and through it check_actual_collisions_and_goal and
        collision_detection_and_reaching_goal.  N <= 512 with a holonomic action keeps CrowdEngine's snp_checks; otherwise one
        snp_large_batch_step call with n_substeps = 0, whose env e gives the flags and checks of a LargeCrowd of env e alone, bit for
        bit.  kinematics="unicycle" sweeps the robot with action (v, r), as step does."""
        if kinematics not in ("holonomic", "unicycle"):
            raise ValueError("kinematics must be 'holonomic' or 'unicycle'")
        if self.N <= 512 and kinematics == "holonomic":
            return super().run_checks(action, pre, post)
        if action is not None:
            a = torch.as_tensor(action, dtype=self.dtype, device=self.device)
            self.action.copy_(a.t() if a.shape == (self.E, 2) else a)
        self._run(self._opts(0.0, 0, robot_mode=1 if kinematics == "holonomic" else 3, pre_checks=pre, post_checks=post))
        return self.decode_flags()

    def renumber(self):
        """Re-numbers the humans of every env among themselves patch by patch (scenarios.spatial_order of the env's current
        positions) and returns perm (int64 [E, N], host): perm[e][k] is the index in env e the human now at k had before,
        new_rows[e] = old_rows[e][perm[e]]; np.argsort(perm[e]) undoes it.  Every per-agent array moves with its human -- state,
        carried desired force, safety, goal list and the index of the current goal; the robots and the walls stay.  Every index
        reported afterwards (rows, laser hits, the swept check's first collision) is in the new numbering: compose perm with any
        bookkeeping of your own.  Env e then steps bit for bit as a LargeCrowd of env e alone re-numbered the same way."""
        return self._renumber().cpu().numpy()

    def _renumber(self):
        """renumber() with perm left on the device."""
        perm = device_spatial_order(self.dyn[L.DYN_PX], self.dyn[L.DYN_PY])
        _gather_crowd(self, perm, 0, _own_arrays(self))
        return perm

    def _unsupported(self, what):
        raise NotImplementedError(f"TiledCrowdEngine: {what} is not available on the tiled path (snp_large_batch_step)")

    def peek(self, dt):
        self._unsupported("peek (and the lookahead and observable states through it)")

    def imitation_learning_step(self, dt=0.0125, n_substeps=20):
        self._unsupported("imitation_learning_step (robot_mode 2)")

    def sim_update(self, dt=0.0125, n_updates=1, robot_every=1, robot_time_step=None, phase=0):
        self._unsupported("sim_update (robot_mode 2, track_touch)")

    def step_host(self, *args, **kwargs):
        self._unsupported("step_host")
