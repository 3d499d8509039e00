"""CrowdEngine: E independent environments of N humans, resident on one B200, stepped by the fused CUDA kernels.

Host-side mirror of the reference's MotionModelManager surface (social_gym/src/motion_model_manager.py):
`update_humans` (:354), `get_human_states` (:285), `set_human_states` (:314), `get_next_human_observable_states` (:691),
`set_safety_space` (:147) -- with a leading env axis on every array -- plus the gym-level fused step
(social_gym/social_nav_gym.py:227-250) and the collision / goal checks (:107-118, social_nav_sim.py:949-1029).

State is held in torch CUDA tensors in structure-of-arrays form (include/snp_b200.h); torch is plumbing only
(memory, streams): all arithmetic happens inside libsnp_b200.so.
"""
import ctypes

import numpy as np
import torch

from . import _lib as L

# social_gym/src/motion_model_manager.py:15-17
SFMS = ["sfm_helbing", "sfm_guo", "sfm_moussaid", "hsfm_farina", "hsfm_guo", "hsfm_moussaid",
        "hsfm_new", "hsfm_new_guo", "hsfm_new_moussaid"]
INFO_NAMES = ["Nothing", "Timeout", "Collision", "ReachGoal", "Danger"]  # social_gym/src/info.py


def model_parameters(title: str) -> np.ndarray:
    """The 20-vector [relax_t,Ai,Aw,Bi,Bw,Ci,Cw,Di,Dw,Ei,k1,k2,lambda,gamma,ns,ns1,ko,kd,alpha,k_lambda] that
    Agent.set_parameters + get_parameters produce for `title` (social_gym/src/agent.py:94-243,268-388)."""
    if title not in SFMS:
        raise Exception(f"The human motion model '{title}' does not exist")  # motion_model_manager.py:252
    t = SFMS.index(title)
    p = np.zeros(20)
    p[0] = 0.5
    p[2], p[4] = 2000.0, 0.08
    p[10], p[11] = 120000.0, 240000.0
    soc = t % 3
    if soc in (0, 1):
        p[1], p[3] = 2000.0, 0.08
    if soc == 1:
        p[5], p[6], p[7], p[8] = 120.0, 120.0, 0.6, 0.6
    if soc == 2:
        p[9], p[12], p[13], p[14], p[15] = 360.0, 2.0, 0.35, 2.0, 3.0
    if t >= 3:
        p[16], p[17], p[18], p[19] = 1.0, 500.0, 3.0, 0.1
    return p


def value_network_layout(model):
    """The packed form snp_value_lookahead takes of a value network: `model`'s leaf modules must be Linear and ReLU alternating and
    end in Linear(., 1) -- CADRL's ValueNetwork (crowd_nav/policy/cadrl.py mlp(input_dim, mlp_dims), last_relu=False), or its
    `value_network` Sequential -- with 13 or 15 inputs, hidden widths in 1..256 and at most 6 Linear layers.  Returns (widths,
    packed): widths [in, h1, ..., 1] and a CPU float32 tensor holding, layer by layer, W transposed ([in][out] row-major,
    weight.t()) then the bias [out] (zeros for a Linear without one).  Anything else raises ValueError."""
    leaves = [m for m in model.modules() if next(m.children(), None) is None]
    kinds = [type(m) for m in leaves]
    if not leaves or len(leaves) % 2 == 0 or any(k is not (torch.nn.Linear if i % 2 == 0 else torch.nn.ReLU) for i, k in enumerate(kinds)):
        raise ValueError("the value network must be Linear / ReLU alternating and end in a Linear layer, got "
                         + ", ".join(k.__name__ for k in kinds))
    linears = leaves[0::2]
    if len(linears) > 6:
        raise ValueError(f"at most 6 Linear layers (got {len(linears)})")
    widths = [linears[0].in_features] + [m.out_features for m in linears]
    if widths[0] not in (13, 15):
        raise ValueError(f"the value network takes the 13 or 15 values of a rotated state, not {widths[0]}")
    if widths[-1] != 1:
        raise ValueError(f"the value network has one output, not {widths[-1]}")
    if any(not 1 <= w <= 256 for w in widths[1:-1]):
        raise ValueError(f"hidden widths must be in 1..256 (got {widths[1:-1]})")
    parts = []
    with torch.no_grad():
        for m in linears:
            parts.append(m.weight.detach().float().cpu().t().reshape(-1))
            parts.append(torch.zeros(m.out_features) if m.bias is None else m.bias.detach().float().cpu().reshape(-1))
    return widths, torch.cat(parts).contiguous()


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class CrowdEngine:
    def __init__(self, model, E, N, G=2, dtype=torch.float64, device="cuda", consider_robot=False, symmetric=True,
                 numba_compat=False, params=None, walls=None, has_robot=True, full_pair_loop=False):
        if model not in SFMS:
            raise Exception(f"The human motion model '{model}' does not exist")
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be torch.float32 or torch.float64")
        self.lib = L.lib()
        self.motion_model_title = model
        self.type = SFMS.index(model)
        self.headed = self.type >= 3
        self.E, self.N, self.G = int(E), int(N), int(G)
        self.dtype, self.device = dtype, torch.device(device)
        self.consider_robot, self.symmetric, self.numba_compat = bool(consider_robot), bool(symmetric), bool(numba_compat)
        # False (default): every unordered pair is evaluated once per warp (Newton's third law); True: every ordered pair in
        # j-ascending order, the reference's own accumulation order (forces.py:145-151).  Same result up to rounding.
        self.full_pair_loop = bool(full_pair_loop)
        self.robot_type, self.robot_params = None, None  # set_robot_motion_model
        self.safety_space = None                         # set_safety_space
        self.respawn_envs = None    # optional int32 [E]: which envs respawn (hybrid scenario); None = all
        self.respawn_bounds = None  # (traffic_length/2, traffic_height/2): parallel-traffic respawn after every update (mmm:407-422)
        self.mapping = 0  # 0 auto, 1 force warp-packed, 2 force block-packed thread mapping (tests / tuning)
        self.params = model_parameters(model) if params is None else np.asarray(params, np.float64).reshape(20)
        kw = dict(dtype=dtype, device=self.device)
        self.dyn = torch.zeros((L.DYN_FIELDS, E, N), **kw)
        self.stat = torch.zeros((L.STAT_FIELDS, E, N), **kw)
        self.goals = torch.zeros((G, 2, E, N), **kw)
        self.goal_idx = torch.zeros((E, N), dtype=torch.int32, device=self.device)
        self.goal_cnt = torch.ones((E, N), dtype=torch.int32, device=self.device)
        self.robot = torch.zeros((L.ROBOT_FIELDS, E), **kw) if (has_robot or consider_robot) else None
        self.agent_params = None
        self.action = torch.zeros((2, E), **kw)
        self.time_now = torch.zeros((E,), dtype=torch.float64, device=self.device)
        self.flags = torch.zeros((E,), dtype=torch.int32, device=self.device)
        self.checks = torch.zeros((E, 4), dtype=torch.float64, device=self.device)
        # reward constants of crowd_nav/configs/env.config: time_limit, collision_penalty, success_reward,
        # discomfort_dist, discomfort_penalty_factor, robot_time_step
        self.consts = [50.0, -0.25, 1.0, 0.2, 0.5, 0.25]
        self._peek_buf, self._peek_idx, self.action_space, self._rotated, self._rewards = None, None, None, None, None
        self._reset_scen, self._reset_draws = None, None
        self._value_net, self._value_out = None, None
        self.walls, self.W, self.S, self.walls_per_env = None, 0, 0, 0
        if walls is not None:
            self.set_walls(walls)

    # ------------------------------------------------------------------ construction from reference arrays
    @classmethod
    def from_reference_arrays(cls, model, states, goals, walls=None, params=None, safety=None, consider_robot=False,
                              all_params_equal=True, numba_compat=False, dtype=torch.float64, device="cuda", robot=None,
                              full_pair_loop=False, **engine_kw):
        """states [E,rows,13] float64 rows (agent.py:256; rows = N + consider_robot), goals [E,N,G,2] NaN padded,
        walls [W,S,2,2] or [E,W,S,2,2] NaN padded, params [20] / [E,N,20], safety [E,rows], robot [E,13] (when the robot is
        not a row of `states` but checks are wanted).  Further keywords go to the constructor (e.g. TiledCrowdEngine's
        unit_capacity)."""
        states = np.ascontiguousarray(states, np.float64)
        goals = np.ascontiguousarray(goals, np.float64)
        E, rows, _ = states.shape
        N, G = goals.shape[1], goals.shape[2]
        if rows != N + int(consider_robot):
            raise ValueError(f"states has {rows} rows per env, expected {N + int(consider_robot)}")
        p_uniform, p_rows = None, None
        if params is not None:
            params = np.asarray(params, np.float64)
            if params.ndim == 1:
                p_uniform = params
            else:
                flat = params.reshape(-1, 20)
                if np.all(flat == flat[0]):
                    p_uniform = flat[0]
                else:
                    p_rows = params.reshape(E, N, 20)
        eng = cls(model, E, N, G, dtype=dtype, device=device, consider_robot=consider_robot, symmetric=all_params_equal,
                  numba_compat=numba_compat, params=p_uniform, walls=walls, has_robot=consider_robot or robot is not None,
                  full_pair_loop=full_pair_loop, **engine_kw)
        if p_rows is not None:
            eng.agent_params = torch.as_tensor(np.ascontiguousarray(p_rows.transpose(2, 0, 1)), dtype=dtype, device=eng.device)
        eng.load_rows(states, safety)
        eng.load_goals(goals)
        if robot is not None and not consider_robot:
            eng.set_robot_rows(robot)
        return eng

    # ------------------------------------------------------------------ descriptors
    def _crowd(self):
        c = L.SnpCrowd()
        c.E, c.N, c.G = self.E, self.N, self.G
        c.dtype = L.SNP_F64 if self.dtype == torch.float64 else L.SNP_F32
        c.dyn, c.stat, c.goals = self.dyn.data_ptr(), self.stat.data_ptr(), self.goals.data_ptr()
        c.goal_idx, c.goal_cnt = self.goal_idx.data_ptr(), self.goal_cnt.data_ptr()
        c.agent_params = None if self.agent_params is None else self.agent_params.data_ptr()
        c.params = (ctypes.c_double * 20)(*self.params.tolist())
        c.robot = None if self.robot is None else self.robot.data_ptr()
        c.walls = None if self.walls is None else self.walls.data_ptr()
        c.W, c.S, c.walls_per_env = self.W, self.S, self.walls_per_env
        return c

    def _opts(self, dt, n_substeps, robot_mode=0, pre_checks=False, post_checks=False, track_touch=False, advance_time=False,
              post_update=True):
        # post_checks: False/True/2 (2 = imitation-learning reward from the actual end state)
        o = L.SnpStepOpts()
        o.type, o.consider_robot, o.symmetric, o.numba_compat = self.type, int(self.consider_robot), int(self.symmetric), int(self.numba_compat)
        o.n_substeps, o.robot_mode, o.dt = int(n_substeps), int(robot_mode), float(dt)
        o.action = self.action.data_ptr()
        o.pre_checks, o.post_checks, o.track_touch = int(pre_checks), int(post_checks), int(track_touch)
        o.reserved = (L.SNP_OPT_FULL_PAIR_LOOP if self.full_pair_loop else 0) | (self.mapping << 2)  # mapping 1 / 2 = SNP_OPT_MAP_WARP / _BLOCK
        o.consts = (ctypes.c_double * 6)(*self.consts)
        o.time_now = self.time_now.data_ptr() if (advance_time or pre_checks or int(post_checks) == 2) else None
        o.flags, o.checks = self.flags.data_ptr(), self.checks.data_ptr()
        if robot_mode == 2:
            o.robot_type = int(self.robot_type)
            o.robot_params = (ctypes.c_double * 20)(*self.robot_params.tolist())
        if self.respawn_bounds is not None and n_substeps > 0 and post_update:
            o.respawn = 1
            o.respawn_bounds = (ctypes.c_double * 2)(*self.respawn_bounds)
            o.respawn_envs = None if self.respawn_envs is None else self.respawn_envs.data_ptr()
        return o

    # ------------------------------------------------------------------ loading / reading in the reference's layouts
    def set_walls(self, walls):
        """walls [W,S,2,2] (shared) or [E,W,S,2,2] float64, NaN padded (motion_model_manager.py:268-276)."""
        walls = np.asarray(walls, np.float64)
        if walls.size == 0 or walls.shape[-4] == 0:
            self.walls, self.W, self.S, self.walls_per_env = None, 0, 0, 0
            return
        per_env = walls.ndim == 5
        self.W, self.S, self.walls_per_env = walls.shape[-4], walls.shape[-3], int(per_env)
        flat = walls.reshape((self.E if per_env else 1), self.W * self.S, 4)
        self.walls = torch.as_tensor(np.ascontiguousarray(flat), dtype=self.dtype, device=self.device)

    def load_rows(self, states, safety=None):
        """Upload reference state rows [E,rows,13] (+ safety [E,rows]) and scatter them into the SoA on the device."""
        states = np.ascontiguousarray(states, np.float64)
        rows = states.shape[1]
        d_rows = torch.from_numpy(states).to(self.device)
        d_saf = None if safety is None else torch.from_numpy(np.ascontiguousarray(safety, np.float64)).to(self.device)
        L.check(self.lib.snp_unpack_states(ctypes.byref(self._crowd()), _ptr(d_rows), rows, _ptr(d_saf), _stream()))

    def load_goals(self, goals):
        d = torch.from_numpy(np.ascontiguousarray(goals, np.float64)).to(self.device)
        L.check(self.lib.snp_unpack_goals(ctypes.byref(self._crowd()), _ptr(d), _ptr(self.goal_cnt), _stream()))

    def set_robot_rows(self, robot_rows, safety=None):
        """robot_rows [E,13] reference rows (robot.get_safe_state(), motion_model_manager.py:359)."""
        r = np.asarray(robot_rows, np.float64).reshape(self.E, 13)
        out = np.zeros((L.ROBOT_FIELDS, self.E))
        out[L.ROBOT_PX], out[L.ROBOT_PY], out[L.ROBOT_TH] = r[:, 0], r[:, 1], r[:, 2]
        out[L.ROBOT_VX], out[L.ROBOT_VY] = r[:, 3], r[:, 4]
        out[L.ROBOT_R], out[L.ROBOT_GX], out[L.ROBOT_GY] = r[:, 8], r[:, 10], r[:, 11]
        out[L.ROBOT_BVX], out[L.ROBOT_BVY], out[L.ROBOT_OM], out[L.ROBOT_M], out[L.ROBOT_VD] = r[:, 5], r[:, 6], r[:, 7], r[:, 9], r[:, 12]
        out[L.ROBOT_GCNT] = 1.0
        if safety is not None:
            out[L.ROBOT_SAFETY] = np.asarray(safety, np.float64).reshape(self.E)
        else:
            out[L.ROBOT_SAFETY] = self.robot[L.ROBOT_SAFETY].double().cpu().numpy()
        self.robot.copy_(torch.as_tensor(out, dtype=self.dtype))

    def set_robot_motion_model(self, title, goals=None):
        """MotionModelManager.set_robot_motion_model (mmm:552-591, Euler only): the robot will be moved by the SFM / HSFM model
        `title` (parameters of agent.py:79-243) in `imitation_learning_step`.  goals: optional [E,1..2,2] robot goal list."""
        if title not in SFMS:
            raise Exception(f"The robot motion model '{title}' does not exist")
        self.robot_motion_model_title = title
        self.robot_type, self.robot_params = SFMS.index(title), model_parameters(title)
        if goals is not None:
            self.set_robot_goals(goals)
        if getattr(self, "safety_space", None) is not None:  # a safety space set earlier now covers the robot too (mmm:159-162)
            self.set_safety_space(self.safety_space)

    def set_robot_goals(self, goals):
        g = np.asarray(goals, np.float64).reshape(self.E, -1, 2)
        if g.shape[1] > 2:
            raise NotImplementedError("the robot's goal list holds at most two goals (every reference scenario: goal and start)")
        t = lambda a: torch.as_tensor(a, dtype=self.dtype, device=self.device)
        self.robot[L.ROBOT_GX].copy_(t(g[:, 0, 0])); self.robot[L.ROBOT_GY].copy_(t(g[:, 0, 1]))
        if g.shape[1] == 2 and not np.isnan(g[:, 1]).any():
            self.robot[L.ROBOT_GX2].copy_(t(g[:, 1, 0])); self.robot[L.ROBOT_GY2].copy_(t(g[:, 1, 1]))
            self.robot[L.ROBOT_GCNT].fill_(2.0)
        else:
            self.robot[L.ROBOT_GCNT].fill_(1.0)

    def imitation_learning_step(self, dt=0.0125, n_substeps=20):
        """SocialNavGym.imitation_learning_step (social_nav_gym.py:252-274): `n_substeps` x (update_robot; update_humans) with
        the robot moved by its own motion model, then the ACTUAL collision / goal checks and the reward at the end time --
        one launch.  Results in self.flags / self.checks (decode_flags) and self.robot."""
        if self.robot_type is None:
            raise ValueError("set_robot_motion_model(title) first")
        o = self._opts(dt, n_substeps, robot_mode=2, post_checks=2, advance_time=True)
        L.check(self.lib.snp_step(ctypes.byref(self._crowd()), ctypes.byref(o), _stream()))

    def sim_update(self, dt=0.0125, n_updates=1, robot_every=1, robot_time_step=None, phase=0):
        """`n_updates` x SocialNavSim.update (social_nav_sim.py:476-492) with the robot driven by its motion model through
        control_robot (:500-529), the loop behind run_k_steps -- one launch.  The humans see the robot's state from before its
        update.  robot_every = ROBOT_SAMPLING_TIME / SAMPLING_TIME: 1 -> update_robot(dt) every update (:521); k > 1 -> the pose
        advances every update with the last velocity (update_robot_pose, motion_model_manager.py:655) and every k-th update
        (update index `phase` + i a multiple of k) update_robot(robot_time_step, just_velocities=True) refreshes the velocities
        (:523-524).  `track_touch` reports run_k_steps' collision test (:702-703) in decode_flags()["touched"]."""
        if self.robot_type is None:
            raise ValueError("set_robot_motion_model(title) first")
        if int(robot_every) < 1:
            raise ValueError("robot_every must be >= 1 (robot sampling time as a multiple of the environment's)")
        keep = self.consts[5]
        self.consts[5] = float(robot_time_step if robot_time_step is not None else dt * int(robot_every))
        try:
            o = self._opts(dt, n_updates, robot_mode=2, track_touch=True, advance_time=True)
            o.robot_every, o.robot_phase = int(robot_every), int(phase) % int(robot_every)
            L.check(self.lib.snp_step(ctypes.byref(self._crowd()), ctypes.byref(o), _stream()))
        finally:
            self.consts[5] = keep

    def robot_rows(self):
        """Robot state as reference rows [E,13] + carried desired force [E,2]."""
        r = self.robot.double().cpu().numpy()
        rows = np.zeros((self.E, 13))
        rows[:, 0], rows[:, 1], rows[:, 2] = r[L.ROBOT_PX], r[L.ROBOT_PY], r[L.ROBOT_TH]
        rows[:, 3], rows[:, 4], rows[:, 5], rows[:, 6], rows[:, 7] = r[L.ROBOT_VX], r[L.ROBOT_VY], r[L.ROBOT_BVX], r[L.ROBOT_BVY], r[L.ROBOT_OM]
        rows[:, 8], rows[:, 9], rows[:, 10], rows[:, 11], rows[:, 12] = r[L.ROBOT_R], r[L.ROBOT_M], r[L.ROBOT_GX], r[L.ROBOT_GY], r[L.ROBOT_VD]
        return rows, np.stack([r[L.ROBOT_DFX], r[L.ROBOT_DFY]], 1)

    def rows(self, template):
        """Download the state in reference row form: `template` [E,rows,13] provides the static columns and the robot row
        (as update_humans_parallel's np.copy does, forces_parallel.py:214); columns 0..7 and 10..11 of human rows are replaced."""
        d = torch.from_numpy(np.ascontiguousarray(template, np.float64)).to(self.device)
        L.check(self.lib.snp_pack_states(ctypes.byref(self._crowd()), _ptr(d), template.shape[1], _stream()))
        return d.cpu().numpy()

    def desired_force(self):
        return torch.stack([self.dyn[L.DYN_DFX], self.dyn[L.DYN_DFY]], -1).double().cpu().numpy()

    def set_desired_force(self, df):
        df = torch.as_tensor(np.asarray(df, np.float64), dtype=self.dtype, device=self.device)
        self.dyn[L.DYN_DFX].copy_(df[..., 0]); self.dyn[L.DYN_DFY].copy_(df[..., 1])

    def current_goals(self, goal_idx=None):
        idx = (self.goal_idx if goal_idx is None else goal_idx).long()[None, None]  # [1,1,E,N]
        return torch.gather(self.goals, 0, idx.expand(1, 2, self.E, self.N))[0].permute(1, 2, 0)  # [E,N,2]

    # ------------------------------------------------------------------ the hot path
    def update_humans(self, t=0.0, dt=0.0125, post_update=True, n_substeps=1):
        """MotionModelManager.update_humans (motion_model_manager.py:354) for every env: `n_substeps` Euler updates in one launch."""
        L.check(self.lib.snp_step(ctypes.byref(self._crowd()), ctypes.byref(self._opts(dt, n_substeps, post_update=post_update)), _stream()))

    def step(self, action=None, dt=0.0125, n_substeps=20, pre_checks=True, post_checks=False, track_touch=False, kinematics="holonomic"):
        """SocialNavGym.step for every env (social_nav_gym.py:227-250): swept collision / goal test and reward on the current
        state, then `n_substeps` x (robot.step(action, dt); update_humans(dt)).  `action` [E,2]: holonomic velocities (vx, vy)
        (ActionXY), or (v, r) with kinematics="unicycle" (ActionRot, robot_agent.py:116-136: the rotation r is applied at every
        sub-step); device tensor or array; None reuses self.action.  Results land in self.flags / self.checks / self.time_now."""
        if kinematics not in ("holonomic", "unicycle"):
            raise ValueError("kinematics must be 'holonomic' or 'unicycle'")
        if action is not None:
            a = torch.as_tensor(action, dtype=self.dtype, device=self.device)
            self.action.copy_(a.t() if a.shape == (self.E, 2) else a)
        o = self._opts(dt, n_substeps, robot_mode=1 if kinematics == "holonomic" else 3, pre_checks=pre_checks, post_checks=post_checks,
                       track_touch=track_touch, advance_time=True)
        L.check(self.lib.snp_step(ctypes.byref(self._crowd()), ctypes.byref(o), _stream()))

    def step_host(self, action_host, obs_host, flags_host, checks_host, dt=0.0125, n_substeps=20, pre_checks=True, post_checks=False,
                  track_touch=False, staged=False):
        """The same gym step through ONE C-ABI call with host buffers (snp_gym_step_host): `action_host` [2,E] is copied in, the
        fused step runs, observation [4,E,N] (px,py,vx,vy), flags [E] int32 and checks [E,4] float64 land in the host buffers and the
        stream is synchronised.  The buffers are CPU tensors or NumPy arrays of the engine's dtype.  PINNED result buffers are written
        by the kernel itself (zero-copy: no D2H transfer after the launch); pageable ones -- or staged=True -- get D2H copies."""
        # the two descriptor blocks are rebuilt only when something they describe changed (a gym loop calls this every 0.25 s of
        # simulated time with the same arguments; building them costs more host time than the launch)
        key = (float(dt), int(n_substeps), bool(pre_checks), int(post_checks), bool(track_touch), bool(staged), self.full_pair_loop, self.mapping,
               self.consider_robot, self.symmetric, self.numba_compat, tuple(self.consts), self.respawn_bounds,
               None if self.respawn_envs is None else self.respawn_envs.data_ptr(), self.params.tobytes(),
               self.dyn.data_ptr(), self.stat.data_ptr(), self.goals.data_ptr(), self.goal_idx.data_ptr(), self.goal_cnt.data_ptr(),
               None if self.agent_params is None else self.agent_params.data_ptr(), None if self.robot is None else self.robot.data_ptr(),
               None if self.walls is None else self.walls.data_ptr(), self.W, self.S, self.walls_per_env, self.action.data_ptr(),
               self.time_now.data_ptr(), self.flags.data_ptr(), self.checks.data_ptr())
        cached = getattr(self, "_host_call", None)
        if cached is None or cached[0] != key:
            o = self._opts(dt, n_substeps, robot_mode=1, pre_checks=pre_checks, post_checks=post_checks, track_touch=track_touch, advance_time=True)
            if staged:
                o.reserved |= L.SNP_OPT_STAGED_COPIES
            cached = self._host_call = (key, self._crowd(), o)
        hp = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr() if torch.is_tensor(t) else t.ctypes.data)
        L.check(self.lib.snp_gym_step_host(ctypes.byref(cached[1]), ctypes.byref(cached[2]), hp(action_host), hp(obs_host), hp(flags_host),
                                           hp(checks_host), _stream()))

    def run_checks(self, action=None, pre=True, post=True):
        """collision_detection_and_reaching_goal + compute_reward_and_infos (social_nav_sim.py:949-1029) and
        check_actual_collisions_and_goal (social_nav_gym.py:107-118) on the current state, without stepping."""
        if action is not None:
            a = torch.as_tensor(action, dtype=self.dtype, device=self.device)
            self.action.copy_(a.t() if a.shape == (self.E, 2) else a)
        o = self._opts(0.0, 0, pre_checks=pre, post_checks=post)
        L.check(self.lib.snp_checks(ctypes.byref(self._crowd()), ctypes.byref(o), _stream()))
        return self.decode_flags()

    def collision_detection_and_reaching_goal(self, action, time_step=None):
        """SocialNavSim.collision_detection_and_reaching_goal(action, time_step) (social_nav_sim.py:949-984) for every env at once:
        (collision, dmin, reaching_goal) of the swept test over one robot step with `action` [E,2]; humans keep their last velocity."""
        keep = self.consts[5]
        if time_step is not None:
            self.consts[5] = float(time_step)
        try:
            r = self.run_checks(action, pre=True, post=False)
        finally:
            self.consts[5] = keep
        return r["collision"], r["dmin"], r["reaching_goal"]

    def decode_flags(self):
        f = self.flags.cpu().numpy()
        c = self.checks.cpu().numpy()
        return dict(collision=(f & L.FLAG_COLLISION) != 0, dmin=c[:, 0], reaching_goal=(f & L.FLAG_REACHING_GOAL) != 0,
                    reward=c[:, 1], terminated=(f & L.FLAG_TERMINATED) != 0, truncated=(f & L.FLAG_TRUNCATED) != 0,
                    info=(f >> L.FLAG_INFO_SHIFT) & 7, actual_collision=(f & L.FLAG_ACTUAL_COLLISION) != 0, actual_dmin=c[:, 2],
                    actual_goal=(f & L.FLAG_ACTUAL_GOAL) != 0, touched=(f & L.FLAG_TOUCHED) != 0)

    def robot_check_collisions(self):
        """RobotAgent.check_collisions(humans, walls) (robot_agent.py:35-48) for every env: the robot is pushed out of the humans it
        overlaps (in index order), then out of the walls; updates self.robot's position in place."""
        L.check(self.lib.snp_robot_push_out(ctypes.byref(self._crowd()), _stream()))

    def check_actual_collisions_and_goal(self):
        r = self.run_checks(pre=False, post=True)
        return r["actual_collision"], r["actual_dmin"], r["actual_goal"]

    # ------------------------------------------------------------------ MotionModelManager surface
    def get_human_states(self, include_goal=True, headed=False):
        """[E,N,8] / [E,N,6] / [E,N,4] in the layouts of motion_model_manager.py:285-312."""
        d = self.dyn
        if include_goal:
            g = self.current_goals()
            v = (d[L.DYN_BVX], d[L.DYN_BVY]) if headed else (d[L.DYN_VX], d[L.DYN_VY])
            out = torch.stack([d[L.DYN_PX], d[L.DYN_PY], d[L.DYN_TH], v[0], v[1], d[L.DYN_OM], g[..., 0], g[..., 1]], -1)
        elif headed:
            out = torch.stack([d[L.DYN_PX], d[L.DYN_PY], d[L.DYN_TH], d[L.DYN_BVX], d[L.DYN_BVY], d[L.DYN_OM]], -1)
        else:
            out = torch.stack([d[L.DYN_PX], d[L.DYN_PY], d[L.DYN_VX], d[L.DYN_VY]], -1)
        return out.double().cpu().numpy()

    def set_human_states(self, state, just_visual=False):
        """motion_model_manager.py:314-352: state [E,N,8] = [x,y,yaw,Vx|BVx,Vy|BVy,Omega,Gx,Gy]; the goal list is rewound so
        that its head equals (Gx,Gy) (rewind_goals, :57-64); for headed models v = R(yaw) bv is refreshed (:324)."""
        s = torch.as_tensor(np.asarray(state, np.float64), device=self.device)
        d = self.dyn
        d[L.DYN_PX].copy_(s[..., 0]); d[L.DYN_PY].copy_(s[..., 1]); d[L.DYN_TH].copy_(s[..., 2])
        if just_visual:
            return
        if self.headed:
            d[L.DYN_BVX].copy_(s[..., 3]); d[L.DYN_BVY].copy_(s[..., 4])
            c, sn = torch.cos(s[..., 2]), torch.sin(s[..., 2])
            d[L.DYN_VX].copy_(c * s[..., 3] - sn * s[..., 4]); d[L.DYN_VY].copy_(sn * s[..., 3] + c * s[..., 4])
        else:
            d[L.DYN_VX].copy_(s[..., 3]); d[L.DYN_VY].copy_(s[..., 4])
        d[L.DYN_OM].copy_(s[..., 5])
        # goal rewind: first slot whose goal equals (Gx, Gy); unknown goals overwrite the list (parallel traffic, :58)
        g = self.goals.double().permute(2, 3, 0, 1)  # [E,N,G,2]
        match = (g == s[..., None, 6:8]).all(-1) & (torch.arange(self.G, device=self.device) < self.goal_cnt[..., None])
        has = match.any(-1)
        self.goal_idx.copy_(torch.where(has, match.int().argmax(-1), torch.zeros_like(self.goal_idx)).int())
        if (~has).any():
            e, n = torch.nonzero(~has, as_tuple=True)
            self.goals[0, 0, e, n] = s[e, n, 6].to(self.dtype); self.goals[0, 1, e, n] = s[e, n, 7].to(self.dtype)
            self.goal_cnt[e, n] = 1

    def peek(self, dt):
        """One update of length dt into a side buffer (snp_step with dyn_out): returns the [DYN_FIELDS,E,N] device tensor of the
        humans one step ahead; pose, velocities and goal index of the crowd are untouched.  As in the reference
        (motion_model_manager.py:691-709) the carried desired force IS updated.  No clone / restore traffic."""
        if self._peek_buf is None:
            self._peek_buf, self._peek_idx = torch.empty_like(self.dyn), torch.empty_like(self.goal_idx)
        o = self._opts(dt, 1, post_update=False)
        o.dyn_out, o.goal_idx_out = self._peek_buf.data_ptr(), self._peek_idx.data_ptr()
        L.check(self.lib.snp_step(ctypes.byref(self._crowd()), ctypes.byref(o), _stream()))
        return self._peek_buf

    def get_next_human_observable_states(self, dt, theta_and_omega_visible=False):
        """motion_model_manager.py:691-709: the humans' observable states one update of length dt ahead, [E,N,4] = x,y,Vx,Vy or
        [E,N,8] = x,y,yaw,Vx,Vy,Omega,Gx,Gy (:288,:307).  As in the reference, the carried desired force is NOT restored."""
        nx = self.peek(dt)
        if not theta_and_omega_visible:
            return torch.stack([nx[L.DYN_PX], nx[L.DYN_PY], nx[L.DYN_VX], nx[L.DYN_VY]], -1).double().cpu().numpy()
        ho = nx if self.headed else self.dyn  # non-headed models do not integrate yaw / omega
        g = self.current_goals(self._peek_idx)  # read before the restore (mmm:705-707): the goal the peeked update arrived at
        return torch.stack([nx[L.DYN_PX], nx[L.DYN_PY], ho[L.DYN_TH], nx[L.DYN_VX], nx[L.DYN_VY], ho[L.DYN_OM], g[..., 0], g[..., 1]],
                           -1).double().cpu().numpy()

    # ------------------------------------------------------------------ on-device reset (SURVEY 8f-4)
    def reset_scenario(self, scenario, seeds=None, seed0=0, mask=None, randomize_attributes=False, circle_radius=7.0, robot_radius=0.3,
                       traffic_length=14.0, traffic_height=3.0, human_mass=75.0, robot_mass=80.0, robot_desired_speed=1.0,
                       force_cta=False):
        """SocialNavGym.reset (social_nav_gym.py:120-225) for every env -- or those selected by `mask` [E] bool -- without leaving the
        device: env e replays the reference's generator for `scenario` on NumPy's MT19937 stream seeded with seeds[e] (default
        seed0 + e), as np.random.seed(offset[phase] + case) does (:135-137).  Returns (scenario_of_env int32 [E], draws int32 [E])
        device tensors; parallel-traffic envs get their respawn switched on (mmm:407-422).  A warp generates an env up to 1,522
        humans, a CTA above that (up to 6,322); force_cta=True takes the CTA kernel at any N (the same bits; for tests and
        measurement)."""
        if self.robot is None:
            raise ValueError("the scenarios place a robot: build the engine with has_robot=True")
        g = L.SnpResetArgs()
        g.scenario = L.RESET_SCENARIOS[scenario] if isinstance(scenario, str) else int(scenario)
        g.randomize_attributes = int(randomize_attributes)
        dev = self.device
        if seeds is not None:
            if torch.is_tensor(seeds):   # device-side seeds (e.g. a running case counter): int32 bit patterns are read as uint32
                seeds_t = seeds.to(device=dev, dtype=torch.int32).contiguous()
            else:
                s32 = (np.asarray(seeds, np.int64) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)
                seeds_t = torch.from_numpy(np.ascontiguousarray(s32)).to(dev)
            if seeds_t.numel() != self.E:
                raise ValueError("seeds must have one entry per env")
            g.seeds = seeds_t.data_ptr()
        g.seed0 = int(seed0) & 0xFFFFFFFF
        g.reserved = L.SNP_RESET_FORCE_CTA if force_cta else 0
        mask_t = None
        if mask is not None:
            mask_t = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
            g.mask = mask_t.data_ptr()
        g.circle_radius, g.robot_radius, g.traffic_length, g.traffic_height = float(circle_radius), float(robot_radius), float(traffic_length), float(traffic_height)
        g.human_mass, g.robot_mass, g.robot_desired_speed = float(human_mass), float(robot_mass), float(robot_desired_speed)
        if self._reset_scen is None:
            self._reset_scen = torch.zeros((self.E,), dtype=torch.int32, device=dev)
            self._reset_draws = torch.zeros((self.E,), dtype=torch.int32, device=dev)
        g.time_now, g.flags = self.time_now.data_ptr(), self.flags.data_ptr()
        g.scenario_out, g.draws_out = self._reset_scen.data_ptr(), self._reset_draws.data_ptr()
        L.check(self.lib.snp_reset(ctypes.byref(self._crowd()), ctypes.byref(g), _stream()))
        if g.scenario in (1, 4):   # parallel traffic (all envs, or the coin of the hybrid scenario)
            self.respawn_bounds = (traffic_length / 2, traffic_height / 2)
            self.respawn_envs = self._reset_scen if g.scenario == 4 else None
        elif mask is None:
            self.respawn_bounds, self.respawn_envs = None, None
        return self._reset_scen, self._reset_draws

    def onestep_lookahead(self, action, time_step=0.25, theta_and_omega_visible=False):
        """SocialNavSim.onestep_lookahead (social_nav_sim.py:1031-1049), the per-action form the policies use when they do not
        batch the action space: swept collision / goal test and reward of `action` [E,2] over `time_step` on the current state,
        and the humans' observable states one `time_step` ahead (query_env).  Returns (ob [E,N,4|8], reward [E])."""
        keep = self.consts[5]
        self.consts[5] = float(time_step)
        try:
            reward = self.run_checks(action, pre=True, post=False)["reward"]
        finally:
            self.consts[5] = keep
        return self.get_next_human_observable_states(time_step, theta_and_omega_visible), reward

    # ------------------------------------------------------------------ policy-side lookahead (SURVEY 8f-3)
    def set_action_space(self, actions):
        """actions [A,2] holonomic velocities shared by all envs (crowd_nav/policy/cadrl.py build_action_space)."""
        self.action_space = torch.as_tensor(np.ascontiguousarray(actions, np.float64), device=self.device).reshape(-1, 2).contiguous()
        self._rotated = self._rewards = None

    def lookahead(self, time_step=0.25, theta_and_omega_visible=False, query_env=True, bulk_store=True):
        """What CADRL.predict computes before evaluating its value network (crowd_nav/policy/cadrl.py:235-262), for every env:
        the humans `time_step` ahead -- query_env=True: a peek of the motion model (:257-258); False: the constant-velocity model
        (:92-105, snp_constant_velocity) -- then compute_rotated_states_and_reward (:42-83) for the whole action space.
        Returns device tensors (rotated [E,A,N,13|15] in the engine's dtype, rewards [E,A] float64); two launches."""
        if query_env:
            return self.lookahead_from(self.peek(time_step), time_step, theta_and_omega_visible, bulk_store)
        return self.lookahead_from(self.constant_velocity_next(time_step), time_step, theta_and_omega_visible, bulk_store, yaw_from_next=True)

    def constant_velocity_next(self, dt):
        """propagate_humans_state_with_constant_velocity_model (crowd_nav/policy/cadrl.py:92-105) into the peek buffer: the
        [DYN_FIELDS,E,N] device tensor of the humans one step ahead if nobody changed velocity; the crowd itself is untouched."""
        if self._peek_buf is None:
            self._peek_buf, self._peek_idx = torch.empty_like(self.dyn), torch.empty_like(self.goal_idx)
        L.check(self.lib.snp_constant_velocity(ctypes.byref(self._crowd()), float(dt), ctypes.c_void_p(self._peek_buf.data_ptr()), _stream()))
        return self._peek_buf

    def lookahead_from(self, nxt, time_step=0.25, theta_and_omega_visible=False, bulk_store=True, yaw_from_next=False, split_humans=False):
        """compute_rotated_states_and_reward on a given `nxt` [DYN_FIELDS,E,N].  With theta_and_omega_visible the next yaw / omega are
        read from `nxt` for headed models and from the current state otherwise (what get_next_human_observable_states returns,
        mmm:691-709); yaw_from_next=True reads them from `nxt` whatever the model (the constant-velocity propagation integrates
        theta + omega dt for every model, cadrl.py:103).  Any N: envs whose humans do not fit one CTA's shared memory are split
        into chunks of humans (csrc/snp_lookahead.cu); split_humans=True splits them even where one CTA would hold them (the same
        bits; for tests and measurement, like bulk_store=False)."""
        if getattr(self, "action_space", None) is None:
            raise ValueError("set_action_space(actions) first")
        if self.robot is None:
            raise ValueError("the lookahead needs the robot's state")
        A, ow = self.action_space.shape[0], 15 if theta_and_omega_visible else 13
        if self._rotated is None or self._rotated.shape[-1] != ow:
            self._rotated = torch.empty((self.E, A, self.N, ow), dtype=self.dtype, device=self.device)
            self._rewards = torch.empty((self.E, A), dtype=torch.float64, device=self.device)
        g = L.SnpLookaheadArgs()
        g.type, g.A, g.theta_and_omega_visible, g.reserved = (max(self.type, 3) if yaw_from_next else self.type), A, int(theta_and_omega_visible), (0 if bulk_store else 1) | (2 if split_humans else 0)
        g.next, g.actions, g.dt = nxt.data_ptr(), self.action_space.data_ptr(), float(time_step)
        g.rotated, g.rewards = self._rotated.data_ptr(), self._rewards.data_ptr()
        L.check(self.lib.snp_lookahead(ctypes.byref(self._crowd()), ctypes.byref(g), _stream()))
        return self._rotated, self._rewards

    # ------------------------------------------------------------------ the policy's action choice on the device
    def set_value_network(self, model, gamma):
        """CADRL's value network for predict(): `model` is packed once (value_network_layout) into a device fp32 buffer; `gamma` is
        the policy's discount factor.  Raises ValueError for a network that is not Linear / ReLU alternating ending in Linear(., 1)."""
        widths, packed = value_network_layout(model)
        self._value_net = (widths, packed.to(self.device), float(gamma))

    def predict(self, time_step=0.25, theta_and_omega_visible=False, query_env=True):
        """CADRL.predict (crowd_nav/policy/cadrl.py:235-276) for every env, without the exploration: the humans `time_step` ahead
        (query_env as in lookahead()), the value network on every rotated state, its minimum over the humans, value = reward +
        gamma ^ (time_step * v_pref) * minimum and the first action of largest value.  Returns device tensors (best [E] int64,
        values [E,A] float64, reached [E] bool); where `reached` is set the policy takes the zero action instead of best.  best is -1
        in an env where no value exceeds -inf (a network that outputs NaN): predict's max_action stays None there, and
        action_space[best] must not be taken for it."""
        if query_env:
            return self.predict_from(self.peek(time_step), time_step, theta_and_omega_visible)
        return self.predict_from(self.constant_velocity_next(time_step), time_step, theta_and_omega_visible, yaw_from_next=True)

    def predict_from(self, nxt, time_step=0.25, theta_and_omega_visible=False, yaw_from_next=False, split_humans=False):
        """predict() on a given `nxt` [DYN_FIELDS,E,N] (as lookahead_from).  One fused kernel evaluates the network where each rotated
        row is made and a small one folds rewards, values and the choice (csrc/snp_value.cu); the rows never reach device memory.
        split_humans=True spreads every env's humans over several CTAs in chunks of 32 (the same bits; for tests and measurement)."""
        if getattr(self, "action_space", None) is None:
            raise ValueError("set_action_space(actions) first")
        if self.robot is None:
            raise ValueError("the lookahead needs the robot's state")
        if getattr(self, "_value_net", None) is None:
            raise ValueError("set_value_network(model, gamma) first")
        widths, weights, gamma = self._value_net
        A = self.action_space.shape[0]
        if self._value_out is None or self._value_out[0].shape != (self.E, A):
            dev = self.device
            self._value_out = (torch.empty((self.E, A), dtype=torch.float64, device=dev), torch.empty((self.E,), dtype=torch.int32, device=dev),
                               torch.empty((self.E,), dtype=torch.bool, device=dev))
        values, best, reached = self._value_out
        g = L.SnpValueArgs()
        g.type, g.A, g.theta_and_omega_visible = (max(self.type, 3) if yaw_from_next else self.type), A, int(theta_and_omega_visible)
        g.reserved = 2 if split_humans else 0
        g.next, g.actions, g.dt, g.gamma = nxt.data_ptr(), self.action_space.data_ptr(), float(time_step), gamma
        g.layers = len(widths) - 1
        g.widths = (ctypes.c_int32 * 7)(*(widths + [0] * (7 - len(widths))))
        g.weights, g.values, g.best, g.reached = weights.data_ptr(), values.data_ptr(), best.data_ptr(), reached.data_ptr()
        L.check(self.lib.snp_value_lookahead(ctypes.byref(self._crowd()), ctypes.byref(g), _stream()))
        return best.long(), values, reached

    def set_safety_space(self, safety_space):
        """motion_model_manager.py:147-164: every human gets 0.01 + safety_space; the robot gets it only when it is driven by an
        SFM / HSFM model (robot_motion_model_title, set_robot_motion_model) -- visible or not -- and keeps 0 otherwise.
        None clears both (what a fresh MotionModelManager has)."""
        self.safety_space = safety_space
        value = 0.0 if safety_space is None else 0.01 + safety_space
        self.stat[L.STAT_SAFETY].fill_(value)
        if self.robot is not None:
            self.robot[L.ROBOT_SAFETY].fill_(value if self.robot_type is not None else 0.0)
