"""BatchedSocialNavGym: E copies of the reference's SocialNavGym (social_gym/social_nav_gym.py) stepped in lock-step on one GPU.

Keeps the reference's call surface for the path in scope -- `configure`, `set_safety_space`, `reset(phase, test_case)`,
`step(action)`, `check_actual_collisions_and_goal()` -- with a leading env axis: actions are [E,2] holonomic velocities
(ActionXY), observations [E,N,5] = (px,py,vx,vy,radius) per human (or [E,N,7] with theta, omega), rewards / terminated /
truncated [E] and info codes [E] (0 Nothing, 1 Timeout, 2 Collision, 3 ReachGoal, 4 Danger; social_gym/src/info.py).
Env e of a reset is seeded `offset[phase] + case + e`, the rule of social_nav_gym.py:135-137.

One `step` is ONE kernel launch: swept collision / goal test + reward on the current state, then
`robot_time_step / time_step` fused (robot.step + update_humans) sub-steps (social_nav_gym.py:232-245).

Above 512 humans per env (human_num > MAX_FUSED_HUMANS) the gym runs on a TiledCrowdEngine: `step` is one snp_large_batch_step
call, the checks run on the tiled path and the on-device reset takes a CTA per env above about 1,520 humans (up to about 6,300; the
host reset covers any N).  The scenario generators place humans in random angular order, so every 128-human tile of an env would
span the whole circle and the tiled step's far-tile culling would skip nothing: with `spatial_order` (a configure key, default
True) the gym re-numbers the humans patch by patch after every reset (TiledCrowdEngine.renumber).  That changes only the order of
summation (the last bits) and which colliding human the swept check stops at; rewards, terminated, truncated and info are the
same.  observation() always lists the humans in the generator's order.  spatial_order=False keeps the generator's numbering: the
gym then computes bit for bit what a TiledCrowdEngine built from the same rows computes.  Above 512 humans imitation_learning_step
raises NotImplementedError, and so does `step` in parallel traffic and the hybrid scenario (their respawn is not on the tiled
path).
"""
import numpy as np
import torch

from .engine import CrowdEngine, SFMS, INFO_NAMES  # noqa: F401
from .large import TiledCrowdEngine
from . import scenarios, _lib as L

HUMAN_MODELS = SFMS  # social_nav_gym.py:11-12 minus "orca"
MAX_FUSED_HUMANS = 512  # snp_step's limit: larger envs run on the tiled path


class BatchedSocialNavGym:
    def __init__(self, n_envs, dtype=torch.float64, device="cuda"):
        self.E, self.dtype, self.device = int(n_envs), dtype, device
        self.engine = None
        self.safety_space = 0
        self.case_counter = {"train": 0, "test": 0, "val": 0}
        # social_nav_gym.py:74-76: the counter wraps at case_size (val_size / test_size of env.config; train never wraps in practice)
        self.case_size = {"train": int(np.iinfo(np.uint32).max) - 2000, "val": 100, "test": 500}
        # crowd_nav/configs/env.config defaults
        self.time_limit, self.time_step, self.robot_time_step = 50, 0.0125, 0.25
        self.success_reward, self.collision_penalty, self.discomfort_dist, self.discomfort_penalty_factor = 1.0, -0.25, 0.2, 0.5
        self.human_policy, self.human_num, self.circle_radius, self.robot_radius = "hsfm_farina", 5, 7.0, 0.3
        self.train_val_sim = self.test_sim = "circle_crossing"
        self.traffic_length, self.traffic_height = 14.0, 3.0
        self.robot_visible = False
        self.randomize_attributes = False
        self.robot_motion_model_title = None
        self.robot_kinematics = "holonomic"   # or "unicycle" (robot_agent.py:95: the robot policy's kinematics)
        self._robot_goals = None
        self.walls = None
        self.spatial_order = True  # above MAX_FUSED_HUMANS: re-number the humans patch by patch after every reset
        self._order = None         # [E, N] int64 device: the generator's index of the human at each row (None: the identity)

    def configure(self, config):
        """config: a configparser object with the reference's sections (social_nav_gym.py:59-84) or a flat dict."""
        if hasattr(config, "getfloat"):
            self.time_limit = config.getint("env", "time_limit")
            self.case_size["val"], self.case_size["test"] = config.getint("env", "val_size"), config.getint("env", "test_size")
            self.time_step, self.robot_time_step = config.getfloat("env", "time_step"), config.getfloat("env", "robot_time_step")
            self.success_reward, self.collision_penalty = config.getfloat("reward", "success_reward"), config.getfloat("reward", "collision_penalty")
            self.discomfort_dist = config.getfloat("reward", "discomfort_dist")
            self.discomfort_penalty_factor = config.getfloat("reward", "discomfort_penalty_factor")
            self.human_policy = config.get("humans", "policy")
            self.robot_radius = config.getfloat("robot", "radius")
            self.robot_visible = config.getboolean("robot", "visible")
            self.train_val_sim, self.test_sim = config.get("sim", "train_val_sim"), config.get("sim", "test_sim")
            self.circle_radius, self.human_num = config.getfloat("sim", "circle_radius"), config.getint("sim", "human_num")
            self.traffic_length, self.traffic_height = config.getfloat("sim", "traffic_length"), config.getfloat("sim", "traffic_height")
        else:
            for k, v in config.items():
                setattr(self, k, v)
        if self.human_policy not in HUMAN_MODELS:
            raise NotImplementedError
        ratio = self.robot_time_step / self.time_step
        if abs(ratio - round(ratio)) > 1e-7:
            raise ValueError("Robot time step must be a multiple of time step")
        self.time_step_factor = int(self.robot_time_step / self.time_step)

    def set_safety_space(self, safety_space):
        self.safety_space = safety_space

    def reset(self, phase="test", test_case=None, on_device=True):
        """SocialNavGym.reset (social_nav_gym.py:120-225) for the whole batch: env e gets case `case_counter + e`, i.e. the seed
        offset[phase] + case + e (:135-137).  on_device=True generates the scenarios with the reset kernel (snp_reset: the reference's
        generators on NumPy's MT19937 stream, a warp per env, or a CTA per env above about 1,520 humans, up to about 6,300); False
        builds them on the host (scenarios.py, any N) and uploads."""
        assert phase in ["train", "val", "test"]
        if test_case is not None:
            self.case_counter[phase] = test_case
        offset = {"train": 2000, "val": 0, "test": 1000}[phase]                  # social_nav_gym.py:135
        sim = self.test_sim if phase == "test" else self.train_val_sim
        # env e plays case (counter + e) mod case_size: the reference's counter, advanced once per env (social_nav_gym.py:197)
        cases = (self.case_counter[phase] + np.arange(self.E, dtype=np.int64)) % self.case_size[phase]
        seed0 = offset + cases
        if on_device:
            return self._reset_on_device(sim, 0, phase, seeds=seed0)
        if sim == "hybrid_scenario":
            raise NotImplementedError("the hybrid scenario is generated on the device only (reset(on_device=True))")
        if self.randomize_attributes and sim != "circle_crossing":
            raise NotImplementedError("randomize_attributes on the host path covers circle_crossing only (use reset(on_device=True))")
        if sim == "circle_crossing":
            sc = scenarios.circular_crossing(self.E, self.human_num, seed0, self.circle_radius, self.robot_radius,
                                             randomize_attributes=self.randomize_attributes)
        elif sim == "circular_crossing_with_static_obstacles":
            # the reference's generator (social_nav_sim.py:364-431) only terminates for small crowds; above 10 humans the 3 static
            # obstacles are combined with the circular-crossing sampler (SURVEY.md 8(d) config 3)
            gen = scenarios.circular_crossing_with_static_obstacles if self.human_num <= 10 else scenarios.ccso_synthetic
            sc = gen(self.E, self.human_num, seed0, self.circle_radius, self.robot_radius)
        elif sim == "parallel_traffic":
            sc = scenarios.parallel_traffic(self.E, self.human_num, seed0, self.traffic_length, self.traffic_height, self.robot_radius)
        else:
            raise NotImplementedError(f"scenario {sim}: the hybrid scenario mixes generators per env (social_nav_gym.py:155-167)")
        self.case_counter[phase] = (self.case_counter[phase] + self.E) % self.case_size[phase]
        robot = sc["robot"].copy()
        # robot goal list of the reference scenarios: [goal, start] (social_nav_sim.py:237,309)
        self._robot_goals = np.stack([robot[:, 10:12], robot[:, 0:2]], 1)
        robot[:, 3:5] = 0.0                                                      # robot.set(..., vx=0, vy=0) (social_nav_gym.py:213)
        states = np.concatenate([sc["states"], robot[:, None]], 1) if self.robot_visible else sc["states"]
        self.engine = self._engine_class().from_reference_arrays(self.human_policy, states, sc["goals"], walls=self.walls, consider_robot=self.robot_visible,
                                                        all_params_equal=True, dtype=self.dtype, device=self.device,
                                                        robot=None if self.robot_visible else robot)
        self.engine.respawn_bounds = sc.get("respawn_bounds")   # parallel traffic: respawn at the right end (mmm:407-422)
        self.engine.consts = [float(self.time_limit), self.collision_penalty, self.success_reward, self.discomfort_dist,
                              self.discomfort_penalty_factor, self.robot_time_step]
        if self.safety_space > 0:
            self.engine.set_safety_space(self.safety_space)
        self._spatial_order()
        return self.observation(), np.zeros(self.E, int)

    def _engine_class(self):
        return TiledCrowdEngine if self.human_num > MAX_FUSED_HUMANS else CrowdEngine

    def _spatial_order(self, mask=None):
        """After a reset of all envs (mask None) or of those of `mask`: rows of reset envs are in the generator's order again; on
        the tiled path with spatial_order, every env is then re-numbered patch by patch and the permutation composed into _order."""
        if mask is None or self._order is None:
            self._order = None
        else:
            ident = torch.arange(self.human_num, device=self._order.device).expand_as(self._order)
            self._order = torch.where(mask.bool()[:, None], ident, self._order)
        if not (isinstance(self.engine, TiledCrowdEngine) and self.spatial_order):
            return
        perm = self.engine._renumber()  # new_rows[e] = old_rows[e][perm[e]]
        self._order = perm if self._order is None else torch.gather(self._order, 1, perm)

    def _reset_on_device(self, sim, seed0, phase, mask=None, seeds=None):
        e = self.engine
        cls = self._engine_class()
        fresh = (e is None or type(e) is not cls or e.N != self.human_num or e.motion_model_title != self.human_policy or
                 e.consider_robot != self.robot_visible)
        if fresh:
            e = self.engine = cls(self.human_policy, self.E, self.human_num, G=2, dtype=self.dtype, device=self.device,
                                          consider_robot=self.robot_visible, symmetric=True, walls=self.walls, has_robot=True)
        e.consts = [float(self.time_limit), self.collision_penalty, self.success_reward, self.discomfort_dist,
                    self.discomfort_penalty_factor, self.robot_time_step]
        name = "ccso_synthetic" if (sim == "circular_crossing_with_static_obstacles" and self.human_num > 10) else sim
        e.reset_scenario(name, seeds=seeds, seed0=seed0, mask=mask, randomize_attributes=self.randomize_attributes,
                         circle_radius=self.circle_radius, robot_radius=self.robot_radius, traffic_length=self.traffic_length,
                         traffic_height=self.traffic_height)
        if mask is None:
            self.case_counter[phase] = (self.case_counter[phase] + self.E) % self.case_size[phase]
        # always rewritten: snp_reset keeps the safety columns, so a safety space from an earlier episode must not survive (gym:215)
        if self.robot_motion_model_title is not None and e.robot_type is None:
            e.set_robot_motion_model(self.robot_motion_model_title)
        e.set_safety_space(self.safety_space if self.safety_space > 0 else None)
        # robot goal list of the reference scenarios: [goal, start] (social_nav_sim.py:237,309)
        r = e.robot
        self._robot_goals = torch.stack([torch.stack([r[L.ROBOT_GX], r[L.ROBOT_GY]], -1), torch.stack([r[L.ROBOT_GX2], r[L.ROBOT_GY2]], -1)], 1).double().cpu().numpy()
        if self.robot_motion_model_title is not None:
            e.set_robot_motion_model(self.robot_motion_model_title)
        self._spatial_order(None if fresh else mask)
        return self.observation(), np.zeros(self.E, int)

    def reset_finished(self, finished, phase="train"):
        """Restart only the envs whose episode ended (`finished` [E] bool: terminated | truncated), each with the next unused case
        of `phase` -- the vectorised form of calling reset() again on those envs.  Stays on the device."""
        fin = torch.as_tensor(finished, device=self.device).bool()
        offset = {"train": 2000, "val": 0, "test": 1000}[phase]
        order = torch.cumsum(fin.int(), 0) - 1
        seeds = (offset + (self.case_counter[phase] + order.long()) % self.case_size[phase]).to(torch.int32)
        n = int(fin.sum().item())
        sim = self.test_sim if phase == "test" else self.train_val_sim
        self._reset_on_device(sim, 0, phase, mask=fin, seeds=seeds)
        self.case_counter[phase] = (self.case_counter[phase] + n) % self.case_size[phase]
        return self.observation()

    def observation(self, theta_and_omega_visible=False):
        """[E,N,5] (or [E,N,7]) with the humans in the generator's order, whatever the engine's numbering."""
        e = self.engine
        cols = [e.dyn[L.DYN_PX], e.dyn[L.DYN_PY], e.dyn[L.DYN_VX], e.dyn[L.DYN_VY], e.stat[L.STAT_R]]
        if theta_and_omega_visible:
            cols += [e.dyn[L.DYN_TH], e.dyn[L.DYN_OM]]
        obs = torch.stack(cols, -1)
        if self._order is not None:
            obs = torch.empty_like(obs).scatter_(1, self._order[..., None].expand_as(obs), obs)
        return obs.double().cpu().numpy()

    def step(self, action):
        """SocialNavGym.step (social_nav_gym.py:227-250) for every env.  `action` [E,2]: (vx, vy) for a holonomic robot (ActionXY) or
        (v, r) for a unicycle one (ActionRot; set `robot_kinematics = "unicycle"`, what RobotAgent takes from its policy,
        robot_agent.py:95).  Above 512 humans per env, parallel traffic and the hybrid scenario raise NotImplementedError here
        (their respawn is not on the tiled path)."""
        self.engine.step(action, self.time_step, n_substeps=self.time_step_factor, pre_checks=True, kinematics=self.robot_kinematics)
        r = self.engine.decode_flags()
        return self.observation(), r["reward"], r["terminated"], r["truncated"], r["info"]

    def set_robot_motion_model(self, title):
        """The robot will be moved by the SFM / HSFM model `title` in imitation_learning_step (mmm:552-591, Euler)."""
        self.robot_motion_model_title = title
        if self.engine is not None:
            self.engine.set_robot_motion_model(title, goals=self._robot_goals)

    def imitation_learning_step(self):
        """social_nav_gym.py:252-274 for every env: time_step_factor x (update_robot; update_humans), then the ACTUAL collision /
        goal checks and the reward at the end time -- one launch.  Above 512 humans per env it raises NotImplementedError (the
        tiled path has no robot moved by its own motion model)."""
        if self.engine.robot_type is None:
            self.engine.set_robot_motion_model(self.robot_motion_model_title, goals=self._robot_goals)
        self.engine.imitation_learning_step(self.time_step, n_substeps=self.time_step_factor)
        r = self.engine.decode_flags()
        return self.observation(), r["reward"], r["terminated"], r["truncated"], r["info"]

    def check_actual_collisions_and_goal(self):
        return self.engine.check_actual_collisions_and_goal()

    @property
    def global_time(self):
        return self.engine.time_now.cpu().numpy()
