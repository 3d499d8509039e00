/*
 * snp_b200.h -- C ABI of libsnp_b200.so: the B200 (sm_100a) batched crowd-stepping engine that drops in for the
 * per-step human motion update of Social-Navigation-PyEnvs.
 *
 * Everything here is plain C: pointers, ints, doubles.  No torch / C++ types cross this boundary.  Device-pointer
 * entry points are stream-ordered, allocate nothing and never synchronise; host-pointer entry points (suffix _host)
 * copy in, run the same kernels, copy out and synchronise the stream they use.
 *
 * Every function returns 0 on success or a negative snp_status; snp_last_error() gives the message
 * (the Python adapter turns it into ValueError / RuntimeError, matching the reference's exceptions,
 * social_gym/src/forces_parallel.py:211).
 *
 * Reference interfaces replaced (paths relative to the reference's social_gym/):
 *   snp_step / snp_update_humans_parallel_host   <- src/forces_parallel.py:184-284 update_humans_parallel  (sole call
 *                                                   site src/motion_model_manager.py:360), and the serial path it
 *                                                   shadows: motion_model_manager.py:354-373,424-459 + src/forces.py
 *   fused sub-step loop + robot motion            <- social_nav_gym.py:240-245 (20 x robot.step + update_humans),
 *                                                   src/robot_agent.py:126-136
 *   snp_gym_step_host                             <- social_nav_gym.py:227-250 SocialNavGym.step with host action / observation buffers
 *   snp_checks (+ fused into snp_step)            <- social_nav_sim.py:949-984 collision_detection_and_reaching_goal,
 *                                                   :986-1029 compute_reward_and_infos, :702-703;
 *                                                   social_nav_gym.py:107-118 check_actual_collisions_and_goal
 *   snp_laser / snp_laser_host                    <- src/sensors.py:53-69 LaserSensor.get_laser_measurements
 *                                                   (:24-33 circle, :35-51 segment), src/robot_agent.py:77-82
 *   respawn option of snp_step                    <- motion_model_manager.py:407-422 (parallel-traffic post_update)
 *   robot_mode 2 of snp_step                      <- motion_model_manager.py:593-653 update_robot / compute_robot_forces,
 *                                                   social_nav_gym.py:252-274 imitation_learning_step
 *   snp_lookahead (+ dyn_out peek of snp_step)    <- crowd_nav/policy/cadrl.py:42-83 compute_rotated_states_and_reward, :13-40;
 *                                                   motion_model_manager.py:691-709 get_next_human_observable_states
 *   snp_value_lookahead                           <- crowd_nav/policy/cadrl.py:235-276 CADRL.predict (value network, min, argmax)
 *   snp_robot_push_out                            <- src/robot_agent.py:35-48 RobotAgent.check_collisions (social_nav_sim.py:509)
 *   snp_reset                                     <- social_nav_gym.py:120-225 reset, social_nav_sim.py:200-431 scenario generators
 *   snp_pack_states / snp_unpack_states           <- src/agent.py:256-266 get_safe_state / set_state row layout
 *   snp_large_run_p2p                             <- same update for one very large crowd (tiled all-pairs), with its robot
 *   snp_large_checks                              <- the checks above for the robot of one very large crowd
 *   snp_spatial_order / snp_gather_crowd          <- scenarios.spatial_order (+ deal_tiles) and new_rows = old_rows[perm], mid-run
 */
#ifndef SNP_B200_H
#define SNP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNP_ABI_VERSION 4

typedef enum snp_status {
    SNP_OK = 0,
    SNP_ERR_INVALID = -1, /* bad argument (type outside 0..8, sizes, null pointers) -> ValueError */
    SNP_ERR_CUDA = -2,    /* CUDA runtime error */
    SNP_ERR_UNSUPPORTED = -3
} snp_status;

enum { SNP_F32 = 0, SNP_F64 = 1 };
enum { SNP_OPT_FULL_PAIR_LOOP = 1, SNP_OPT_NO_CULLING = 2, SNP_OPT_MAP_WARP = 4, SNP_OPT_MAP_BLOCK = 8,
       SNP_OPT_STAGED_COPIES = 16, /* snp_gym_step_host: D2H copies after the launch even for pinned result buffers */
       SNP_OPT_UNIT_SCRATCH = 32   /* snp_large_run_p2p / snp_large_batch_step: the scratch was sized by snp_large_*scratch_bytes_units */ };

/* Field order of the structure-of-arrays buffers (each field is a contiguous run of E*N elements). */
enum { SNP_DYN_PX = 0, SNP_DYN_PY, SNP_DYN_VX, SNP_DYN_VY, SNP_DYN_TH, SNP_DYN_BVX, SNP_DYN_BVY, SNP_DYN_OM,
       SNP_DYN_DFX, SNP_DYN_DFY, SNP_DYN_FIELDS };                        /* dfx,dfy: carried desired force (forces.py:12-15) */
enum { SNP_STAT_R = 0, SNP_STAT_M, SNP_STAT_VD, SNP_STAT_SAFETY, SNP_STAT_FIELDS };
enum { SNP_ROBOT_PX = 0, SNP_ROBOT_PY, SNP_ROBOT_VX, SNP_ROBOT_VY, SNP_ROBOT_R, SNP_ROBOT_SAFETY, SNP_ROBOT_GX,
       SNP_ROBOT_GY, SNP_ROBOT_TH,
       /* only used when the robot is driven by a motion model (robot_mode == 2): */
       SNP_ROBOT_BVX, SNP_ROBOT_BVY, SNP_ROBOT_OM, SNP_ROBOT_M, SNP_ROBOT_VD, SNP_ROBOT_DFX, SNP_ROBOT_DFY,
       SNP_ROBOT_GX2, SNP_ROBOT_GY2,   /* the other goal of the robot's (at most two-entry) goal list */
       SNP_ROBOT_GCNT,                 /* 1 or 2 goals */
       SNP_ROBOT_SPARE, SNP_ROBOT_FIELDS };

/* Bits of the per-env flags word written by snp_step / snp_checks. */
enum {
    SNP_FLAG_COLLISION = 1 << 0,        /* swept test over one robot step (social_nav_sim.py:949-979) */
    SNP_FLAG_REACHING_GOAL = 1 << 1,    /* social_nav_sim.py:980-983 */
    SNP_FLAG_TERMINATED = 1 << 2,       /* social_nav_sim.py:986-1029 */
    SNP_FLAG_TRUNCATED = 1 << 3,
    SNP_FLAG_INFO_SHIFT = 4,            /* 3 bits: 0 Nothing 1 Timeout 2 Collision 3 ReachGoal 4 Danger */
    SNP_FLAG_ACTUAL_COLLISION = 1 << 7, /* social_nav_gym.py:107-118 on the post-step state */
    SNP_FLAG_ACTUAL_GOAL = 1 << 8,
    SNP_FLAG_TOUCHED = 1 << 9           /* |p_h - p_r| < r_h + r_r after any sub-step (social_nav_sim.py:702-703) */
};

/* A batch of E independent environments with N humans each, resident in device memory.
 * `dtype` selects float or double for every `void*` array below. */
typedef struct snp_crowd {
    int32_t E, N, G;          /* envs, humans per env, goal slots per human */
    int32_t dtype;            /* SNP_F32 / SNP_F64 */
    void *dyn;                /* [SNP_DYN_FIELDS][E*N]   updated in place */
    const void *stat;         /* [SNP_STAT_FIELDS][E*N] */
    const void *goals;        /* [G][2][E*N]  goal lists; slots >= goal_cnt are ignored */
    int32_t *goal_idx;        /* [E*N] index of the current goal (the reference rotates the list instead,
                                 motion_model_manager.py:66-70); updated in place */
    const int32_t *goal_cnt;  /* [E*N] number of valid goals (>= 1) */
    const void *agent_params; /* optional [20][E*N] per-agent parameter rows (agent.py:269); NULL -> `params` for all */
    double params[20];        /* uniform parameter row used when agent_params == NULL */
    void *robot;              /* optional [SNP_ROBOT_FIELDS][E]; required when consider_robot or checks are on */
    const void *walls;        /* optional [walls_per_env ? E : 1][W*S][4] = ax,ay,bx,by per segment slot, NaN-padded
                                 (motion_model_manager.py:268-276), endpoints ordered as obstacle.py:31-32 */
    int32_t W, S;             /* wall polygons, segment slots per polygon */
    int32_t walls_per_env;
} snp_crowd;

typedef struct snp_step_opts {
    int32_t type;             /* 0..8 index into SFMS (motion_model_manager.py:15-17) */
    int32_t consider_robot;   /* robot exerts force on humans (motion_model_manager.py:35) */
    int32_t symmetric;        /* all_equal_humans: pair (i,j), i<j evaluated with i as agent1 and applied +/- (forces.py:130-151);
                                 0 -> per-agent path (forces.py:153-218) */
    int32_t numba_compat;     /* 0: serial Python/NumPy semantics (oracle of record); 1: forces_parallel.py semantics
                                 ('<=' goal test, zeroed desired force, Guo wall force / W, first-wins closest segment) */
    int32_t n_substeps;       /* fused update_humans calls per launch (20 in SocialNavGym.step) */
    int32_t robot_mode;       /* 0: robot row fixed during the launch; 1: holonomic action: before every sub-step
                                 p += a*dt, v = a (robot_agent.py:126-131); 2: the robot is moved by its own SFM / HSFM model
                                 before every human update (motion_model_manager.py:593-653 update_robot, as in
                                 SocialNavGym.imitation_learning_step, social_nav_gym.py:260-265); 3: unicycle action (v, r):
                                 before every sub-step p += v (cos, sin)(yaw + r) dt, yaw = (yaw + r) % 2 pi, velocity along the
                                 new yaw (robot_agent.py:116-136); the swept check uses v (cos, sin)(yaw + r) (social_nav_sim.py:973,
                                 with the robot's yaw where the reference reads its never-assigned `theta`) */
    double dt;
    const void *action;       /* [2][E] (dtype of the crowd) when robot_mode == 1 / 3 or pre_checks: (vx, vy), or (v, r) in mode 3 */
    int32_t pre_checks;       /* swept collision / goal / reward on the PRE-step state (social_nav_gym.py:232-234) */
    int32_t post_checks;      /* 1: actual collision / goal on the POST-step state (social_nav_gym.py:107-118); 2: also reward, terminated,
                                 truncated and info code from them at the end time (imitation_learning_step, social_nav_gym.py:269-271) */
    int32_t track_touch;      /* OR of the run_k_steps collision test after every sub-step */
    int32_t reserved;         /* bit 0 (SNP_OPT_FULL_PAIR_LOOP): evaluate every ordered pair in j-ascending order (the reference's
                                 accumulation order) instead of each unordered pair once per warp;
                                 bits 2-3 (SNP_OPT_MAP_WARP / SNP_OPT_MAP_BLOCK): force the warp-packed / block-packed thread mapping */
    double consts[6];         /* time_limit, collision_penalty, success_reward, discomfort_dist,
                                 discomfort_penalty_factor, robot_time_step */
    double *time_now;         /* optional [E] global_time; read by the reward, advanced by dt per sub-step */
    int32_t *flags;           /* [E] out, required when any check is on */
    double *checks;           /* [E][4] out: dmin (swept), reward, dmin (actual), unused */
    double respawn_bounds[2]; /* (traffic_length / 2, traffic_height / 2)  (social_nav_sim.py:360) */
    int32_t respawn;          /* parallel-traffic respawn after every sub-step (motion_model_manager.py:407-422): humans within 3 m of
                                 their goal restart at the right end; rewrites goals[0], goal_cnt (N <= 32 only) */
    int32_t robot_type;       /* robot_mode 2: the robot's model, 0..8 (may differ from the humans') */
    double robot_params[20];  /* robot_mode 2: the robot's parameter row (agent.py:269 for its model) */
    void *dyn_out;            /* optional [SNP_DYN_FIELDS][E*N]: PEEK (motion_model_manager.py:691-709 get_next_human_observable_states):
                                 the updated px..omega fields are written here instead of in place and the goal index is not
                                 advanced; the carried desired force is still updated in place (the reference does not restore it) */
    const int32_t *respawn_envs; /* optional [E], with respawn: only envs with a non-zero entry respawn (hybrid scenario: the parallel-traffic
                                 envs of a mixed batch; snp_reset's scenario_out works as is) */
    int32_t *goal_idx_out;    /* optional [E*N], with dyn_out: the goal index the update arrived at (the peek reports the goal after it) */
    int32_t robot_every;      /* robot_mode 2 only.  0: SocialNavGym.imitation_learning_step order (update_robot, then humans that see the
                                 moved robot).  >= 1: SocialNavSim.update / control_robot (social_nav_sim.py:476-529): the humans see the
                                 robot's state from BEFORE its update (:484-491); 1 = equal sampling times, update_robot(dt) every
                                 sub-step (:521); k > 1 = the pose advances every sub-step with the last velocity, yaw unwrapped
                                 (update_robot_pose, motion_model_manager.py:655-657) and every k-th sub-step the velocities are refreshed
                                 by update_robot(..., consts[5] = ROBOT_SAMPLING_TIME, just_velocities=True) (:523-524, mmm:72-85) */
    int32_t robot_phase;      /* robot_every > 1: index of this launch's first sub-step in that schedule (n_updates of the simulator) */
} snp_step_opts;

typedef struct snp_laser_args {
    int32_t E, N;             /* envs, circles (humans) per env */
    int32_t dtype;
    int32_t samples;
    const void *px, *py, *radius; /* [E*N] each (SoA fields of a crowd work as is) */
    const void *walls;        /* as snp_crowd.walls */
    int32_t W, S, walls_per_env;
    int32_t reserved;
    const void *pose;         /* [3][E] x, y, yaw of the sensor */
    double range, max_distance, robot_radius; /* robot_radius is subtracted from the ranges (robot_agent.py:81); 0 for raw */
    void *ranges;             /* [E][samples] out */
    int32_t *hits;            /* [E][samples] out (optional): human index, N + segment ordinal, or -1 */
    /* ABI 3 (appended): LaserSensor.add_uncertainty (sensors.py:71-74) on the device -- every range becomes
     * clip(N(range, uncertainty), 0, max_distance) before the robot radius is subtracted.  The reference draws from the caller's global
     * np.random stream, one normal per ray in ray order; here ray (env, k) of scan `noise_scan` takes its normal from the counter-based
     * Philox4x32-10 stream keyed by `noise_seed` (counter = k, env, scan): same distribution, reproducible, independent of the launch
     * geometry.  uncertainty <= 0 (or NaN): no noise, as with uncertainty=None. */
    double uncertainty;
    uint64_t noise_seed;
    uint64_t noise_scan;
} snp_laser_args;

/* One-step lookahead of the value-network policies (crowd_nav/policy/cadrl.py:42-83 compute_rotated_states_and_reward,
 * called from CADRL.predict :235-262) for every env of a crowd and every action of the action space. */
typedef struct snp_lookahead_args {
    int32_t type;             /* the humans' model 0..8 (headed models take yaw / omega from `next`, the others from the crowd) */
    int32_t A;                /* number of actions */
    int32_t theta_and_omega_visible; /* 0: 13 values per (action, human); 1: 15 (cadrl.py:14-21) */
    int32_t reserved;         /* bit 0: write the rows with per-thread vector stores instead of bulk asynchronous copies (A/B measurement);
                                 bit 1: split every env's humans into chunks of 256 over several CTAs, which is what runs by itself
                                 where one CTA's shared memory cannot hold an env (fp64 N > 673 / > 609 visible, fp32 > 1312 / > 1190);
                                 the same bits either way (tests and measurement).  Any N; the outputs may exceed 2^31 words */
    const void *next;         /* [SNP_DYN_FIELDS][E*N] the humans one policy time step ahead: output of the peek (snp_step with dyn_out) */
    const double *actions;    /* [A][2] holonomic velocities (vx, vy), shared by all envs (cadrl.py build_action_space) */
    double dt;                /* the policy's time step (0.25) */
    void *rotated;            /* out [E][A][N][13|15] in the crowd's dtype: dg, v_pref, theta, radius, vx, vy, px1, py1, vx1, vy1, radius1, da,
                                 radius_sum (, theta1, omega1) */
    double *rewards;          /* out [E][A]: -0.25 collision, 1 goal, (dmin - 0.2) * 0.5 * dt discomfort, 0 (cadrl.py:68-72), bit-exact */
} snp_lookahead_args;

/* CADRL's action choice (crowd_nav/policy/cadrl.py:235-276 CADRL.predict) for every env of a crowd, with the value network evaluated
 * on the device where the lookahead's rows are made (csrc/snp_value.cu): rotated rows (as snp_lookahead, rounded to fp32) -> MLP ->
 * minimum over the humans -> value = reward + gamma ^ (dt * v_pref) * (double) minimum in double -> first action of largest value.
 * The rows and the network's activations never reach device memory. */
typedef struct snp_value_args {
    int32_t type;             /* the humans' model 0..8, as snp_lookahead_args.type */
    int32_t A;                /* number of actions, 1..65535 */
    int32_t theta_and_omega_visible; /* 0: 13 values per row; 1: 15 -- must equal widths[0] */
    int32_t reserved;         /* bit 1: split every env's humans into chunks of 32 over several CTAs (the same bits; tests and measurement) */
    const void *next;         /* [SNP_DYN_FIELDS][E*N] the humans one policy time step ahead (as snp_lookahead_args.next) */
    const double *actions;    /* [A][2] holonomic velocities (vx, vy) */
    double dt;                /* the policy's time step (0.25) */
    double gamma;             /* the policy's discount factor */
    int32_t layers;           /* Linear layers, 1..6, with ReLU between them and none after the last */
    int32_t widths[7];        /* widths[0] = 13 | 15 inputs, widths[1..layers-1] hidden widths in 1..256, widths[layers] = 1 */
    const float *weights;     /* device fp32, layer by layer: W transposed ([in][out] row-major, i.e. torch's weight.t()) then b [out] */
    double *values;           /* out [E][A] */
    int32_t *best;            /* out [E]: first index of the largest value (-1 if no value exceeds -inf) */
    uint8_t *reached;         /* out [E]: 1 where the robot is within its radius of its goal now (predict returns the zero action there) */
} snp_value_args;

/* SocialNavGym.reset for every (selected) environment of a crowd, on the device (social_gym/social_nav_gym.py:120-225): env e replays
 * the reference's scenario generator (social_gym/social_nav_sim.py:200-299 circular crossing, :301-362 parallel traffic, :364-431
 * circular crossing with static obstacles; insert_robot = True, randomize_human_positions = True) on NumPy's own MT19937 stream seeded
 * with seeds[e] (the gym seeds np.random with offset[phase] + case, social_nav_gym.py:135-137): same draws, same accept / reject
 * decisions, positions equal up to the last ulp of cos / sin. */
enum { SNP_RESET_CIRCULAR_CROSSING = 0, SNP_RESET_PARALLEL_TRAFFIC = 1, SNP_RESET_CCSO = 2,
       SNP_RESET_CCSO_SYNTHETIC = 3, /* 3 static humans + the circular-crossing sampler: the 25-human crowd of SURVEY.md 8(d) config 3 */
       SNP_RESET_HYBRID = 4          /* np.random.choice between the first two, then re-seed (social_nav_gym.py:155-157) */ };
enum { SNP_RESET_FORCE_CTA = 1 };
typedef struct snp_reset_args {
    int32_t scenario;
    int32_t randomize_attributes; /* desired speed ~ U(0.5,1.5), radius ~ U(0.3,0.5) per human, drawn first (social_nav_sim.py:217-220) */
    const uint32_t *seeds;        /* optional [E] device: np.random.seed argument of each env; NULL -> seed0 + env index */
    uint32_t seed0;
    uint32_t reserved;            /* bit 0 (SNP_RESET_FORCE_CTA): use the CTA-per-env kernel even where the warp kernel fits */
    const uint8_t *mask;          /* optional [E] device: only envs with a non-zero entry are reset (restart of finished episodes) */
    double circle_radius, robot_radius, traffic_length, traffic_height;
    double human_mass, robot_mass, robot_desired_speed; /* 75 (social_nav_sim.py:141), 80 (robot_agent.py:16), 1 */
    double *time_now;             /* optional [E]: set to 0 (social_nav_gym.py:129) */
    int32_t *flags;               /* optional [E]: cleared */
    int32_t *scenario_out;        /* optional [E]: the scenario generated (the hybrid scenario's coin) */
    int32_t *draws_out;           /* optional [E]: number of uniforms the generator consumed */
} snp_reset_args;

int snp_abi_version(void);
const char *snp_last_error(void);
/* Device properties the host side sizes grids with: sm_count, cc_major, cc_minor, l2_bytes. */
int snp_device_info(int32_t *out4);

/* ---- device-pointer API ---- */
int snp_step(const snp_crowd *crowd, const snp_step_opts *opts, void *cuda_stream);
int snp_checks(const snp_crowd *crowd, const snp_step_opts *opts, void *cuda_stream);
int snp_laser(const snp_laser_args *args, void *cuda_stream);
/* RobotAgent.check_collisions (src/robot_agent.py:35-48): crowd->robot's position is pushed out of the humans it overlaps (in index
 * order), then out of the wall polygons it overlaps; sequential per env, bit-identical to the reference for fp64 state. */
int snp_robot_push_out(const snp_crowd *crowd, void *cuda_stream);
/* Rewrites crowd->dyn, stat (radius, mass, desired speed; the safety space is kept), goals, goal_idx, goal_cnt and crowd->robot.
 * One warp per env while four envs' scratch (624 generator words + 32 bytes per human) fits 200 KB of shared memory, N <= 1522;
 * above that one CTA of 16 warps per env, which splits the test of a candidate against the placed humans between its warps, up to
 * N = 6322; larger N is SNP_ERR_UNSUPPORTED before any launch (the host generators cover any N).  args->reserved bit 0
 * (SNP_RESET_FORCE_CTA) takes the CTA kernel at any N up to that limit.  Both kernels give the same bits in every output. */
int snp_reset(const snp_crowd *crowd, const snp_reset_args *args, void *cuda_stream);
/* Uses crowd->dyn (current px,py,vx,vy,theta,omega), crowd->stat (radius) and crowd->robot (px,py,r,gx,gy,vd). */
int snp_lookahead(const snp_crowd *crowd, const snp_lookahead_args *args, void *cuda_stream);
/* Uses what snp_lookahead uses; values / best / reached only.  SNP_ERR_INVALID before any launch for null pointers, E or N < 1,
 * E > 65535, A outside 1..65535, a bad type or dtype, layers outside 1..6, widths[0] != 13 | 15 (theta_and_omega_visible), a hidden
 * width outside 1..256 or widths[layers] != 1. */
int snp_value_lookahead(const snp_crowd *crowd, const snp_value_args *args, void *cuda_stream);
/* The policies' query_env = False branch (crowd_nav/policy/cadrl.py:92-105 propagate_humans_state_with_constant_velocity_model):
 * `next` [SNP_DYN_FIELDS][E*N] (crowd dtype) = the humans one step of length dt ahead under constant velocity (x + vx dt, y + vy dt,
 * theta + omega dt, velocities carried over) -- the `next` input of snp_lookahead when the env is not queried. */
int snp_constant_velocity(const snp_crowd *crowd, double dt, void *next, void *cuda_stream);
/* AoS <-> SoA: rows are the reference's 13-wide float64 state rows [E][rows][13] with the robot (if any) as row N. */
int snp_unpack_states(const snp_crowd *crowd, const double *rows_dev, int32_t rows_per_env, const double *safety_dev,
                      void *cuda_stream);
int snp_pack_states(const snp_crowd *crowd, double *rows_dev, int32_t rows_per_env, void *cuda_stream);
/* Goal lists: reference rows [E][N][G][2] NaN padded (motion_model_manager.py:262-267) -> crowd->goals / goal_idx (= 0) and
 * goal_cnt_dev (writable alias of crowd->goal_cnt).  snp_rotate_goal_rows applies the rotation the reference would have
 * performed in place (forces_parallel.py:229-232) to the caller's float64 rows, given the crowd's goal_idx. */
int snp_unpack_goals(const snp_crowd *crowd, const double *goal_rows_dev, int32_t *goal_cnt_dev, void *cuda_stream);
int snp_rotate_goal_rows(const snp_crowd *crowd, double *goal_rows_dev, void *cuda_stream);
/* One very large crowd (the crowd's E*N agents form ONE environment), shared-memory tiled all-pairs: `n_substeps` sub-steps in ONE
 * call (the loop SocialNavGym.step runs, social_nav_gym.py:240-245), all enqueued on `cuda_stream` without returning to the host.
 * The crowd is this rank's slice of agents of a view of M entities exerting force (x,y,vx,vy,r+safety, SoA), starting at entity
 * `self_offset`; a crowd not sharded over GPUs is the whole view (world = 1, rank = 0, self_offset = 0).  Own state is updated in
 * place and the updated entries of the own agents are stored into the next view of every rank.  Buffers, as host arrays of `world`
 * device pointers indexed by rank (peer-mapped over NVLink when world > 1, e.g. torch symmetric memory): `peer_views_a` /
 * `peer_views_b` = the two view buffers, each [5][M] entities followed by the view's [ceil(M/128)][5] tile-box table; `peer_flags` =
 * uint64[world] barrier slots per rank, zero-initialised once.  `first_is_b` selects the buffer that holds the current view;
 * `epoch_base` must grow by `n_substeps` from call to call.  Per sub-step: the tiled pair phase, the finish kernel and, when
 * world > 1, one single-warp barrier kernel; `error_flag` (device int32) is set if a peer never reached a barrier.  When this slice
 * is a whole number of 128-entity tiles and the `world` slices make up the view, the producers also write the next view's tile boxes;
 * otherwise every sub-step recomputes the boxes of the view it reads (one more launch).  An exchange of its own (e.g. an all-gather
 * of the slices) runs between calls of one sub-step with world = 1.  `scratch` = 16-byte aligned device workspace of at least
 * snp_large_scratch_bytes(n_local, M, dtype) bytes (per-chunk partial sums, the map and lists of the (agent block, entity chunk)
 * units in reach, the work queues' counters).  opts->reserved bit 1 (SNP_OPT_NO_CULLING) disables the exact far-tile culling.
 * opts->reserved bit 5 (SNP_OPT_UNIT_SCRATCH): the scratch was sized by snp_large_scratch_bytes_units(n_local, M, dtype, units); a culled
 * step then keeps the partial sums of a unit in reach in slot k = its position on the work list, of floor(extra bytes / (2 * 128 *
 * sizeof(T))) slots (0 or more), so memory follows the units in reach instead of n_local * M.  A unit without a slot is evaluated by
 * the finish kernel in its place in the order: the result is bit for bit that of the default scratch whatever the slot count; it only
 * costs time.  With the bit, before any launch, what needs the static grid is SNP_ERR_UNSUPPORTED: Moussaid types (2, 5, 8),
 * SNP_OPT_NO_CULLING, pair-law parameters without a culling distance, a self_offset that is not a multiple of 128,
 * ceil(n_local/128) * ceil(M/128) >= 2^31 units; and the scratch must be at least the size for 0 units.  Unit counts of the call (with
 * the bit): int32 word 1 of the scratch = the most units listed in one sub-step, word 2 = the units the finish kernel evaluated for
 * want of a slot; the call's first launch zeroes them, and nothing synchronises.  Without the bit the scratch and the kernels are
 * the default ones, and words 1 and 2 hold nothing.
 * The robot of SocialNavGym.step (crowd->robot, one env): opts->robot_mode 0 (fixed), 1 (holonomic action) or 3 (unicycle action)
 * moves it before every sub-step as snp_step does, and opts->consider_robot adds its pair force to every human (never culled).  Every
 * rank recomputes the robot of each sub-step from crowd->robot, so no exchange is needed; after the last sub-step crowd->robot holds
 * the end state and opts->time_now (optional) has advanced by dt per sub-step.  The checks are snp_large_checks.  robot_mode 2,
 * track_touch, pre_checks / post_checks, dyn_out and respawn are SNP_ERR_UNSUPPORTED, before any launch. */
int64_t snp_large_scratch_bytes(int64_t n_local, int64_t M, int32_t dtype);
/* The scratch of a culled step with `units` slots of partial sums (SNP_OPT_UNIT_SCRATCH); host arithmetic, -1 for bad arguments
 * (n_local < 1, M < n_local, units < 0, bad dtype).  At units = ceil(n_local/128) * ceil(M/128) and n_local a multiple of 128 it
 * equals snp_large_scratch_bytes. */
int64_t snp_large_scratch_bytes_units(int64_t n_local, int64_t M, int32_t dtype, int64_t units);
int snp_large_run_p2p(const snp_crowd *crowd, const snp_step_opts *opts, const void *const *peer_views_a, const void *const *peer_views_b,
                      int32_t first_is_b, int64_t M, int64_t self_offset, int32_t world, int32_t rank, const void *const *peer_flags,
                      uint64_t epoch_base, int32_t n_substeps, int32_t *error_flag, void *scratch, int64_t scratch_bytes, void *cuda_stream);
/* The collision / goal / reward checks of SocialNavGym.step for the robot crowd->robot (one env) against the M humans of a view
 * buffer `view` [5][M] (x, y, vx, vy, r+safety; as snp_large_run_p2p reads and writes it) with radii `radius` [M], both in the
 * crowd's dtype.  opts->pre_checks: the swept test over one robot step of length consts[5] with opts->action (v (cos, sin)(yaw + r)
 * for robot_mode 3), stopping at the first colliding human in index order, dmin, the goal test and the reward / info code at
 * opts->time_now (social_nav_sim.py:949-1029).  opts->post_checks = 1: actual dmin, collision and goal (social_nav_gym.py:107-118).
 * Writes the bits and checks fields of the checks it runs into opts->flags[0] / opts->checks[0..3] (as snp_step; the other bits and
 * fields are left as they are).  Double arithmetic, formula-exact; one CTA, no workspace, no host synchronisation. */
int snp_large_checks(const snp_crowd *crowd, const snp_step_opts *opts, const void *view, const void *radius, int64_t M, void *cuda_stream);
/* SocialNavGym.step (social_nav_gym.py:227-250) for E environments of N humans each, any N >= 1 (snp_step's limit is 512), through
 * the tiled kernels of snp_large_run_p2p with an environment axis: tiles, chunks and agent blocks are per env, so a human only ever
 * meets humans of its own env, and env e's result is bit for bit that of snp_large_run_p2p / snp_large_checks on env e alone.  One
 * call, all enqueued on `cuda_stream` without host synchronisation: the entity view is published from crowd->dyn (as
 * snp_large_publish: v = R(yaw) bv for headed models), the swept
 * pre-checks run (opts->pre_checks), then n_substeps x (robot step; tiled update), the robot's end state and the clock
 * (opts->time_now, optional, [E]), and the actual post-checks (opts->post_checks = 1).  Honours type, consider_robot, symmetric,
 * numba_compat, n_substeps, robot_mode 0 / 1 / 3, action [2][E], dt, consts, flags [E], checks [E][4] and reserved bit 1
 * (SNP_OPT_NO_CULLING); crowd->robot is [SNP_ROBOT_FIELDS][E]; walls are shared or per env (walls_per_env).  When a check runs the
 * env's flags and checks are rewritten from zero (as snp_step); otherwise they are left as they are.  `scratch` = 16-byte aligned
 * device workspace of at least snp_large_batch_scratch_bytes(E, N, dtype) bytes: the two view buffers, their tile boxes, the
 * partial sums [ceil(N/128)][2][E*N], the live map and the work lists; nothing is carried from one call to the next.  Before any
 * launch: robot_mode 2, robot_every, track_touch, post_checks 2, dyn_out, respawn and crowd->agent_params are SNP_ERR_UNSUPPORTED;
 * bad E / N / G / dtype / type, missing arrays, a missing robot / action / flags and too small a scratch are SNP_ERR_INVALID.
 * snp_large_batch_scratch_bytes returns -1 for bad arguments.  SNP_OPT_UNIT_SCRATCH and the unit counts in words 1 and 2 of the
 * scratch are as for snp_large_run_p2p, with a scratch of snp_large_batch_scratch_bytes_units(E, N, dtype, units) bytes (units of
 * E * ceil(N/128) * ceil(N/128); Moussaid types and SNP_OPT_NO_CULLING refused); the same bits whatever the slot count.
 * With n_substeps = 0 a call is the checks alone, at any N (what snp_checks does for N <= 512): publish, then the pre- and / or
 * post-checks on the current state; crowd->dyn, the robot and the clock are left as they are. */
int64_t snp_large_batch_scratch_bytes(int32_t E, int32_t N, int32_t dtype);
int64_t snp_large_batch_scratch_bytes_units(int32_t E, int32_t N, int32_t dtype, int64_t units);
int snp_large_batch_step(const snp_crowd *crowd, const snp_step_opts *opts, void *scratch, int64_t scratch_bytes, void *cuda_stream);
/* Writes this crowd's [5][.] entity view (x,y,vx,vy,r+safety; v = R(yaw) bv for headed models) into `view` (field stride
 * `stride` elements, starting at element `offset`). */
int snp_large_publish(const snp_crowd *crowd, int32_t type, void *view, int64_t stride, int64_t offset, void *cuda_stream);
/* The [ceil(M/128)][5] tile-box table (xmin, xmax, ymin, ymax, max r+safety of every 128-entity tile) of a view buffer `view` =
 * [5][M] entities followed by that table, as the first sub-step of a snp_large_run_p2p call computes it: a view republished between
 * calls (e.g. after a re-numbering) then carries the boxes of its own entities. */
int snp_large_tile_boxes(void *view, int64_t M, int32_t dtype, void *cuda_stream);

/* ---- re-numbering the humans patch by patch (csrc/snp_order.cu) ----
 * The far-tile culling of the tiled path compares bounding boxes of runs of 128 consecutive humans, so it skips more when
 * consecutive humans stand close together.  A crowd that walks for long mixes; re-numbering it now and then keeps its tiles compact.
 * snp_spatial_order: for each of E envs of N humans (positions px, py [E*N] in `dtype`), perm [E][N] int64 = the permutation
 * scenarios.spatial_order(positions) returns with block = 256 -- max(1, round_half_even(sqrt(N / 256))) strips of equal head count
 * (the first N % strips one human more, as np.array_split) cut from the humans in ascending x, each walked in ascending y, every
 * sort stable (ties keep index order), -0.0 equal to +0.0, fp32 positions ordered as their float64 widening.  perm[e][k] is the
 * env-local index the human going to place k has now: new rows = old rows[perm].  world > 1 (N a whole number of 128-human tiles)
 * then deals the tiles round-robin to `world` ranks (scenarios.deal_tiles).  *nonfinite (device int32) is set to 1 when a position
 * is NaN or infinite, to 0 otherwise; perm is then meaningless.  Stable CUB radix sorts on `cuda_stream`, no host synchronisation;
 * `scratch` = 16-byte aligned device workspace of at least snp_spatial_order_scratch_bytes(E, N) bytes (which asks CUB for its
 * temporary storage: it needs the CUDA device; -1 for bad arguments or a CUDA error).  E * N < 2^31. */
int64_t snp_spatial_order_scratch_bytes(int32_t E, int32_t N);
int snp_spatial_order(const void *px, const void *py, int32_t E, int32_t N, int32_t dtype, int32_t world, int64_t *perm,
                      int32_t *nonfinite, void *scratch, int64_t scratch_bytes, void *cuda_stream);
/* Applies a re-numbering to every per-agent array of `dst` (dyn, all SNP_DYN_FIELDS fields with the carried desired force; stat;
 * goals; goal_idx; goal_cnt) from `src`, a crowd of the same E, G and dtype with src->N >= offset + dst->N humans per env: agent k
 * of env e of dst = agent perm[e * src->N + offset + k] of env e of src.  So a rank of an agent-sharded crowd takes its slice
 * [offset, offset + n_local) of the re-numbered whole crowd from a gathered copy of it, and one crowd (offset 0, same N) from a
 * copy of itself; dst and src must not overlap.  The robot, walls and parameters are not per-agent arrays and are not touched;
 * agent_params is SNP_ERR_UNSUPPORTED.  An entry of perm outside 0..src->N-1 sets *error_flag (optional device int32) and leaves
 * that agent unwritten.  One launch, no host synchronisation. */
int snp_gather_crowd(const snp_crowd *dst, const snp_crowd *src, const int64_t *perm, int64_t offset, int32_t *error_flag,
                     void *cuda_stream);

/* ---- host-pointer API (the reference operator, batched over a leading env axis) ----
 * update_humans_parallel(type, agents_state, goals, obstacles, agents_params, dt, safety_space,
 *                        all_params_equal, last_is_robot) -> updated_state        forces_parallel.py:184
 * agents_state [E][rows][13] (rows = N + last_is_robot), goals [E][N][G][2] NaN-padded and ROTATED IN PLACE on goal
 * reach, agents_state[:,:,10:12] refreshed and (headed models) [:,:,3:5] overwritten as the reference does
 * (fp:229-234,256); obstacles [W][S][2][2] NaN-padded or NULL; agents_params [E][N][20]; safety_space [E][rows];
 * desired_force [E][N][2] in/out or NULL (zeros; only the serial semantics carry it); out_state [E][rows][13]. */
int snp_update_humans_parallel_host(int32_t type, int32_t E, int32_t N, int32_t G, double *agents_state, double *goals,
                                    const double *obstacles, int32_t W, int32_t S, const double *agents_params, double dt,
                                    const double *safety_space, int32_t all_params_equal, int32_t last_is_robot,
                                    int32_t numba_compat, int32_t dtype, int32_t n_substeps, double *desired_force,
                                    double *out_state);
/* SocialNavGym.step (social_gym/social_nav_gym.py:227-250) for a crowd that stays RESIDENT on the device, with host buffers for what
 * crosses the boundary every step: `action_host` [2][E] (crowd dtype; copied into opts->action), then snp_step, then the observation
 * `obs_host` [4][E*N] = px, py, vx, vy of every human (crowd dtype), `flags_host` [E] and `checks_host` [E][4] (dmin, reward, actual
 * dmin, -) are copied back and the stream is synchronised.  Pass pinned host memory for asynchronous copies; any of the host
 * pointers may be NULL. */
int snp_gym_step_host(const snp_crowd *crowd, const snp_step_opts *opts, const void *action_host, void *obs_host, int32_t *flags_host,
                      double *checks_host, void *cuda_stream);
/* LaserSensor.get_laser_measurements over E sensors: humans [E][N][3] = x,y,r; walls [W][S][2][2]; pose [E][3];
 * ranges [E][samples]; hits [E][samples] or NULL. */
int snp_laser_host(int32_t E, int32_t N, const double *humans, const double *walls, int32_t W, int32_t S, const double *pose,
                   double range, int32_t samples, double max_distance, double robot_radius, int32_t dtype, double *ranges,
                   int32_t *hits);

/* ---- measurement helpers (bench.py) ---- */
/* Runs a register-resident FMA / MUFU loop on every SM and returns achieved TFLOP/s (kind 0 fp32 FMA, 1 fp64 FMA)
 * or Gop/s (kind 2 MUFU.EX2).  Used as the measured denominator of the compute roofline. */
int snp_measure_pipe_peak(int32_t kind, double *out);
/* Test hook: y[i] = the kernels' table-based fp64 exp (csrc/snp_math.cuh exp_tbl) of x[i]; device pointers. */
int snp_debug_exp(const double *x_dev, double *y_dev, int32_t n, void *cuda_stream);
/* Test hook for the kernels' own fp64 elementary functions (csrc/snp_math.cuh); device pointers, n elements each.
 * kind 0: out[i] = exp2_scaled(x[i]) = 2^(x[i] / 2048);  1: out[i] = atan2_poly(y[i], x[i]);
 * 2: out[i] = sin, out[n + i] = cos of x[i] by sincos_bounded (|x| <= pi + 1);  3: out[i] = rsqrt_(x[i]);  4: out[i] = clamp01_(x[i]). */
int snp_debug_math(int32_t kind, const double *x_dev, const double *y_dev, double *out_dev, int32_t n, void *cuda_stream);
/* Launch statistics since the last reset: number of kernels this library launched. */
int64_t snp_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* SNP_B200_H */
