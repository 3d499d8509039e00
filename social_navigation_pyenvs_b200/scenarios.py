"""Synthetic initial conditions in the reference's array layouts (host side, NumPy; inputs of the hot path, not part of it).

`circular_crossing` replays the reference generator's draw sequence (social_gym/social_nav_sim.py:200-299, the
`insert_robot=True, randomize_human_positions=True` branch used by SocialNavGym.reset, social_nav_gym.py:141-144) on a private
`np.random.RandomState(seed)`, so env e seeded with 2000+e is the environment the reference's gym would build for train case e
(social_nav_gym.py:135-137).  `ccso_synthetic` is the 25-human static-obstacle crowd of SURVEY.md section 8(d) config 3 (the
reference's own CCSO generator does not terminate for 25 actors, SURVEY.md section 7).
"""
import math
import os

import numpy as np

# social_gym/custom_config/config_example.py:20-22 -- three wall polygons (vertices, counter-clockwise)
EXAMPLE_WALLS = [
    [[1 - 7.5, 1 - 7.5], [1.5 - 7.5, 1 - 7.5], [1.5 - 7.5, 3 - 7.5], [1 - 7.5, 3 - 7.5], [0.5 - 7.5, 2 - 7.5]],
    [[3 - 7.5, 9 - 7.5], [5 - 7.5, 7 - 7.5], [6 - 7.5, 9 - 7.5], [6 - 7.5, 9.5 - 7.5], [3 - 7.5, 9.5 - 7.5]],
    [[7 - 7.5, 5 - 7.5], [9 - 7.5, 5 - 7.5], [9 - 7.5, 7 - 7.5], [7 - 7.5, 5.5 - 7.5]],
]


def bound_angle(angle):  # social_gym/src/utils.py:7-13
    two_pi = 2 * math.pi
    if angle >= two_pi:
        angle %= two_pi
    if angle <= -two_pi:
        angle %= -two_pi
    if angle > math.pi:
        angle -= two_pi
    if angle < -math.pi:
        angle += two_pi
    return angle


def pack_walls(polygons):
    """Vertex lists -> [W,S,2,2] NaN padded segment array with endpoints in lexicographic order (obstacle.py:26-32,
    motion_model_manager.py:268-276)."""
    if not polygons:
        return np.zeros((0, 1, 2, 2))
    smax = max(len(p) for p in polygons)
    out = np.full((len(polygons), smax, 2, 2), np.nan)
    for w, verts in enumerate(polygons):
        for i in range(len(verts)):
            a, b = list(verts[i]), list(verts[(i + 1) % len(verts)])
            out[w, i, 0], out[w, i, 1] = min(a, b), max(a, b)
    return out


def _state_row(pos, yaw, radius, mass, goal, vd):
    # [px,py,theta,vx,vy,bvx,bvy,omega,r,m,gx,gy,vd]  (social_gym/src/agent.py:256-258)
    return [pos[0], pos[1], yaw, 0.0, 0.0, 0.0, 0.0, 0.0, radius, mass, goal[0], goal[1], vd]


def _cc_sample(rs, humans_pos, static_upto, i, radius, des_speed, r_i, radii, robot_r):
    """One accepted draw of the circular-crossing rejection sampler (social_nav_sim.py:271-295).  Same draw order and same
    accept/reject decisions as the reference's loop; the per-candidate distance tests are evaluated as array ops."""
    robot_pos, robot_goal = np.array([0.0, -radius]), np.array([0.0, radius])
    k = len(humans_pos)
    if k:
        others = np.asarray(humans_pos, np.float64)
        other_goals = others.copy()
        other_goals[static_upto:] = -others[static_upto:]
        min_dist = r_i + np.asarray(radii[:k], np.float64) + 0.2
    rmin = r_i + robot_r + 0.2
    while True:
        angle = rs.random_sample() * np.pi * 2
        n0 = (rs.random_sample() - 0.5) * des_speed
        n1 = (rs.random_sample() - 0.5) * des_speed
        pos = np.array([radius * np.cos(angle) + n0, radius * np.sin(angle) + n1])
        if k:
            d1 = np.sqrt(((pos - others) ** 2).sum(1))
            d2 = np.sqrt(((pos - other_goals) ** 2).sum(1))
            if ((d1 < min_dist) | (d2 < min_dist)).any():
                continue
        if math.hypot(pos[0] - robot_pos[0], pos[1] - robot_pos[1]) < rmin or math.hypot(pos[0] - robot_goal[0], pos[1] - robot_goal[1]) < rmin:
            continue
        return pos, angle


def _env_seed(seed0, e):
    """Seed of env e: seed0 + e, or seed0[e] when the caller passes one seed per env (a case counter that wraps inside the batch)."""
    return int(seed0[e]) if np.ndim(seed0) else int(seed0) + e


def _map_envs(fn, E, args):
    """Run fn(e, *args) for every env, on all host cores when the batch is large (scenario generation is host-side setup)."""
    if E < 256:
        return [fn(e, *args) for e in range(E)]
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as pool:
        return pool.starmap(fn, [(e, *args) for e in range(E)], chunksize=max(1, E // 256))


def _attributes(rs, N, randomize):
    """humans_des_speed / humans_radius (social_nav_sim.py:217-224): uniform(0.5, 1.5) and uniform(0.3, 0.5) per human, drawn
    interleaved BEFORE any position, or the fixed 1.0 / 0.3."""
    if not randomize:
        return [1.0] * N, [0.3] * N
    vd, radii = [], []
    for _ in range(N):
        vd.append(0.5 + (1.5 - 0.5) * rs.random_sample())   # RandomState.uniform = low + (high - low) * random_sample()
        radii.append(0.3 + (0.5 - 0.3) * rs.random_sample())
    return vd, radii


def _cc_env(e, N, seed0, circle_radius, robot_radius, mass, randomize_attributes=False):
    rs = np.random.RandomState(_env_seed(seed0, e))
    st, gl = np.zeros((N, 13)), np.zeros((N, 2, 2))
    vd, radii = _attributes(rs, N, randomize_attributes)
    pos_list = []
    for i in range(N):
        pos, angle = _cc_sample(rs, pos_list, 0, i, circle_radius, vd[i], radii[i], radii, robot_radius)
        pos_list.append([pos[0], pos[1]])
        st[i] = _state_row(pos, bound_angle(math.pi + angle), radii[i], mass, -pos, vd[i])
        gl[i, 0], gl[i, 1] = -pos, pos
    return st, gl


def circular_crossing(E, N, seed0=2000, circle_radius=7.0, robot_radius=0.3, mass=75.0, randomize_attributes=False):
    """E environments of N humans on a circle, goals at the antipodes and back (G = 2).
    Returns dict(states [E,N,13], goals [E,N,2,2], robot [E,13])."""
    res = _map_envs(_cc_env, E, (N, seed0, circle_radius, robot_radius, mass, randomize_attributes))
    return dict(states=np.stack([r[0] for r in res]), goals=np.stack([r[1] for r in res]),
                robot=robot_rows(E, circle_radius, robot_radius))


def robot_rows(E, circle_radius=7.0, robot_radius=0.3, velocity=(0.0, 1.0)):
    """Robot of the reference scenarios (social_nav_sim.py:270): starts at (0,-R) heading to (0,R); mass 80 (robot_agent.py:16)."""
    r = np.zeros((E, 13))
    r[:, 1] = -circle_radius
    r[:, 2] = math.pi / 2
    r[:, 3], r[:, 4] = velocity
    r[:, 8], r[:, 9] = robot_radius, 80.0
    r[:, 11] = circle_radius
    r[:, 12] = 1.0
    return r


def _ccso_env(e, N, seed0, circle_radius, robot_radius, mass):
    rs = np.random.RandomState(_env_seed(seed0, e))
    st, gl = np.zeros((N, 13)), np.zeros((N, 2, 2))
    inner = circle_radius - 3.0
    radii = [1 + (rs.random_sample() - 1) * 0.4 for _ in range(3)] + [0.3] * (N - 3)
    pos_list = []
    for i in range(N):
        if i < 3:
            while True:
                angle = (np.pi / 4) * (-0.5 + 2 * i + (rs.random_sample() - 0.5) * 0.5)
                noise = np.array([(rs.random_sample() - 0.5) * 0.1, (rs.random_sample() - 0.5) * 0.1])
                pos = np.array([inner * np.cos(angle) + noise[0], inner * np.sin(angle) + noise[1]])
                if all(np.linalg.norm(pos - np.array(o)) >= radii[i] + radii[j] + 0.2 for j, o in enumerate(pos_list)):
                    break
            goal, vd = pos, 0.0
            gl[i, 0], gl[i, 1] = pos, pos
        else:
            pos, angle = _cc_sample(rs, pos_list, 3, i, circle_radius, 1.0, 0.3, radii, robot_radius)
            goal, vd = -pos, 1.0
            gl[i, 0], gl[i, 1] = -pos, pos
        pos_list.append([pos[0], pos[1]])
        st[i] = _state_row(pos, bound_angle(math.pi + angle), radii[i], mass, goal, vd)
    return st, gl


def ccso_synthetic(E, N=25, seed0=2000, circle_radius=7.0, robot_radius=0.3, mass=75.0):
    """SURVEY.md 8(d) config 3: humans 0-2 are static obstacles (vd = 0, r = 1 + (u-1)*0.4, on the inner circle R-3 at
    (pi/4)(-0.5 + 2i + noise), goals [p, p]; social_nav_sim.py:381-399,416-417), humans 3.. are the circular-crossing
    sampler on R (social_nav_sim.py:271-295)."""
    res = _map_envs(_ccso_env, E, (N, seed0, circle_radius, robot_radius, mass))
    return dict(states=np.stack([r[0] for r in res]), goals=np.stack([r[1] for r in res]),
                robot=robot_rows(E, circle_radius, robot_radius))


def _ccso_ref_env(e, N, seed0, circle_radius, robot_radius, mass):
    """generate_circular_crossing_with_static_obstacles (social_nav_sim.py:364-431), insert_robot=True: humans 0-2 static on the
    inner circle R-3, the others in angular slots (pi / int(N/2)) (0.5 + 2i + noise) of the circle R."""
    rs = np.random.RandomState(_env_seed(seed0, e))
    st, gl = np.zeros((N, 13)), np.zeros((N, 2, 2))
    inner = circle_radius - 3.0
    radii = [(1 + (rs.random_sample() - 1) * 0.4) if i < 3 else 0.3 for i in range(N)]
    robot_pos, robot_goal = np.array([0.0, -circle_radius]), np.array([0.0, circle_radius])
    slot = np.pi / int(N / 2)
    pos_list = []
    for i in range(N):
        while True:
            if i < 3:
                angle = slot * (-0.5 + 2 * i + (rs.random_sample() - 0.5) * 0.5)
                n0 = (rs.random_sample() - 0.5) * 0.1
                n1 = (rs.random_sample() - 0.5) * 0.1
                pos = np.array([inner * np.cos(angle) + n0, inner * np.sin(angle) + n1])
            else:
                angle = slot * (0.5 + 2 * i + (rs.random_sample() - 0.5) * 0.5)
                n0 = (rs.random_sample() - 0.5) * 0.7
                n1 = (rs.random_sample() - 0.5) * 0.7
                pos = np.array([circle_radius * np.cos(angle) + n0, circle_radius * np.sin(angle) + n1])
            collide = False
            for j, o in enumerate(pos_list):
                o = np.asarray(o)
                og = o if j < 3 else -o
                md = radii[i] + radii[j] + 0.2
                if np.linalg.norm(pos - o) < md or np.linalg.norm(pos - og) < md:
                    collide = True
                    break
            rmin = radii[i] + robot_radius + 0.2
            if np.linalg.norm(pos - robot_pos) < rmin or np.linalg.norm(pos - robot_goal) < rmin:
                collide = True
            if not collide:
                break
        pos_list.append([pos[0], pos[1]])
        goal, vd = (pos, 0.0) if i < 3 else (-pos, 1.0)
        gl[i, 0], gl[i, 1] = goal, pos
        st[i] = _state_row(pos, bound_angle(math.pi + angle), radii[i], mass, goal, vd)
    return st, gl


def circular_crossing_with_static_obstacles(E, N, seed0=2000, circle_radius=7.0, robot_radius=0.3, mass=75.0):
    """The reference's own CCSO generator (social_nav_sim.py:364-431); terminates only for small crowds (N <= ~10: the slots of
    humans 3.. wrap around the circle and collide for larger N, SURVEY.md section 7)."""
    res = _map_envs(_ccso_ref_env, E, (N, seed0, circle_radius, robot_radius, mass))
    return dict(states=np.stack([r[0] for r in res]), goals=np.stack([r[1] for r in res]),
                robot=robot_rows(E, circle_radius, robot_radius))


def _pt_env(e, N, seed0, traffic_length, traffic_height, robot_radius, mass, randomize_attributes=False):
    rs = np.random.RandomState(_env_seed(seed0, e))
    st, gl = np.zeros((N, 13)), np.zeros((N, 1, 2))
    robot_pos = np.array([-(traffic_length / 2) + 1, 0.0])
    vd, radii = _attributes(rs, N, randomize_attributes)
    if sum(math.pi * r ** 2 for r in radii) > traffic_length * traffic_height * 0.4:   # social_nav_sim.py:327-329
        raise ValueError("Number of humans specified is too big for desided traffic height and length")
    placed = []
    for i in range(N):
        while True:
            a, b = -(traffic_length / 2) + radii[i], traffic_length / 2 - radii[i]
            pos = np.array([(b - a) * rs.random_sample() + a, (rs.random_sample() - 0.5) * traffic_height])
            if any(np.linalg.norm(pos - o) - radii[i] - radii[j] - 0.1 < 0 for j, o in enumerate(placed)):
                continue
            if np.linalg.norm(pos - robot_pos) - radii[i] - robot_radius - 0.1 < 0:
                continue
            break
        placed.append(pos)
        goal = [-(traffic_length / 2) - 3, pos[1]]
        st[i] = _state_row(pos, bound_angle(-math.pi), radii[i], mass, goal, vd[i])
        gl[i, 0] = goal
    return st, gl


def parallel_traffic(E, N, seed0=2000, traffic_length=14.0, traffic_height=3.0, robot_radius=0.3, mass=75.0, randomize_attributes=False):
    """Parallel-traffic scenario (social_nav_sim.py:301-362, insert_robot=True): humans walk towards x = -L/2 - 3 and are respawned
    at the right end when they get within 3 m of it (motion_model_manager.py:407-422).  Returns states, goals [E,N,1,2], robot rows
    and `respawn_bounds` = (L/2, H/2)."""
    res = _map_envs(_pt_env, E, (N, seed0, traffic_length, traffic_height, robot_radius, mass, randomize_attributes))
    robot = np.zeros((E, 13))
    robot[:, 0] = -(traffic_length / 2) + 1
    robot[:, 8], robot[:, 9], robot[:, 12] = robot_radius, 80.0, 1.0
    robot[:, 10] = (traffic_length / 2) - 1
    return dict(states=np.stack([r[0] for r in res]), goals=np.stack([r[1] for r in res]), robot=robot,
                respawn_bounds=(traffic_length / 2, traffic_height / 2))


def hybrid_choice(seed):
    """The coin of the hybrid scenario (social_nav_gym.py:155-156): np.random.seed(seed); np.random.choice([cc, pt]) -> 0 / 1.  The
    legacy choice draws randint(0, 2) = the first 32-bit output of MT19937 masked to one bit."""
    return int.from_bytes(np.random.RandomState(int(seed)).bytes(4), "little") & 1


def spatial_order(positions, block=256):
    """Permutation that numbers the agents of ONE large crowd patch by patch: the crowd is cut into sqrt(n / block) vertical
    strips of equal head count (sorted by x) and every strip is walked in y, so that a run of consecutive agents (a 128-entity
    tile, a 256-agent block of the tiled all-pairs kernels) covers a compact patch of the plane instead of a long strip.  The
    exact far-tile culling of snp_large_run_p2p tests bounding boxes of such runs and skips ~2x more of them.  The numbering of
    the agents is the caller's (the reference keeps humans in insertion order, social_nav_sim.py:271-295, and no force depends
    on it), so this is applied to the rows BEFORE they are handed to LargeCrowd; `np.argsort(perm)` undoes it."""
    pos = np.asarray(positions, np.float64).reshape(-1, 2)
    n = len(pos)
    strips = max(1, int(round(math.sqrt(n / float(block)))))
    by_x = np.argsort(pos[:, 0], kind="stable")
    out = []
    for s in np.array_split(by_x, strips):
        out.append(s[np.argsort(pos[s, 1], kind="stable")])
    return np.concatenate(out) if out else by_x


def deal_tiles(perm, world, tile=128):
    """Load balance of an agent-sharded large crowd: the `tile`-human runs of `perm` (compact patches after spatial_order) are dealt
    to the `world` ranks round-robin, so that the contiguous slice rank r owns (agent_shard) is made of patches from all over the crowd
    instead of one block of strips -- an interior block has ~25 % more near neighbours than a corner one.  Needs len(perm) to be a
    whole number of tiles; like spatial_order this only re-numbers the caller's rows."""
    perm = np.asarray(perm)
    if world <= 1:
        return perm
    if len(perm) % tile:
        raise ValueError(f"deal_tiles: {len(perm)} agents are not a whole number of {tile}-agent tiles")
    tiles = perm.reshape(-1, tile)
    return np.concatenate([tiles[r::world] for r in range(world)]).reshape(-1)


def jittered_grid_crowd(n_side, pitch=2.0, jitter=0.5, seed=0, mass=75.0):
    """SURVEY.md 8(d) config 5: n_side x n_side jittered grid, every goal mirrored through the crowd centre (G = 2)."""
    rs = np.random.RandomState(seed)
    n = n_side * n_side
    ix, iy = np.meshgrid(np.arange(n_side), np.arange(n_side), indexing="ij")
    c = (n_side - 1) * pitch / 2
    pos = np.stack([ix.ravel() * pitch - c, iy.ravel() * pitch - c], 1) + rs.uniform(-jitter, jitter, (n, 2))
    states = np.zeros((1, n, 13))
    states[0, :, 0:2] = pos
    states[0, :, 2] = np.arctan2(-pos[:, 1], -pos[:, 0])
    states[0, :, 8], states[0, :, 9], states[0, :, 12] = 0.3, mass, 1.0
    states[0, :, 10:12] = -pos
    goals = np.zeros((1, n, 2, 2))
    goals[0, :, 0], goals[0, :, 1] = -pos, pos
    return dict(states=states, goals=goals)
