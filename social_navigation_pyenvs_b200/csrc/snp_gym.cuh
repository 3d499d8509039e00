// snp_gym.cuh -- pieces of SocialNavGym.step shared by the small-crowd kernel (snp_step_small.inl) and the large-crowd path
// (snp_step_large.cu): the reward / info code of a check, and the robot's holonomic and unicycle steps.
#pragma once
#include "snp_kernels.cuh"

namespace snp {
namespace {

// social_nav_sim.py:986-1029.  Returns info code, writes reward / terminated / truncated.  (Double arithmetic, formula-exact; see
// snp_math.cuh.)
__device__ __forceinline__ int reward_and_info(bool collision, double dmin, bool goal, double t, const double *c, double &reward,
                                               bool &terminated, bool &truncated) {
    if (t >= __dsub_rn(c[0], 1.0)) { reward = 0.0; truncated = true; terminated = false; return 1; }
    if (collision) { reward = c[1]; truncated = false; terminated = true; return 2; }
    if (goal) { reward = c[2]; truncated = false; terminated = true; return 3; }
    if (dmin < c[3]) { reward = __dmul_rn(__dmul_rn(__dsub_rn(dmin, c[3]), c[4]), c[5]); truncated = false; terminated = false; return 4; }
    reward = 0.0; truncated = false; terminated = false; return 0;
}

// RobotAgent.step with holonomic kinematics (robot_agent.py:126-131), one coordinate: p = p + a dt (the velocity becomes a).
template <typename T> __device__ __forceinline__ T robot_holonomic_step(T p, T a, T dt) {
    if (sizeof(T) == 8) return (T)__dadd_rn((double)p, __dmul_rn((double)a, (double)dt));
    return p + a * dt;
}

// RobotAgent.step with unicycle kinematics (robot_agent.py:116-136), action = ActionRot(v, r): the position advances along
// yaw + r, the yaw becomes (yaw + r) % 2 pi -- r is added at EVERY call, whatever delta_t -- and the velocity points along the new
// yaw.  Double arithmetic (what the reference computes in); by one thread, out of line.  `rb` is indexed by SNP_ROBOT_*.
template <typename T> __device__ __noinline__ void robot_unicycle_step(T *rb, double v, double r, double dt) {
    const double two_pi = 6.283185307179586;
    const double yaw = (double)rb[SNP_ROBOT_TH] + r;
    double sn, cs;
    sincos(yaw, &sn, &cs);
    rb[SNP_ROBOT_PX] = (T)__dadd_rn((double)rb[SNP_ROBOT_PX], __dmul_rn(__dmul_rn(cs, v), dt));
    rb[SNP_ROBOT_PY] = (T)__dadd_rn((double)rb[SNP_ROBOT_PY], __dmul_rn(__dmul_rn(sn, v), dt));
    double w = fmod(yaw, two_pi);   // Python's float %: the result takes the divisor's sign
    if (w < 0.0) w += two_pi;
    sincos(w, &sn, &cs);
    rb[SNP_ROBOT_TH] = (T)w;
    rb[SNP_ROBOT_VX] = (T)__dmul_rn(cs, v); rb[SNP_ROBOT_VY] = (T)__dmul_rn(sn, v);
}

}  // namespace
}  // namespace snp
