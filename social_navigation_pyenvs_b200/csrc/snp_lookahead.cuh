// snp_lookahead.cuh -- the per-(action, human) arithmetic of the policies' one-step lookahead (crowd_nav/policy/cadrl.py:42-83),
// shared by k_lookahead (snp_lookahead.cu, which writes the rotated rows out) and k_value (snp_value.cu, which feeds them to the
// value network where they are made): one copy of each expression, so a row and a reward are the same bits in both kernels.
#pragma once
#include "snp_kernels.cuh"

namespace snp {

// cadrl.py:56-72 from the folded swept test: the reward of action (axd, ayd) for the robot at (rpx, rpy) with goal (rgx, rgy)
__device__ __forceinline__ double look_reward(bool collision, double dmin, double axd, double ayd, double dt, double rpx, double rpy,
                                              double rgx, double rgy, double rr) {
    const double npx = __dadd_rn(rpx, __dmul_rn(axd, dt)), npy = __dadd_rn(rpy, __dmul_rn(ayd, dt));
    const bool reached = xnorm_plain(__dsub_rn(npx, rgx), __dsub_rn(npy, rgy)) < rr;
    if (collision) return -0.25;
    if (reached) return 1.0;
    if (dmin < 0.2) return __dmul_rn(__dmul_rn(__dsub_rn(dmin, 0.2), 0.5), dt);
    return 0.0;
}

// The swept test of several humans folded into one signed 64-bit key whose minimum over any split of the humans is the whole test:
// -1 for a collision (some d < 0), else the bits of the smallest d >= 0 plus 0.0 (positive doubles order like their bits); NaN takes
// part in neither.  look_key_cap is the key of the reference's initial dmin, np.iinfo(np.int64).max as a double.
constexpr double kLookDminCap = 9223372036854775807.0;
__device__ __forceinline__ long long look_key(bool collision, double dmin) {
    return collision ? -1LL : __double_as_longlong(__dadd_rn(dmin, 0.0));  // -0.0 -> +0.0
}
__device__ __forceinline__ double look_key_reward(long long key, double axd, double ayd, double dt, double rpx, double rpy, double rgx,
                                                  double rgy, double rr) {
    const double d = __longlong_as_double(key);
    return look_reward(key < 0, d < kLookDminCap ? d : kLookDminCap, axd, ayd, dt, rpx, rpy, rgx, rgy, rr);
}

// Per-action quantities shared by the humans of an env: next robot position, (cos, sin) of the rotation, distance to goal.
template <typename T> struct PerAction { double axd, ayd; T npx, npy, c, s, dg, ax, ay, pad; };

// next robot position (cadrl.py:54), rotation (:22), distance to goal of action (axd, ayd) for the robot at (rpx, rpy), goal (rgx, rgy).
// (cos rot, sin rot) with rot = atan2(gy, gx) is the unit vector towards the goal: g / |g| (and (1, 0) for g = 0, atan2(0,0) = 0)
// -- one division instead of an atan2 + sincos chain; agrees with the reference's libm round trip to ~1e-16.
template <typename T>
__device__ __forceinline__ PerAction<T> look_action(double axd, double ayd, double dt, T rpx, T rpy, T rgx, T rgy) {
    PerAction<T> p;
    p.axd = axd; p.ayd = ayd;
    p.ax = (T)p.axd; p.ay = (T)p.ayd; p.pad = T(0);
    if (sizeof(T) == 8) {  // no contraction: p + a * dt
        p.npx = (T)__dadd_rn((double)rpx, __dmul_rn(p.axd, dt)); p.npy = (T)__dadd_rn((double)rpy, __dmul_rn(p.ayd, dt));
        const double gx = __dsub_rn((double)rgx, (double)p.npx), gy = __dsub_rn((double)rgy, (double)p.npy);
        const double dg = xnorm_plain(gx, gy);
        p.dg = (T)dg;
        const double inv = dg > 0.0 ? 1.0 / dg : 0.0;
        p.c = (T)(dg > 0.0 ? gx * inv : 1.0); p.s = (T)(gy * inv);
    } else {
        const T dtT = (T)dt;
        p.npx = rpx + p.ax * dtT; p.npy = rpy + p.ay * dtT;
        const T gx = rgx - p.npx, gy = rgy - p.npy;
        p.dg = Real<T>::sqrt_exact(gx * gx + gy * gy);
        const T inv = p.dg > T(0) ? T(1) / p.dg : T(0);
        p.c = p.dg > T(0) ? gx * inv : T(1); p.s = gy * inv;
    }
    return p;
}

// What a human contributes to every action's pair: its next state and the action-independent part of the swept test.
template <typename T> struct LookHuman { T hr, nxx, nxy, nvx, nvy, th, om; double dx, dy, hvx, hvy, rsum; };

// cur = (px, py, vx, vy, r) now, next = (x, y, vx, vy, theta, omega) one policy step ahead, robot at (rpx, rpy)
template <typename T>
__device__ __forceinline__ LookHuman<T> look_human(T px, T py, T vx, T vy, T r, T nxx, T nxy, T nvx, T nvy, T th, T om, T rpx, T rpy) {
    LookHuman<T> h;
    h.hr = r;
    h.nxx = nxx; h.nxy = nxy; h.nvx = nvx; h.nvy = nvy; h.th = th; h.om = om;
    h.dx = __dsub_rn((double)px, (double)rpx); h.dy = __dsub_rn((double)py, (double)rpy);  // sim:962 difference
    h.hvx = (double)vx; h.hvy = (double)vy;
    h.rsum = (double)h.hr;
    return h;
}

// swept distance of one (action, human) pair (social_nav_sim.py:962-976 via utils.py:22-36, formula-exact)
template <typename T>
__device__ __forceinline__ double look_swept(const LookHuman<T> &h, const PerAction<T> &q, double dt, T rr) {
    const double vx = __dsub_rn(h.hvx, q.axd), vy = __dsub_rn(h.hvy, q.ayd);
    const double ex = __dadd_rn(h.dx, __dmul_rn(vx, dt)), ey = __dadd_rn(h.dy, __dmul_rn(vy, dt));
    return __dsub_rn(__dsub_rn(origin_to_segment(h.dx, h.dy, ex, ey), h.rsum), (double)rr);
}

// the rotated row of one (action, human) pair (cadrl.py:13-40): 13 values, 15 when `visible`
template <typename T>
__device__ __forceinline__ void look_row(const LookHuman<T> &h, const PerAction<T> &q, T rvd, T rr, int visible, T *o) {
    const T ddx = h.nxx - q.npx, ddy = h.nxy - q.npy;
    o[0] = q.dg; o[1] = rvd; o[2] = T(0); o[3] = rr;
    o[4] = q.ax * q.c + q.ay * q.s; o[5] = q.ay * q.c - q.ax * q.s;
    o[6] = ddx * q.c + ddy * q.s; o[7] = ddy * q.c - ddx * q.s;
    o[8] = h.nvx * q.c + h.nvy * q.s; o[9] = h.nvy * q.c - h.nvx * q.s;
    o[10] = h.hr;
    o[11] = Real<T>::sqrt_(ddx * ddx + ddy * ddy);  // < 1.5 ulp (snp_math.cuh); the rotated states carry the 1e-9 / 1e-4 tolerance
    o[12] = rr + h.hr;
    if (visible) { o[13] = h.th - T(0); o[14] = h.om; }
}

}  // namespace snp
