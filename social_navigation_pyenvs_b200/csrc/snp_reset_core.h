// snp_reset_core.h -- the reference's scenario generators as host/device code driven by NumPy's own random stream.
//
// SocialNavGym.reset (social_gym/social_nav_gym.py:120-225) seeds the GLOBAL np.random with `offset[phase] + case` (:135-137) and
// calls one of the rejection samplers of social_gym/social_nav_sim.py: :200-299 circular crossing, :301-362 parallel traffic,
// :364-431 circular crossing with static obstacles; the hybrid scenario first flips np.random.choice between the first two and
// re-seeds (social_nav_gym.py:155-157).  All of them draw through np.random.random() / np.random.uniform() only, i.e. through
// MT19937 + random_double of the legacy RandomState.  Reproducing that generator per environment makes an on-device reset
// consume EXACTLY the reference's draw sequence: same accept / reject decisions, same number of draws, positions equal to the
// last ulp of cos / sin.  (SURVEY.md 8f-4 expected distribution-level parity only.)
//
// The code below is shared by the CUDA kernel (snp_reset.cu) and by a host harness the CPU tests compile with g++
// (tests/reset_core_host.cpp), so the logic is checked against the recorded reference outputs without a GPU.  It is written for a
// GROUP of cooperating lanes that execute it in lock step: the group splits the generator's twist, and it SPECULATES on the
// rejection sampler -- lane l evaluates the l-th next attempt (the stream is random access inside a 624-word block: attempt l reads
// the words the sequential algorithm would read if the l previous attempts were rejected), the first accepted attempt wins and
// the stream advances past exactly the words a sequential run would have consumed.  Same draws, same result, but the serial latency
// of an unlucky environment (hundreds of rejected attempts) shrinks by up to the group size.  On the host the group is one lane
// (SoloGroup) and the code is the plain sequential algorithm; on the device it is a warp per environment, or, for crowds whose
// scratch does not fit one warp's share of shared memory, a CTA per environment (CtaGroup, snp_reset.cu): every warp of the CTA
// speculates on the same 32 attempts, tests them against its own STRIPE of the humans placed so far (j = j0(), j0() + jstep(), ...),
// and first() / all() combine the warps' verdicts.  The collision test is a pure OR over j, so a striped test rejects exactly what a
// full one rejects.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SNP_HD __host__ __device__ __forceinline__
#else
#define SNP_HD inline
#endif

namespace snp {

enum { SNP_SCEN_CIRCULAR_CROSSING = 0, SNP_SCEN_PARALLEL_TRAFFIC = 1, SNP_SCEN_CCSO = 2, SNP_SCEN_CCSO_SYNTHETIC = 3, SNP_SCEN_HYBRID = 4 };

// numpy/random/src/mt19937/mt19937.c: mt19937_seed (np.random.seed(int)), mt19937_gen, and random_double of the legacy
// distributions: (a >> 5, b >> 6) -> (a * 2^26 + b) / 2^53.
struct SoloGroup {  // one lane: the sequential algorithm
    static constexpr bool kStriped = false;  // true: several warps share the candidates, see CtaGroup (snp_reset.cu)
    SNP_HD int lane() const { return 0; }
    SNP_HD int size() const { return 1; }
    SNP_HD bool leader() const { return true; }            // the one member that does the group's sequential writes
    SNP_HD int j0() const { return 0; }                    // the stripe of placed humans this member tests: j0, j0 + jstep, ...
    SNP_HD int jstep() const { return 1; }
    SNP_HD int first(bool v) const { return v ? 0 : -1; }  // lowest lane whose flag is set (in every stripe), or -1
    SNP_HD bool all(bool v) const { return v; }            // v holds in every stripe (every lane tests the same candidate)
    SNP_HD double bcast(double v, int) const { return v; }
    SNP_HD void sync() const {}
};

template <class Group> struct Mt19937 {
    uint32_t *mt;
    int pos;
    long long draws;
    Group g;
    SNP_HD uint32_t &at(int i) { return mt[i]; }
    SNP_HD void seed(uint32_t s) {  // sequential recurrence: one lane writes, everybody waits
        g.sync();                   // nobody is still reading the previous state
        if (g.leader())
            for (int i = 0; i < 624; ++i) { at(i) = s; s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)(i + 1); }
        g.sync();
        pos = 624;
    }
    // mt19937_gen's regeneration of all 624 words.  Word kk needs the OLD words kk, kk+1 and, for kk < 227, the OLD word kk+397,
    // else the NEW word kk-227 (and the new word 0 for kk = 623): a batch of `size` consecutive words reads everything it needs
    // before any of them is written, and what it reads as new was written by an earlier batch (a batch must not exceed 227 words).
    // A striped group twists in its first warp, between barriers of the whole group.
    SNP_HD void twist() {
        if constexpr (Group::kStriped) {
            g.sync();
            if (g.twister()) twist_by(g.warp());
            g.sync();
        } else {
            twist_by(g);
        }
        pos = 0;
    }
    template <class W> SNP_HD void twist_by(const W &t) {
        const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, A = 0x9908b0dfu;
        for (int base = 0; base < 624; base += t.size()) {
            const int kk = base + t.lane();
            uint32_t v = 0;
            if (kk < 624) {
                const uint32_t y = (at(kk) & UP) | (at(kk + 1 == 624 ? 0 : kk + 1) & LO);
                v = at(kk < 624 - 397 ? kk + 397 : kk - (624 - 397)) ^ (y >> 1) ^ ((y & 1u) ? A : 0u);
            }
            t.sync();
            if (kk < 624) at(kk) = v;
            t.sync();
        }
    }
    SNP_HD uint32_t peek32(int i) {  // tempered output of state word i (the output next32() returns when pos == i)
        uint32_t y = at(i);
        y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
        return y;
    }
    SNP_HD uint32_t next32() {
        if (pos == 624) twist();
        return peek32(pos++);
    }
    SNP_HD double peek_double(int i) {  // the double random() returns when pos == i (needs i + 1 < 624)
        const uint32_t a = peek32(i) >> 5, b = peek32(i + 1) >> 6;
        return (a * 67108864.0 + b) / 9007199254740992.0;
    }
    SNP_HD double random() {  // np.random.random()
        const uint32_t a = next32() >> 5, b = next32() >> 6;
        ++draws;
        return (a * 67108864.0 + b) / 9007199254740992.0;
    }
    SNP_HD double uniform(double lo, double hi) { return lo + (hi - lo) * random(); }  // np.random.uniform
};

struct ResetParams {
    int scenario, N, randomize_attributes;
    double circle_radius, robot_radius, traffic_length, traffic_height;
};

// Scratch of one environment: positions, radii and desired speeds of the humans placed so far.  Every member of the group writes the
// same value to the same slot (benign), reads happen after a group sync.
struct ResetScratch {
    double *px, *py, *rad, *vd;
    SNP_HD double &X(int i) { return px[i]; }
    SNP_HD double &Y(int i) { return py[i]; }
    SNP_HD double &R(int i) { return rad[i]; }
    SNP_HD double &V(int i) { return vd[i]; }
};

SNP_HD double reset_norm(double x, double y) { return sqrt(fma(y, y, x * x)); }  // np.linalg.norm of a length-2 vector
SNP_HD double reset_bound_angle(double a) {                                         // utils.py:7-13
    const double pi = 3.141592653589793, two_pi = 2 * pi;
    if (a >= two_pi) a = fmod(a, two_pi);
    if (a <= -two_pi) a = fmod(a, -two_pi);
    if (a > pi) a -= two_pi;
    if (a < -pi) a += two_pi;
    return a;
}

// One human of the result: state-row fields (agent.py:256) that differ from zero, and its goal list.
struct ResetHuman { double x, y, yaw, radius, vd, g0x, g0y, g1x, g1y; int goal_count; };

// One accepted sample of a rejection sampler that draws DRAWS uniforms per attempt: cand(u, x, y, angle) builds the candidate from
// the uniforms, collides(x, y) tests it against everything placed so far.  Lane l of the group speculates on attempt l; see the
// header comment.  When fewer words than one attempt needs are left before the twist, that attempt is made sequentially by every
// lane alike.
template <int DRAWS, class Group, class Cand, class Coll>
SNP_HD void reset_place(Mt19937<Group> &rng, Cand &cand, Coll &collides, double &x, double &y, double &angle) {
    const Group g = rng.g;
    for (;;) {
        if (rng.pos == 624) rng.twist();
        const int avail = (624 - rng.pos) / (2 * DRAWS);
        if (avail == 0) {
            double u[DRAWS];
            for (int d = 0; d < DRAWS; ++d) u[d] = rng.random();
            cand(u, x, y, angle);
            if (g.all(!collides(x, y))) return;
            continue;
        }
        const int width = avail < g.size() ? avail : g.size();
        const int l = g.lane();
        bool ok = false;
        double cx = 0.0, cy = 0.0, ca = 0.0;
        if (l < width) {
            double u[DRAWS];
            for (int d = 0; d < DRAWS; ++d) u[d] = rng.peek_double(rng.pos + 2 * DRAWS * l + 2 * d);
            cand(u, cx, cy, ca);
            ok = !collides(cx, cy);
        }
        const int first = g.first(ok);
        const int used = first >= 0 ? first + 1 : width;
        rng.pos += 2 * DRAWS * used;
        rng.draws += DRAWS * used;
        if (first >= 0) { x = g.bcast(cx, first); y = g.bcast(cy, first); angle = g.bcast(ca, first); return; }
    }
}

// Runs the generator of `p.scenario` for one environment seeded with `seed`; calls emit(i, ResetHuman) for every human in order.
// Returns the scenario that was generated (the coin of the hybrid scenario, else p.scenario).
template <class Group, class Emit>
SNP_HD int reset_generate(const ResetParams &p, uint32_t seed, Mt19937<Group> &rng, ResetScratch &w, Emit &emit) {
    const Group g = rng.g;
    const double pi = 3.141592653589793;
    const int N = p.N;
    rng.draws = 0;
    rng.seed(seed);
    int scen = p.scenario;
    if (scen == SNP_SCEN_HYBRID) {  // np.random.choice(['circle_crossing', 'parallel_traffic']); np.random.seed(...) again (gym:155-157)
        scen = (rng.next32() & 1u) ? SNP_SCEN_PARALLEL_TRAFFIC : SNP_SCEN_CIRCULAR_CROSSING;
        rng.seed(seed);
    }
    // ---- attributes (sim:217-224, :318-326, :381-388) ----
    if (scen == SNP_SCEN_CCSO || scen == SNP_SCEN_CCSO_SYNTHETIC) {
        if (scen == SNP_SCEN_CCSO) {
            for (int i = 0; i < N; ++i) { w.V(i) = i < 3 ? 0.0 : 1.0; w.R(i) = i < 3 ? 1 + (rng.random() - 1) * 0.4 : 0.3; }
        } else {
            for (int i = 0; i < N; ++i) { w.V(i) = i < 3 ? 0.0 : 1.0; w.R(i) = 0.3; }
            for (int i = 0; i < 3 && i < N; ++i) w.R(i) = 1 + (rng.random() - 1) * 0.4;
        }
    } else if (p.randomize_attributes) {
        for (int i = 0; i < N; ++i) { w.V(i) = rng.uniform(0.5, 1.5); w.R(i) = rng.uniform(0.3, 0.5); }
    } else {
        for (int i = 0; i < N; ++i) { w.V(i) = 1.0; w.R(i) = 0.3; }
    }
    g.sync();
    if (scen == SNP_SCEN_PARALLEL_TRAFFIC) {  // sim:330-352
        const double half = p.traffic_length / 2;
        const double rx = -half + 1, ry = 0.0;
        for (int i = 0; i < N; ++i) {
            const double ri = w.R(i);
            auto cand = [&](const double *u, double &x, double &y, double &angle) {
                const double a = -half + ri, b = half - ri;
                x = (b - a) * u[0] + a;
                y = (u[1] - 0.5) * p.traffic_height;
                angle = 0.0;
            };
            auto collides = [&](double x, double y) {  // any hit rejects (the reference's `break` only ends its loop)
                for (int j = g.j0(); j < i; j += g.jstep())
                    if (reset_norm(x - w.X(j), y - w.Y(j)) - ri - w.R(j) - 0.1 < 0) return true;
                return g.j0() == 0 && reset_norm(x - rx, y - ry) - ri - p.robot_radius - 0.1 < 0;  // the robot: once, in stripe 0
            };
            double x, y, angle;
            reset_place<2>(rng, cand, collides, x, y, angle);
            w.X(i) = x; w.Y(i) = y;
            g.sync();
            ResetHuman h{x, y, reset_bound_angle(-pi), ri, w.V(i), -half - 3, y, 0.0, 0.0, 1};
            h.g1x = h.g0x; h.g1y = h.g0y;
            emit(i, h);
        }
        return scen;
    }
    // ---- the circular scenarios ----
    const double R = p.circle_radius, inner = R - 3.0;
    const double slot = scen == SNP_SCEN_CCSO ? pi / (double)(N / 2) : pi / 4;
    const bool with_statics = scen == SNP_SCEN_CCSO || scen == SNP_SCEN_CCSO_SYNTHETIC;
    for (int i = 0; i < N; ++i) {
        const bool is_static = with_statics && i < 3;
        // the synthetic 25-human crowd tests its static humans against positions only (scenarios.py ccso_synthetic)
        const bool positions_only = scen == SNP_SCEN_CCSO_SYNTHETIC && is_static;
        const double ri = w.R(i), vi = w.V(i);
        auto cand = [&](const double *u, double &x, double &y, double &angle) {
            if (is_static) {                      // sim:393-396
                angle = slot * (-0.5 + 2 * i + (u[0] - 0.5) * 0.5);
                const double n0 = (u[1] - 0.5) * 0.1, n1 = (u[2] - 0.5) * 0.1;
                x = inner * cos(angle) + n0; y = inner * sin(angle) + n1;
            } else if (scen == SNP_SCEN_CCSO) {   // sim:397-400
                angle = slot * (0.5 + 2 * i + (u[0] - 0.5) * 0.5);
                const double n0 = (u[1] - 0.5) * 0.7, n1 = (u[2] - 0.5) * 0.7;
                x = R * cos(angle) + n0; y = R * sin(angle) + n1;
            } else {                              // sim:274-276
                angle = u[0] * pi * 2;
                const double n0 = (u[1] - 0.5) * vi, n1 = (u[2] - 0.5) * vi;
                x = R * cos(angle) + n0; y = R * sin(angle) + n1;
            }
        };
        auto collides = [&](double x, double y) {
            for (int j = g.j0(); j < i; j += g.jstep()) {
                const double md = ri + w.R(j) + 0.2;
                const double ox = w.X(j), oy = w.Y(j);
                if (reset_norm(x - ox, y - oy) < md) return true;
                if (!positions_only) {
                    const bool other_static = with_statics && j < 3;
                    const double gx = other_static ? ox : -ox, gy = other_static ? oy : -oy;
                    if (reset_norm(x - gx, y - gy) < md) return true;
                }
            }
            if (!positions_only && g.j0() == 0) {  // the robot: once, in stripe 0
                const double rm = ri + p.robot_radius + 0.2;
                if (reset_norm(x - 0.0, y - (-R)) < rm || reset_norm(x - 0.0, y - R) < rm) return true;
            }
            return false;
        };
        double x, y, angle;
        reset_place<3>(rng, cand, collides, x, y, angle);
        w.X(i) = x; w.Y(i) = y;
        g.sync();
        ResetHuman h{x, y, reset_bound_angle(pi + angle), ri, vi, is_static ? x : -x, is_static ? y : -y, x, y, 2};
        emit(i, h);
    }
    return scen;
}

}  // namespace snp
