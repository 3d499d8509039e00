// snp_lookahead.cu -- the policy-side one-step lookahead producer (SURVEY.md 8f-3): for every env and every action of the
// policy's action space, the swept collision / goal reward and the agent-centric ("rotated") joint state the value network
// consumes.  Reference: crowd_nav/policy/cadrl.py:42-83 compute_rotated_states_and_reward, :13-40
// transform_state_to_agent_centric (both Numba, float64), called once per decision from CADRL.predict (:235-262) after the
// peek get_next_human_observable_states (motion_model_manager.py:691-709, here snp_step with opts.dyn_out).
//
// Output volume dominates: [E][A][N][13|15] words (4096 x 81 x 25 x 13 doubles = 862 MB) against ~3 kB of input per env, so
// this is a pure HBM-WRITE kernel.  One CTA produces the rows of one (env, chunk of actions): a thread per (action, human)
// computes its 13 / 15 values into a shared-memory tile laid out exactly like the output, then the tile leaves as ONE bulk
// asynchronous copy (cp.async.bulk shared -> global, the TMA engine) -- no per-thread global stores, full 128-byte lines.
// The tile starts in shared memory at the same offset modulo 16 as its destination so that both sides of the bulk copy are
// 16-byte aligned; the (at most 15-byte) head and tail are written with scalar stores.
// Rewards are computed in double with formula-exact operations (snp_math.cuh) so that they are bit-identical to the
// reference for fp64 state; in fp32 mode from the widened fp32 state.
//
// Any N.  The CTA above stages all N humans of its env; once that layout needs more than 200 KB of shared memory even for one
// action per CTA (fp64: N > 673 with 13 values, > 609 with 15; fp32: > 1312 / > 1190) the humans are split instead:
// k_lookahead<T, true> covers (env, range of actions, chunk of H = kLookThreads humans), stages only its chunk, and writes the
// rows [e][a][j0 : j0+H] of each action as one tile -- contiguous, so it leaves through the same bulk copy with the same 16-byte
// head / tail handling and double buffering.  A thread owns one human of the chunk for all the CTA's actions, so a rotated row is
// computed by the same code from the same operands whatever the decomposition.  Actions per CTA: split the action range until
// E x chunks x ranges reaches 12 CTAs per SM, then further while shared memory exceeds 200 KB.
// The reward needs collision = (some d < 0) and dmin = min over d >= 0 across all chunks, NaN taking part in neither: the
// rewards are first filled with 0x7F bytes (as an int64 key 0x7F7F...7F, as a double a positive value above the reference's
// initial dmin 9223372036854775807.0), every CTA folds its chunk into one signed 64-bit atomicMin per action (-1 for a
// collision, else the bits of its smallest d >= 0 plus 0.0 -- positive doubles order like their bits), and k_lookahead_fold
// decodes the key and applies the same reward expression (look_reward) as the whole-env kernel: bit-identical rewards, in
// any order of the atomics.  snp_lookahead_args.reserved bit 1 forces the split where one CTA would hold the env (tests and
// measurement), as bit 0 forces the vector stores.
#include "snp_lookahead.cuh"

namespace snp {
namespace {

constexpr int kLookThreads = 256;

struct LookArgs {
    int E, N, A, visible, headed;
    int chunk;   // actions per tile (one bulk copy)
    int aper;    // actions per CTA (a CTA walks its range tile by tile)
    long long EN;
    const void *dyn, *stat, *next, *robot;
    const double *actions;
    double dt;
    void *rotated;
    double *rewards;
    int bulk;  // 1: tiles leave through cp.async.bulk; 0: cooperative vector stores (A/B comparison)
    int H, nhc;  // split kernel: humans per chunk, chunks per env (blockIdx.x = action range * nhc + chunk)
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

template <typename T> struct LookSmem {
    size_t pa, dist, tile, tile_stride, total;
    __host__ __device__ LookSmem(int N, int OW, int chunk, int aper) {
        size_t off = (sizeof(T) * 11 * (size_t)N + 15) & ~size_t(15);
        pa = off; off = (off + sizeof(PerAction<T>) * (size_t)aper + 15) & ~size_t(15);
        dist = off; off = (off + sizeof(double) * (size_t)aper * N + 15) & ~size_t(15);  // swept distances of the CTA's whole action range
        tile = off;
        tile_stride = ((size_t)chunk * N * OW * sizeof(T) + 16 + 15) & ~size_t(15);  // + 16: room for the alignment offset
        total = off + 2 * tile_stride;
    }
};

// kSplit = false: one CTA per (env, range of actions) with all N humans; true: per (env, range of actions, chunk of a.H humans),
// the rewards folded by atomicMin (header comment).  N below is the number of humans the CTA stages.  An fp64 split CTA stages 256
// humans and two tiles of 256 rows (> 75 KB of shared memory): 2 CTAs per SM, so it may use the registers of 2 without spilling.
template <typename T, bool kSplit>
__global__ void __launch_bounds__(kLookThreads, sizeof(T) == 4 ? 4 : (kSplit ? 2 : 3)) k_lookahead(const LookArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int OW = a.visible ? 15 : 13;
    const int e = blockIdx.y;
    const int hc = kSplit ? (int)(blockIdx.x % (unsigned)a.nhc) : 0;
    const int j0 = kSplit ? hc * a.H : 0;
    const int N = kSplit ? min(a.H, a.N - j0) : a.N;
    const int abeg = (kSplit ? (int)(blockIdx.x / (unsigned)a.nhc) : (int)blockIdx.x) * a.aper;
    const int acnt = min(a.aper, a.A - abeg);
    const T *dyn = (const T *)a.dyn, *stat = (const T *)a.stat, *nxt = (const T *)a.next, *robot = (const T *)a.robot;
    const long long EN = a.EN, base = (long long)e * a.N + j0;

    // shared memory: [cur: px py vx vy r | N each][next: x y vx vy th om | N each][per-action][dist x2][tile x2]
    const LookSmem<T> lay(N, OW, a.chunk, a.aper);
    T *cur = reinterpret_cast<T *>(smem_raw);
    T *nx = cur + 5 * N;
    PerAction<T> *pa = reinterpret_cast<PerAction<T> *>(smem_raw + lay.pa);
    double *dist_all = reinterpret_cast<double *>(smem_raw + lay.dist);

    // ---- stage the env's humans (coalesced SoA loads) and the robot ----
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        cur[0 * N + j] = dyn[SNP_DYN_PX * EN + base + j]; cur[1 * N + j] = dyn[SNP_DYN_PY * EN + base + j];
        cur[2 * N + j] = dyn[SNP_DYN_VX * EN + base + j]; cur[3 * N + j] = dyn[SNP_DYN_VY * EN + base + j];
        cur[4 * N + j] = stat[SNP_STAT_R * EN + base + j];
        nx[0 * N + j] = nxt[SNP_DYN_PX * EN + base + j]; nx[1 * N + j] = nxt[SNP_DYN_PY * EN + base + j];
        nx[2 * N + j] = nxt[SNP_DYN_VX * EN + base + j]; nx[3 * N + j] = nxt[SNP_DYN_VY * EN + base + j];
        // non-headed models do not integrate yaw / omega: the peek returns the current values (mmm:294-301)
        const T *ho = a.headed ? nxt : dyn;
        nx[4 * N + j] = ho[SNP_DYN_TH * EN + base + j]; nx[5 * N + j] = ho[SNP_DYN_OM * EN + base + j];
    }
    const long long E = a.E;
    const T rpx = robot[SNP_ROBOT_PX * E + e], rpy = robot[SNP_ROBOT_PY * E + e], rr = robot[SNP_ROBOT_R * E + e];
    const T rgx = robot[SNP_ROBOT_GX * E + e], rgy = robot[SNP_ROBOT_GY * E + e], rvd = robot[SNP_ROBOT_VD * E + e];
    // ---- per action, once per CTA: next robot position (cadrl.py:54), rotation (:22), distance to goal (look_action) ----
    for (int k = threadIdx.x; k < acnt; k += blockDim.x)
        pa[k] = look_action<T>(a.actions[2 * (abeg + k)], a.actions[2 * (abeg + k) + 1], a.dt, rpx, rpy, rgx, rgy);
    __syncthreads();

    const size_t row_words = (size_t)a.N * OW;  // one action's rows of the env; a split CTA's tile (chunk = 1) is its part of them
    const int nchunks = (acnt + a.chunk - 1) / a.chunk;
    // A thread keeps the same (action slot k, human j) in every tile (a tile holds at most blockDim pairs unless N > blockDim):
    // the human's state and everything of the swept test that does not depend on the action stay in registers across tiles.
    const int k_own = threadIdx.x / N, j_own = threadIdx.x - k_own * N;
    const bool own = k_own < a.chunk;
    using Human = LookHuman<T>;
    auto load_human = [&](int j) {
        return look_human<T>(cur[j], cur[N + j], cur[2 * N + j], cur[3 * N + j], cur[4 * N + j], nx[j], nx[N + j], nx[2 * N + j], nx[3 * N + j],
                             nx[4 * N + j], nx[5 * N + j], rpx, rpy);
    };
    // one (action, human) pair: swept distance and the rotated row (snp_lookahead.cuh)
    auto do_pair = [&](const Human &h, const PerAction<T> &q, double *dist_out, T *o) {
        *dist_out = look_swept<T>(h, q, a.dt, rr);
        look_row<T>(h, q, rvd, rr, a.visible, o);
    };
    Human mine{};
    if (own) mine = load_human(j_own);

    for (int c = 0; c < nchunks; ++c) {
        const int k0 = c * a.chunk;                    // first action of the tile, relative to abeg
        const int na = min(a.chunk, acnt - k0);
        const int pairs = na * N;
        T *gdst = (T *)a.rotated + ((size_t)e * a.A + abeg + k0) * row_words + (size_t)j0 * OW;
        const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(gdst) & 15);
        // the tile sits in shared memory at the same offset modulo 16 as its destination: both sides of the copy 16-byte aligned
        T *tile = reinterpret_cast<T *>(smem_raw + lay.tile + (size_t)(c & 1) * lay.tile_stride + mis);
        double *dist = dist_all + (size_t)k0 * N;

        // ---- a thread per (action, human) ----
        if (own && k_own < na) do_pair(mine, pa[k0 + k_own], dist + threadIdx.x, tile + (size_t)threadIdx.x * OW);
        for (int p = threadIdx.x + blockDim.x; p < pairs; p += blockDim.x) {  // only when a tile holds more pairs than threads
            const int k = p / N, j = p - k * N;
            do_pair(load_human(j), pa[k0 + k], dist + p, tile + (size_t)p * OW);
        }
        const size_t total = (size_t)pairs * OW * sizeof(T);
        const size_t head = ((16 - mis) & 15) < total ? ((16 - mis) & 15) : total;
        const size_t body = (total - head) & ~size_t(15);
        const size_t tail = total - head - body;
        unsigned char *g8 = reinterpret_cast<unsigned char *>(gdst);
        const unsigned char *s8 = reinterpret_cast<const unsigned char *>(tile);
        if (a.bulk) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy tile writes -> visible to the bulk copy
            // the copy of tile c-1 (other buffer) has had this whole compute phase to drain; the buffer is rewritten in iteration c+1
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        __syncthreads();

        // ---- tile -> global ----
        if (a.bulk) {
            if (threadIdx.x == 0 && body) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g8 + head), "r"(smem_u32(s8 + head)), "r"((unsigned)body)
                             : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            // head and tail (< 16 bytes each) in words of T
            const int hw = (int)(head / sizeof(T)), tw = (int)(tail / sizeof(T));
            if ((int)threadIdx.x >= 32 && (int)threadIdx.x < 32 + hw) gdst[threadIdx.x - 32] = tile[threadIdx.x - 32];
            if ((int)threadIdx.x >= 64 && (int)threadIdx.x < 64 + tw) {
                const size_t w = (head + body) / sizeof(T) + (threadIdx.x - 64);
                gdst[w] = tile[w];
            }
        } else {
            const int hw = (int)(head / sizeof(T));
            if ((int)threadIdx.x < hw) gdst[threadIdx.x] = tile[threadIdx.x];
            const uint4 *sv = reinterpret_cast<const uint4 *>(s8 + head);
            uint4 *gv = reinterpret_cast<uint4 *>(g8 + head);
            for (size_t v = threadIdx.x; v < body / 16; v += blockDim.x) gv[v] = sv[v];
            const int tw = (int)(tail / sizeof(T));
            if ((int)threadIdx.x < tw) { const size_t w = (head + body) / sizeof(T) + threadIdx.x; gdst[w] = tile[w]; }
            __syncthreads();  // single-phase fallback: the tile is reused two iterations later, the dist buffer too
        }

    }

    // ---- rewards (cadrl.py:56-72), once per CTA: a thread per action over the swept distances of all its humans.  (Doing this per
    //      tile made one warp late for every tile barrier: barrier stalls were the top stall reason of the first version.)  `break` in
    //      the reference only cuts its loop short: collision = some swept distance < 0, else dmin = the smallest one ----
    __syncthreads();
    for (int k = threadIdx.x; k < acnt; k += blockDim.x) {
        bool collision = false;
        double dmin = 9223372036854775807.0;  // np.iinfo(np.int64).max
#pragma unroll 5
        for (int j = 0; j < N; ++j) {
            const double d = dist_all[k * N + j];
            collision |= d < 0;
            dmin = (d >= 0 && d < dmin) ? d : dmin;
        }
        if (kSplit) {  // this chunk's part of the swept test as an order-independent key (header comment)
            atomicMin(reinterpret_cast<long long *>(a.rewards) + (size_t)e * a.A + abeg + k, look_key(collision, dmin));
        } else {
            const PerAction<T> q = pa[k];
            a.rewards[(size_t)e * a.A + abeg + k] =
                look_reward(collision, dmin, q.axd, q.ayd, a.dt, (double)rpx, (double)rpy, (double)rgx, (double)rgy, (double)rr);
        }
    }
    if (a.bulk && threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // tiles must outlive the copies' reads
}

// after the split kernel: rewards[e][a] holds the atomicMin key of the whole swept test; a thread per (env, action) decodes it
template <typename T> __global__ void k_lookahead_fold(const LookArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)a.E * a.A) return;
    const int e = (int)(i / a.A), k = (int)(i - (long long)e * a.A);
    const long long key = reinterpret_cast<const long long *>(a.rewards)[i];
    const T *robot = (const T *)a.robot;
    const long long E = a.E;
    a.rewards[i] = look_key_reward(key, a.actions[2 * k], a.actions[2 * k + 1], a.dt, (double)robot[SNP_ROBOT_PX * E + e],
                                   (double)robot[SNP_ROBOT_PY * E + e], (double)robot[SNP_ROBOT_GX * E + e], (double)robot[SNP_ROBOT_GY * E + e],
                                   (double)robot[SNP_ROBOT_R * E + e]);
}

template <typename T> int launch_lookahead_split(LookArgs a, cudaStream_t st) {
    const int N = a.N, OW = a.visible ? 15 : 13;
    a.H = kLookThreads;  // a thread per human of the chunk, which it keeps across the CTA's actions
    a.nhc = (N + a.H - 1) / a.H;
    a.chunk = 1;         // a tile is one action's part of the rows: contiguous in the output
    const int staged = min(N, a.H);
    const int sms = device_sm_count();
    int splits = 1;
    // 12 CTAs per SM: of 6, 12, 24 and 48 the fastest for fp64 at 64 x 1024, 16 x 4096 and 1 x 65536 (DESIGN 4.5)
    while (splits < a.A && (long long)a.E * a.nhc * splits < 12LL * sms) ++splits;
    for (;; ++splits) {
        a.aper = (a.A + splits - 1) / splits;
        if (LookSmem<T>(staged, OW, 1, a.aper).total <= 200 * 1024 || a.aper == 1) break;
    }
    const LookSmem<T> lay(staged, OW, 1, a.aper);
    const long long ctas = (long long)((a.A + a.aper - 1) / a.aper) * a.nhc;
    if (lay.total > 200 * 1024 || ctas > 0x7fffffffLL) {
        set_error("snp_lookahead: %d humans x %d values x %d actions exceed the split decomposition", N, OW, a.A);
        return SNP_ERR_UNSUPPORTED;
    }
    SNP_CUDA_OK(cudaMemsetAsync(a.rewards, 0x7F, sizeof(double) * (size_t)a.E * a.A, st));
    auto kern = k_lookahead<T, true>;
    if (lay.total > 48 * 1024) SNP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
    kern<<<dim3((unsigned)ctas, (unsigned)a.E), kLookThreads, lay.total, st>>>(a);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    const long long EA = (long long)a.E * a.A;
    k_lookahead_fold<T><<<(unsigned)((EA + 255) / 256), 256, 0, st>>>(a);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

template <typename T> int launch_lookahead(LookArgs a, cudaStream_t st, bool split) {
    if (split) return launch_lookahead_split<T>(a, st);
    const int N = a.N, OW = a.visible ? 15 : 13;
    // actions per tile: as many (action, human) pairs as threads, balanced over the tiles of a CTA; capped by shared memory
    int per = kLookThreads / N;
    if (per < 1) per = 1;
    const size_t row = (size_t)N * OW * sizeof(T);
    while (per > 1 && 2 * per * row > 64 * 1024) --per;
    // actions per CTA: whole envs when there are enough of them to fill the machine several times over, else split the action range
    const int sms = device_sm_count();
    int splits = 1;
    while (splits < a.A && (long long)a.E * splits < 8LL * 3 * sms) ++splits;
    for (;; ++splits) {  // ... and until the CTA's swept distances (aper x N doubles) and tiles fit in shared memory
        a.aper = (a.A + splits - 1) / splits;
        const int tiles = (a.aper + per - 1) / per;
        a.chunk = (a.aper + tiles - 1) / tiles;
        if (LookSmem<T>(N, OW, a.chunk, a.aper).total <= 200 * 1024 || a.aper == 1) break;
    }
    const LookSmem<T> lay(N, OW, a.chunk, a.aper);
    if (lay.total > 200 * 1024) return launch_lookahead_split<T>(a, st);  // the env's humans do not fit one CTA
    auto kern = k_lookahead<T, false>;
    if (lay.total > 48 * 1024) SNP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
    kern<<<dim3((unsigned)((a.A + a.aper - 1) / a.aper), (unsigned)a.E), kLookThreads, lay.total, st>>>(a);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

}  // namespace
}  // namespace snp

using namespace snp;

namespace snp {
namespace {
// propagate_humans_state_with_constant_velocity_model (crowd_nav/policy/cadrl.py:92-105), the policies' query_env = False branch:
// x + vx dt, y + vy dt, theta + omega dt with the velocities carried over -- into a [SNP_DYN_FIELDS][E*N] buffer laid out like dyn,
// which is what snp_lookahead takes as `next`.  The reference's expression is a product followed by a sum (no contraction).
template <typename T> __global__ void k_constant_velocity(const T *dyn, T *next, long long EN, T dt) {
    const long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= EN) return;
    const T vx = dyn[SNP_DYN_VX * EN + a], vy = dyn[SNP_DYN_VY * EN + a], om = dyn[SNP_DYN_OM * EN + a];
    if (sizeof(T) == 8) {
        next[SNP_DYN_PX * EN + a] = (T)__dadd_rn((double)dyn[SNP_DYN_PX * EN + a], __dmul_rn((double)vx, (double)dt));
        next[SNP_DYN_PY * EN + a] = (T)__dadd_rn((double)dyn[SNP_DYN_PY * EN + a], __dmul_rn((double)vy, (double)dt));
        next[SNP_DYN_TH * EN + a] = (T)__dadd_rn((double)dyn[SNP_DYN_TH * EN + a], __dmul_rn((double)om, (double)dt));
    } else {
        next[SNP_DYN_PX * EN + a] = (T)__fadd_rn((float)dyn[SNP_DYN_PX * EN + a], __fmul_rn((float)vx, (float)dt));
        next[SNP_DYN_PY * EN + a] = (T)__fadd_rn((float)dyn[SNP_DYN_PY * EN + a], __fmul_rn((float)vy, (float)dt));
        next[SNP_DYN_TH * EN + a] = (T)__fadd_rn((float)dyn[SNP_DYN_TH * EN + a], __fmul_rn((float)om, (float)dt));
    }
    next[SNP_DYN_VX * EN + a] = vx; next[SNP_DYN_VY * EN + a] = vy; next[SNP_DYN_OM * EN + a] = om;
    next[SNP_DYN_BVX * EN + a] = dyn[SNP_DYN_BVX * EN + a]; next[SNP_DYN_BVY * EN + a] = dyn[SNP_DYN_BVY * EN + a];
}
}  // namespace
}  // namespace snp

extern "C" int snp_constant_velocity(const snp_crowd *c, double dt, void *next, void *stream) {
    if (!c || !c->dyn || !next) { set_error("snp_constant_velocity: null argument"); return SNP_ERR_INVALID; }
    if (c->E <= 0 || c->N <= 0) { set_error("snp_constant_velocity: E and N must be positive"); return SNP_ERR_INVALID; }
    const long long EN = (long long)c->E * c->N;
    const unsigned blocks = (unsigned)((EN + 255) / 256);
    if (c->dtype == SNP_F64) snp::k_constant_velocity<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double *)c->dyn, (double *)next, EN, dt);
    else if (c->dtype == SNP_F32) snp::k_constant_velocity<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float *)c->dyn, (float *)next, EN, (float)dt);
    else { set_error("dtype %d is neither SNP_F32 nor SNP_F64", c->dtype); return SNP_ERR_INVALID; }
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

extern "C" int snp_lookahead(const snp_crowd *c, const snp_lookahead_args *g, void *stream) {
    if (!c || !g) { set_error("snp_lookahead: null descriptor"); return SNP_ERR_INVALID; }
    if (c->E <= 0 || c->N <= 0 || g->A <= 0) { set_error("snp_lookahead: E, N and A must be positive"); return SNP_ERR_INVALID; }
    if (c->E > 65535) { set_error("snp_lookahead: at most 65535 envs per call (got %d)", c->E); return SNP_ERR_UNSUPPORTED; }
    if (!c->dyn || !c->stat || !c->robot || !g->next || !g->actions || !g->rotated || !g->rewards) {
        set_error("snp_lookahead: dyn, stat, robot, next, actions, rotated and rewards must be device pointers");
        return SNP_ERR_INVALID;
    }
    if (g->type < 0 || g->type > 8) { set_error("Type %d does not exist for this implementation", g->type); return SNP_ERR_INVALID; }
    LookArgs a;
    a.E = c->E; a.N = c->N; a.A = g->A; a.visible = g->theta_and_omega_visible ? 1 : 0; a.headed = g->type >= 3; a.chunk = 1; a.aper = g->A;
    a.EN = (long long)c->E * c->N;
    a.dyn = c->dyn; a.stat = c->stat; a.next = g->next; a.robot = c->robot;
    a.actions = g->actions; a.dt = g->dt; a.rotated = g->rotated; a.rewards = g->rewards;
    a.bulk = (g->reserved & 1) ? 0 : 1;
    a.H = a.nhc = 0;
    const bool split = (g->reserved & 2) != 0;
    if (c->dtype == SNP_F64) return launch_lookahead<double>(a, (cudaStream_t)stream, split);
    if (c->dtype == SNP_F32) return launch_lookahead<float>(a, (cudaStream_t)stream, split);
    set_error("dtype %d is neither SNP_F32 nor SNP_F64", c->dtype);
    return SNP_ERR_INVALID;
}
