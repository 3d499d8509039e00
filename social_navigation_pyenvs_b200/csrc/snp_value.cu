// snp_value.cu -- CADRL's action choice on the device (crowd_nav/policy/cadrl.py:235-276 CADRL.predict): for every env and every
// action of the action space, the rotated joint state of every human (the rows snp_lookahead writes out) goes through the value
// network -- fp32 Linear layers with ReLU between them and one output (ValueNetwork, cadrl.py mlp(..., last_relu=False)) -- where it
// is made, the outputs are reduced to their minimum over the humans, combined with the lookahead's reward into
//     value[e][a] = reward[e][a] + gamma ^ (dt * v_pref[e]) * (double) min_j MLP(row[e][a][j])
// and the first action of largest value is chosen.  Only values [E][A] (double), best [E] (int32) and reached [E] leave the chip:
// the 862 MB of rows of the benchmark's 4096 x 81 x 25 decision, and the network's activations, never touch HBM.
//
// k_value: a CTA covers (env, range of actions, chunk of humans).  A warp takes the CTA's (action, human) pairs 8 at a time:
// lanes 0..7 build the 8 rotated rows with the lookahead's own code (snp_lookahead.cuh: look_action / look_human / look_row, the
// same bits as the rows k_lookahead writes) and round them to fp32 into the warp's activation buffer [width][8] in shared memory;
// then layer by layer lane l accumulates outputs l, l + 32, ... of all 8 rows in registers (FFMA, fp32 accumulation in input
// order after the bias), reading each input value as a broadcast from shared memory and the weights [in][out] as conflict-free
// shared-memory loads: the packed weights are staged once per CTA, and one persistent CTA per SM walks the work items (CADRL's
// 110 kB of weights and 12 warps' activation buffers take 207 kB).  Weights too large for that are read from L1 / L2 instead,
// one CTA per work item.  ReLU'd outputs go to the
// warp's other buffer; nothing crosses warps, so there is no barrier between layers.  The output of the last layer is folded into a
// per-action running minimum in shared memory (an order-preserving 32-bit key of the float), and at the end the CTA folds each of
// its actions into values[e][a] with one 64-bit atomicMin of an order-preserving key of the double widened from that float
// (negative numbers need the sign flip).  The minimum is exact, so the result does not depend on how the humans were split.
// k_value_fold (a CTA per env) then recomputes the swept test of every (action, human) pair (look_swept, folded into the same
// key as the split lookahead's), the reward (look_key_reward: the lookahead's reward bit for bit), decodes the minimum, writes
// the value and takes the first index of the largest value (predict's strict `>` scan), and the robot's goal test on the current
// pose (`reached`, where predict returns the zero action).
//
// Humans per CTA: all of the env up to 256, chunks of 256 beyond; snp_value_args.reserved bit 1 forces chunks of 32 (tests and
// measurement: the same bits).  Actions per work item: the range is split until there are 8 items per SM.
#include "snp_lookahead.cuh"

namespace snp {
namespace {

constexpr int kValueThreads = 384;  // 12 warps: CADRL's 110 kB of weights and 12 warps' activation buffers fit one SM
constexpr int kValueRows = 8;      // rows a warp carries through the network together
constexpr int kValueMaxWidth = 256;
constexpr int kValueMaxLayers = 6;
constexpr int kValueChunk = 256;  // humans per CTA beyond which an env's humans are split

struct ValueArgs {
    int E, N, A, visible, headed;
    int H, nhc, aper;             // humans per CTA, human chunks per env, actions per CTA (blockIdx.x = action range * nhc + chunk)
    int layers, bufa, bufb;       // Linear layers; floats per row in the warp's two activation buffers
    int items_per_env;            // work items (action ranges x human chunks) of an env
    long long nweights;           // floats in `weights`
    int widths[kValueMaxLayers + 1];
    long long woff[kValueMaxLayers];  // offset of layer l's W [in][out] in `weights` (its bias [out] follows)
    long long EN;
    const void *dyn, *stat, *next, *robot;
    const double *actions;
    double dt, gamma;
    const float *weights;
    double *values;
    int *best;
    unsigned char *reached;
};

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

template <typename T> struct ValueSmem {
    size_t keys, act, total;
    __host__ __device__ ValueSmem(int aper, int bufa, int bufb) {
        keys = align16(sizeof(PerAction<T>) * (size_t)aper);
        act = align16(keys + sizeof(unsigned) * (size_t)aper);
        total = act + sizeof(float) * (size_t)(bufa + bufb) * kValueRows * (kValueThreads / 32);
    }
};

// float <-> unsigned key with the order of the floats (-0.0 below +0.0); double -> 64-bit key likewise
__device__ __forceinline__ unsigned float_key(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
__device__ __forceinline__ unsigned long long double_key(double d) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | (1ull << 63));
}
__device__ __forceinline__ double key_double(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

// One Linear layer for the warp's 8 rows: lane owns outputs o = lane + 32 j, j < NJ.  `in` / `out` are [width][8] row-minor.
template <int NJ>
__device__ __forceinline__ void value_layer(const float *__restrict__ in, float *__restrict__ out, const float *W, int K, int O,
                                            int lane, bool last, float &y0) {
    float acc[kValueRows][NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int o = lane + 32 * j;
        const float b = o < O ? W[(size_t)K * O + o] : 0.f;
#pragma unroll
        for (int r = 0; r < kValueRows; ++r) acc[r][j] = b;
    }
#pragma unroll 1  // unrolling by 2 measured no faster (DESIGN 4.7)
    for (int k = 0; k < K; ++k) {
        const float4 x0 = *reinterpret_cast<const float4 *>(in + k * kValueRows);
        const float4 x1 = *reinterpret_cast<const float4 *>(in + k * kValueRows + 4);
        const float x[kValueRows] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int o = lane + 32 * j;
            const float w = o < O ? W[(size_t)k * O + o] : 0.f;
#pragma unroll
            for (int r = 0; r < kValueRows; ++r) acc[r][j] = __fmaf_rn(x[r], w, acc[r][j]);
        }
    }
    if (last) {  // O == 1: lane 0 holds the network's output of the 8 rows; hand row r's to lane r
#pragma unroll
        for (int r = 0; r < kValueRows; ++r) {
            const float v = __shfl_sync(0xffffffffu, acc[r][0], 0);
            if (lane == r) y0 = v;
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int o = lane + 32 * j;
        if (o < O) {
            float4 *dst = reinterpret_cast<float4 *>(out + o * kValueRows);
            dst[0] = make_float4(fmaxf(acc[0][j], 0.f), fmaxf(acc[1][j], 0.f), fmaxf(acc[2][j], 0.f), fmaxf(acc[3][j], 0.f));
            dst[1] = make_float4(fmaxf(acc[4][j], 0.f), fmaxf(acc[5][j], 0.f), fmaxf(acc[6][j], 0.f), fmaxf(acc[7][j], 0.f));
        }
    }
}

// kStaged: the packed weights are copied into shared memory once per CTA, and the CTA (one per SM, persistent) walks the work items
// (env, range of actions, chunk of humans) blockIdx.x, blockIdx.x + gridDim.x, ...; otherwise (weights too large for shared memory)
// they are read from L1 / L2.  Either way a work item's arithmetic is the same.
template <typename T, bool kStaged> __global__ void __launch_bounds__(kValueThreads, 1) k_value(const ValueArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int OW = a.visible ? 15 : 13;
    const ValueSmem<T> lay(a.aper, a.bufa, a.bufb);
    PerAction<T> *pa = reinterpret_cast<PerAction<T> *>(smem_raw);
    unsigned *mkey = reinterpret_cast<unsigned *>(smem_raw + lay.keys);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *bufa = reinterpret_cast<float *>(smem_raw + lay.act) + (size_t)warp * (a.bufa + a.bufb) * kValueRows;
    float *bufb = bufa + (size_t)a.bufa * kValueRows;
    const float *weights = a.weights;
    if (kStaged) {
        float *ws = reinterpret_cast<float *>(smem_raw + lay.total);
        for (long long i = threadIdx.x; i < a.nweights; i += blockDim.x) ws[i] = __ldg(a.weights + i);
        weights = ws;  // made visible by the first work item's barrier
    }

    const T *dyn = (const T *)a.dyn, *stat = (const T *)a.stat, *nxt = (const T *)a.next, *robot = (const T *)a.robot;
    const T *ho = a.headed ? nxt : dyn;  // non-headed models do not integrate yaw / omega: the peek returns the current values (mmm:294-301)
    const long long E = a.E, EN = a.EN;
    const long long items = (long long)a.E * a.items_per_env;
    for (long long item = blockIdx.x; item < items; item += kStaged ? gridDim.x : items) {
        const int e = (int)(item / a.items_per_env), x = (int)(item - (long long)e * a.items_per_env);
        const int hc = x % a.nhc;
        const int j0 = hc * a.H, nh = min(a.H, a.N - j0);
        const int abeg = (x / a.nhc) * a.aper, acnt = min(a.aper, a.A - abeg);
        const long long base = (long long)e * a.N + j0;
        const T rpx = robot[SNP_ROBOT_PX * E + e], rpy = robot[SNP_ROBOT_PY * E + e], rr = robot[SNP_ROBOT_R * E + e];
        const T rgx = robot[SNP_ROBOT_GX * E + e], rgy = robot[SNP_ROBOT_GY * E + e], rvd = robot[SNP_ROBOT_VD * E + e];
        __syncthreads();  // the previous item's per-action data has been read
        for (int k = threadIdx.x; k < acnt; k += blockDim.x) {
            pa[k] = look_action<T>(a.actions[2 * (abeg + k)], a.actions[2 * (abeg + k) + 1], a.dt, rpx, rpy, rgx, rgy);
            mkey[k] = 0xffffffffu;
        }
        __syncthreads();

        const long long pairs = (long long)acnt * nh, groups = (pairs + kValueRows - 1) / kValueRows;
        for (long long g = warp; g < groups; g += kValueThreads / 32) {
            const long long p = g * kValueRows + lane;
            int k = -1;
            if (lane < kValueRows) {
                T row[15];
                if (p < pairs) {
                    k = (int)(p / nh);
                    const long long i = base + (p - (long long)k * nh);
                    const LookHuman<T> h = look_human<T>(dyn[SNP_DYN_PX * EN + i], dyn[SNP_DYN_PY * EN + i], dyn[SNP_DYN_VX * EN + i],
                                                         dyn[SNP_DYN_VY * EN + i], stat[SNP_STAT_R * EN + i], nxt[SNP_DYN_PX * EN + i],
                                                         nxt[SNP_DYN_PY * EN + i], nxt[SNP_DYN_VX * EN + i], nxt[SNP_DYN_VY * EN + i],
                                                         ho[SNP_DYN_TH * EN + i], ho[SNP_DYN_OM * EN + i], rpx, rpy);
                    look_row<T>(h, pa[k], rvd, rr, a.visible, row);
                } else {
#pragma unroll
                    for (int c = 0; c < 15; ++c) row[c] = T(0);
                }
#pragma unroll
                for (int c = 0; c < 15; ++c)
                    if (c < OW) bufa[c * kValueRows + lane] = (float)row[c];  // round to nearest, as Tensor.float()
            }
            __syncwarp();
            float *in = bufa, *out = bufb, y = 0.f;
            for (int l = 0; l < a.layers; ++l) {
                const int K = a.widths[l], O = a.widths[l + 1];
                const bool last = l + 1 == a.layers;
                const float *W = weights + a.woff[l];
                switch ((O + 31) >> 5) {
                    case 1: value_layer<1>(in, out, W, K, O, lane, last, y); break;
                    case 2: value_layer<2>(in, out, W, K, O, lane, last, y); break;
                    case 3: value_layer<3>(in, out, W, K, O, lane, last, y); break;
                    case 4: value_layer<4>(in, out, W, K, O, lane, last, y); break;
                    case 5: value_layer<5>(in, out, W, K, O, lane, last, y); break;
                    case 6: value_layer<6>(in, out, W, K, O, lane, last, y); break;
                    case 7: value_layer<7>(in, out, W, K, O, lane, last, y); break;
                    default: value_layer<8>(in, out, W, K, O, lane, last, y); break;
                }
                __syncwarp();  // this layer's outputs are the next one's inputs; its inputs are the next one's outputs
                float *t = in; in = out; out = t;
            }
            if (k >= 0) atomicMin(mkey + k, float_key(y));
        }
        __syncthreads();
        for (int k = threadIdx.x; k < acnt; k += blockDim.x)
            atomicMin(reinterpret_cast<unsigned long long *>(a.values) + (size_t)e * a.A + abeg + k, double_key((double)key_float(mkey[k])));
    }
}

// a CTA per env: reward (the swept test over all humans), value, first argmax, goal test of the current pose
template <typename T> __global__ void __launch_bounds__(kValueThreads, 1) k_value_fold(const ValueArgs a) {
    __shared__ double wv[kValueThreads / 32];
    __shared__ int wi[kValueThreads / 32];
    const int e = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T *dyn = (const T *)a.dyn, *stat = (const T *)a.stat, *robot = (const T *)a.robot;
    const long long E = a.E, EN = a.EN, base = (long long)e * a.N;
    const T rpx = robot[SNP_ROBOT_PX * E + e], rpy = robot[SNP_ROBOT_PY * E + e], rr = robot[SNP_ROBOT_R * E + e];
    const T rgx = robot[SNP_ROBOT_GX * E + e], rgy = robot[SNP_ROBOT_GY * E + e], rvd = robot[SNP_ROBOT_VD * E + e];
    const long long nokey = look_key(false, kLookDminCap);
    double bv = -CUDART_INF;
    int bi = -1;
    for (int k = warp; k < a.A; k += kValueThreads / 32) {
        PerAction<T> q{};  // the swept test and the reward read the action's velocity only
        q.axd = a.actions[2 * k]; q.ayd = a.actions[2 * k + 1];
        long long key = nokey;
        for (int j = lane; j < a.N; j += 32) {
            const long long i = base + j;
            const T z = T(0);  // the swept test reads the current state only
            const LookHuman<T> h = look_human<T>(dyn[SNP_DYN_PX * EN + i], dyn[SNP_DYN_PY * EN + i], dyn[SNP_DYN_VX * EN + i],
                                                 dyn[SNP_DYN_VY * EN + i], stat[SNP_STAT_R * EN + i], z, z, z, z, z, z, rpx, rpy);
            const double d = look_swept<T>(h, q, a.dt, rr);
            const long long kd = d < 0 ? -1LL : (d >= 0 ? look_key(false, d) : nokey);
            key = kd < key ? kd : key;
        }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const long long o = __shfl_xor_sync(0xffffffffu, key, s);
            key = o < key ? o : key;
        }
        if (lane == 0) {
            const size_t at = (size_t)e * a.A + k;
            const double m = key_double(reinterpret_cast<const unsigned long long *>(a.values)[at]);
            const double reward = look_key_reward(key, q.axd, q.ayd, a.dt, (double)rpx, (double)rpy, (double)rgx, (double)rgy, (double)rr);
            const double disc = pow(a.gamma, __dmul_rn(a.dt, (double)rvd));  // pow(self.gamma, self.time_step * state.self_state.v_pref)
            const double v = __dadd_rn(reward, __dmul_rn(disc, m));
            a.values[at] = v;
            if (v > bv) { bv = v; bi = k; }  // ascending k within the warp: the first of equal values stays
        }
    }
    if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = -CUDART_INF;
        int b = -1;
        for (int w = 0; w < kValueThreads / 32; ++w)
            if (wi[w] >= 0 && (wv[w] > v || (wv[w] == v && wi[w] < b))) { v = wv[w]; b = wi[w]; }
        a.best[e] = b;
        a.reached[e] = xnorm_plain(__dsub_rn((double)rpx, (double)rgx), __dsub_rn((double)rpy, (double)rgy)) < (double)rr ? 1 : 0;
    }
}

template <typename T> int launch_value(ValueArgs a, cudaStream_t st, bool force_split) {
    a.H = force_split ? 32 : (a.N <= kValueChunk ? a.N : kValueChunk);
    a.nhc = (a.N + a.H - 1) / a.H;
    const int sms = device_sm_count();
    int splits = 1;
    while (splits < a.A && (long long)a.E * a.nhc * splits < 8LL * sms) ++splits;
    for (;; ++splits) {
        a.aper = (a.A + splits - 1) / splits;
        if (a.aper <= 1024) break;
    }
    const ValueSmem<T> lay(a.aper, a.bufa, a.bufb);
    a.items_per_env = ((a.A + a.aper - 1) / a.aper) * a.nhc;
    const long long items = (long long)a.E * a.items_per_env;
    const size_t staged = lay.total + sizeof(float) * (size_t)a.nweights;
    SNP_CUDA_OK(cudaMemsetAsync(a.values, 0xFF, sizeof(double) * (size_t)a.E * a.A, st));  // the largest key: every minimum lands below it
    if (staged <= 220 * 1024) {  // weights in shared memory, one persistent CTA per SM
        auto kern = k_value<T, true>;
        SNP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged));
        const long long grid = items < sms ? items : sms;
        kern<<<(unsigned)grid, kValueThreads, staged, st>>>(a);
    } else {
        if (items > 0x7fffffffLL) {
            set_error("snp_value_lookahead: %d humans x %d actions exceed the grid", a.N, a.A);
            return SNP_ERR_UNSUPPORTED;
        }
        auto kern = k_value<T, false>;
        if (lay.total > 48 * 1024) SNP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
        kern<<<(unsigned)items, kValueThreads, lay.total, st>>>(a);
    }
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    k_value_fold<T><<<(unsigned)a.E, kValueThreads, 0, st>>>(a);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

}  // namespace
}  // namespace snp

using namespace snp;

extern "C" int snp_value_lookahead(const snp_crowd *c, const snp_value_args *g, void *stream) {
    if (!c || !g) { set_error("snp_value_lookahead: null descriptor"); return SNP_ERR_INVALID; }
    if (c->E <= 0 || c->N <= 0) { set_error("snp_value_lookahead: E and N must be positive"); return SNP_ERR_INVALID; }
    if (c->E > 65535) { set_error("snp_value_lookahead: at most 65535 envs per call (got %d)", c->E); return SNP_ERR_INVALID; }
    if (g->A < 1 || g->A > 65535) { set_error("snp_value_lookahead: A must be in 1..65535 (got %d)", g->A); return SNP_ERR_INVALID; }
    if (!c->dyn || !c->stat || !c->robot || !g->next || !g->actions || !g->weights || !g->values || !g->best || !g->reached) {
        set_error("snp_value_lookahead: dyn, stat, robot, next, actions, weights, values, best and reached must be device pointers");
        return SNP_ERR_INVALID;
    }
    if (g->type < 0 || g->type > 8) { set_error("snp_value_lookahead: type %d does not exist for this implementation", g->type); return SNP_ERR_INVALID; }
    if (c->dtype != SNP_F32 && c->dtype != SNP_F64) { set_error("snp_value_lookahead: dtype %d is neither SNP_F32 nor SNP_F64", c->dtype); return SNP_ERR_INVALID; }
    if (g->layers < 1 || g->layers > kValueMaxLayers) {
        set_error("snp_value_lookahead: %d Linear layers (1..%d supported)", g->layers, kValueMaxLayers);
        return SNP_ERR_INVALID;
    }
    const int OW = g->theta_and_omega_visible ? 15 : 13;
    if (g->widths[0] != OW) {
        set_error("snp_value_lookahead: the network takes %d inputs, the rotated state has %d (theta_and_omega_visible = %d)", g->widths[0], OW,
                  g->theta_and_omega_visible);
        return SNP_ERR_INVALID;
    }
    for (int l = 1; l < g->layers; ++l)
        if (g->widths[l] < 1 || g->widths[l] > kValueMaxWidth) {
            set_error("snp_value_lookahead: hidden width %d of layer %d is outside 1..%d", g->widths[l], l, kValueMaxWidth);
            return SNP_ERR_INVALID;
        }
    if (g->widths[g->layers] != 1) { set_error("snp_value_lookahead: the last layer has %d outputs, the value network one", g->widths[g->layers]); return SNP_ERR_INVALID; }

    ValueArgs a{};
    a.E = c->E; a.N = c->N; a.A = g->A; a.visible = g->theta_and_omega_visible ? 1 : 0; a.headed = g->type >= 3;
    a.layers = g->layers;
    long long off = 0;
    for (int l = 0; l <= g->layers; ++l) a.widths[l] = g->widths[l];
    for (int l = 0; l < g->layers; ++l) {
        a.woff[l] = off;
        off += (long long)a.widths[l] * a.widths[l + 1] + a.widths[l + 1];
        a.nweights = off;
        // activation l (the input of layer l) lives in buffer a for even l, b for odd l
        if (l % 2 == 0) a.bufa = a.widths[l] > a.bufa ? a.widths[l] : a.bufa;
        else a.bufb = a.widths[l] > a.bufb ? a.widths[l] : a.bufb;
    }
    a.EN = (long long)c->E * c->N;
    a.dyn = c->dyn; a.stat = c->stat; a.next = g->next; a.robot = c->robot;
    a.actions = g->actions; a.dt = g->dt; a.gamma = g->gamma; a.weights = g->weights;
    a.values = g->values; a.best = g->best; a.reached = g->reached;
    const bool split = (g->reserved & 2) != 0;
    if (c->dtype == SNP_F64) return launch_value<double>(a, (cudaStream_t)stream, split);
    return launch_value<float>(a, (cudaStream_t)stream, split);
}
