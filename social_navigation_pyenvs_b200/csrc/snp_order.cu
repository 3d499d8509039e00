// snp_order.cu -- re-numbering a crowd patch by patch on the device (snp_spatial_order) and applying a re-numbering to every
// per-agent array of a crowd (snp_gather_crowd).
//
// snp_spatial_order is scenarios.spatial_order (block = 256) per env, as four stable CUB radix sorts of the whole batch:
//   1. (x key, index) over all E*N humans, then stably by env: the humans of every env in ascending x, ties in index order;
//   2. (y key, position in that order), then stably by segment = env * strips + strip of the position (np.array_split: the first
//      N % strips strips get one human more): every strip in ascending y, ties in x order -- np.argsort(kind="stable") of the strip.
// Keys are the order-preserving unsigned images of the positions widened to double, with -0.0 folded into +0.0, so that the order
// and the ties are NumPy's for fp64 and for fp32 positions alike.  A last kernel writes perm[e][k] = the env-local index of the
// human that goes to place k, after dealing the 128-human tiles round-robin to `world` ranks (scenarios.deal_tiles) when asked.
#include <cub/device/device_radix_sort.cuh>

#include <cmath>

#include "snp_kernels.cuh"

namespace snp {
namespace {

constexpr int kOrderBlock = 256;     // the agents per patch spatial_order aims at (its `block` argument)
constexpr int kDealTile = 128;       // the tile deal_tiles deals (the tiled kernels' entity tile)
constexpr size_t kAlign = 256;

size_t up(size_t b) { return (b + kAlign - 1) & ~(kAlign - 1); }

// Python's max(1, int(round(sqrt(n / 256)))): round half to even, which nearbyint does in the default rounding mode.
int order_strips(int n) {
    const int s = (int)std::nearbyint(std::sqrt((double)n / (double)kOrderBlock));
    return s < 1 ? 1 : s;
}

int key_bits(long long max_key) {
    int b = 1;
    while (b < 32 && (1LL << b) <= max_key) ++b;
    return b;
}

struct OrderScratch {
    size_t keys_a, keys_b, vals_a, vals_b, by_x, temp, temp_bytes, bytes;
};

// Regions of the scratch; `temp_bytes` is the larger of CUB's two temporary-storage sizes (64-bit and 32-bit keys).
int order_scratch(long long EN, OrderScratch *s) {
    size_t t64 = 0, t32 = 0;
    cub::DoubleBuffer<unsigned long long> k64(nullptr, nullptr);
    cub::DoubleBuffer<unsigned int> k32(nullptr, nullptr);
    cub::DoubleBuffer<int> v(nullptr, nullptr);
    SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, t64, k64, v, (int)EN));
    SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, t32, k32, v, (int)EN));
    s->temp_bytes = t64 > t32 ? t64 : t32;
    size_t o = 0;
    s->keys_a = o; o += up(sizeof(unsigned long long) * EN);
    s->keys_b = o; o += up(sizeof(unsigned long long) * EN);
    s->vals_a = o; o += up(sizeof(int) * EN);
    s->vals_b = o; o += up(sizeof(int) * EN);
    s->by_x = o; o += up(sizeof(int) * EN);
    s->temp = o; o += up(s->temp_bytes);
    s->bytes = o;
    return SNP_OK;
}

// The order-preserving unsigned image of v (as a double): ascending keys = ascending values, -0.0 and +0.0 the same key.
__device__ __forceinline__ unsigned long long order_key(double v) {
    if (v == 0.0) v = 0.0;
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

// Pass 1 input: key of x of human g, value g; any non-finite x or y raises the flag.
template <typename T>
__global__ void k_order_x_keys(const T *px, const T *py, long long EN, unsigned long long *keys, int *vals, int *nonfinite) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= EN) return;
    const double x = (double)px[g], y = (double)py[g];
    if (!isfinite(x) || !isfinite(y)) *nonfinite = 1;
    keys[g] = order_key(x);
    vals[g] = (int)g;
}

// The env of every sorted index (the key of the stable sort that groups the envs back together).
__global__ void k_order_env_keys(const int *vals, long long EN, int N, unsigned int *keys) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < EN) keys[p] = (unsigned)(vals[p] / N);
}

// Pass 2 input: key of y of the human at x-order position p, value p.
template <typename T>
__global__ void k_order_y_keys(const T *py, const int *by_x, long long EN, unsigned long long *keys, int *vals) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= EN) return;
    keys[p] = order_key((double)py[by_x[p]]);
    vals[p] = (int)p;
}

// Segment (env * strips + strip) of x-order position p; strips as np.array_split cuts N positions into `strips` parts.
__global__ void k_order_strip_keys(const int *vals, long long EN, int N, int strips, unsigned int *keys) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= EN) return;
    const int v = vals[p], e = v / N, k = v - e * N;
    const int q = N / strips, r = N % strips, big = r * (q + 1);
    const int s = k < big ? k / (q + 1) : r + (k - big) / q;
    keys[p] = (unsigned)e * (unsigned)strips + (unsigned)s;
}

// perm[e][k'] = env-local index of the human at place k of env e, k' = k or its place after the tiles are dealt to `world` ranks.
__global__ void k_order_write(const int *vals, const int *by_x, long long EN, int N, int world, long long *perm) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= EN) return;
    const int e = (int)(p / N), k = (int)(p - (long long)e * N);
    const int old = by_x[vals[p]] - e * N;
    int dst = k;
    if (world > 1) {  // tile t goes to rank t % world, as that rank's (t / world)-th tile
        const int T = N / kDealTile, t = k / kDealTile, r = t % world;
        const int start = r * (T / world) + (r < T % world ? r : T % world);
        dst = (start + t / world) * kDealTile + (k - t * kDealTile);
    }
    perm[(long long)e * N + dst] = old;
}

template <typename T>
__global__ void k_gather_crowd(const snp_crowd dst, const snp_crowd src, const long long *perm, long long offset, int *error_flag) {
    const long long n = dst.N, M = src.N, En = (long long)dst.E * n, EM = (long long)src.E * M;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= En) return;
    const long long e = t / n, k = t - e * n;
    const long long p = perm[e * M + offset + k];
    if (p < 0 || p >= M) {
        if (error_flag) *error_flag = 1;
        return;
    }
    const long long s = e * M + p;
    const T *sd = (const T *)src.dyn, *ss = (const T *)src.stat, *sg = (const T *)src.goals;
    T *dd = (T *)dst.dyn, *ds = (T *)dst.stat, *dg = (T *)dst.goals;
#pragma unroll
    for (int f = 0; f < SNP_DYN_FIELDS; ++f) dd[f * En + t] = sd[f * EM + s];
#pragma unroll
    for (int f = 0; f < SNP_STAT_FIELDS; ++f) ds[f * En + t] = ss[f * EM + s];
    for (int f = 0; f < 2 * dst.G; ++f) dg[f * En + t] = sg[f * EM + s];
    dst.goal_idx[t] = src.goal_idx[s];
    const_cast<int32_t *>(dst.goal_cnt)[t] = src.goal_cnt[s];
}

unsigned blocks_of(long long n) { return (unsigned)((n + 255) / 256); }

template <typename T>
int spatial_order(const T *px, const T *py, int E, int N, int world, long long *perm, int *nonfinite, unsigned char *scratch,
                  const OrderScratch &s, cudaStream_t st) {
    const long long EN = (long long)E * N;
    const unsigned nb = blocks_of(EN);
    auto *ka = (unsigned long long *)(scratch + s.keys_a), *kb = (unsigned long long *)(scratch + s.keys_b);
    int *va = (int *)(scratch + s.vals_a), *vb = (int *)(scratch + s.vals_b), *by_x = (int *)(scratch + s.by_x);
    void *temp = scratch + s.temp;
    size_t tb = s.temp_bytes;
    SNP_CUDA_OK(cudaMemsetAsync(nonfinite, 0, sizeof(int), st));
    // 1. by x, then (stably) by env
    k_order_x_keys<T><<<nb, 256, 0, st>>>(px, py, EN, ka, va, nonfinite);
    count_launch();
    cub::DoubleBuffer<unsigned long long> k64(ka, kb);
    cub::DoubleBuffer<int> v(va, vb);
    SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(temp, tb, k64, v, (int)EN, 0, 64, st));
    cub::DoubleBuffer<unsigned int> k32((unsigned *)ka, (unsigned *)kb);
    if (E > 1) {
        k_order_env_keys<<<nb, 256, 0, st>>>(v.Current(), EN, N, k32.Current());
        count_launch();
        SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(temp, tb, k32, v, (int)EN, 0, key_bits(E - 1), st));
    }
    SNP_CUDA_OK(cudaMemcpyAsync(by_x, v.Current(), sizeof(int) * EN, cudaMemcpyDeviceToDevice, st));
    // 2. by y, then (stably) by strip
    k64 = cub::DoubleBuffer<unsigned long long>(ka, kb);
    v = cub::DoubleBuffer<int>(va, vb);
    k_order_y_keys<T><<<nb, 256, 0, st>>>(py, by_x, EN, k64.Current(), v.Current());
    count_launch();
    SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(temp, tb, k64, v, (int)EN, 0, 64, st));
    const int strips = order_strips(N);
    if ((long long)E * strips > 1) {
        k32 = cub::DoubleBuffer<unsigned int>((unsigned *)ka, (unsigned *)kb);
        k_order_strip_keys<<<nb, 256, 0, st>>>(v.Current(), EN, N, strips, k32.Current());
        count_launch();
        SNP_CUDA_OK(cub::DeviceRadixSort::SortPairs(temp, tb, k32, v, (int)EN, 0, key_bits((long long)E * strips - 1), st));
    }
    k_order_write<<<nb, 256, 0, st>>>(v.Current(), by_x, EN, N, world, perm);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

}  // namespace
}  // namespace snp

using namespace snp;

extern "C" {

int64_t snp_spatial_order_scratch_bytes(int32_t E, int32_t N) {
    if (E < 1 || N < 1 || (long long)E * N >= (1LL << 31)) {
        set_error("snp_spatial_order_scratch_bytes: E=%d N=%d (1 <= E, N and E * N < 2^31)", E, N);
        return -1;
    }
    OrderScratch s;
    if (order_scratch((long long)E * N, &s)) return -1;
    return (int64_t)s.bytes;
}

int snp_spatial_order(const void *px, const void *py, int32_t E, int32_t N, int32_t dtype, int32_t world, int64_t *perm,
                      int32_t *nonfinite, void *scratch, int64_t scratch_bytes, void *stream) {
    if (!px || !py || !perm || !nonfinite || !scratch) { set_error("snp_spatial_order: null argument"); return SNP_ERR_INVALID; }
    if (E < 1 || N < 1 || (long long)E * N >= (1LL << 31)) { set_error("snp_spatial_order: E=%d N=%d (1 <= E, N and E * N < 2^31)", E, N); return SNP_ERR_INVALID; }
    if (dtype != SNP_F64 && dtype != SNP_F32) { set_error("snp_spatial_order: bad dtype %d", dtype); return SNP_ERR_INVALID; }
    if (world < 1 || (world > 1 && N % kDealTile)) {
        set_error("snp_spatial_order: world %d needs world >= 1 and, above 1, a whole number of %d-human tiles (N = %d)", world, kDealTile, N);
        return SNP_ERR_INVALID;
    }
    if (reinterpret_cast<uintptr_t>(scratch) % 16) { set_error("snp_spatial_order: the scratch must be 16-byte aligned"); return SNP_ERR_INVALID; }
    OrderScratch s;
    if (order_scratch((long long)E * N, &s)) return SNP_ERR_CUDA;
    if (scratch_bytes < (int64_t)s.bytes) {
        set_error("snp_spatial_order: scratch of %lld bytes needed, %lld given", (long long)s.bytes, (long long)scratch_bytes);
        return SNP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return dtype == SNP_F64 ? spatial_order<double>((const double *)px, (const double *)py, E, N, world, (long long *)perm, nonfinite,
                                                    (unsigned char *)scratch, s, st)
                            : spatial_order<float>((const float *)px, (const float *)py, E, N, world, (long long *)perm, nonfinite,
                                                   (unsigned char *)scratch, s, st);
}

int snp_gather_crowd(const snp_crowd *dst, const snp_crowd *src, const int64_t *perm, int64_t offset, int32_t *error_flag, void *stream) {
    if (!dst || !src || !perm) { set_error("snp_gather_crowd: null argument"); return SNP_ERR_INVALID; }
    const snp_crowd *cs[2] = {dst, src};
    for (const snp_crowd *c : cs)
        if (!c->dyn || !c->stat || !c->goals || !c->goal_idx || !c->goal_cnt) { set_error("snp_gather_crowd: crowd arrays missing"); return SNP_ERR_INVALID; }
    if (dst->dtype != src->dtype || (dst->dtype != SNP_F64 && dst->dtype != SNP_F32)) {
        set_error("snp_gather_crowd: dtypes %d and %d (both SNP_F32 or both SNP_F64)", dst->dtype, src->dtype);
        return SNP_ERR_INVALID;
    }
    if (dst->E < 1 || dst->E != src->E || dst->G < 1 || dst->G != src->G || dst->N < 1 || src->N < 1) {
        set_error("snp_gather_crowd: E=%d/%d G=%d/%d N=%d/%d (same E >= 1 and G >= 1, N >= 1)", dst->E, src->E, dst->G, src->G, dst->N, src->N);
        return SNP_ERR_INVALID;
    }
    if (offset < 0 || offset + dst->N > src->N) {
        set_error("snp_gather_crowd: slice [%lld, %lld) outside the source's %d humans", (long long)offset, (long long)offset + dst->N, src->N);
        return SNP_ERR_INVALID;
    }
    if (dst->agent_params || src->agent_params) { set_error("snp_gather_crowd: per-agent parameter rows are not supported"); return SNP_ERR_UNSUPPORTED; }
    const unsigned nb = blocks_of((long long)dst->E * dst->N);
    cudaStream_t st = (cudaStream_t)stream;
    if (dst->dtype == SNP_F64) k_gather_crowd<double><<<nb, 256, 0, st>>>(*dst, *src, (const long long *)perm, offset, error_flag);
    else k_gather_crowd<float><<<nb, 256, 0, st>>>(*dst, *src, (const long long *)perm, offset, error_flag);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

}  // extern "C"
