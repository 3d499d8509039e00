// snp_step_large.cu -- one very large crowd: shared-memory tiled all-pairs (N-body style) social force, then the same wall /
// desired / torque / Euler epilogue as the small-crowd kernel.  One sub-step on one stream:
//
//   k_tile_boxes    bounding box (+ max r+safety) of every 128-entity tile of the `others` view  [5][M] = x, y, vx, vy, r+s
//                   (every sub-step, or -- when the producers of a call write every tile of the next view -- the first sub-step
//                   of a call only: afterwards the finish kernel writes the boxes of the tiles it produces)
//   pair phase      unit of work = (i-block of 128 or 256 agents, j-chunk of 128 entities): every agent accumulates the force of
//                   the chunk's entities in ascending j from a shared-memory tile and writes ONE partial sum per chunk.  A tile
//                   is skipped when its box is farther from the i-block's box than reach = max(r+s) of the i-block + max(r+s)
//                   of the tile + 700 B in fp64, + 88 B in fp32 (Guo: max(B, D)).  Beyond that every exponential of the pair
//                   law is below e^-700 (fp64) / e^-88 (fp32) times its amplitude, so a skipped pair contributes at most about
//                   A e^-700 ~ 2e-301 (fp64; the exponent clamp of exp2_scaled_times keeps even far pairs near 2^-1010) or
//                   A e^-88 ~ 1.2e-35 and C e^-88 ~ 7e-37 (fp32: normal floats, not flushed by ex2.approx.ftz) -- NOT an
//                   identically zero force.  Any other force on the agent absorbs terms that small, so culling on and off agree
//                   bit for bit in practice; only an agent with no other force in reach sees them.
//                     all pairs:  k_large_pairs on the static (i-block, chunk) grid;
//                     culled:     k_large_cull lists the units in reach, persistent k_large_pairs_list CTAs work the list off.
//   k_large_finish  per agent: partial sums of the live chunks added in ascending chunk order (fixed, so the result does not depend
//                   on how the crowd is sharded over GPUs), goal switch, wall force, desired force, torque, Euler; writes the
//                   state in place and the agent's entry (and its tile's box) of the NEXT entity view -- on every rank.
//                   With a visible robot (a separate instantiation) the robot's pair force is added after the chunk sums.
//   k_large_robot_end  after the last sub-step of a call, one thread: the robot's end state into crowd->robot, the clock advanced.
//
// The robot (SocialNavGym.step, social_nav_gym.py:240-245: robot.step, then update_humans, per sub-step) is entity M of the
// reference's ordered loop, the last one: the finish kernel adds its pair force after every chunk, never culls it, and for
// Moussaid's symmetric path the human is agent 1 (the robot has the highest index).  Its motion does not depend on the humans
// (robot_mode 0 fixed, 1 holonomic, 3 unicycle), so every finish thread of every rank recomputes the robot of its sub-step from the
// call's start state in crowd->robot with k_step's expressions: the same bits everywhere, no exchange and no scratch.
// k_large_checks is the swept / actual check of the robot against a view of the whole crowd (snp_large_checks).
//
// Invariant: a chunk the finish kernel adds was written in this sub-step.  On the static grid a unit that culled every tile says
// so in `live` and the finish kernel skips it; every unit on the work list writes its partial sums, zeros when it culled every
// tile (k_large_cull builds the i-block's box from tile boxes, which can be larger than the box of the slice's own agents).
//
// Small chunks matter once culling is on and the crowd is sharded: only a few percent of the units have anything to evaluate, and
// what one rank of an 8-way split keeps must still fill 148 SMs evenly (history: 4096-entity chunks 2.6 ms per sub-step at 65536
// humans and no gain from a second GPU; 512: 2.0 / 1.1 ms; 256 + exact culling on compact tiles + one agent per thread: 0.75 ms on
// one GPU, 0.158 on eight; 128 + the work list + grouped evaluation: 0.59 / 0.125).  The price is J = M/128 partial sums per LIVE chunk and agent.
// Reference: same as snp_step_small.cu (motion_model_manager.py:354-373,424-459; forces.py:63-151).
#include "snp_gym.cuh"

namespace snp {
namespace {

constexpr int kTile = 128;           // entities per shared-memory tile == threads per block
// Register tiling of the pairs kernel: every staged entity is used for APT agents of the thread.  2 halves the shared-memory
// loads per pair (best when every ordered pair is evaluated: 7.8 vs 8.4 ms per sub-step at 65536 humans); 1 doubles the number of
// work units, which is what a culled fp64 step needs once the crowd is sharded.  The summation order per agent does not depend
// on it, so results stay bit-identical.
constexpr int kMaxAgentsPerThread = 2;
#ifndef SNP_LARGE_CHUNK
#define SNP_LARGE_CHUNK 128
#endif
// Culled steps (one agent per thread): entities evaluated together between two contact votes.  Measured in fp64 on one rank's slice
// of an 8-way split / on the whole 65536 crowd: 1 -> 0.1229 / 0.657 ms per sub-step, 2 -> 0.1167 / 0.621, 4 -> 0.1136 / 0.616,
// 8 -> 0.1106 / 0.604 (more registers, fewer resident CTAs per SM, but independent chains per warp when few warps are left on an SM).
#ifndef SNP_LARGE_GROUP
#define SNP_LARGE_GROUP 8
#endif
constexpr int kChunk = SNP_LARGE_CHUNK;  // entities per j-chunk (one partial sum each); fixed so results are sharding-independent

template <typename T> struct LargeArgs {
    KArgs<T> k;
    const T *others;
    long long M, self_offset;
    T *peers[8];  // next-view buffers of every rank (peer-mapped device pointers; one buffer: n_peers = 1); the finish kernel stores into all of them
    int n_peers;
    T *partial;   // [J][2][N_local]
    T *boxes;     // [n_tiles][5] xmin, xmax, ymin, ymax, max(r+s) of the tiles of `others` (the view buffer's own table)
    T *peer_boxes[8];  // the NEXT view's tile boxes on every rank, or null: the finish kernel writes its own tiles' boxes there
    unsigned char *live;  // [i-blocks][J]: 1 when the (i-block, chunk) CTA evaluated at least one tile and wrote its partial sums
    int J, n_tiles;
    int Jp;  // row stride of the `live` map: J rounded up to 16 (the finish kernel reads 16 flags per load)
    T cull_margin;  // distance beyond r+s sums at which the pair law is exactly zero; < 0 disables culling
    int boxes_ready;  // the tile boxes of `others` are already in `boxes` (written by the previous sub-step's producer)
    int apt;          // agents per thread of the pairs kernel (1 or 2): fixes the i-block size the `live` map is indexed by
    // culled steps: the (i-block, chunk) pairs that are near each other, listed by k_large_cull and handed out to persistent CTAs
    int *work;            // [i-blocks * J] entries i-block * J + chunk
    int *work_counters;   // [0] entries listed, [4 + q] entries handed out from queue q; zeroed by the finish kernel for the next sub-step
    int use_list;
    int *live_cnt, *live_list;  // per i-block: how many chunks are in reach, and which, ascending ([i-blocks], [i-blocks][Jp]) -- what the
                                // finish kernel walks instead of scanning the flags
    int robot_steps;  // robot.step calls of this call up to and including this sub-step's (0 for a fixed robot)
    // A batch of k.E environments (the kBatch instantiations, snp_large_batch_step): env_n humans each, human i of env e at e * env_n + i
    // in the view, the SoA and the partial sums.  Tiles, chunks and i-blocks are per env (clipped at the env's end), so a unit
    // (i-block, chunk) only ever pairs humans of one env; the global tile of env e's tile t is e * env_tiles + t.
    long long env_n;
    int env_tiles, env_iblocks, env_fblocks;  // per env: 128-entity tiles (= chunks), i-blocks of the pair phase, finish CTAs
    // Work list: entry k writes its partial sums to slot k of the [cap][2][128] region `partial`.  An entry k >= cap has no slot: the
    // pairs kernel skips it, the i-block's list holds -1 - chunk, and the finish kernel evaluates the chunk itself.
    int cap;
};
constexpr int kMaxQueues = 256;                 // one queue of list entries per SM (entry k belongs to queue k mod n_queues)
// The counter block (the first ints of the scratch): [0] entries listed in this sub-step, [1] most entries listed in one sub-step of
// the call, [2] units the finish kernel evaluated in the call, [3] unused, [4 + q] entries handed out from queue q.
constexpr int kWorkCounters = 4 + kMaxQueues;

template <typename T> __device__ __forceinline__ T warp_min(T v) {
    for (int o = 16; o > 0; o >>= 1) { const T w = __shfl_xor_sync(0xffffffffu, v, o); v = w < v ? w : v; }
    return v;
}
template <typename T> __device__ __forceinline__ T warp_max(T v) {
    for (int o = 16; o > 0; o >>= 1) { const T w = __shfl_xor_sync(0xffffffffu, v, o); v = w > v ? w : v; }
    return v;
}

// Block-wide (128 threads) box of per-thread (xmin, xmax, ymin, ymax, rsmax); result broadcast through `sbox`.
template <typename T> __device__ __forceinline__ void block_box(T xmin, T xmax, T ymin, T ymax, T rs, T *sbox /*[4][5]*/, T *out /*[5]*/) {
    xmin = warp_min(xmin); xmax = warp_max(xmax); ymin = warp_min(ymin); ymax = warp_max(ymax); rs = warp_max(rs);
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { sbox[w * 5 + 0] = xmin; sbox[w * 5 + 1] = xmax; sbox[w * 5 + 2] = ymin; sbox[w * 5 + 3] = ymax; sbox[w * 5 + 4] = rs; }
    __syncthreads();
    out[0] = min(min(sbox[0], sbox[5]), min(sbox[10], sbox[15]));
    out[1] = max(max(sbox[1], sbox[6]), max(sbox[11], sbox[16]));
    out[2] = min(min(sbox[2], sbox[7]), min(sbox[12], sbox[17]));
    out[3] = max(max(sbox[3], sbox[8]), max(sbox[13], sbox[18]));
    out[4] = max(max(sbox[4], sbox[9]), max(sbox[14], sbox[19]));
    __syncthreads();
}

template <typename T, bool kBatch>
__global__ void __launch_bounds__(kTile) k_tile_boxes(const T *others, long long M, T *boxes, long long env_n, int env_tiles) {
    __shared__ T sbox[20];
    long long j;
    bool ok;
    if constexpr (kBatch) {  // block = global tile e * env_tiles + t
        const int e = blockIdx.x / env_tiles;
        const long long r = (long long)(blockIdx.x - e * env_tiles) * kTile + threadIdx.x;
        j = e * env_n + r; ok = r < env_n;
    } else {
        j = (long long)blockIdx.x * kTile + threadIdx.x; ok = j < M;
    }
    const T big = Real<T>::inf();
    const T x = ok ? others[j] : T(0), y = ok ? others[M + j] : T(0), rs = ok ? others[4 * M + j] : T(0);
    T out[5];
    block_box<T>(ok ? x : big, ok ? x : -big, ok ? y : big, ok ? y : -big, rs, sbox, out);
    if (threadIdx.x < 5) boxes[(size_t)blockIdx.x * 5 + threadIdx.x] = out[threadIdx.x];
}

// The box of an i-block from the tile boxes alone: its agents are the entities of kAgentsPerThread consecutive tiles, whose union
// box contains them.
template <typename T, bool kBatch> __device__ __forceinline__ void iblock_box(const LargeArgs<T> &la, int iblock, int apt, T *u /*[5]*/) {
    long long t0, t_end = la.n_tiles;
    if constexpr (kBatch) {  // the i-block's tiles, clipped at its env's last
        const int e = iblock / la.env_iblocks;
        t0 = (long long)e * la.env_tiles + (long long)(iblock - e * la.env_iblocks) * apt;
        t_end = (long long)(e + 1) * la.env_tiles;
    } else {
        t0 = (la.self_offset + (long long)iblock * apt * kTile) / kTile;
    }
    const T inf = Real<T>::inf();
    u[0] = inf; u[1] = -inf; u[2] = inf; u[3] = -inf; u[4] = T(0);
    for (int q = 0; q < apt; ++q)
        if (t0 + q < t_end) {
            const T *b = la.boxes + (size_t)(t0 + q) * 5;
            u[0] = min(u[0], b[0]); u[1] = max(u[1], b[1]); u[2] = min(u[2], b[2]); u[3] = max(u[3], b[3]); u[4] = max(u[4], b[4]);
        }
}
// Is any tile of chunk `chunk` (of env e in a batch) within reach of the box u?  (Beyond reach the pair law is below the bound in
// the header.)
template <typename T, bool kBatch> __device__ __forceinline__ bool chunk_near(const LargeArgs<T> &la, const T *u, int chunk, int e) {
    long long base = 0, end = la.M, tile0 = 0;  // the env's first entity, its end and its first tile
    if constexpr (kBatch) { base = e * la.env_n; end = base + la.env_n; tile0 = (long long)e * la.env_tiles; }
    const long long j_begin = base + (long long)chunk * kChunk, j_end = min(end, j_begin + kChunk);
    bool near = false;
    for (long long j0 = j_begin; j0 < j_end; j0 += kTile) {
        const T *b = la.boxes + (size_t)(tile0 + (j0 - base) / kTile) * 5;
        const T gx = max(T(0), max(u[0] - b[1], b[0] - u[1]));
        const T gy = max(T(0), max(u[2] - b[3], b[2] - u[3]));
        const T reach = u[4] + b[4] + la.cull_margin;
        near |= !(fma_<T>(gx, gx, gy * gy) > reach * reach);
    }
    return near;
}

template <typename T> struct PairsSmem {
    alignas(16) unsigned char tile_raw[sizeof(Ent<T>) * kTile];
    T tile_rs[kTile];
    alignas(16) double exp_tbl_s[kExpN];
    T sbox[20];
    int item, steal;
};
// What the finish kernel stages besides its exp table to evaluate a unit the partial sums had no slot for: one tile and the box
// reduction's scratch.
template <typename T> struct TileSmem {
    alignas(16) unsigned char tile_raw[sizeof(Ent<T>) * kTile];
    T tile_rs[kTile];
    T sbox[20];
};

// One (i-block, chunk) unit of the pair phase: the i-block's agents against the chunk's entities, one partial sum per agent, from
// zero in ascending entity order.  All 128 threads of the CTA take part.  In a batch the i-block and the chunk are those of one env:
// agents and entities are numbered from the env's first (base), so that Moussaid's jj < idx compares indices in the same numbering.
// Where the sums go (kOut): kToGrid [J][2][N_local] by chunk and agent (the static grid); kToSlot slot `slot` of the [cap][2][128]
// region, agent = thread (the work list, one agent per thread); kToCaller *out_x / *out_y (the finish kernel's units without a
// slot: one agent per thread, the `live` map left alone).
enum { kToGrid = 0, kToSlot = 1, kToCaller = 2 };
template <typename T, int SOC, int kAgentsPerThread, bool kBatch, int kOut = kToGrid>
__device__ __forceinline__ void pairs_chunk(const LargeArgs<T> &la, unsigned char *tile_raw, T *tile_rs, double *exp_tbl_s, T *sbox, int iblock,
                                            int chunk, bool &have_tbl, int slot = 0, T *out_x = nullptr, T *out_y = nullptr) {
    Ent<T> *tile = reinterpret_cast<Ent<T> *>(tile_raw);
    const KArgs<T> &a = la.k;
    const long long N = a.EN, M = la.M;
    const Params<T> &P = a.P;
    long long base = 0, n_env = N, end = M, tile0 = 0;  // the env's first entity, its humans, its end and its first tile
    int ib = iblock;                                     // the i-block within its env
    if constexpr (kBatch) {
        const int e = iblock / la.env_iblocks;
        ib = iblock - e * la.env_iblocks;
        base = e * la.env_n; n_env = la.env_n; end = base + la.env_n; tile0 = (long long)e * la.env_tiles;
    }
    const long long j_begin = base + (long long)chunk * kChunk;
    const long long j_end = min(end, j_begin + kChunk);
    unsigned char *live_flag = la.live + (size_t)iblock * la.Jp + chunk;
    T mx[kAgentsPerThread], my[kAgentsPerThread], mvx[kAgentsPerThread], mvy[kAgentsPerThread], mrs[kAgentsPerThread];
    long long idx[kAgentsPerThread];
    T fsx[kAgentsPerThread], fsy[kAgentsPerThread];
    const T big = Real<T>::inf();
    T bx0 = big, bx1 = -big, by0 = big, by1 = -big, brs = T(0);
#pragma unroll
    for (int q = 0; q < kAgentsPerThread; ++q) {
        idx[q] = ((long long)ib * kAgentsPerThread + q) * kTile + threadIdx.x;
        const bool live = idx[q] < n_env;
        const long long o = la.self_offset + base + (live ? idx[q] : 0);
        mx[q] = la.others[o]; my[q] = la.others[M + o]; mvx[q] = la.others[2 * M + o]; mvy[q] = la.others[3 * M + o]; mrs[q] = la.others[4 * M + o];
        fsx[q] = T(0); fsy[q] = T(0);
        if (live) { bx0 = min(bx0, mx[q]); bx1 = max(bx1, mx[q]); by0 = min(by0, my[q]); by1 = max(by1, my[q]); brs = max(brs, mrs[q]); }
    }
    T ibox[5];
    block_box<T>(bx0, bx1, by0, by1, brs, sbox, ibox);

    const bool sym = a.symmetric != 0;
    bool any_tile = false;
    for (long long j0 = j_begin; j0 < j_end; j0 += kTile) {
        if (la.cull_margin >= T(0)) {  // uniform across the CTA
            const T *b = la.boxes + (size_t)(tile0 + (j0 - base) / kTile) * 5;
            const T gx = max(T(0), max(ibox[0] - b[1], b[0] - ibox[1]));
            const T gy = max(T(0), max(ibox[2] - b[3], b[2] - ibox[3]));
            const T reach = ibox[4] + b[4] + la.cull_margin;
            if (fma_<T>(gx, gx, gy * gy) > reach * reach) continue;
        }
        if (sizeof(T) == 8 && !have_tbl) { exp_table_init(exp_tbl_s); have_tbl = true; }
        any_tile = true;
        __syncthreads();
        const long long j = j0 + threadIdx.x;
        if (j < j_end) {
            tile[threadIdx.x] = Ent<T>{la.others[j], la.others[M + j], la.others[2 * M + j], la.others[3 * M + j]};
            tile_rs[threadIdx.x] = la.others[4 * M + j];
        }
        __syncthreads();
        const int cnt = (int)min((long long)kTile, j_end - j0);
        int t_first = 0;
#if SNP_LARGE_GROUP > 1
        if constexpr (kAgentsPerThread == 1 && SOC != 2) {
            // one agent per thread (culled steps): SNP_LARGE_GROUP consecutive entities are evaluated branch-free and share ONE contact vote
            // (independent chains in flight when few warps are left on the SM); added in entity order, so the sum is unchanged
            for (; t_first + SNP_LARGE_GROUP <= cnt; t_first += SNP_LARGE_GROUP) {
                T fx[SNP_LARGE_GROUP], fy[SNP_LARGE_GROUP];
                bool contact = false;
#pragma unroll
                for (int u = 0; u < SNP_LARGE_GROUP; ++u) {
                    const Ent<T> o = tile[t_first + u];
                    contact |= Real<T>::positive_(pair_eval<T, SOC, false>(P, exp_tbl_s, mx[0], my[0], mvx[0], mvy[0], mrs[0], o.x, o.y, o.vx, o.vy, tile_rs[t_first + u], fx[u], fy[u]));
                }
                if (__any_sync(0xffffffffu, contact)) {
#pragma unroll
                    for (int u = 0; u < SNP_LARGE_GROUP; ++u) {
                        const Ent<T> o = tile[t_first + u];
                        pair_eval<T, SOC, true>(P, exp_tbl_s, mx[0], my[0], mvx[0], mvy[0], mrs[0], o.x, o.y, o.vx, o.vy, tile_rs[t_first + u], fx[u], fy[u]);
                    }
                }
#pragma unroll
                for (int u = 0; u < SNP_LARGE_GROUP; ++u) { fsx[0] += fx[u]; fsy[0] += fy[u]; }
            }
        }
#endif
#pragma unroll 2
        for (int t = t_first; t < cnt; ++t) {
            const Ent<T> o = tile[t];
            const T rsj = tile_rs[t];
            const long long jj = j0 + t - la.self_offset - base;  // index of the entity in this crowd's (env's) numbering
            // the self pair (jj == idx[q]) contributes exactly zero by construction (tiny_ in pair_eval)
            if constexpr (sizeof(T) == 4) {
                // the evaluations of the thread's agents are independent and branch-free; ONE vote covers the rare contact
                // re-evaluation of all of them
                T fx[kAgentsPerThread], fy[kAgentsPerThread];
                bool contact = false;
#pragma unroll
                for (int q = 0; q < kAgentsPerThread; ++q) {
                    const bool sw = SOC == 2 && sym && jj < idx[q];
                    if (SOC == 2) {
                        contact |= pair_eval<T, SOC, false>(P, exp_tbl_s, sw ? o.x : mx[q], sw ? o.y : my[q], sw ? o.vx : mvx[q], sw ? o.vy : mvy[q], sw ? rsj : mrs[q],
                                                            sw ? mx[q] : o.x, sw ? my[q] : o.y, sw ? mvx[q] : o.vx, sw ? mvy[q] : o.vy, sw ? mrs[q] : rsj, fx[q], fy[q]) > T(0);
                        fx[q] = sw ? -fx[q] : fx[q]; fy[q] = sw ? -fy[q] : fy[q];
                    } else {
                        contact |= pair_eval<T, SOC, false>(P, exp_tbl_s, mx[q], my[q], mvx[q], mvy[q], mrs[q], o.x, o.y, o.vx, o.vy, rsj, fx[q], fy[q]) > T(0);
                    }
                }
                if (__any_sync(0xffffffffu, contact)) {
#pragma unroll
                    for (int q = 0; q < kAgentsPerThread; ++q) {
                        const bool sw = SOC == 2 && sym && jj < idx[q];
                        if (SOC == 2) {
                            pair_eval<T, SOC, true>(P, exp_tbl_s, sw ? o.x : mx[q], sw ? o.y : my[q], sw ? o.vx : mvx[q], sw ? o.vy : mvy[q], sw ? rsj : mrs[q],
                                                    sw ? mx[q] : o.x, sw ? my[q] : o.y, sw ? mvx[q] : o.vx, sw ? mvy[q] : o.vy, sw ? mrs[q] : rsj, fx[q], fy[q]);
                            fx[q] = sw ? -fx[q] : fx[q]; fy[q] = sw ? -fy[q] : fy[q];
                        } else {
                            pair_eval<T, SOC, true>(P, exp_tbl_s, mx[q], my[q], mvx[q], mvy[q], mrs[q], o.x, o.y, o.vx, o.vy, rsj, fx[q], fy[q]);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < kAgentsPerThread; ++q) { fsx[q] += fx[q]; fsy[q] += fy[q]; }
            } else {  // fp64, two agents per thread (all pairs) or the tail of a tile: one evaluation at a time
#pragma unroll
                for (int q = 0; q < kAgentsPerThread; ++q) {
                    T fx, fy;
                    if (SOC == 2) {
                        const bool sw = sym && jj < idx[q];
                        pair_force<T, SOC>(P, exp_tbl_s, 0xffffffffu, sw ? o.x : mx[q], sw ? o.y : my[q], sw ? o.vx : mvx[q], sw ? o.vy : mvy[q], sw ? rsj : mrs[q],
                                           sw ? mx[q] : o.x, sw ? my[q] : o.y, sw ? mvx[q] : o.vx, sw ? mvy[q] : o.vy, sw ? mrs[q] : rsj, fx, fy);
                        fx = sw ? -fx : fx; fy = sw ? -fy : fy;
                    } else {
                        pair_force<T, SOC>(P, exp_tbl_s, 0xffffffffu, mx[q], my[q], mvx[q], mvy[q], mrs[q], o.x, o.y, o.vx, o.vy, rsj, fx, fy);
                    }
                    fsx[q] += fx; fsy[q] += fy;
                }
            }
        }
    }
    if constexpr (kOut == kToCaller) {
        static_assert(kAgentsPerThread == 1, "the finish kernel runs one agent per thread");
        *out_x = fsx[0]; *out_y = fsy[0];
        return;
    }
    if (threadIdx.x == 0) *live_flag = any_tile ? 1 : 0;
    // Every tile culled: on the static grid the finish kernel reads `live` and skips the chunk, so nothing is written.  A unit on
    // the work list is added whatever happened here, and k_large_cull listed it from the tile box of the i-block, which for the
    // last, partly foreign tile of a slice ending inside the view is larger than the box of the agents tested above: such a unit
    // writes its (zero) partial sums.
    if constexpr (kOut == kToSlot) {
        static_assert(kAgentsPerThread == 1, "the work list runs one agent per thread");
        if (idx[0] < n_env) {
            la.partial[((size_t)slot * 2 + 0) * kTile + threadIdx.x] = fsx[0];
            la.partial[((size_t)slot * 2 + 1) * kTile + threadIdx.x] = fsy[0];
        }
        return;
    }
    if (!any_tile && !la.use_list) return;
#pragma unroll
    for (int q = 0; q < kAgentsPerThread; ++q)
        if (idx[q] < n_env) {
            la.partial[((size_t)chunk * 2 + 0) * N + base + idx[q]] = fsx[q];
            la.partial[((size_t)chunk * 2 + 1) * N + base + idx[q]] = fsy[q];
        }
}

// Regular grid (i-block, chunk): every ordered pair, or -- with culling, for a slice the work list does not take -- every tile
// tested against the box of the i-block's agents.  A CTA that culled every tile leaves its partial sums unwritten and says so in
// `live`.
template <typename T, int SOC, int kAgentsPerThread, bool kBatch>
__global__ void __launch_bounds__(kTile) k_large_pairs(const LargeArgs<T> la) {
    __shared__ PairsSmem<T> sm;
    bool have_tbl = false;  // the 16 kB exp table is staged only by CTAs that evaluate at least one tile (most are culled)
    pairs_chunk<T, SOC, kAgentsPerThread, kBatch>(la, sm.tile_raw, sm.tile_rs, sm.exp_tbl_s, sm.sbox, blockIdx.x, blockIdx.y, have_tbl);
}

// Culled steps of a wide crowd: of the i-blocks x J grid only a few percent of the CTAs have anything to evaluate (65536 humans on
// 512 m: 12 800 of 131 072), and what is left is too uneven for a static grid -- a rank of an 8-way split ends with 1 600 CTAs
// for 888 resident slots.  So the reach test runs first, one thread per (i-block, chunk), and lists the pairs that are near;
// persistent CTAs (one per resident slot, exp table staged once) then work the list off.  WHICH CTA takes which entry matters: with
// one shared counter the ~400 entries left when every CTA has had its first land on the SMs at random -- some get 7, some none --
// and the slowest SM sets the time (measured: 45 % over the ideal).  So entry k belongs to queue k mod n_SMs, a CTA serves the
// queue of the SM it runs on (%smid) and only when that is empty looks for another queue with entries left: every SM gets the
// same number of entries whatever the placement of the CTAs, and every entry is taken whichever CTAs exist.  Partial sums land
// where the grid version puts them: results are bit-identical.
// kSlots (SNP_OPT_UNIT_SCRATCH): the i-block's list holds each unit's slot of the partial sums (its index on the work list), or
// -1 - chunk when the index is beyond the slots; otherwise the chunk.
template <typename T, bool kBatch, bool kSlots> __global__ void __launch_bounds__(256) k_large_cull(const LargeArgs<T> la) {
    __shared__ int warp_cnt[8];
    T u[5];
    iblock_box<T, kBatch>(la, blockIdx.x, la.apt, u);
    const int env = kBatch ? (int)blockIdx.x / la.env_iblocks : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int *mine = la.live_list + (size_t)blockIdx.x * la.Jp;
    int listed = 0;  // chunks of this i-block listed so far (uniform)
    for (int c0 = 0; c0 < la.J; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x;
        const bool near = c < la.J && chunk_near<T, kBatch>(la, u, c, env);
        if (c < la.J) la.live[(size_t)blockIdx.x * la.Jp + c] = near ? 1 : 0;
        const unsigned m = __ballot_sync(0xffffffffu, near);
        const int below = __popc(m & ((1u << lane) - 1u));
        [[maybe_unused]] int slot = 0;
        if (m) {  // the global list of work units (any order)
            int base = 0;
            if (lane == __ffs(m) - 1) base = atomicAdd(la.work_counters, __popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if constexpr (kSlots) slot = base + below;
            if (near) la.work[base + below] = blockIdx.x * la.J + c;
        }
        // this i-block's own list, ascending: the order the finish kernel adds the partial sums in
        if (lane == 0) warp_cnt[warp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { const int v = warp_cnt[w]; before += w < warp ? v : 0; total += v; }
        if constexpr (kSlots) {
            if (near) mine[listed + before + below] = slot < la.cap ? slot : -1 - c;
        } else {
            if (near) mine[listed + before + below] = c;
        }
        listed += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) la.live_cnt[blockIdx.x] = listed;
}

// kSlots (SNP_OPT_UNIT_SCRATCH): entry k writes slot k of the partial sums, and entries beyond the slots are left to the finish kernel.
template <typename T, int SOC, int kAgentsPerThread, bool kBatch, bool kSlots>
__global__ void __launch_bounds__(kTile) k_large_pairs_list(const LargeArgs<T> la, const int n_queues) {
    __shared__ PairsSmem<T> sm;
    bool have_tbl = false;
    const int n_items = kSlots ? min(la.work_counters[0], la.cap) : la.work_counters[0];
    int *cursor = la.work_counters + 4;
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    int q = (int)(smid % (unsigned)n_queues);
    for (;;) {
        __syncthreads();  // the previous unit is done with the tile, the boxes and sm.item
        if (threadIdx.x == 0) {
            const long long k = (long long)q + (long long)atomicAdd(cursor + q, 1) * n_queues;
            sm.item = k < n_items ? (int)k : -1;
            sm.steal = 0x7fffffff;
        }
        __syncthreads();
        const int item = sm.item;
        if (item >= 0) {
            const int w = la.work[item];
            pairs_chunk<T, SOC, kAgentsPerThread, kBatch, kSlots ? kToSlot : kToGrid>(la, sm.tile_raw, sm.tile_rs, sm.exp_tbl_s, sm.sbox, w / la.J, w % la.J, have_tbl, item);
            continue;
        }
        // this queue is empty (and stays so: the counters only grow): move to the nearest queue that still has entries, if any
        for (int t = threadIdx.x; t < n_queues; t += kTile) {
            const int c = *reinterpret_cast<volatile int *>(cursor + t);
            if ((long long)t + (long long)c * n_queues < n_items) atomicMin(&sm.steal, (t - q + n_queues) % n_queues);
        }
        __syncthreads();
        if (sm.steal == 0x7fffffff) return;
        q = (q + sm.steal) % n_queues;
    }
}

// The robot after `steps` robot.step calls from the state in a.robot (robot_agent.py:116-136), stepped as k_step does: rb[] gets
// SNP_ROBOT_PX, PY, VX, VY and TH.  In a batch env e's robot is a.robot[field * E + e] and its action a.action[e], a.action[E + e].
template <typename T, bool kBatch> __device__ __forceinline__ void large_robot_replay(const KArgs<T> &a, int steps, T *rb, int e) {
    const long long RE = kBatch ? a.E : 1;
    rb[SNP_ROBOT_PX] = a.robot[SNP_ROBOT_PX * RE + e]; rb[SNP_ROBOT_PY] = a.robot[SNP_ROBOT_PY * RE + e];
    rb[SNP_ROBOT_VX] = a.robot[SNP_ROBOT_VX * RE + e]; rb[SNP_ROBOT_VY] = a.robot[SNP_ROBOT_VY * RE + e]; rb[SNP_ROBOT_TH] = a.robot[SNP_ROBOT_TH * RE + e];
    if (steps <= 0) return;
    const T dt = a.dt;
    if (a.robot_mode == 1) {  // holonomic: v = a
        const T ax = a.action[e], ay = a.action[RE + e];
        T px = rb[SNP_ROBOT_PX], py = rb[SNP_ROBOT_PY];
        for (int s = 0; s < steps; ++s) { px = robot_holonomic_step<T>(px, ax, dt); py = robot_holonomic_step<T>(py, ay, dt); }
        rb[SNP_ROBOT_PX] = px; rb[SNP_ROBOT_PY] = py; rb[SNP_ROBOT_VX] = ax; rb[SNP_ROBOT_VY] = ay;
    } else if (a.robot_mode == 3) {  // unicycle (v, r)
        for (int s = 0; s < steps; ++s) robot_unicycle_step<T>(rb, (double)a.action[e], (double)a.action[RE + e], (double)dt);
    }
}

// The sum of the partial sums on i-block `row`'s ascending list (the order is what makes the result independent of the sharding and
// of which units had a slot), added to fsx, fsy.  Sixteen entries per step, the next sixteen already on their way while the partial
// sums of the current ones are loaded.  FSOC < 0: the entries are chunks of the [J][2][N_local] sums, agent i.  FSOC >= 0 (the CTA
// is the whole i-block, every thread present): the entries are slots of the [cap][2][128] sums, agent = lane; an entry -1 - chunk
// had no slot, and the chunk is evaluated here with the pairs kernel's code, in its place in the order.
template <typename T, int FSOC, bool kBatch>
__device__ __forceinline__ void sum_listed(const LargeArgs<T> &la, long long row, long long n, long long lane, T &fsx, T &fsy, double *exp_tbl_s, TileSmem<T> *ts) {
    const int4 *ll = reinterpret_cast<const int4 *>(la.live_list + (size_t)row * la.Jp);
    const int cnt = la.live_cnt[row];
    int4 nxt[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) nxt[u] = ll[u];  // (a row is Jp >= 16 entries long; entries beyond cnt are ignored)
    for (int k = 0; k < cnt; k += 16) {
        int4 cur[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) cur[u] = nxt[u];
        if (k + 16 < cnt) {
#pragma unroll
            for (int u = 0; u < 4; ++u) nxt[u] = ll[(k >> 2) + 4 + u];
        }
        const int idx[16] = {cur[0].x, cur[0].y, cur[0].z, cur[0].w, cur[1].x, cur[1].y, cur[1].z, cur[1].w,
                             cur[2].x, cur[2].y, cur[2].z, cur[2].w, cur[3].x, cur[3].y, cur[3].z, cur[3].w};
        if constexpr (FSOC >= 0) {
            bool miss = false;  // (uniform: the list is the CTA's)
#pragma unroll
            for (int b = 0; b < 16; ++b) miss |= k + b < cnt && idx[b] < 0;
            if (miss) {  // one entry at a time
#pragma unroll 1
                for (int b = k; b < k + 16 && b < cnt; ++b) {
                    const int s = la.live_list[(size_t)row * la.Jp + b];
                    T vx, vy;
                    if (s >= 0) {
                        vx = la.partial[((size_t)s * 2 + 0) * n + lane]; vy = la.partial[((size_t)s * 2 + 1) * n + lane];
                    } else {
                        bool have_tbl = true;  // staged by the caller
                        pairs_chunk<T, FSOC, 1, kBatch, kToCaller>(la, ts->tile_raw, ts->tile_rs, exp_tbl_s, ts->sbox, (int)row, -1 - s, have_tbl, 0, &vx, &vy);
                        if (threadIdx.x == 0) atomicAdd(la.work_counters + 2, 1);
                    }
                    fsx += vx; fsy += vy;
                }
                continue;
            }
        }
        T vx[16], vy[16];
#pragma unroll
        for (int b = 0; b < 16; ++b)
            if (k + b < cnt) { vx[b] = la.partial[((size_t)idx[b] * 2 + 0) * n + lane]; vy[b] = la.partial[((size_t)idx[b] * 2 + 1) * n + lane]; }
#pragma unroll
        for (int b = 0; b < 16; ++b)
            if (k + b < cnt) { fsx += vx[b]; fsy += vy[b]; }
    }
}

// RSOC: the pair law of the visible robot's force (SOC of the humans' model), or -1 for no robot -- a separate instantiation, so
// that the common ones keep their registers.  kBatch: CTA b of env e is block e * env_fblocks + b and covers humans 128 b ... of env
// e only, so that it stages its own env's walls.  FSOC >= 0 (steps with SNP_OPT_UNIT_SCRATCH, another instantiation): the list holds
// slots of the [cap][2][128] partial sums, and -1 - chunk for a unit without one, which this kernel evaluates with the pair law FSOC
// (sum_listed; a tile staged in TileSmem after the segment counts, and the exp table).
template <typename T, int OBS, int HEADED, int RSOC, bool kBatch, int FSOC = -1>
__global__ void __launch_bounds__(kTile) k_large_finish(const LargeArgs<T> la) {
    using R = Real<T>;
    const KArgs<T> &a = la.k;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int nseg = a.W * a.S;
    double *exp_tbl_s = reinterpret_cast<double *>(smem_raw);
    constexpr size_t kTbl = sizeof(double) * kExpN;
    Seg<T> *segs = reinterpret_cast<Seg<T> *>(smem_raw + kTbl);
    int *seg_cnt = reinterpret_cast<int *>(smem_raw + kTbl + ((sizeof(Seg<T>) * (size_t)nseg + 15) & ~size_t(15)));
    if (sizeof(T) == 8 && (nseg > 0 || RSOC >= 0 || FSOC >= 0)) exp_table_init(exp_tbl_s);  // only the wall force, the robot and units without a slot evaluate exp here
    int env = 0;
    const T *walls = a.walls;
    if constexpr (kBatch) {
        env = blockIdx.x / la.env_fblocks;
        if (a.walls_per_env) walls += (size_t)env * nseg * 4;
    }
    for (int k = threadIdx.x; k < nseg; k += blockDim.x) {
        const T *w = walls + (size_t)k * 4;
        segs[k] = make_seg<T>(w[0], w[1], w[2], w[3]);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < a.W; k += blockDim.x) {
        int c = 0;
        while (c < a.S && segs[(size_t)k * a.S + c].ax == segs[(size_t)k * a.S + c].ax) ++c;
        seg_cnt[k] = c;
    }
    __syncthreads();
    const long long N = a.EN, M = la.M;
    long long i, r = 0;  // the agent; in a batch also its index in its env
    bool gone;
    if constexpr (kBatch) {
        r = (long long)(blockIdx.x - env * la.env_fblocks) * kTile + threadIdx.x;
        i = env * la.env_n + r; gone = r >= la.env_n;
    } else {
        i = (long long)blockIdx.x * kTile + threadIdx.x; gone = i >= N;
    }
    if constexpr (FSOC < 0) {
        if (la.use_list && blockIdx.x == 0)  // the pair phase is over: empty list and queues for the next sub-step
            for (int k = threadIdx.x; k < kWorkCounters; k += kTile) la.work_counters[k] = 0;
    } else if (blockIdx.x == 0) {  // the same, but the call's unit counts (words 1-3) stay; word 1 keeps the most units listed
        if (threadIdx.x == 0) la.work_counters[1] = max(la.work_counters[1], la.work_counters[0]);
        for (int k = threadIdx.x; k < kWorkCounters; k += kTile)
            if (k == 0 || k >= 4) la.work_counters[k] = 0;
    }
    [[maybe_unused]] T listed_x = T(0), listed_y = T(0);
    if constexpr (FSOC >= 0) {  // before any thread leaves: the units without a slot are evaluated by the whole CTA (= the i-block)
        const size_t seg_end = kTbl + ((sizeof(Seg<T>) * (size_t)nseg + 15) & ~size_t(15)) + ((sizeof(int) * (size_t)(a.W + 1) + 15) & ~size_t(15));
        sum_listed<T, FSOC, kBatch>(la, blockIdx.x, kTile, threadIdx.x, listed_x, listed_y, exp_tbl_s, reinterpret_cast<TileSmem<T> *>(smem_raw + seg_end));
    }
    const bool fold_boxes = la.peer_boxes[0] != nullptr;  // uniform; only offered when N is a whole number of tiles, so that every
    if (gone) return;                                      // thread of every block reaches the box reduction at the end
    const unsigned vote_mask = __activemask();  // the lanes that own an agent (the tail warp is partial)
    const Params<T> &P = a.P;
    Agent<T> m;
    m.px = a.dyn[SNP_DYN_PX * N + i]; m.py = a.dyn[SNP_DYN_PY * N + i];
    m.vx = a.dyn[SNP_DYN_VX * N + i]; m.vy = a.dyn[SNP_DYN_VY * N + i];
    m.dfx = a.dyn[SNP_DYN_DFX * N + i]; m.dfy = a.dyn[SNP_DYN_DFY * N + i];
    if (HEADED) {
        m.th = a.dyn[SNP_DYN_TH * N + i]; m.bvx = a.dyn[SNP_DYN_BVX * N + i]; m.bvy = a.dyn[SNP_DYN_BVY * N + i];
        m.om = a.dyn[SNP_DYN_OM * N + i];
        R::sincos_(m.th, &m.sn, &m.cs);
        m.vx = np_mv(m.cs, -m.sn, m.bvx, m.bvy);  // mmm:448; the same value k_large_publish / the previous step put in the view
        m.vy = np_mv(m.sn, m.cs, m.bvx, m.bvy);
    } else { m.th = m.bvx = m.bvy = m.om = T(0); m.cs = T(1); m.sn = T(0); }
    m.r = a.stat[SNP_STAT_R * N + i]; m.m = a.stat[SNP_STAT_M * N + i]; m.vd = a.stat[SNP_STAT_VD * N + i];
    m.rs = m.r + a.stat[SNP_STAT_SAFETY * N + i];
    agent_static<T>(P, m);
    int gidx = a.goal_idx[i];
    const int gcnt = a.goal_cnt[i];
    m.gx = a.goals[((size_t)gidx * 2 + 0) * N + i]; m.gy = a.goals[((size_t)gidx * 2 + 1) * N + i];
    T fsx = T(0), fsy = T(0);
    if constexpr (FSOC >= 0) { fsx = listed_x; fsy = listed_y; }
    // Sum of the live chunks' partial sums in ascending chunk order (the order is what makes the result independent of the
    // sharding).  On the work list the cull kernel left them as the i-block's ascending list.  On the static grid the flags are the
    // same for the whole CTA and live chunks come in runs; they are read 64 at a time, and for every 16 flags with a live one the
    // loads of all live partial sums are issued together before the (ordered) additions -- a flag-by-flag loop serialised one L2
    // round trip per live chunk.
    const long long row = kBatch ? (long long)env * la.env_iblocks + r / (kTile * la.apt) : i / (kTile * la.apt);  // the agent's i-block
    const uint4 *lv = reinterpret_cast<const uint4 *>(la.live + (size_t)row * la.Jp);
    const int n_words = la.use_list ? 0 : la.Jp >> 4;
    if (FSOC < 0 && la.use_list) sum_listed<T, FSOC, kBatch>(la, row, N, i, fsx, fsy, exp_tbl_s, nullptr);
    for (int w0 = 0; w0 < n_words; w0 += 4) {
        uint4 f[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) f[u] = (w0 + u < n_words) ? lv[w0 + u] : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (!(f[u].x | f[u].y | f[u].z | f[u].w)) continue;
            const unsigned word[4] = {f[u].x, f[u].y, f[u].z, f[u].w};  // sixteen flags, one per byte
            const int p0 = (w0 + u) << 4;
            T vx[16], vy[16];
            bool on[16];
#pragma unroll
            for (int b = 0; b < 16; ++b) {
                on[b] = ((word[b >> 2] >> (8 * (b & 3))) & 0xffu) != 0 && p0 + b < la.J;  // (bytes beyond J are padding nobody wrote)
                if (on[b]) { vx[b] = la.partial[((size_t)(p0 + b) * 2 + 0) * N + i]; vy[b] = la.partial[((size_t)(p0 + b) * 2 + 1) * N + i]; }
            }
#pragma unroll
            for (int b = 0; b < 16; ++b)
                if (on[b]) { fsx += vx[b]; fsy += vy[b]; }
        }
    }
    if constexpr (RSOC >= 0) {
        // the robot: the last entity of the ordered loop, after every chunk; never culled (one pair per human)
        T rb[SNP_ROBOT_FIELDS];
        large_robot_replay<T, kBatch>(a, la.robot_steps, rb, env);
        const long long RE = kBatch ? a.E : 1;
        const T rrs = a.robot[SNP_ROBOT_R * RE + env] + a.robot[SNP_ROBOT_SAFETY * RE + env];
        T fx, fy;
        pair_force<T, RSOC>(P, exp_tbl_s, vote_mask, m.px, m.py, m.vx, m.vy, m.rs, rb[SNP_ROBOT_PX], rb[SNP_ROBOT_PY], rb[SNP_ROBOT_VX],
                            rb[SNP_ROBOT_VY], rrs, fx, fy);
        fsx += fx; fsy += fy;
    }

    const T dg = np_norm(m.gx - m.px, m.gy - m.py);
    if (a.numba ? (dg <= m.r) : (dg < m.r)) {
        gidx = (gidx + 1 >= gcnt) ? 0 : gidx + 1;
        m.gx = a.goals[((size_t)gidx * 2 + 0) * N + i]; m.gy = a.goals[((size_t)gidx * 2 + 1) * N + i];
    }
    T fox = T(0), foy = T(0);
    if (a.W > 0) obstacle_force<T, OBS>(P, exp_tbl_s, vote_mask, segs, seg_cnt, a.W, a.S, a.numba != 0, m.px, m.py, m.vx, m.vy, m.rs, fox, foy);
    desired_force<T>(P, m, a.numba != 0);
    integrate<T, HEADED>(P, m, fox, foy, fsx, fsy, a.dt);
    a.dyn[SNP_DYN_PX * N + i] = m.px; a.dyn[SNP_DYN_PY * N + i] = m.py;
    a.dyn[SNP_DYN_VX * N + i] = m.vx; a.dyn[SNP_DYN_VY * N + i] = m.vy;
    a.dyn[SNP_DYN_DFX * N + i] = m.dfx; a.dyn[SNP_DYN_DFY * N + i] = m.dfy;
    if (HEADED) {
        a.dyn[SNP_DYN_TH * N + i] = m.th; a.dyn[SNP_DYN_BVX * N + i] = m.bvx; a.dyn[SNP_DYN_BVY * N + i] = m.bvy;
        a.dyn[SNP_DYN_OM * N + i] = m.om;
    }
    a.goal_idx[i] = gidx;
    // the all-gather of the entity view fused into the producer: every rank's copy of the NEXT view receives this agent's entry
    // through peer (NVLink) stores, so no separate collective runs between sub-steps -- only a barrier
    const long long o = la.self_offset + i;
    for (int p = 0; p < la.n_peers; ++p) {
        T *v = la.peers[p];
        v[o] = m.px; v[M + o] = m.py; v[2 * M + o] = m.vx; v[3 * M + o] = m.vy; v[4 * M + o] = m.rs;
    }
    if (fold_boxes) {
        // k_tile_boxes folded into the producer: this block's agents ARE one tile of the next view (self_offset is a multiple of
        // the tile size), so its bounding box goes to every rank's next-box table with the entries themselves
        __shared__ T sbox2[20];
        T out[5];
        block_box<T>(m.px, m.px, m.py, m.py, m.rs, sbox2, out);
        if (threadIdx.x < 5) {
            const long long tile = la.self_offset / kTile + blockIdx.x;
            for (int p = 0; p < la.n_peers; ++p) la.peer_boxes[p][tile * 5 + threadIdx.x] = out[threadIdx.x];
        }
    }
}

// Cross-rank barrier of our own between sub-steps (one tiny kernel instead of a host-driven collective): slot [r] of every rank's
// flag array receives rank r's epoch through a peer store; a rank passes once all its slots have reached the epoch.  Epochs only
// grow, so nothing is ever reset and a fast rank that is already signalling the next barrier cannot release a slow one early.
// The kernel boundary orders the finish kernel's peer stores before the signal (fence.sc.sys + release store); the acquire loads
// order the next sub-step's reads after it.  A rank that never arrives trips the time-out instead of hanging the GPU.
struct BarrierArgs {
    unsigned long long *flags[8];  // every rank's flag array [world] (peer-mapped), index = rank
    int world, rank;
    unsigned long long epoch;
    int *error;
};

__global__ void k_rank_barrier(const BarrierArgs b) {
    const int t = threadIdx.x;
    if (t < b.world) {
        __threadfence_system();
        unsigned long long *dst = b.flags[t] + b.rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(b.epoch) : "memory");
        const unsigned long long *src = b.flags[b.rank] + t;
        const long long t0 = clock64();
        unsigned long long seen = 0;
        while (true) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(src) : "memory");
            if (seen >= b.epoch) break;
            if (clock64() - t0 > 40000000000LL) { *b.error = 1; break; }  // ~20 s: a peer died; report instead of spinning forever
        }
    }
    __syncthreads();
    __threadfence_system();
}

// x, y, vx, vy, r+safety of every agent into a [5][stride] view (v = R(yaw) bv for headed models, mmm:448).
template <typename T> __global__ void k_large_publish(const T *dyn, const T *stat, long long N, int headed, T *view, long long stride, long long offset) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    T vx = dyn[SNP_DYN_VX * N + i], vy = dyn[SNP_DYN_VY * N + i];
    if (headed) {
        T s, c;
        Real<T>::sincos_(dyn[SNP_DYN_TH * N + i], &s, &c);
        const T bx = dyn[SNP_DYN_BVX * N + i], by = dyn[SNP_DYN_BVY * N + i];
        vx = np_mv(c, -s, bx, by); vy = np_mv(s, c, bx, by);
    }
    const long long o = offset + i;
    view[o] = dyn[SNP_DYN_PX * N + i]; view[stride + o] = dyn[SNP_DYN_PY * N + i];
    view[2 * stride + o] = vx; view[3 * stride + o] = vy;
    view[4 * stride + o] = stat[SNP_STAT_R * N + i] + stat[SNP_STAT_SAFETY * N + i];
}

// unit_slots (SNP_OPT_UNIT_SCRATCH, never Moussaid): the culled step through the slot instantiations of the cull, pairs and finish
// kernels; `first`: the call's first sub-step.
template <typename T, int SOC, int OBS, int HEADED, bool kBatch> int launch_large(const LargeArgs<T> &la, bool unit_slots, bool first, cudaStream_t st) {
    const long long N = la.k.EN;
    const int nseg = la.k.W * la.k.S;
    if (sizeof(T) == 8) SNP_CUDA_OK(ensure_exp_table());
    if (!la.boxes_ready) k_tile_boxes<T, kBatch><<<(unsigned)la.n_tiles, kTile, 0, st>>>(la.others, la.M, la.boxes, la.env_n, la.env_tiles);
    const long long per_block = (long long)kTile * la.apt;
    dim3 grid((unsigned)(kBatch ? (long long)la.k.E * la.env_iblocks : (N + per_block - 1) / per_block), (unsigned)la.J);
    if constexpr (SOC == 2) {  // Moussaid's pair law has no culling distance (run_large): every pair, two agents per thread
        k_large_pairs<T, SOC, kMaxAgentsPerThread, kBatch><<<grid, kTile, 0, st>>>(la);
    } else if (la.use_list) {  // (culled: one agent per thread)
        // the counters start empty: zeroed here, else by the previous sub-step's finish kernel.  With slots on the call's first
        // sub-step (the call's unit counts too), without on a sub-step that computes the tile boxes.
        if (unit_slots ? first : !la.boxes_ready) SNP_CUDA_OK(cudaMemsetAsync(la.work_counters, 0, kWorkCounters * sizeof(int), st));
        const auto cull = unit_slots ? k_large_cull<T, kBatch, true> : k_large_cull<T, kBatch, false>;
        const auto pairs = unit_slots ? k_large_pairs_list<T, SOC, 1, kBatch, true> : k_large_pairs_list<T, SOC, 1, kBatch, false>;
        cull<<<grid.x, 256, 0, st>>>(la);
        static int slots[2] = {0, 0};  // resident CTAs per SM of each pairs kernel
        int &sl = slots[unit_slots ? 1 : 0];
        const int n_queues = device_sm_count() < kMaxQueues ? device_sm_count() : kMaxQueues;
        if (!sl) SNP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sl, pairs, kTile, 0));
        pairs<<<(unsigned)(device_sm_count() * (sl > 0 ? sl : 1)), kTile, 0, st>>>(la, n_queues);
        count_launch();
    } else if (la.apt == 1) k_large_pairs<T, SOC, 1, kBatch><<<grid, kTile, 0, st>>>(la);
    else k_large_pairs<T, SOC, 2, kBatch><<<grid, kTile, 0, st>>>(la);
    size_t smem = sizeof(double) * kExpN + ((sizeof(Seg<T>) * (size_t)nseg + 15) & ~size_t(15)) + sizeof(int) * (la.k.W + 1) + 16;
    auto fin = la.k.consider_robot ? k_large_finish<T, OBS, HEADED, SOC, kBatch> : k_large_finish<T, OBS, HEADED, -1, kBatch>;
    if constexpr (SOC != 2) {
        // partial sums in slots: the finish instantiation that reads them and evaluates the units without one (a tile staged after
        // the segment counts)
        if (la.use_list && unit_slots) {
            fin = la.k.consider_robot ? k_large_finish<T, OBS, HEADED, SOC, kBatch, SOC> : k_large_finish<T, OBS, HEADED, -1, kBatch, SOC>;
            smem = sizeof(double) * kExpN + ((sizeof(Seg<T>) * (size_t)nseg + 15) & ~size_t(15)) + ((sizeof(int) * (size_t)(la.k.W + 1) + 15) & ~size_t(15)) +
                   sizeof(TileSmem<T>);
        }
    }
    if (smem > 48 * 1024) SNP_CUDA_OK(cudaFuncSetAttribute(fin, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fin<<<(unsigned)(kBatch ? (long long)la.k.E * la.env_fblocks : (N + kTile - 1) / kTile), kTile, smem, st>>>(la);
    count_launch(la.boxes_ready ? 2 : 3);
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

inline long long large_J(long long M) { return (M + kChunk - 1) / kChunk; }
inline long long large_tiles(long long M) { return (M + kTile - 1) / kTile; }
inline long long large_iblocks(long long N) { return (N + kTile - 1) / kTile; }  // sized for one agent per thread (the finer split)

inline long long up16(long long b) { return (b + 15) & ~15LL; }

// The scratch of `blocks` i-blocks against J chunks with `partial_bytes` of partial sums: byte offsets of its regions (the counters
// at 0) and its size.  Every region starts 16-byte aligned (the finish kernel reads the live map and the lists 16 bytes at a time).
// The partial sums are [J][2][n_local] on the static grid (the default size) or, on the work list, [cap][2][128] slots; a multiple
// of 16 bytes more of them moves every later region by exactly that much.
struct LargeScratch { long long partial, live, work, live_cnt, live_list, bytes; };
inline LargeScratch large_scratch_regions(long long partial_bytes, long long J, long long blocks) {
    const long long Jp = (J + 15) & ~15LL;
    LargeScratch s;
    s.partial = up16(4 * kWorkCounters);               // counters and queues (kWorkCounters ints), then the partial sums
    s.live = up16(s.partial + partial_bytes);          // [blocks][Jp] live map
    s.work = up16(s.live + blocks * Jp);               // [blocks * J] list of the units in reach
    s.live_cnt = up16(s.work + 4 * blocks * J);        // [blocks] live chunks per i-block
    s.live_list = up16(s.live_cnt + 4 * blocks);       // [blocks][Jp] their slots (or -1 - chunk), ascending by chunk
    s.bytes = s.live_list + 4 * blocks * Jp;
    return s;
}
inline long long unit_bytes(long long elem_bytes) { return 2 * kTile * elem_bytes; }  // one slot: [2][128]
// One crowd: n_local agents against M entities; units < 0: the default size, [J][2][n_local] partial sums.
inline LargeScratch large_scratch(long long n_local, long long M, long long elem_bytes, long long units = -1) {
    const long long J = large_J(M);
    return large_scratch_regions(units < 0 ? elem_bytes * J * 2 * n_local : units * unit_bytes(elem_bytes), J, large_iblocks(n_local));
}
// A batch of E envs of N humans: the regions above (chunks and i-blocks per env), then the two view buffers, each [5][E N] entities
// and the [E ceil(N/128)][5] tile boxes.
struct LargeBatchScratch { LargeScratch s; long long view_a, view_b, bytes; };
inline LargeBatchScratch large_batch_scratch(long long E, long long N, long long elem_bytes, long long units = -1) {
    LargeBatchScratch b;
    const long long J = large_J(N);
    b.s = large_scratch_regions(units < 0 ? elem_bytes * J * 2 * E * N : units * unit_bytes(elem_bytes), J, E * large_iblocks(N));
    const long long view = up16(elem_bytes * 5 * (E * N + E * large_tiles(N)));
    b.view_a = up16(b.s.bytes);
    b.view_b = b.view_a + view;
    b.bytes = b.view_b + view;
    return b;
}
// The slots a scratch of `scratch_bytes` holds (SNP_OPT_UNIT_SCRATCH): what is left after the regions of a scratch with none.
inline long long units_in(long long scratch_bytes, long long bytes_for_none, long long elem_bytes) {
    return scratch_bytes < bytes_for_none ? -1 : (scratch_bytes - bytes_for_none) / unit_bytes(elem_bytes);
}
// The longest decay length of a step's pair law (Helbing B, Guo max(B, D)) when the step is culled, else -1: SNP_OPT_NO_CULLING,
// Moussaid (no culling distance) or a decay length that is not positive.
inline double large_cull_length(const snp_crowd *c, const snp_step_opts *o) {
    const int soc = o->type % 3;
    const double B = c->params[3], D = c->params[7];
    if ((o->reserved & SNP_OPT_NO_CULLING) || soc == 2 || !(B > 0) || (soc == 1 && !(D > 0))) return -1.0;
    return soc == 1 && D > B ? D : B;
}

// Does a step take the work list (culled, one agent per thread) and hence the slot layout?  Otherwise the static grid.
inline bool large_uses_list(const snp_crowd *c, const snp_step_opts *o, long long self_offset, long long blocks, long long J) {
    return large_cull_length(c, o) > 0.0 && self_offset % kTile == 0 && blocks * J < (1LL << 31);
}

template <typename T, bool kBatch> int dispatch_large(int type, const LargeArgs<T> &la, bool unit_slots, bool first, cudaStream_t st) {
    switch (type) {
        case 0: return launch_large<T, 0, 0, 0, kBatch>(la, unit_slots, first, st);
        case 1: return launch_large<T, 1, 1, 0, kBatch>(la, unit_slots, first, st);
        case 2: return launch_large<T, 2, 0, 0, kBatch>(la, unit_slots, first, st);
        case 3: return launch_large<T, 0, 0, 1, kBatch>(la, unit_slots, first, st);
        case 4: return launch_large<T, 1, 1, 1, kBatch>(la, unit_slots, first, st);
        case 5: return launch_large<T, 2, 0, 1, kBatch>(la, unit_slots, first, st);
        case 6: return launch_large<T, 0, 0, 2, kBatch>(la, unit_slots, first, st);
        case 7: return launch_large<T, 1, 1, 2, kBatch>(la, unit_slots, first, st);
        case 8: return launch_large<T, 2, 0, 2, kBatch>(la, unit_slots, first, st);
    }
    set_error("Type %d does not exist for this implementation", type);
    return SNP_ERR_INVALID;
}

// One sub-step: `cur` = the view buffer read ([5][M] entities + their [n_tiles][5] tile boxes), `next` = the n_peers buffers the
// finish kernel stores the updated entries into, and their tile boxes too when `fold_boxes`.  `boxes_ready`: `cur`'s tile boxes
// were written by the previous sub-step's producers.  `sub`: index of the sub-step in the call (how far a moving robot has gone).
// units: the slots of the partial sums (SNP_OPT_UNIT_SCRATCH), or -1 for the default size.  env_n > 0: the crowd is a batch of c->E
// envs of env_n = c->N humans (M = E N, self_offset 0, one next buffer).
template <typename T> int run_large(const snp_crowd *c, const snp_step_opts *o, const void *cur, const void *const *next, int n_peers,
                                    long long M, long long self_offset, bool fold_boxes, bool boxes_ready, void *scratch, int sub, cudaStream_t st,
                                    long long units, long long env_n = 0) {
    const bool batch = env_n > 0;
    LargeArgs<T> la;
    la.n_peers = n_peers;
    for (int p = 0; p < 8; ++p) la.peers[p] = (p < n_peers) ? (T *)next[p] : nullptr;
    for (int p = 0; p < 8; ++p) la.peer_boxes[p] = (fold_boxes && p < n_peers) ? (T *)next[p] + 5 * M : nullptr;
    la.boxes_ready = boxes_ready ? 1 : 0;
    KArgs<T> &a = la.k;
    a.E = 1; a.N = 0; a.G = c->G; a.EN = (long long)c->E * c->N;
    a.dyn = (T *)c->dyn; a.stat = (const T *)c->stat; a.goals = (const T *)c->goals; a.goal_idx = c->goal_idx; a.goal_cnt = c->goal_cnt;
    a.agent_params = nullptr; a.P = make_params<T>(c->params); a.robot = (T *)c->robot;
    a.walls = (const T *)c->walls; a.W = c->W; a.S = c->W > 0 ? c->S : 0; a.walls_per_env = 0;
    if (batch) { a.E = c->E; a.N = c->N; a.walls_per_env = c->walls_per_env; }
    a.consider_robot = o->consider_robot; a.symmetric = o->symmetric; a.numba = o->numba_compat; a.n_substeps = 1; a.robot_mode = o->robot_mode;
    a.dt = (T)o->dt; a.dt_d = o->dt; a.action = (const T *)o->action; a.pre_checks = a.post_checks = a.track_touch = 0;
    a.time_now = nullptr; a.flags = nullptr; a.checks = nullptr; a.epw = 1; a.gpb = 1; a.mapping = 0; a.full_pair_loop = 1; a.respawn = 0; a.robot_type = 0; a.RP = a.P; a.robot_every = 0; a.robot_phase = 0; a.robot_dt = T(0);
    la.robot_steps = (o->robot_mode == 1 || o->robot_mode == 3) ? sub + 1 : 0;
    la.others = (const T *)cur; la.M = M; la.self_offset = self_offset;
    la.boxes = (T *)cur + 5 * M;
    la.env_n = env_n; la.env_tiles = (int)large_tiles(env_n);
    la.J = (int)large_J(batch ? env_n : M); la.n_tiles = (int)(batch ? c->E * large_tiles(env_n) : large_tiles(M));
    la.Jp = (la.J + 15) & ~15;
    const long long blocks = batch ? c->E * large_iblocks(env_n) : large_iblocks(a.EN);  // rows of the live map
    const long long partial_bytes = units < 0 ? (long long)sizeof(T) * la.J * 2 * a.EN : units * unit_bytes(sizeof(T));
    const LargeScratch sc = large_scratch_regions(partial_bytes, la.J, blocks);
    char *base = (char *)scratch;
    la.partial = (T *)(base + sc.partial);
    la.live = (unsigned char *)(base + sc.live);
    la.work_counters = (int *)base;
    la.work = (int *)(base + sc.work);
    la.live_cnt = (int *)(base + sc.live_cnt);
    la.live_list = (int *)(base + sc.live_list);
    // culling distance beyond the r+s sums: where exp(rd/B) has fallen below e^-700 (fp64) / e^-88 (fp32), see the header
    const double under = sizeof(T) == 8 ? 700.0 : 88.0;
    const double cull_length = large_cull_length(c, o);
    const double margin = cull_length > 0.0 ? under * cull_length : -1.0;
    la.cull_margin = (T)margin;
    // culled steps: one agent per thread (twice the units to hand out).  Round 2 kept two for fp32 on the static grid, where the
    // finer split only added CTAs to launch; on the work list one rank's slice of an 8-way split runs 0.0552 -> 0.0408 ms in fp32
    la.apt = margin >= 0.0 ? 1 : kMaxAgentsPerThread;  // fp32 pair evaluations are short: the finer split only adds launch overhead there
    la.use_list = large_uses_list(c, o, self_offset, blocks, la.J) ? 1 : 0;
    // SNP_OPT_UNIT_SCRATCH: the slots the partial sums hold, at most one per unit (the default size keeps [J][2][N_local])
    const long long cap = partial_bytes / unit_bytes(sizeof(T));
    la.cap = la.use_list && units >= 0 ? (int)(cap < blocks * la.J ? cap : blocks * la.J) : 0;
    const long long per_block = (long long)kTile * la.apt;
    la.env_iblocks = (int)((env_n + per_block - 1) / per_block);
    la.env_fblocks = (int)large_iblocks(env_n);
    return batch ? dispatch_large<T, true>(o->type, la, units >= 0, sub == 0, st) : dispatch_large<T, false>(o->type, la, units >= 0, sub == 0, st);
}

// After the last sub-step of a call: the robot's end state (robot_mode 1 / 3; the finish kernels of the call read the start state
// until they are done) and the clock, advanced by dt per sub-step as k_step does.  One thread (per env in a batch).
template <typename T, bool kBatch> __global__ void k_large_robot_end(const KArgs<T> a, int n_substeps) {
    int e = 0;
    long long RE = 1;
    if constexpr (kBatch) {
        e = blockIdx.x * blockDim.x + threadIdx.x; RE = a.E;
        if (e >= a.E) return;
    }
    if (a.robot && (a.robot_mode == 1 || a.robot_mode == 3)) {
        T rb[SNP_ROBOT_FIELDS];
        large_robot_replay<T, kBatch>(a, n_substeps, rb, e);
        a.robot[SNP_ROBOT_PX * RE + e] = rb[SNP_ROBOT_PX]; a.robot[SNP_ROBOT_PY * RE + e] = rb[SNP_ROBOT_PY];
        a.robot[SNP_ROBOT_VX * RE + e] = rb[SNP_ROBOT_VX]; a.robot[SNP_ROBOT_VY * RE + e] = rb[SNP_ROBOT_VY];
        a.robot[SNP_ROBOT_TH * RE + e] = rb[SNP_ROBOT_TH];
    }
    if (a.time_now) {
        double t = a.time_now[e];
        for (int s = 0; s < n_substeps; ++s) t = __dadd_rn(t, a.dt_d);
        a.time_now[e] = t;
    }
}

template <typename T, bool kBatch> int launch_large_robot_end(const snp_crowd *c, const snp_step_opts *o, int n_substeps, cudaStream_t st) {
    KArgs<T> a{};
    a.E = c->E; a.robot = (T *)c->robot; a.action = (const T *)o->action; a.robot_mode = o->robot_mode;
    a.dt = (T)o->dt; a.dt_d = o->dt; a.time_now = o->time_now;
    if (kBatch) k_large_robot_end<T, true><<<(unsigned)((c->E + 127) / 128), 128, 0, st>>>(a, n_substeps);
    else k_large_robot_end<T, false><<<1, 1, 0, st>>>(a, n_substeps);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

// ---- snp_large_checks: the robot against M humans of a view (social_nav_sim.py:949-1029, social_nav_gym.py:107-118) ----
// One CTA.  Thread t scans the contiguous run [t * per, (t + 1) * per) in index order; the runs are combined in index order (a shuffle
// tree that only ever puts a run's summary to the LEFT of the next one's, then the same over the warps), so the result is that of
// the reference's sequential loop: the swept test stops at the first colliding human and dmin is the minimum over the humans before
// it, the first of equal minima kept ('<'), NaN distances never taken.
constexpr int kCheckThreads = 1024;

// E envs of M humans (one crowd: E = 1), view [5][stride = E M], radius [E M]; clear: start from zero flags and checks.
template <typename T> struct CheckArgs {
    const T *robot, *action, *view, *radius;
    long long M, stride;
    int E, mode, pre, post, clear;
    double consts[6];
    const double *time_now;
    int *flags;
    double *checks;
};

// (dmin, hit) of a run on the left combined with the run on its right
__device__ __forceinline__ void swept_combine(double &dmin, int &hit, double dmin_r, int hit_r) {
    if (hit) return;
    dmin = dmin_r < dmin ? dmin_r : dmin;
    hit = hit_r;
}

// One CTA per env (blockIdx.x = env).
template <typename T> __global__ void __launch_bounds__(kCheckThreads) k_large_checks(const CheckArgs<T> c) {
    __shared__ double s_dmin[kCheckThreads / 32], s_admin[kCheckThreads / 32];
    __shared__ int s_hit[kCheckThreads / 32];
    const int env = blockIdx.x;
    const long long RE = c.E, stride = c.stride;
    const T *rbt = c.robot + env;
    const T rpx = rbt[SNP_ROBOT_PX * RE], rpy = rbt[SNP_ROBOT_PY * RE], rr = rbt[SNP_ROBOT_R * RE], rgx = rbt[SNP_ROBOT_GX * RE], rgy = rbt[SNP_ROBOT_GY * RE];
    T ax = T(0), ay = T(0);
    if (c.pre) {
        ax = c.action[env]; ay = c.action[RE + env];
        if (c.mode == 3) {  // unicycle action (v, r): the swept test and the goal test use v (cos, sin)(yaw + r) (sim:973)
            const double uv = (double)ax, ur = (double)ay;
            double sn_, cs_;
            sincos((double)rbt[SNP_ROBOT_TH * RE] + ur, &sn_, &cs_);
            ax = (T)__dmul_rn(uv, cs_); ay = (T)__dmul_rn(uv, sn_);
        }
    }
    const long long M = c.M, per = (M + kCheckThreads - 1) / kCheckThreads;
    const long long b = (long long)threadIdx.x * per, e = min(M, b + per);
    const T *view = c.view + env * M, *radius = c.radius + env * M;
    const T *px = view, *py = view + stride, *vx = view + 2 * stride, *vy = view + 3 * stride;
    double dmin = CUDART_INF, admin = 10000.0;
    int hit = 0;
    if (c.pre)
        for (long long k = b; k < e; ++k) {
            const double cd = swept_distance((double)px[k], (double)py[k], (double)vx[k], (double)vy[k], (double)radius[k], (double)rpx, (double)rpy,
                                             (double)rr, (double)ax, (double)ay, c.consts[5]);
            if (cd < 0) { hit = 1; break; }
            else if (cd < dmin) dmin = cd;
        }
    if (c.post)
        for (long long k = b; k < e; ++k) {
            double d = __dsub_rn(__dsub_rn(xnorm_np(__dsub_rn((double)px[k], (double)rpx), __dsub_rn((double)py[k], (double)rpy)), (double)radius[k]), (double)rr);
            if (!(d < 10000.0)) d = 10000.0;
            admin = d < admin ? d : admin;
        }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int off = 1; off < 32; off <<= 1) {  // lane l ends up with the runs of lanes [l, l + 2 off) in order
        const double dr = __shfl_down_sync(0xffffffffu, dmin, off), ar = __shfl_down_sync(0xffffffffu, admin, off);
        const int hr = __shfl_down_sync(0xffffffffu, hit, off);
        if (lane + off < 32) { swept_combine(dmin, hit, dr, hr); admin = ar < admin ? ar : admin; }
    }
    if (lane == 0) { s_dmin[warp] = dmin; s_admin[warp] = admin; s_hit[warp] = hit; }
    __syncthreads();
    if (threadIdx.x != 0) return;
    dmin = CUDART_INF; admin = 10000.0; hit = 0;
    for (int w = 0; w < kCheckThreads / 32; ++w) { swept_combine(dmin, hit, s_dmin[w], s_hit[w]); admin = s_admin[w] < admin ? s_admin[w] : admin; }
    int *flags = c.flags + env;
    double *checks = c.checks ? c.checks + 4 * env : nullptr;
    int f = *flags;
    if (c.clear) {
        f = 0;
        if (checks) checks[0] = checks[1] = checks[2] = checks[3] = 0.0;
    }
    if (c.pre) {
        const double endx = __dadd_rn((double)rpx, __dmul_rn((double)ax, c.consts[5]));
        const double endy = __dadd_rn((double)rpy, __dmul_rn((double)ay, c.consts[5]));
        const bool goal = xnorm_np(__dsub_rn(endx, (double)rgx), __dsub_rn(endy, (double)rgy)) < (double)rr;
        const double tnow = c.time_now ? c.time_now[env] : 0.0;
        double reward;
        bool term, trunc;
        const int code = reward_and_info(hit != 0, dmin, goal, tnow, c.consts, reward, term, trunc);
        f &= ~(SNP_FLAG_COLLISION | SNP_FLAG_REACHING_GOAL | SNP_FLAG_TERMINATED | SNP_FLAG_TRUNCATED | (7 << SNP_FLAG_INFO_SHIFT));
        f |= (hit ? SNP_FLAG_COLLISION : 0) | (goal ? SNP_FLAG_REACHING_GOAL : 0) | (term ? SNP_FLAG_TERMINATED : 0) | (trunc ? SNP_FLAG_TRUNCATED : 0) |
             (code << SNP_FLAG_INFO_SHIFT);
        if (checks) { checks[0] = dmin; checks[1] = reward; }
    }
    if (c.post) {
        const bool agoal = xnorm_np(__dsub_rn((double)rpx, (double)rgx), __dsub_rn((double)rpy, (double)rgy)) < (double)rr;
        f &= ~(SNP_FLAG_ACTUAL_COLLISION | SNP_FLAG_ACTUAL_GOAL);
        f |= (admin <= 0.0 ? SNP_FLAG_ACTUAL_COLLISION : 0) | (agoal ? SNP_FLAG_ACTUAL_GOAL : 0);
        if (checks) checks[2] = admin;
    }
    *flags = f;
}

// E envs of M humans each, the checks selected by pre / post; `clear` zeroes each env's flags and checks first.
template <typename T> int launch_large_checks(const snp_crowd *cr, const snp_step_opts *o, const void *view, const void *radius, int E, long long M,
                                              cudaStream_t st, bool pre = true, bool post = true, bool clear = false) {
    CheckArgs<T> c;
    c.robot = (const T *)cr->robot; c.action = (const T *)o->action; c.view = (const T *)view; c.radius = (const T *)radius;
    c.M = M; c.stride = (long long)E * M; c.E = E; c.clear = clear;
    c.mode = o->robot_mode; c.pre = pre && o->pre_checks != 0; c.post = post && o->post_checks != 0;
    for (int k = 0; k < 6; ++k) c.consts[k] = o->consts[k];
    c.time_now = o->time_now; c.flags = o->flags; c.checks = o->checks;
    k_large_checks<T><<<(unsigned)E, kCheckThreads, 0, st>>>(c);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

// snp_large_batch_step after validation: publish, pre-checks, n_substeps x (robot step, tiled update) between the two view buffers of
// the scratch, the robot's end state and the clock, post-checks.
template <typename T> int large_batch_step(const snp_crowd *c, const snp_step_opts *o, void *scratch, long long units, cudaStream_t st) {
    const long long E = c->E, N = c->N, EN = E * N;
    const LargeBatchScratch sb = large_batch_scratch(E, N, sizeof(T), units);
    void *views[2] = {(char *)scratch + sb.view_a, (char *)scratch + sb.view_b};
    k_large_publish<T><<<(unsigned)((EN + 255) / 256), 256, 0, st>>>((const T *)c->dyn, (const T *)c->stat, EN, o->type >= 3, (T *)views[0], EN, 0);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    const T *radius = (const T *)c->stat + SNP_STAT_R * EN;
    if (o->pre_checks) {
        const int rc = launch_large_checks<T>(c, o, views[0], radius, c->E, N, st, true, false, true);
        if (rc) return rc;
    }
    // the finish kernel writes the next view's tile boxes when its CTAs are whole tiles (LargeCrowd's rule)
    const bool fold_boxes = N % kTile == 0;
    for (int s = 0; s < o->n_substeps; ++s) {
        const void *next[1] = {views[(s + 1) & 1]};
        const int rc = run_large<T>(c, o, views[s & 1], next, 1, EN, 0, fold_boxes, fold_boxes && s > 0, scratch, s, st, units, N);
        if (rc) return rc;
    }
    if (o->n_substeps > 0 && ((c->robot && (o->robot_mode == 1 || o->robot_mode == 3)) || o->time_now)) {
        const int rc = launch_large_robot_end<T, true>(c, o, o->n_substeps, st);
        if (rc) return rc;
    }
    if (o->post_checks) return launch_large_checks<T>(c, o, views[o->n_substeps & 1], radius, c->E, N, st, false, true, !o->pre_checks);
    return SNP_OK;
}

}  // namespace
}  // namespace snp

using namespace snp;

extern "C" {

int64_t snp_large_scratch_bytes(int64_t n_local, int64_t M, int32_t dtype) {
    return large_scratch(n_local, M, dtype == SNP_F64 ? 8 : 4).bytes;
}

int64_t snp_large_scratch_bytes_units(int64_t n_local, int64_t M, int32_t dtype, int64_t units) {
    if (n_local < 1 || M < n_local || units < 0 || (dtype != SNP_F64 && dtype != SNP_F32)) {
        set_error("snp_large_scratch_bytes_units: n_local=%lld M=%lld dtype=%d units=%lld", (long long)n_local, (long long)M, dtype, (long long)units);
        return -1;
    }
    return large_scratch(n_local, M, dtype == SNP_F64 ? 8 : 4, units).bytes;
}

// SNP_OPT_UNIT_SCRATCH: the refusals of a step whose partial sums are slots of the work list (`what` names the entry point), or SNP_OK.
static int unit_scratch_refusals(const char *what, const snp_crowd *c, const snp_step_opts *o, long long self_offset, long long blocks, long long J) {
    if (o->type % 3 == 2) { set_error("%s: SNP_OPT_UNIT_SCRATCH: Moussaid's pair law (type %d) is never culled and needs the default scratch", what, o->type); return SNP_ERR_UNSUPPORTED; }
    if (o->reserved & SNP_OPT_NO_CULLING) { set_error("%s: SNP_OPT_UNIT_SCRATCH with SNP_OPT_NO_CULLING: every unit is evaluated, use the default scratch", what); return SNP_ERR_UNSUPPORTED; }
    if (self_offset % kTile) { set_error("%s: SNP_OPT_UNIT_SCRATCH needs a slice starting on a 128-entity tile (self_offset %lld)", what, self_offset); return SNP_ERR_UNSUPPORTED; }
    if (blocks * J >= (1LL << 31)) { set_error("%s: SNP_OPT_UNIT_SCRATCH: %lld units exceed the int32 unit index", what, blocks * J); return SNP_ERR_UNSUPPORTED; }
    if (!large_uses_list(c, o, self_offset, blocks, J)) { set_error("%s: SNP_OPT_UNIT_SCRATCH: these pair-law parameters have no culling distance", what); return SNP_ERR_UNSUPPORTED; }
    return SNP_OK;
}

int snp_large_run_p2p(const snp_crowd *c, const snp_step_opts *o, const void *const *peer_views_a, const void *const *peer_views_b,
                      int32_t first_is_b, int64_t M, int64_t self_offset, int32_t world, int32_t rank, const void *const *peer_flags,
                      uint64_t epoch_base, int32_t n_substeps, int32_t *error_flag, void *scratch, int64_t scratch_bytes, void *stream) {
    if (!c || !o || !peer_views_a || !peer_views_b || !peer_flags || !error_flag || !scratch) { set_error("snp_large_run_p2p: null argument"); return SNP_ERR_INVALID; }
    if (world < 1 || world > 8 || rank < 0 || rank >= world) { set_error("snp_large_run_p2p: 1..8 ranks (got world %d rank %d)", world, rank); return SNP_ERR_INVALID; }
    if (!c->dyn || !c->stat || !c->goals || !c->goal_idx || !c->goal_cnt) { set_error("snp_large_run_p2p: crowd arrays missing"); return SNP_ERR_INVALID; }
    if (c->agent_params || c->walls_per_env) { set_error("snp_large_run_p2p: uniform parameters and one wall set only"); return SNP_ERR_UNSUPPORTED; }
    if (c->dtype != SNP_F64 && c->dtype != SNP_F32) { set_error("bad dtype %d", c->dtype); return SNP_ERR_INVALID; }
    // the robot of SocialNavGym.step: fixed (0), holonomic (1) or unicycle (3), visible or not; the checks are a call of their own
    if (o->robot_mode < 0 || o->robot_mode > 3) { set_error("snp_large_run_p2p: robot_mode must be 0, 1 or 3 (got %d)", o->robot_mode); return SNP_ERR_INVALID; }
    if (o->robot_mode == 2) { set_error("snp_large_run_p2p: robot_mode 2 (a robot moved by its own motion model) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->track_touch) { set_error("snp_large_run_p2p: track_touch is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->pre_checks || o->post_checks) { set_error("snp_large_run_p2p: run the collision / goal checks with snp_large_checks"); return SNP_ERR_UNSUPPORTED; }
    if (o->dyn_out) { set_error("snp_large_run_p2p: dyn_out (peek) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->respawn) { set_error("snp_large_run_p2p: respawn is not supported"); return SNP_ERR_UNSUPPORTED; }
    if ((o->consider_robot || o->robot_mode) && !c->robot) { set_error("snp_large_run_p2p: consider_robot / robot_mode need crowd->robot"); return SNP_ERR_INVALID; }
    if (o->robot_mode && !o->action) { set_error("snp_large_run_p2p: robot_mode %d needs opts->action", o->robot_mode); return SNP_ERR_INVALID; }
    const long long N = (long long)c->E * c->N;
    if (self_offset < 0 || self_offset + N > M) { set_error("snp_large_run_p2p: M=%lld offset=%lld N=%lld", (long long)M, (long long)self_offset, N); return SNP_ERR_INVALID; }
    const int w = c->dtype == SNP_F64 ? 8 : 4;
    const bool unit_scratch = (o->reserved & SNP_OPT_UNIT_SCRATCH) != 0;
    if (unit_scratch) {
        const int rc = unit_scratch_refusals("snp_large_run_p2p", c, o, self_offset, large_iblocks(N), large_J(M));
        if (rc) return rc;
    }
    const long long need = large_scratch(N, M, w, unit_scratch ? 0 : -1).bytes;  // with the bit: the size for no slot at all
    const long long units = unit_scratch ? units_in(scratch_bytes, need, w) : -1;
    if (scratch_bytes < need || reinterpret_cast<uintptr_t>(scratch) % 16) {
        set_error("snp_large_run_p2p: 16-byte aligned scratch of %lld bytes needed, %lld given", need, (long long)scratch_bytes);
        return SNP_ERR_INVALID;
    }
    // The producers write the next view's tile boxes only when together they write every tile of it: this slice is a whole number
    // of tiles and the `world` slices make up the view.  Otherwise every sub-step recomputes the boxes of the view it reads.
    const bool fold_boxes = self_offset % kTile == 0 && N % kTile == 0 && world * N == M;
    cudaStream_t st = (cudaStream_t)stream;
    BarrierArgs b;
    for (int p = 0; p < 8; ++p) b.flags[p] = p < world ? (unsigned long long *)peer_flags[p] : nullptr;
    b.world = world; b.rank = rank; b.error = error_flag;
    int cur_is_b = first_is_b ? 1 : 0;
    for (int s = 0; s < n_substeps; ++s) {
        const void *const *cur = cur_is_b ? peer_views_b : peer_views_a, *const *nxt = cur_is_b ? peer_views_a : peer_views_b;
        const bool boxes_ready = fold_boxes && s > 0;  // sub-step 0 computes the tile boxes of the view it was handed
        const int rc = c->dtype == SNP_F64 ? run_large<double>(c, o, cur[rank], nxt, world, M, self_offset, fold_boxes, boxes_ready, scratch, s, st, units)
                                           : run_large<float>(c, o, cur[rank], nxt, world, M, self_offset, fold_boxes, boxes_ready, scratch, s, st, units);
        if (rc) return rc;
        if (world > 1) {
            b.epoch = epoch_base + (unsigned long long)s + 1;
            k_rank_barrier<<<1, 32, 0, st>>>(b);
            count_launch();
            SNP_CUDA_OK(cudaGetLastError());
        }
        cur_is_b ^= 1;
    }
    // the robot's end state and the clock: after every finish kernel of the call has read the start state
    if (n_substeps > 0 && ((c->robot && (o->robot_mode == 1 || o->robot_mode == 3)) || o->time_now))
        return c->dtype == SNP_F64 ? launch_large_robot_end<double, false>(c, o, n_substeps, st) : launch_large_robot_end<float, false>(c, o, n_substeps, st);
    return SNP_OK;
}

int snp_large_checks(const snp_crowd *c, const snp_step_opts *o, const void *view, const void *radius, int64_t M, void *stream) {
    if (!c || !o || !view || !radius) { set_error("snp_large_checks: null argument"); return SNP_ERR_INVALID; }
    if (c->dtype != SNP_F64 && c->dtype != SNP_F32) { set_error("snp_large_checks: bad dtype %d", c->dtype); return SNP_ERR_INVALID; }
    if (M < 1) { set_error("snp_large_checks: M must be >= 1 (got %lld)", (long long)M); return SNP_ERR_INVALID; }
    if (!c->robot) { set_error("snp_large_checks: crowd->robot is required"); return SNP_ERR_INVALID; }
    if (!o->pre_checks && !o->post_checks) { set_error("snp_large_checks: neither pre_checks nor post_checks is set"); return SNP_ERR_INVALID; }
    if (o->post_checks != 0 && o->post_checks != 1) { set_error("snp_large_checks: post_checks 2 (imitation-learning reward) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->robot_mode != 0 && o->robot_mode != 1 && o->robot_mode != 3) { set_error("snp_large_checks: robot_mode must be 0, 1 or 3 (got %d)", o->robot_mode); return SNP_ERR_INVALID; }
    if (o->pre_checks && !o->action) { set_error("snp_large_checks: pre_checks needs opts->action"); return SNP_ERR_INVALID; }
    if (!o->flags) { set_error("snp_large_checks: opts->flags is required"); return SNP_ERR_INVALID; }
    return c->dtype == SNP_F64 ? launch_large_checks<double>(c, o, view, radius, 1, M, (cudaStream_t)stream)
                               : launch_large_checks<float>(c, o, view, radius, 1, M, (cudaStream_t)stream);
}

int64_t snp_large_batch_scratch_bytes(int32_t E, int32_t N, int32_t dtype) {
    if (E < 1 || N < 1 || (dtype != SNP_F64 && dtype != SNP_F32)) { set_error("snp_large_batch_scratch_bytes: E=%d N=%d dtype=%d", E, N, dtype); return -1; }
    return large_batch_scratch(E, N, dtype == SNP_F64 ? 8 : 4).bytes;
}

int64_t snp_large_batch_scratch_bytes_units(int32_t E, int32_t N, int32_t dtype, int64_t units) {
    if (E < 1 || N < 1 || units < 0 || (dtype != SNP_F64 && dtype != SNP_F32)) {
        set_error("snp_large_batch_scratch_bytes_units: E=%d N=%d dtype=%d units=%lld", E, N, dtype, (long long)units);
        return -1;
    }
    return large_batch_scratch(E, N, dtype == SNP_F64 ? 8 : 4, units).bytes;
}

int snp_large_batch_step(const snp_crowd *c, const snp_step_opts *o, void *scratch, int64_t scratch_bytes, void *stream) {
    if (!c || !o || !scratch) { set_error("snp_large_batch_step: null argument"); return SNP_ERR_INVALID; }
    if (c->E < 1 || c->N < 1 || c->G < 1) { set_error("snp_large_batch_step: E, N and G must be positive (E=%d N=%d G=%d)", c->E, c->N, c->G); return SNP_ERR_INVALID; }
    if (c->dtype != SNP_F64 && c->dtype != SNP_F32) { set_error("snp_large_batch_step: bad dtype %d", c->dtype); return SNP_ERR_INVALID; }
    if (o->type < 0 || o->type > 8) { set_error("snp_large_batch_step: type %d does not exist for this implementation", o->type); return SNP_ERR_INVALID; }
    if (!c->dyn || !c->stat || !c->goals || !c->goal_idx || !c->goal_cnt) { set_error("snp_large_batch_step: crowd arrays missing"); return SNP_ERR_INVALID; }
    if (c->W < 0 || c->S < 0 || (c->W > 0 && (!c->walls || c->S == 0))) { set_error("snp_large_batch_step: walls W=%d S=%d but no segment array", c->W, c->S); return SNP_ERR_INVALID; }
    if (o->n_substeps < 0) { set_error("snp_large_batch_step: n_substeps must be >= 0"); return SNP_ERR_INVALID; }
    if (o->robot_mode < 0 || o->robot_mode > 3) { set_error("snp_large_batch_step: robot_mode must be 0, 1 or 3 (got %d)", o->robot_mode); return SNP_ERR_INVALID; }
    if (large_J(c->N) > 65535) { set_error("snp_large_batch_step: at most %d humans per env", 65535 * kChunk); return SNP_ERR_INVALID; }
    if (o->robot_mode == 2) { set_error("snp_large_batch_step: robot_mode 2 (a robot moved by its own motion model) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->robot_every) { set_error("snp_large_batch_step: robot_every is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->track_touch) { set_error("snp_large_batch_step: track_touch is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->post_checks != 0 && o->post_checks != 1) { set_error("snp_large_batch_step: post_checks 2 (imitation-learning reward) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->dyn_out) { set_error("snp_large_batch_step: dyn_out (peek) is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (o->respawn) { set_error("snp_large_batch_step: respawn is not supported"); return SNP_ERR_UNSUPPORTED; }
    if (c->agent_params) { set_error("snp_large_batch_step: per-agent parameter rows are not supported (uniform parameters only)"); return SNP_ERR_UNSUPPORTED; }
    if ((o->consider_robot || o->robot_mode || o->pre_checks || o->post_checks) && !c->robot) {
        set_error("snp_large_batch_step: consider_robot, robot_mode and the checks need crowd->robot"); return SNP_ERR_INVALID;
    }
    if ((o->robot_mode || o->pre_checks) && !o->action) { set_error("snp_large_batch_step: robot_mode 1 / 3 and pre_checks need opts->action"); return SNP_ERR_INVALID; }
    if ((o->pre_checks || o->post_checks) && !o->flags) { set_error("snp_large_batch_step: the checks need opts->flags"); return SNP_ERR_INVALID; }
    const int w = c->dtype == SNP_F64 ? 8 : 4;
    const bool unit_scratch = (o->reserved & SNP_OPT_UNIT_SCRATCH) != 0;
    if (unit_scratch) {
        const int rc = unit_scratch_refusals("snp_large_batch_step", c, o, 0, (long long)c->E * large_iblocks(c->N), large_J(c->N));
        if (rc) return rc;
    }
    const long long need = large_batch_scratch(c->E, c->N, w, unit_scratch ? 0 : -1).bytes;  // with the bit: the size for no slot at all
    if (scratch_bytes < need || reinterpret_cast<uintptr_t>(scratch) % 16) {
        set_error("snp_large_batch_step: 16-byte aligned scratch of %lld bytes needed, %lld given", need, (long long)scratch_bytes);
        return SNP_ERR_INVALID;
    }
    const long long units = unit_scratch ? units_in(scratch_bytes, need, w) : -1;
    return c->dtype == SNP_F64 ? large_batch_step<double>(c, o, scratch, units, (cudaStream_t)stream)
                               : large_batch_step<float>(c, o, scratch, units, (cudaStream_t)stream);
}

int snp_large_publish(const snp_crowd *c, int32_t type, void *view, int64_t stride, int64_t offset, void *stream) {
    if (!c || !view || !c->dyn || !c->stat) { set_error("snp_large_publish: null argument"); return SNP_ERR_INVALID; }
    if (type < 0 || type > 8) { set_error("Type %d does not exist for this implementation", type); return SNP_ERR_INVALID; }
    const long long N = (long long)c->E * c->N;
    const unsigned blocks = (unsigned)((N + 255) / 256);
    if (c->dtype == SNP_F64) k_large_publish<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double *)c->dyn, (const double *)c->stat, N, type >= 3, (double *)view, stride, offset);
    else k_large_publish<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float *)c->dyn, (const float *)c->stat, N, type >= 3, (float *)view, stride, offset);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

int snp_large_tile_boxes(void *view, int64_t M, int32_t dtype, void *stream) {
    if (!view) { set_error("snp_large_tile_boxes: null argument"); return SNP_ERR_INVALID; }
    if (M < 1) { set_error("snp_large_tile_boxes: M must be >= 1 (got %lld)", (long long)M); return SNP_ERR_INVALID; }
    if (dtype != SNP_F64 && dtype != SNP_F32) { set_error("snp_large_tile_boxes: bad dtype %d", dtype); return SNP_ERR_INVALID; }
    const unsigned n_tiles = (unsigned)((M + kTile - 1) / kTile);
    if (dtype == SNP_F64) k_tile_boxes<double, false><<<n_tiles, kTile, 0, (cudaStream_t)stream>>>((const double *)view, M, (double *)view + 5 * M, 0, 0);
    else k_tile_boxes<float, false><<<n_tiles, kTile, 0, (cudaStream_t)stream>>>((const float *)view, M, (float *)view + 5 * M, 0, 0);
    count_launch();
    SNP_CUDA_OK(cudaGetLastError());
    return SNP_OK;
}

}  // extern "C"
