// mapf_env_kernels.cu — the environment hot path as hand-written CUDA for sm_100a.
//
//   (K1+K2, the fused step + observe kernel, lives in mapf_step_kernels.cu)
//   K3     bfs_navi_kernel       Environment.get_navi_map (environment.py:217-276): bit-parallel
//                                wavefront BFS, one warp per (env, agent), lane = map row.
//   pack / unpack helpers        Environment.load (environment.py:198-215) and attribute reads.
//
// None of this is a dense contraction: no tensor cores.  K1+K2 is bound by the HBM write of the
// observation bytes (486 B per agent-step); everything else stays in shared memory / registers.
#include <type_traits>

#include "mapf_bfs_device.cuh"
#include "mapf_common.cuh"

namespace {

constexpr int kBfsWarps = 4;

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// ---------------------------------------------------------------------------------------------
// pack: u8 maps -> padded obstacle bitmaps; copy coordinates; steps = 0      (environment.py:198-215)
// SIZED: instance i has in_n[i] agents on an in_l[i] map (NULL: N and L); map cells outside it and agent rows beyond it are
// ignored -- the bitmap is zero there, the rows read 255 -- and the slot's sizes are recorded.
// ---------------------------------------------------------------------------------------------
template <bool SIZED>
__device__ __forceinline__ void pack_load_body(const EnvDims &d, const int32_t *__restrict__ env_ids, int n, const uint8_t *__restrict__ maps,
                                               const uint8_t *__restrict__ agents, const uint8_t *__restrict__ goals,
                                               uint32_t *__restrict__ obst, uint8_t *__restrict__ pos, uint8_t *__restrict__ goal,
                                               int32_t *__restrict__ steps, int32_t *__restrict__ err, const uint8_t *in_n = nullptr,
                                               const uint8_t *in_l = nullptr, uint8_t *sz_n = nullptr, uint8_t *sz_l = nullptr)
{
    int i = blockIdx.x;
    if (i >= n) return;
    int e = env_ids ? env_ids[i] : i;
    if (e < 0 || e >= d.B) {  // a slot id outside the batch: nothing is written (the reference would raise IndexError)
        if (threadIdx.x == 0) atomicOr(err, MAPF_ERRBIT_STATE);
        return;
    }
    const int NA = SIZED && in_n ? (int)in_n[i] : d.N, LM = SIZED && in_l ? (int)in_l[i] : d.L;
    const uint8_t *m = maps + (size_t)i * d.L * d.L;
    uint32_t *o = obst + (size_t)e * d.obst_stride;
    for (int w = threadIdx.x; w < d.obst_stride; w += blockDim.x) {
        int row = w / d.RWS, ww = w - row * d.RWS;
        uint32_t bits = 0;
        int x = row - 4;
        if (row < d.R && ww < d.RW && x >= 0 && x < LM) {
            for (int b = 0; b < 32; ++b) {
                int y = ww * 32 + b - 4;
                if (y >= 0 && y < LM && m[x * d.L + y] != 0) bits |= 1u << b;
            }
        }
        o[w] = bits;
    }
    for (int k = threadIdx.x; k < 2 * d.N; k += blockDim.x) {
        const bool present = !SIZED || k < 2 * NA;
        pos[(size_t)e * 2 * d.N + k] = present ? agents[(size_t)i * 2 * d.N + k] : (uint8_t)255;
        goal[(size_t)e * 2 * d.N + k] = present ? goals[(size_t)i * 2 * d.N + k] : (uint8_t)255;
    }
    if (threadIdx.x == 0) {
        steps[e] = 0;
        if constexpr (SIZED) sz_n[e] = (uint8_t)NA, sz_l[e] = (uint8_t)LM;
    }
}

__global__ void pack_load_kernel(EnvDims d, const int32_t *__restrict__ env_ids, int n, const uint8_t *__restrict__ maps,
                                 const uint8_t *__restrict__ agents, const uint8_t *__restrict__ goals,
                                 uint32_t *__restrict__ obst, uint8_t *__restrict__ pos, uint8_t *__restrict__ goal,
                                 int32_t *__restrict__ steps, int32_t *__restrict__ err)
{
    pack_load_body<false>(d, env_ids, n, maps, agents, goals, obst, pos, goal, steps, err);
}

__global__ void pack_load_sized_kernel(EnvDims d, const int32_t *__restrict__ env_ids, int n, const uint8_t *__restrict__ maps,
                                       const uint8_t *__restrict__ agents, const uint8_t *__restrict__ goals,
                                       uint32_t *__restrict__ obst, uint8_t *__restrict__ pos, uint8_t *__restrict__ goal,
                                       int32_t *__restrict__ steps, int32_t *__restrict__ err, const uint8_t *__restrict__ in_n,
                                       const uint8_t *__restrict__ in_l, uint8_t *__restrict__ sz_n, uint8_t *__restrict__ sz_l)
{
    pack_load_body<true>(d, env_ids, n, maps, agents, goals, obst, pos, goal, steps, err, in_n, in_l, sz_n, sz_l);
}

// ---------------------------------------------------------------------------------------------
// state validation after load / set_state: the step kernel indexes shared memory with the coordinates, so a coordinate
// outside the map must never reach it.  Out-of-range coordinates are clamped into the map and latched as
// MAPF_ERRBIT_STATE (the reference raises IndexError on the same input); two agents on one cell are latched as
// MAPF_ERRBIT_UNIQUE (the reference raises RuntimeError('unique') at the next step, environment.py:424-428).
// One warp per environment.  SIZED: against the slot's own side, over its present agents; absent rows are set to 255.
// ---------------------------------------------------------------------------------------------
template <bool SIZED>
__device__ __forceinline__ void validate_state_body(const EnvDims &d, const int32_t *__restrict__ env_ids, int n, uint8_t *__restrict__ pos,
                                                    uint8_t *__restrict__ goal, int32_t *__restrict__ err,
                                                    const uint8_t *sz_n = nullptr, const uint8_t *sz_l = nullptr)
{
    const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (i >= n) return;
    const int lane = threadIdx.x & 31;
    const int e = env_ids ? env_ids[i] : i;
    if (e < 0 || e >= d.B) return;  // latched by pack_load_kernel
    const int NA = SIZED ? (int)sz_n[e] : d.N, LM = SIZED ? (int)sz_l[e] : d.L;
    uchar2 *pp = reinterpret_cast<uchar2 *>(pos) + (size_t)e * d.N;
    uchar2 *gg = reinterpret_cast<uchar2 *>(goal) + (size_t)e * d.N;
    bool bad = false;
    for (int a = lane; a < d.N; a += 32) {
        if (SIZED && a >= NA) {
            pp[a] = gg[a] = make_uchar2(255, 255);
            continue;
        }
        uchar2 p = pp[a], g = gg[a];
        if (p.x >= LM || p.y >= LM) {
            bad = true;
            p.x = min((int)p.x, LM - 1), p.y = min((int)p.y, LM - 1);
            pp[a] = p;
        }
        if (g.x >= LM || g.y >= LM) {
            bad = true;
            g.x = min((int)g.x, LM - 1), g.y = min((int)g.y, LM - 1);
            gg[a] = g;
        }
    }
    __syncwarp();
    bool dup = false;
    for (int a = lane; a < NA; a += 32) {
        const uchar2 p = pp[a];
        for (int b = 0; b < a; ++b) {
            const uchar2 q = pp[b];
            if (q.x == p.x && q.y == p.y) dup = true;
        }
    }
    bad = __any_sync(MAPF_FULL_MASK, bad);
    dup = __any_sync(MAPF_FULL_MASK, dup);
    if (lane == 0 && (bad || dup)) atomicOr(err, (bad ? MAPF_ERRBIT_STATE : 0) | (dup ? MAPF_ERRBIT_UNIQUE : 0));
}

__global__ void validate_state_kernel(EnvDims d, const int32_t *__restrict__ env_ids, int n, uint8_t *__restrict__ pos,
                                      uint8_t *__restrict__ goal, int32_t *__restrict__ err)
{
    validate_state_body<false>(d, env_ids, n, pos, goal, err);
}

__global__ void validate_state_sized_kernel(EnvDims d, const int32_t *__restrict__ env_ids, int n, uint8_t *__restrict__ pos,
                                            uint8_t *__restrict__ goal, int32_t *__restrict__ err, const uint8_t *__restrict__ sz_n,
                                            const uint8_t *__restrict__ sz_l)
{
    validate_state_body<true>(d, env_ids, n, pos, goal, err, sz_n, sz_l);
}

// ---------------------------------------------------------------------------------------------
// K3: bit-parallel wavefront BFS (environment.py:217-276): one warp per APW agents, see mapf_bfs_device.cuh
// ---------------------------------------------------------------------------------------------
template <int RW, int RPL, int APW>
__global__ void __launch_bounds__(kBfsWarps * 32, RW * RPL <= 9 ? 8 : 1)  // <= 64 registers (32 resident warps per SM)
                                                                          // wherever that does not spill
bfs_navi_kernel(EnvDims d, const int32_t *__restrict__ env_ids, const uint8_t *__restrict__ env_mask, int n,
                const uint32_t *__restrict__ obst, const uint8_t *__restrict__ goal, uint32_t *__restrict__ navi,
                uint32_t *__restrict__ navi_alt, const uint8_t *__restrict__ navi_sel, int32_t *__restrict__ dist_out)
{
    constexpr int LW = 32 / APW;
    const int g = (blockIdx.x * kBfsWarps + (threadIdx.x >> 5)) * APW + lane_id() / LW;
    bool alive = g < n * d.N;
    const int i = alive ? g / d.N : 0, a = alive ? g - i * d.N : 0;
    int e = env_ids ? env_ids[i] : i;
    if (e < 0 || e >= d.B) alive = false, e = 0;           // bad slot id: latched by pack_load_kernel
    if (alive && env_mask && !env_mask[e]) alive = false;  // masked re-computation after a device-side reset
    if (!__any_sync(MAPF_FULL_MASK, alive)) return;
    // the slot's live buffer (mapf_common.cuh)
    uint32_t *nv = (navi_alt && navi_sel[e]) ? navi_alt : navi;
    bfs_navi_warp<RW, RPL, APW>(d, e, a, i, alive, obst, goal, nv, dist_out);
}

// The same on a sized handle: the free cells are clipped to the slot's side l_e, and only its n_e present agents search
// (groups of absent agents own no rows and store nothing; a warp with none present leaves).  With dist_out every agent's
// distances are written: an absent agent searches an empty map, so its rows read MAPF_DIST_UNREACHABLE.  The free rows are
// kept in registers (KEEP): the side differs from group to group of a warp.
template <int RW, int RPL, int APW>
__global__ void __launch_bounds__(kBfsWarps * 32, RW * RPL <= 9 ? 8 : 1)
bfs_navi_sized_kernel(EnvDims d, const int32_t *__restrict__ env_ids, const uint8_t *__restrict__ env_mask, int n,
                      const uint32_t *__restrict__ obst, const uint8_t *__restrict__ goal, uint32_t *__restrict__ navi,
                      int32_t *__restrict__ dist_out, const uint8_t *__restrict__ sz_n, const uint8_t *__restrict__ sz_l)
{
    constexpr int LW = 32 / APW;
    const int g = (blockIdx.x * kBfsWarps + (threadIdx.x >> 5)) * APW + lane_id() / LW;
    bool alive = g < n * d.N;
    const int i = alive ? g / d.N : 0, a = alive ? g - i * d.N : 0;
    int e = env_ids ? env_ids[i] : i;
    if (e < 0 || e >= d.B) alive = false, e = 0;           // bad slot id: latched by pack_load_kernel
    if (alive && env_mask && !env_mask[e]) alive = false;  // masked re-computation after a device-side reset
    const bool present = a < (int)sz_n[e];
    if (!dist_out && !present) alive = false;
    if (!__any_sync(MAPF_FULL_MASK, alive)) return;
    EnvDims df = d;  // the free cells: l_e x l_e, none for an absent agent
    df.L = present ? (int)sz_l[e] : 0;
    const uint32_t *ob = obst + (size_t)e * d.obst_stride;
    const uchar2 gg = present ? __ldcg(reinterpret_cast<const uchar2 *>(goal) + (size_t)e * d.N + a) : make_uchar2(0, 0);
    BfsFree<RW, RPL> F;
    bfs_load_free<RW, RPL, APW>(df, ob, F);
    if (dist_out) bfs_navi_search<RW, RPL, APW, false, true, true>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, dist_out);
    else if (d.L < LW * RPL) bfs_navi_search<RW, RPL, APW, true, false, true>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, nullptr);
    else bfs_navi_search<RW, RPL, APW, false, false, true>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, nullptr);
}

// The heuristic maps of the pre-generated NEXT instances of the listed slots (episode handling of mapf_env_rollout): reads
// the staged obstacle bitmaps / goals, writes the buffer the slot's live instance does not use.  The list's length is only
// known on the device, so a fixed grid claims (slot, agent group) items from a counter.
template <int RW, int RPL, int APW>
__global__ void __launch_bounds__(kBfsWarps * 32, RW * RPL <= 9 ? 8 : 4)
pregen_bfs_kernel(EnvDims d, const uint32_t *__restrict__ list, int min_count, unsigned long long *__restrict__ counter,
                  const uint32_t *__restrict__ pg_obst, const uint8_t *__restrict__ pg_goal, uint32_t *__restrict__ navi,
                  uint32_t *__restrict__ navi_alt, const uint8_t *__restrict__ navi_sel, const uint32_t *__restrict__ pg_n,
                  uint32_t *__restrict__ pg_cnt, uint32_t *__restrict__ pg_epi)
{
    constexpr int LW = 32 / APW;
    const int lane = lane_id();
    const unsigned groups = (unsigned)(d.N + APW - 1) / APW;
    if (list[0] < (unsigned)min_count) return;
    const unsigned long long items = (unsigned long long)list[0] * groups;
    for (;;) {
        unsigned long long it = 0;
        if (lane == 0) it = atomicAdd(counter, 1ull);
        it = __shfl_sync(MAPF_FULL_MASK, it, 0);
        if (it >= items) break;
        const unsigned i = (unsigned)(it / groups);
        const int a = (int)(it - (unsigned long long)i * groups) * APW + lane / LW;
        const int e = (int)list[1 + i];
        const bool alive = a < d.N;
        // (the slot's selector only changes when THIS instance is adopted, i.e. after the last group has published it)
        uint32_t *nv = __ldcg(navi_sel + e) ? navi : navi_alt;
        bfs_navi_warp<RW, RPL, APW>(d, e, alive ? a : 0, 0, alive, pg_obst, pg_goal, nv, nullptr);
        __syncwarp();
        if (lane == 0) {
            __threadfence();  // the tiles (and, through the generator's launch, the staged state) before the count
            if (atomicAdd(pg_cnt + e, 1u) + 1u == groups) {
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(pg_epi + e), "r"(__ldcg(pg_n + e)) : "memory");
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// communication mask of the actor-side inference glue                    (model.py:196-208)
//
// comm_mask[i][j] = (|dx| <= obs_radius and |dy| <= obs_radius) and j is among the k nearest agents of i
// (Euclidean, i itself included at distance 0).  torch.topk leaves the order of equal distances
// unspecified; here ties go to the lower agent id (key = d^2 << 8 | j).  One warp per environment,
// lane = agent; positions of the env sit in shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int kCommWarps = 4;

// SIZED: only the n_e present agents take part; rows and columns of absent agents are 0
// PACKED: also writes the mask as packed rows (include/mapf_b200.h) at row bits_rows[e] (NULL: e) of `bits`; `out` is optional
template <bool SIZED, bool PACKED = false>
__device__ __forceinline__ void comm_mask_body(const EnvDims &d, const uint8_t *__restrict__ pos, int k_nearest, uint8_t *__restrict__ out,
                                               const int tid, const uint8_t *sz_n = nullptr, uint8_t *__restrict__ bits = nullptr,
                                               const int64_t *__restrict__ bits_rows = nullptr)
{
    __shared__ uint16_t s_pos[kCommWarps][MAPF_MAX_AGENTS];
    __shared__ uint32_t s_bits[kCommWarps][MAPF_MAX_AGENTS][MAPF_MAX_AGENTS / 32];
    const int lane = tid & 31, warp = tid >> 5;  // (tid read by the kernel, within its launch bounds)
    const int e = blockIdx.x * kCommWarps + warp;
    if (e >= d.B) return;
    const int N = d.N;
    const int NA = SIZED ? (int)sz_n[e] : N;
    for (int a = lane; a < N; a += 32) s_pos[warp][a] = reinterpret_cast<const uint16_t *>(pos)[(size_t)e * N + a];
    __syncwarp();
    if constexpr (SIZED) {
        for (int i = NA + lane; i < N; i += 32)
#pragma unroll
            for (int w = 0; w < MAPF_MAX_AGENTS / 32; ++w) s_bits[warp][i][w] = 0;
    }
    for (int i = lane; i < NA; i += 32) {
        const int xi = s_pos[warp][i] & 0xff, yi = s_pos[warp][i] >> 8;
        // three smallest keys, ascending.  Only agents inside the field of view can end up in the mask, and those lie within
        // d^2 <= 2 r^2; an agent farther away can neither be one nor displace one from the three nearest: start at that bound
        // (the insertion below then runs for the few close agents only)
        constexpr uint32_t kFar = (uint32_t)(2 * MAPF_OBS_RADIUS * MAPF_OBS_RADIUS + 1) << 8;
        uint32_t b0 = kFar, b1 = kFar, b2 = kFar;
        for (int j = 0; j < NA; ++j) {
            const int dx = xi - (s_pos[warp][j] & 0xff), dy = yi - (s_pos[warp][j] >> 8);
            uint32_t key = ((uint32_t)(dx * dx + dy * dy) << 8) | (uint32_t)j;
            if (key < b2) {
                b2 = key;
                if (b2 < b1) { const uint32_t t = b1; b1 = b2; b2 = t; }
                if (b1 < b0) { const uint32_t t = b0; b0 = b1; b1 = t; }
            }
        }
        uint32_t row[MAPF_MAX_AGENTS / 32] = {0, 0, 0, 0};
        const uint32_t best[3] = {b0, b1, b2};
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            if (q < k_nearest && best[q] < kFar) {
                const int j = best[q] & 0xff;
                const int dx = abs(xi - (s_pos[warp][j] & 0xff)), dy = abs(yi - (s_pos[warp][j] >> 8));
                if (dx <= MAPF_OBS_RADIUS && dy <= MAPF_OBS_RADIUS) {
#pragma unroll
                    for (int w = 0; w < MAPF_MAX_AGENTS / 32; ++w)
                        if ((j >> 5) == w) row[w] |= 1u << (j & 31);
                }
            }
        }
#pragma unroll
        for (int w = 0; w < MAPF_MAX_AGENTS / 32; ++w) s_bits[warp][i][w] = row[w];
    }
    __syncwarp();
    if constexpr (PACKED) {
        // byte m of row i = bits 8m .. 8m+7 of the row (bits j >= N are 0)
        const int CW = (N + 7) >> 3;
        uint8_t *ob = bits + (size_t)(bits_rows ? bits_rows[e] : (int64_t)e) * N * CW;
        for (int idx = lane; idx < N * CW; idx += 32) {
            const int i = idx / CW, m = idx - i * CW;
            ob[idx] = (uint8_t)(s_bits[warp][i][m >> 2] >> (8 * (m & 3)));
        }
        if (!out) return;
    }
    uint8_t *o = out + (size_t)e * N * N;
    if ((N & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        // 16 mask bytes (16 consecutive j of one row) per lane and store: bits -> bool bytes as in the observation path
        const int per_row = N >> 4;
        for (int c = lane; c < N * per_row; c += 32) {
            const int i = c / per_row, j0 = (c - i * per_row) << 4;
            const uint32_t b = (s_bits[warp][i][j0 >> 5] >> (j0 & 31)) & 0xffffu;
            uint4 v;
            v.x = ((b & 0xfu) * 0x00204081u) & 0x01010101u;
            v.y = (((b >> 4) & 0xfu) * 0x00204081u) & 0x01010101u;
            v.z = (((b >> 8) & 0xfu) * 0x00204081u) & 0x01010101u;
            v.w = ((b >> 12) * 0x00204081u) & 0x01010101u;
            reinterpret_cast<uint4 *>(o)[c] = v;
        }
    } else {
        for (int idx = lane; idx < N * N; idx += 32) {
            const int i = idx / N, j = idx - i * N;
            o[idx] = (s_bits[warp][i][j >> 5] >> (j & 31)) & 1u;
        }
    }
}

__global__ void __launch_bounds__(kCommWarps * 32)
comm_mask_kernel(EnvDims d, const uint8_t *__restrict__ pos, int k_nearest, uint8_t *__restrict__ out)
{
    comm_mask_body<false>(d, pos, k_nearest, out, threadIdx.x);
}

__global__ void __launch_bounds__(kCommWarps * 32)
comm_mask_sized_kernel(EnvDims d, const uint8_t *__restrict__ pos, int k_nearest, uint8_t *__restrict__ out,
                       const uint8_t *__restrict__ sz_n)
{
    comm_mask_body<true>(d, pos, k_nearest, out, threadIdx.x, sz_n);
}

template <bool SIZED>
__global__ void __launch_bounds__(kCommWarps * 32)
comm_mask_packed_kernel(EnvDims d, const uint8_t *__restrict__ pos, int k_nearest, uint8_t *__restrict__ out,
                        uint8_t *__restrict__ bits, const int64_t *__restrict__ bits_rows, const uint8_t *__restrict__ sz_n)
{
    comm_mask_body<SIZED, true>(d, pos, k_nearest, out, threadIdx.x, sz_n, bits, bits_rows);
}

// ---------------------------------------------------------------------------------------------
// attribute reads: unpack state for parity dumps / drop-in attributes
// ---------------------------------------------------------------------------------------------
__global__ void unpack_map_kernel(EnvDims d, const uint32_t *__restrict__ obst, uint8_t *__restrict__ map_out)
{
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)d.B * d.L * d.L;
    if (idx >= total) return;
    int y = idx % d.L;
    int x = (idx / d.L) % d.L;
    int e = idx / ((size_t)d.L * d.L);
    uint32_t w = obst[(size_t)e * d.obst_stride + (x + 4) * d.RWS + ((y + 4) >> 5)];
    map_out[idx] = (w >> ((y + 4) & 31)) & 1u;
}

// SIZED: absent agents read 0 (their maps are not recomputed once a slot has fewer agents)
template <bool SIZED>
__device__ __forceinline__ void unpack_navi_body(const EnvDims &d, const uint32_t *__restrict__ navi, const uint32_t *__restrict__ navi_alt,
                                                 const uint8_t *__restrict__ navi_sel, uint8_t *__restrict__ navi_out,
                                                 const uint8_t *sz_n = nullptr)
{
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)d.B * d.N * 4 * d.L * d.L;
    if (idx >= total) return;
    int y = idx % d.L;
    int x = (idx / d.L) % d.L;
    int k = (idx / ((size_t)d.L * d.L)) % 4;
    size_t ea = idx / ((size_t)4 * d.L * d.L);
    if constexpr (SIZED) {
        if ((int)(ea % d.N) >= (int)sz_n[ea / d.N]) {
            navi_out[idx] = 0;
            return;
        }
    }
    const int pr = x + 4, pc = y + 4;
    const int bx = min(pr >> 3, d.NB - 1), by = min(pc >> 3, d.NB - 1);
    const uint32_t *live = (navi_alt && navi_sel[ea / d.N]) ? navi_alt : navi;
    const uint2 v = reinterpret_cast<const uint2 *>(live + ea * d.navi_agent_stride)[((size_t)(bx * d.NB + by) << 4) + (pr - 8 * bx)];
    const uint32_t half = k < 2 ? v.x : v.y;
    navi_out[idx] = (half >> (16 * (k & 1) + (pc - 8 * by))) & 1u;
}

__global__ void unpack_navi_kernel(EnvDims d, const uint32_t *__restrict__ navi, const uint32_t *__restrict__ navi_alt,
                                   const uint8_t *__restrict__ navi_sel, uint8_t *__restrict__ navi_out)
{
    unpack_navi_body<false>(d, navi, navi_alt, navi_sel, navi_out);
}

__global__ void unpack_navi_sized_kernel(EnvDims d, const uint32_t *__restrict__ navi, const uint32_t *__restrict__ navi_alt,
                                         const uint8_t *__restrict__ navi_sel, uint8_t *__restrict__ navi_out,
                                         const uint8_t *__restrict__ sz_n)
{
    unpack_navi_body<true>(d, navi, navi_alt, navi_sel, navi_out, sz_n);
}

}  // namespace

// ---- entry points used by mapf_abi.cu -----------------------------------------------------------
int mapf_launch_pack_load(mapf_env *env, const int32_t *d_env_ids, int n, const uint8_t *d_maps,
                          const uint8_t *d_agents, const uint8_t *d_goals, cudaStream_t st)
{
    pack_load_kernel<<<n, 128, 0, st>>>(env->d, d_env_ids, n, d_maps, d_agents, d_goals, env->obst, env->pos, env->goal,
                                        env->steps, env->err);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

// sized handle: d_n / d_l u8[n] per instance (NULL: N and L)
int mapf_launch_pack_load_sized(mapf_env *env, const int32_t *d_env_ids, int n, const uint8_t *d_maps, const uint8_t *d_agents,
                                const uint8_t *d_goals, const uint8_t *d_n, const uint8_t *d_l, cudaStream_t st)
{
    pack_load_sized_kernel<<<n, 128, 0, st>>>(env->d, d_env_ids, n, d_maps, d_agents, d_goals, env->obst, env->pos, env->goal,
                                              env->steps, env->err, d_n, d_l, env->sz_n, env->sz_l);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

// slots env_ids[0..n) (NULL: slots 0..n-1)
int mapf_launch_validate_state(mapf_env *env, const int32_t *d_env_ids, int n, cudaStream_t st)
{
    if (n <= 0) return MAPF_OK;
    if (env->sz_n)
        validate_state_sized_kernel<<<(n + 3) / 4, 128, 0, st>>>(env->d, d_env_ids, n, env->pos, env->goal, env->err, env->sz_n, env->sz_l);
    else
        validate_state_kernel<<<(n + 3) / 4, 128, 0, st>>>(env->d, d_env_ids, n, env->pos, env->goal, env->err);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

// pregen_min >= 0: pregen_bfs_kernel over the list in env->ro_prio (ids / mask / n / dist unused)
template <int RW>
static int launch_bfs_rw(mapf_env *env, const int32_t *ids, const uint8_t *mask, int n, int32_t *dist, int pregen_min, cudaStream_t st)
{
    const bool pregen = pregen_min >= 0;
    const EnvDims &d = env->d;
    // four agents per warp (8 lanes x up to 5 rows each) for two-word maps of up to 40 cells a side, two (16 lanes x up to 6 rows)
    // for every other map of up to 88 cells, else one
    const int apw = d.bfs_apw;
    const int rpl = (d.L + 32 / apw - 1) / (32 / apw);
    const long warps = ((long)n * d.N + apw - 1) / apw;
    const int grid = pregen ? env->num_sms * 8 : (int)((warps + kBfsWarps - 1) / kBfsWarps);
#define MAPF_BFS_LAUNCH(RPL, APW)                                                                                                   \
    do {                                                                                                                            \
        if (pregen)                                                                                                                 \
            pregen_bfs_kernel<RW, RPL, APW><<<grid, kBfsWarps * 32, 0, st>>>(d, env->ro_prio, pregen_min, env->ro_work + 3, env->pg_obst, \
                                                                             env->pg_goal, env->navi, env->navi_alt, env->navi_sel, \
                                                                             env->pg_n, env->pg_cnt, env->pg_epi);                   \
        else if (env->sz_n)                                                                                                         \
            bfs_navi_sized_kernel<RW, RPL, APW><<<grid, kBfsWarps * 32, 0, st>>>(d, ids, mask, n, env->obst, env->goal, env->navi,   \
                                                                                 dist, env->sz_n, env->sz_l);                        \
        else                                                                                                                        \
            bfs_navi_kernel<RW, RPL, APW><<<grid, kBfsWarps * 32, 0, st>>>(d, ids, mask, n, env->obst, env->goal, env->navi,         \
                                                                           env->navi_alt, env->navi_sel, dist);                      \
    } while (0)
    bool ok = true;
    if constexpr (RW == 1) {
        switch (rpl) {
            case 1: MAPF_BFS_LAUNCH(1, 2); break;
            case 2: MAPF_BFS_LAUNCH(2, 2); break;
            default: ok = false;
        }
    } else if constexpr (RW == 2) {
        if (apw == 4) {
            if (rpl <= 4) MAPF_BFS_LAUNCH(4, 4);
            else MAPF_BFS_LAUNCH(5, 4);
        } else {
            switch (rpl) {
                case 2: MAPF_BFS_LAUNCH(2, 2); break;
                case 3: MAPF_BFS_LAUNCH(3, 2); break;
                case 4: MAPF_BFS_LAUNCH(4, 2); break;
                default: ok = false;
            }
        }
    } else if constexpr (RW == 3) {
        switch (rpl) {
            case 4: MAPF_BFS_LAUNCH(4, 2); break;
            case 5: MAPF_BFS_LAUNCH(5, 2); break;
            case 6: MAPF_BFS_LAUNCH(6, 2); break;
            default: ok = false;
        }
    } else {
        switch (rpl) {
            case 3: MAPF_BFS_LAUNCH(3, 1); break;
            case 4: MAPF_BFS_LAUNCH(4, 1); break;
            default: ok = false;
        }
    }
#undef MAPF_BFS_LAUNCH
    if (!ok) {
        mapf_set_error("unsupported map size");
        return MAPF_EINVAL;
    }
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

static int launch_bfs(mapf_env *env, const int32_t *d_env_ids, const uint8_t *d_mask, int n, int32_t *d_dist_out, int pregen_min,
                      cudaStream_t st)
{
    switch (env->d.RW) {
        case 1: return launch_bfs_rw<1>(env, d_env_ids, d_mask, n, d_dist_out, pregen_min, st);
        case 2: return launch_bfs_rw<2>(env, d_env_ids, d_mask, n, d_dist_out, pregen_min, st);
        case 3: return launch_bfs_rw<3>(env, d_env_ids, d_mask, n, d_dist_out, pregen_min, st);
        case 4: return launch_bfs_rw<4>(env, d_env_ids, d_mask, n, d_dist_out, pregen_min, st);
    }
    mapf_set_error("unsupported map size");
    return MAPF_EINVAL;
}

int mapf_launch_bfs(mapf_env *env, const int32_t *d_env_ids, int n, int32_t *d_dist_out, cudaStream_t st)
{
    return launch_bfs(env, d_env_ids, nullptr, n, d_dist_out, -1, st);
}

// all B slots, skipping those whose mask byte is zero (NULL mask = all)
int mapf_launch_bfs_masked(mapf_env *env, const uint8_t *d_mask, cudaStream_t st)
{
    return launch_bfs(env, nullptr, d_mask, env->d.B, nullptr, -1, st);
}

// heuristic maps of the staged next instances listed in env->ro_prio (mapf_launch_pregen, mapf_reset_kernels.cu)
int mapf_launch_pregen_bfs(mapf_env *env, int min_count, cudaStream_t st)
{
    return launch_bfs(env, nullptr, nullptr, 0, nullptr, min_count < 0 ? 0 : min_count, st);
}

int mapf_launch_comm_mask(mapf_env *env, int k_nearest, uint8_t *d_out, cudaStream_t st)
{
    const int grid = (env->d.B + kCommWarps - 1) / kCommWarps;
    if (env->sz_n) comm_mask_sized_kernel<<<grid, kCommWarps * 32, 0, st>>>(env->d, env->pos, k_nearest, d_out, env->sz_n);
    else comm_mask_kernel<<<grid, kCommWarps * 32, 0, st>>>(env->d, env->pos, k_nearest, d_out);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_comm_mask_packed(mapf_env *env, int k_nearest, uint8_t *d_out, uint8_t *d_bits, const int64_t *d_rows, cudaStream_t st)
{
    const int grid = (env->d.B + kCommWarps - 1) / kCommWarps;
    if (env->sz_n) comm_mask_packed_kernel<true><<<grid, kCommWarps * 32, 0, st>>>(env->d, env->pos, k_nearest, d_out, d_bits, d_rows, env->sz_n);
    else comm_mask_packed_kernel<false><<<grid, kCommWarps * 32, 0, st>>>(env->d, env->pos, k_nearest, d_out, d_bits, d_rows, nullptr);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_unpack(mapf_env *env, uint8_t *d_map, uint8_t *d_navi, cudaStream_t st)
{
    const EnvDims &d = env->d;
    if (d_map) {
        size_t total = (size_t)d.B * d.L * d.L;
        unpack_map_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d, env->obst, d_map);
        MAPF_CUDA(cudaGetLastError());
    }
    if (d_navi) {
        size_t total = (size_t)d.B * d.N * 4 * d.L * d.L;
        if (env->sz_n)
            unpack_navi_sized_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d, env->navi, env->navi_alt, env->navi_sel, d_navi,
                                                                                      env->sz_n);
        else
            unpack_navi_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d, env->navi, env->navi_alt, env->navi_sel, d_navi);
        MAPF_CUDA(cudaGetLastError());
    }
    return MAPF_OK;
}
