// mapf_plan_kernels.cu — prioritized planning (PP) on the device: a collision-free plan for every environment of a batch in
// one launch (mapf_env_plan_prioritized, DESIGN.md §8 (f)5).
//
// Agents a = 0 .. n-1 are planned in index order.  Agent a takes the earliest-arrival space-time path that avoids the paths
// of agents 0 .. a-1, which are reserved in three tables over t = 0 .. H:
//   Occ(t)      cells the reserved agents occupy at time t (an agent parks on its goal from its arrival to H)
//   SB_k(t)     cells v from which a reserved agent moves to v - delta_k between t and t+1: arriving at v by action k over
//               the same step would swap with it
//   last_busy   the largest t with goal in Occ(t)
// and searched with a bit-parallel frontier over time, the wave loop of the heuristic-map BFS with a reservation mask:
//   F(0) = {start},  F(t+1) = (F(t) | OR_k (shift_k F(t) & ~SB_k(t))) & Free & ~Occ(t+1)
//   arrival t* = min { t <= H : goal in F(t), t > last_busy(goal) }
// The path is read back from the stored frontiers (from (goal, t*) down: the first action id k whose predecessor
// v - delta_k is in F(t-1) and, for a move, v is not in SB_k(t-1)) and committed to the tables.
//
// One warp per environment, lane l owns map rows RPL*l .. RPL*l + RPL - 1 (APW = 1 in mapf_bfs_device.cuh terms), RW words
// of padded column bits per row.  The tables and the frontier history live in per-warp global scratch owned by the handle;
// environments are handed out through a work counter, and a warp clears its tables before each environment, so a result
// does not depend on which warp planned it or what that warp planned before.
#include <algorithm>

#include "mapf_bfs_device.cuh"
#include "mapf_common.cuh"

namespace {

constexpr int kPlanWarps = 4;
constexpr int kPlanTables = 6;                          // Occ, SB_1 .. SB_4, F
constexpr size_t kPlanCounterWords = 64;                // the work counter, ahead of the warps' tables
// scratch bytes at most, whatever the horizon and map size.  Each warp's search is a chain of dependent table loads, so
// the launch is latency-bound and more resident warps plan a batch faster: a 1 GB cap takes 2.0x (8192 x 32 @ 40) and 2.9x
// (4096 x 64 @ 80) the time of this one (DESIGN.md §8 (f)5; -DMAPF_PLAN_SCRATCH_MB=1024 builds the A/B partner)
#ifndef MAPF_PLAN_SCRATCH_MB
#define MAPF_PLAN_SCRATCH_MB 4096
#endif
constexpr int64_t kPlanScratchCap = (int64_t)MAPF_PLAN_SCRATCH_MB << 20;

struct PlanArgs {
    EnvDims d;
    const uint32_t *obst;
    const uint8_t *pos, *goal;
    const uint8_t *sz_n, *sz_l;  // NULL: uniform handle
    int H;
    size_t warp_words;           // scratch words per warp
    uint32_t *scratch;           // [0]: work counter; the warps' tables from kPlanCounterWords on
    uint8_t *actions;            // u8[H, B, N], zeroed before the launch
    int32_t *arrival;            // i32[B, N]
};

// offsets of action k (environment.py:12): 0 stay, 1 x-1, 2 x+1, 3 y-1, 4 y+1
__device__ __forceinline__ int act_dx(int k) { return k == 1 ? -1 : (k == 2 ? 1 : 0); }
__device__ __forceinline__ int act_dy(int k) { return k == 3 ? -1 : (k == 4 ? 1 : 0); }

template <int RW, int RPL>
__global__ void __launch_bounds__(kPlanWarps * 32) plan_pp_kernel(const PlanArgs p)
{
    __shared__ uint16_t s_path[kPlanWarps][MAPF_PLAN_MAX_HORIZON + 1];  // x << 8 | y of the current agent at t = 0 .. t*
    constexpr int WPT = 32 * RPL * RW;  // words of one time slice of a table: [q][w][lane]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const EnvDims &d = p.d;
    const int H = p.H;
    const size_t tbl = (size_t)(H + 1) * WPT;  // words of one table
    uint32_t *const occ = p.scratch + kPlanCounterWords + (size_t)(blockIdx.x * kPlanWarps + wid) * p.warp_words;
    uint32_t *const sb = occ;               // SB_k = sb + k * tbl, k = 1 .. 4
    uint32_t *const fh = occ + 5 * tbl;     // frontier history F(0 .. t*)
    uint16_t *const path = s_path[wid];
    auto cell = [](int x, int y) -> size_t { return (size_t)((x % RPL) * RW + ((y + 4) >> 5)) * 32 + x / RPL; };
    auto bit = [](int y) -> uint32_t { return 1u << ((y + 4) & 31); };

    for (;;) {
        unsigned e = 0;
        if (lane == 0) e = atomicAdd(p.scratch, 1u);
        e = __shfl_sync(MAPF_FULL_MASK, e, 0);
        if (e >= (unsigned)d.B) break;

        // clean reservation tables: Occ and SB_1 .. SB_4 over t = 0 .. H
        {
            uint4 *z = reinterpret_cast<uint4 *>(occ);
            const size_t n4 = 5 * tbl / 4;
            for (size_t i = lane; i < n4; i += 32) __stcg(z + i, make_uint4(0u, 0u, 0u, 0u));
        }
        const int n = p.sz_n ? (int)__ldcg(p.sz_n + e) : d.N;
        EnvDims df = d;  // the free cells: l_e x l_e on a sized handle
        if (p.sz_l) df.L = (int)__ldcg(p.sz_l + e);
        BfsFree<RW, RPL> F;
        bfs_load_free<RW, RPL, 1>(df, p.obst + (size_t)e * d.obst_stride, F);
        int32_t *const arr = p.arrival + (size_t)e * d.N;
        for (int a = n + lane; a < d.N; a += 32) arr[a] = 0;  // absent agents
        __syncwarp();

        for (int a = 0; a < n; ++a) {
            const uchar2 s = __ldcg(reinterpret_cast<const uchar2 *>(p.pos) + (size_t)e * d.N + a);
            const uchar2 g = __ldcg(reinterpret_cast<const uchar2 *>(p.goal) + (size_t)e * d.N + a);
            const size_t gi = cell(g.x, g.y);
            const uint32_t gb = bit(g.y);
            const int gl = g.x / RPL, gq = g.x % RPL, gw = (g.y + 4) >> 5;
            // last_busy(goal)
            int lb = -1;
#pragma unroll 4
            for (int t = lane; t <= H; t += 32)
                if (__ldcg(occ + (size_t)t * WPT + gi) & gb) lb = t;
            lb = __reduce_max_sync(MAPF_FULL_MASK, lb);

            uint32_t f[RPL][RW];
#pragma unroll
            for (int q = 0; q < RPL; ++q)
#pragma unroll
                for (int w = 0; w < RW; ++w) {
                    f[q][w] = (lane * RPL + q == s.x && ((s.y + 4) >> 5) == w) ? bit(s.y) : 0u;
                    __stcg(fh + (q * RW + w) * 32 + lane, f[q][w]);
                }
            auto at_goal = [&](int t) -> bool {
                uint32_t x = 0;
#pragma unroll
                for (int q = 0; q < RPL; ++q)
#pragma unroll
                    for (int w = 0; w < RW; ++w)
                        if (q == gq && w == gw) x = f[q][w];
                return __any_sync(MAPF_FULL_MASK, lane == gl && (x & gb)) && t > lb;
            };

            int tstar = -1;
            if (at_goal(0)) {
                tstar = 0;
            } else if (lb < H) {
                for (int t = 0; t < H; ++t) {
                    uint32_t on[RPL][RW], sbk[4][RPL][RW];
#pragma unroll
                    for (int q = 0; q < RPL; ++q)
#pragma unroll
                        for (int w = 0; w < RW; ++w) {
                            const size_t o = (size_t)(q * RW + w) * 32 + lane;
                            on[q][w] = __ldcg(occ + (size_t)(t + 1) * WPT + o);
#pragma unroll
                            for (int k = 0; k < 4; ++k) sbk[k][q][w] = __ldcg(sb + (k + 1) * tbl + (size_t)t * WPT + o);
                        }
                    uint32_t nf[RPL][RW];
                    uint32_t any = 0;
#pragma unroll
                    for (int w = 0; w < RW; ++w) {
                        uint32_t above, below;
                        bfs_rows_around<RW, RPL, 32, false>(f, w, lane, above, below);
#pragma unroll
                        for (int q = 0; q < RPL; ++q) {
                            const uint32_t c = f[q][w];
                            const uint32_t from_dn = q < RPL - 1 ? f[q < RPL - 1 ? q + 1 : q][w] : below;  // action 1 (x-1)
                            const uint32_t from_up = q > 0 ? f[q > 0 ? q - 1 : 0][w] : above;              // action 2 (x+1)
                            const uint32_t from_rt = w < RW - 1 ? __funnelshift_r(c, f[q][w < RW - 1 ? w + 1 : w], 1) : c >> 1;  // 3
                            const uint32_t from_lt = w > 0 ? __funnelshift_l(f[q][w > 0 ? w - 1 : 0], c, 1) : c << 1;            // 4
                            const uint32_t x = (c | (from_dn & ~sbk[0][q][w]) | (from_up & ~sbk[1][q][w]) | (from_rt & ~sbk[2][q][w]) |
                                                (from_lt & ~sbk[3][q][w])) & F.v[q][w] & ~on[q][w];
                            nf[q][w] = x;
                            any |= x;
                        }
                    }
#pragma unroll
                    for (int q = 0; q < RPL; ++q)
#pragma unroll
                        for (int w = 0; w < RW; ++w) {
                            f[q][w] = nf[q][w];
                            __stcg(fh + (size_t)(t + 1) * WPT + (q * RW + w) * 32 + lane, nf[q][w]);
                        }
                    if (!__any_sync(MAPF_FULL_MASK, any != 0)) break;
                    if (at_goal(t + 1)) {
                        tstar = t + 1;
                        break;
                    }
                }
            }
            __syncwarp();

            if (tstar < 0) {  // the environment fails: no plan, no actions, arrival row -1
                for (int t = lane; t < H; t += 32)
                    for (int b = 0; b < a; ++b) p.actions[((size_t)t * d.B + e) * d.N + b] = 0;
                for (int b = lane; b < d.N; b += 32) arr[b] = -1;
                break;
            }

            // back from (goal, t*): lane k < 5 tests action k, the lowest admissible id wins
            int vx = g.x, vy = g.y;
            if (lane == 0) path[tstar] = (uint16_t)(vx << 8 | vy);
            for (int t = tstar; t >= 1; --t) {
                bool ok = false;
                if (lane < 5) {
                    const int ux = vx - act_dx(lane), uy = vy - act_dy(lane);
                    if (ux >= 0 && ux < d.L && uy >= 0 && uy < d.L) {
                        ok = (__ldcg(fh + (size_t)(t - 1) * WPT + cell(ux, uy)) & bit(uy)) != 0;
                        if (ok && lane > 0) ok = (__ldcg(sb + lane * tbl + (size_t)(t - 1) * WPT + cell(vx, vy)) & bit(vy)) == 0;
                    }
                }
                const unsigned m = __ballot_sync(MAPF_FULL_MASK, ok);
                const int k = m ? __ffs(m) - 1 : 0;
                vx -= act_dx(k), vy -= act_dy(k);
                if (lane == 0) path[t - 1] = (uint16_t)(vx << 8 | vy);
            }
            __syncwarp();

            // commit: the path into Occ(0 .. t*), the goal into Occ(t* .. H), each move's origin into SB_opposite(k)
            for (int t = lane; t <= H; t += 32) {
                const int c = t <= tstar ? path[t] : (g.x << 8 | g.y);
                const int x = c >> 8, y = c & 255;
                uint32_t *o = occ + (size_t)t * WPT + cell(x, y);
                __stcg(o, __ldcg(o) | bit(y));
                if (t < tstar) {
                    const int x2 = path[t + 1] >> 8, y2 = path[t + 1] & 255;
                    const int k = x2 < x ? 1 : (x2 > x ? 2 : (y2 < y ? 3 : (y2 > y ? 4 : 0)));
                    if (k) {
                        p.actions[((size_t)t * d.B + e) * d.N + a] = (uint8_t)k;
                        uint32_t *r = sb + (k & 1 ? k + 1 : k - 1) * tbl + (size_t)t * WPT + cell(x, y);
                        __stcg(r, __ldcg(r) | bit(y));
                    }
                }
            }
            if (lane == 0) arr[a] = tstar;
            __syncwarp();
        }
    }
}

template <int RW, int RPL>
int launch_plan(mapf_env *env, int H, uint8_t *d_actions, int32_t *d_arrival, cudaStream_t st)
{
    const EnvDims &d = env->d;
    const size_t warp_words = (size_t)kPlanTables * (H + 1) * 32 * RPL * RW;
    int per_sm = 0;
    MAPF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, plan_pp_kernel<RW, RPL>, kPlanWarps * 32, 0));
    const int64_t block_bytes = (int64_t)kPlanWarps * warp_words * 4;
    int64_t blocks = std::min<int64_t>((int64_t)std::max(per_sm, 1) * env->num_sms, (d.B + kPlanWarps - 1) / kPlanWarps);
    blocks = std::max<int64_t>(1, std::min<int64_t>(blocks, kPlanScratchCap / block_bytes));
    const int64_t bytes = (int64_t)kPlanCounterWords * 4 + blocks * block_bytes;
    if (bytes > env->pp_bytes) {  // first use, or a larger horizon / grid than before
        if (env->pp_scratch) {
            MAPF_CUDA(cudaStreamSynchronize(st));
            cudaFree(env->pp_scratch);
            env->arena_bytes -= env->pp_bytes;
            env->pp_scratch = nullptr, env->pp_bytes = 0;
        }
        const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&env->pp_scratch), (size_t)bytes);
        if (e != cudaSuccess) {
            mapf_cuda_fail(e, "mapf_env_plan_prioritized: scratch");
            env->pp_scratch = nullptr;
            return MAPF_ENOMEM;
        }
        env->pp_bytes = bytes;
        env->arena_bytes += bytes;
    }
    MAPF_CUDA(cudaMemsetAsync(env->pp_scratch, 0, 4, st));
    MAPF_CUDA(cudaMemsetAsync(d_actions, 0, (size_t)H * d.B * d.N, st));
    PlanArgs p;
    p.d = d;
    p.obst = env->obst, p.pos = env->pos, p.goal = env->goal;
    p.sz_n = env->sz_n, p.sz_l = env->sz_l;
    p.H = H;
    p.warp_words = warp_words;
    p.scratch = env->pp_scratch;
    p.actions = d_actions, p.arrival = d_arrival;
    plan_pp_kernel<RW, RPL><<<(unsigned)blocks, kPlanWarps * 32, 0, st>>>(p);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

}  // namespace

// rows per lane RPL = ceil(L / 32) next to the handle's RW: L <= 24 (1, 1), <= 56 (2, 1..2), <= 88 (3, 2..3), <= 120 (4, 3..4)
int mapf_launch_plan(mapf_env *env, int H, uint8_t *d_actions, int32_t *d_arrival, cudaStream_t st)
{
    const int rpl = (env->d.L + 31) / 32;
    switch (env->d.RW * 8 + rpl) {
        case 1 * 8 + 1: return launch_plan<1, 1>(env, H, d_actions, d_arrival, st);
        case 2 * 8 + 1: return launch_plan<2, 1>(env, H, d_actions, d_arrival, st);
        case 2 * 8 + 2: return launch_plan<2, 2>(env, H, d_actions, d_arrival, st);
        case 3 * 8 + 2: return launch_plan<3, 2>(env, H, d_actions, d_arrival, st);
        case 3 * 8 + 3: return launch_plan<3, 3>(env, H, d_actions, d_arrival, st);
        case 4 * 8 + 3: return launch_plan<4, 3>(env, H, d_actions, d_arrival, st);
        case 4 * 8 + 4: return launch_plan<4, 4>(env, H, d_actions, d_arrival, st);
    }
    mapf_set_error("mapf_env_plan_prioritized: unsupported map size");
    return MAPF_EINVAL;
}
