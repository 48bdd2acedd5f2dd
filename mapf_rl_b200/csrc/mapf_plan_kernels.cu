// mapf_plan_kernels.cu — prioritized planning (PP) on the device: a collision-free plan for every environment of a batch in
// one launch (mapf_env_plan_prioritized, DESIGN.md §8 (f)5), and the best of R priority orders per environment
// (mapf_env_plan_prioritized_orders).
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
//
// Several orders: order 0 is index order, order r >= 1 sorts the agents by (Philox key of (g, PURPOSE_ORDER | r << 8, a), a).
// Pass 1 plans every (environment, order) pair as a work item without writing actions and folds (sum of costs, r) of a
// solved order into the environment's selection word with atomicMin, so the smallest sum of costs wins and ties go to the
// smallest r whatever the schedule.  Pass 2 re-plans each environment's winning order and writes its results.
#include <algorithm>

#include "mapf_bfs_device.cuh"
#include "mapf_common.cuh"
#include "mapf_reset_device.cuh"

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
constexpr unsigned long long kNoOrder = ~0ull;  // selection word of an environment no order has solved

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

struct OrderArgs {
    int R;                       // priority orders per environment
    uint2 key;                   // Philox key (seed)
    uint64_t env_offset;         // global index of environment 0
    unsigned long long *sel;     // u64[B]: (sum of costs << 32 | r) of the best solved order, kNoOrder before pass 1
    int32_t *order;              // i32[B]: the winning r, -1
    uint8_t *rank;               // u8[B, N]: agent a's position in the winning order, 255
};

// offsets of action k (environment.py:12): 0 stay, 1 x-1, 2 x+1, 3 y-1, 4 y+1
__device__ __forceinline__ int act_dx(int k) { return k == 1 ? -1 : (k == 2 ? 1 : 0); }
__device__ __forceinline__ int act_dy(int k) { return k == 3 ? -1 : (k == 4 ? 1 : 0); }

// The planner of one warp, all three kernels' code:
//   kPlanIndex        plan_pp_kernel: environment e is a work item, its agents planned in index order, results written
//   kPlanOrders       pass 1 of plan_orders_kernel: item i = (e, r) = (i / R, i % R), agents in order r, nothing written but
//                     (sum of costs << 32 | r) of a solved order, folded into the selection word ord.sel[e] with atomicMin
//   kPlanOrdersFinal  pass 2: environment e is a work item, its winning order re-planned with results, rank and order
//                     written, or the failure rows where no order solved it
enum : int { kPlanIndex = 0, kPlanOrders = 1, kPlanOrdersFinal = 2 };

template <int RW, int RPL, int MODE>
__device__ __forceinline__ void plan_body(const PlanArgs &p, const OrderArgs &ord)
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

    uint8_t *agent = nullptr;  // the agent at each position of the order
    uint32_t *key = nullptr;
    if constexpr (MODE != kPlanIndex) {
        __shared__ uint8_t s_agent[kPlanWarps][MAPF_MAX_AGENTS];
        __shared__ uint32_t s_key[kPlanWarps][MAPF_MAX_AGENTS];
        agent = s_agent[wid], key = s_key[wid];
    }

    for (;;) {
        unsigned e = 0;
        int oi = 0;  // the order
        if constexpr (MODE == kPlanIndex) {
            if (lane == 0) e = atomicAdd(p.scratch, 1u);
            e = __shfl_sync(MAPF_FULL_MASK, e, 0);
            if (e >= (unsigned)d.B) break;
        } else {
            // 64-bit counters (B * R items): words 0 .. 1 for pass 1, 2 .. 3 for pass 2
            unsigned long long i = 0;
            if (lane == 0) i = atomicAdd(reinterpret_cast<unsigned long long *>(p.scratch) + (MODE == kPlanOrdersFinal), 1ull);
            i = __shfl_sync(MAPF_FULL_MASK, i, 0);
            if (i >= (unsigned long long)d.B * (MODE == kPlanOrders ? ord.R : 1)) break;
            e = MODE == kPlanOrders ? (unsigned)(i / ord.R) : (unsigned)i;
            oi = MODE == kPlanOrders ? (int)(i % ord.R) : 0;
            if constexpr (MODE == kPlanOrdersFinal) {
                const unsigned long long sel = __ldcg(ord.sel + e);
                if (sel == kNoOrder) {  // every order failed: arrival row -1, rank 255, actions 0 (zeroed before the launch)
                    for (int b = lane; b < d.N; b += 32) p.arrival[(size_t)e * d.N + b] = -1, ord.rank[(size_t)e * d.N + b] = 255;
                    if (lane == 0) ord.order[e] = -1;
                    continue;
                }
                oi = (int)(uint32_t)sel;
            }
        }

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
        if constexpr (MODE != kPlanOrders)
            for (int a = n + lane; a < d.N; a += 32) arr[a] = 0;  // absent agents
        if constexpr (MODE != kPlanIndex) {
            // order oi: agent a goes to position #{b < n : (k_b, b) < (k_a, a)}; order 0 has every key 0, i.e. index order
            const uint64_t ge = ord.env_offset + e;  // the environment's global index
            for (int a = lane; a < n; a += 32)
                key[a] = oi ? philox4x32_10(make_uint4((uint32_t)ge, (uint32_t)(ge >> 32), PURPOSE_ORDER | ((uint32_t)oi << 8), (uint32_t)a), ord.key).x
                           : 0u;
            __syncwarp();
            for (int a = lane; a < n; a += 32) {
                const uint32_t ka = key[a];
                int pos = 0;
                for (int b = 0; b < n; ++b) pos += key[b] < ka || (key[b] == ka && b < a);
                agent[pos] = (uint8_t)a;
                if constexpr (MODE == kPlanOrdersFinal) ord.rank[(size_t)e * d.N + a] = (uint8_t)pos;
            }
            if constexpr (MODE == kPlanOrdersFinal)
                for (int a = n + lane; a < d.N; a += 32) ord.rank[(size_t)e * d.N + a] = 255;
        }
        __syncwarp();

        int soc = 0;
        bool solved = true;
        for (int j = 0; j < n; ++j) {  // an order stops at its first failing agent
            const int a = MODE == kPlanIndex ? j : agent[j];
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

            if (tstar < 0) {  // the environment (the order) fails: no plan, no actions, arrival row -1
                if constexpr (MODE == kPlanIndex) {
                    for (int t = lane; t < H; t += 32)
                        for (int b = 0; b < a; ++b) p.actions[((size_t)t * d.B + e) * d.N + b] = 0;
                    for (int b = lane; b < d.N; b += 32) arr[b] = -1;
                }
                solved = false;
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
                        if constexpr (MODE != kPlanOrders) p.actions[((size_t)t * d.B + e) * d.N + a] = (uint8_t)k;
                        uint32_t *r = sb + (k & 1 ? k + 1 : k - 1) * tbl + (size_t)t * WPT + cell(x, y);
                        __stcg(r, __ldcg(r) | bit(y));
                    }
                }
            }
            if (MODE != kPlanOrders && lane == 0) arr[a] = tstar;
            soc += tstar;
            __syncwarp();
        }
        if constexpr (MODE != kPlanIndex) {
            if (lane == 0) {
                if (MODE == kPlanOrdersFinal) ord.order[e] = oi;
                else if (solved) atomicMin(ord.sel + e, (unsigned long long)soc << 32 | (unsigned)oi);
            }
            __syncwarp();
        }
    }
}

template <int RW, int RPL>
__global__ void __launch_bounds__(kPlanWarps * 32) plan_pp_kernel(const PlanArgs p)
{
    plan_body<RW, RPL, kPlanIndex>(p, OrderArgs{});
}

template <int RW, int RPL, int MODE>
__global__ void __launch_bounds__(kPlanWarps * 32) plan_orders_kernel(const PlanArgs p, const OrderArgs o)
{
    plan_body<RW, RPL, MODE>(p, o);
}

// The handle's planner scratch: at least `bytes`, allocated on first use and grown when a call needs more
int reserve_plan_scratch(mapf_env *env, int64_t bytes, cudaStream_t st, const char *what)
{
    if (bytes <= env->pp_bytes) return MAPF_OK;
    if (env->pp_scratch) {
        MAPF_CUDA(cudaStreamSynchronize(st));
        cudaFree(env->pp_scratch);
        env->arena_bytes -= env->pp_bytes;
        env->pp_scratch = nullptr, env->pp_bytes = 0;
    }
    const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&env->pp_scratch), (size_t)bytes);
    if (e != cudaSuccess) {
        mapf_cuda_fail(e, what);
        env->pp_scratch = nullptr;
        return MAPF_ENOMEM;
    }
    env->pp_bytes = bytes;
    env->arena_bytes += bytes;
    return MAPF_OK;
}

// blocks of a planner launch over `items` warp work items: the resident blocks, at most the scratch cap
template <typename Kernel>
int plan_blocks(mapf_env *env, Kernel kernel, int64_t items, int64_t block_bytes, int64_t &blocks)
{
    int per_sm = 0;
    MAPF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kPlanWarps * 32, 0));
    blocks = std::min<int64_t>((int64_t)std::max(per_sm, 1) * env->num_sms, (items + kPlanWarps - 1) / kPlanWarps);
    blocks = std::max<int64_t>(1, std::min<int64_t>(blocks, kPlanScratchCap / block_bytes));
    return MAPF_OK;
}

PlanArgs plan_args(mapf_env *env, int H, size_t warp_words, uint8_t *d_actions, int32_t *d_arrival)
{
    PlanArgs p;
    p.d = env->d;
    p.obst = env->obst, p.pos = env->pos, p.goal = env->goal;
    p.sz_n = env->sz_n, p.sz_l = env->sz_l;
    p.H = H;
    p.warp_words = warp_words;
    p.scratch = env->pp_scratch;
    p.actions = d_actions, p.arrival = d_arrival;
    return p;
}

template <int RW, int RPL>
int launch_plan(mapf_env *env, int H, uint8_t *d_actions, int32_t *d_arrival, cudaStream_t st)
{
    const EnvDims &d = env->d;
    const size_t warp_words = (size_t)kPlanTables * (H + 1) * 32 * RPL * RW;
    const int64_t block_bytes = (int64_t)kPlanWarps * warp_words * 4;
    int64_t blocks = 0;
    int rc = plan_blocks(env, plan_pp_kernel<RW, RPL>, d.B, block_bytes, blocks);
    if (rc != MAPF_OK) return rc;
    rc = reserve_plan_scratch(env, (int64_t)kPlanCounterWords * 4 + blocks * block_bytes, st,
                                        "mapf_env_plan_prioritized: scratch");
    if (rc != MAPF_OK) return rc;
    MAPF_CUDA(cudaMemsetAsync(env->pp_scratch, 0, 4, st));
    MAPF_CUDA(cudaMemsetAsync(d_actions, 0, (size_t)H * d.B * d.N, st));
    plan_pp_kernel<RW, RPL><<<(unsigned)blocks, kPlanWarps * 32, 0, st>>>(plan_args(env, H, warp_words, d_actions, d_arrival));
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

template <int RW, int RPL>
int launch_plan_orders(mapf_env *env, int H, int R, uint64_t seed, uint64_t env_offset, uint8_t *d_actions, int32_t *d_arrival,
                       int32_t *d_order, uint8_t *d_rank, cudaStream_t st)
{
    const EnvDims &d = env->d;
    const size_t warp_words = (size_t)kPlanTables * (H + 1) * 32 * RPL * RW;
    const int64_t block_bytes = (int64_t)kPlanWarps * warp_words * 4;
    int64_t blocks = 0, blocks2 = 0;
    int rc = plan_blocks(env, plan_orders_kernel<RW, RPL, kPlanOrders>, (int64_t)d.B * R, block_bytes, blocks);
    if (rc == MAPF_OK) rc = plan_blocks(env, plan_orders_kernel<RW, RPL, kPlanOrdersFinal>, d.B, block_bytes, blocks2);
    if (rc != MAPF_OK) return rc;
    // the selection words follow the warps' tables
    const int64_t sel_off = (int64_t)kPlanCounterWords * 4 + blocks * block_bytes;
    rc = reserve_plan_scratch(env, sel_off + (int64_t)d.B * 8, st, "mapf_env_plan_prioritized_orders: scratch");
    if (rc != MAPF_OK) return rc;
    OrderArgs o;
    o.R = R;
    o.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    o.env_offset = env_offset;
    o.sel = reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(env->pp_scratch) + sel_off);
    o.order = d_order, o.rank = d_rank;
    MAPF_CUDA(cudaMemsetAsync(env->pp_scratch, 0, 16, st));
    MAPF_CUDA(cudaMemsetAsync(o.sel, 0xff, (size_t)d.B * 8, st));
    MAPF_CUDA(cudaMemsetAsync(d_actions, 0, (size_t)H * d.B * d.N, st));
    const PlanArgs p = plan_args(env, H, warp_words, d_actions, d_arrival);
    plan_orders_kernel<RW, RPL, kPlanOrders><<<(unsigned)blocks, kPlanWarps * 32, 0, st>>>(p, o);
    MAPF_CUDA(cudaGetLastError());
    // pass 2 uses the tables of the first blocks2 <= blocks blocks of pass 1
    plan_orders_kernel<RW, RPL, kPlanOrdersFinal><<<(unsigned)std::min(blocks, blocks2), kPlanWarps * 32, 0, st>>>(p, o);
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

int mapf_launch_plan_orders(mapf_env *env, int H, int R, uint64_t seed, uint64_t env_offset, uint8_t *d_actions, int32_t *d_arrival,
                            int32_t *d_order, uint8_t *d_rank, cudaStream_t st)
{
    const int rpl = (env->d.L + 31) / 32;
#define MAPF_PLAN_ORDERS_CASE(rw, r) \
    case rw * 8 + r: return launch_plan_orders<rw, r>(env, H, R, seed, env_offset, d_actions, d_arrival, d_order, d_rank, st)
    switch (env->d.RW * 8 + rpl) {
        MAPF_PLAN_ORDERS_CASE(1, 1);
        MAPF_PLAN_ORDERS_CASE(2, 1);
        MAPF_PLAN_ORDERS_CASE(2, 2);
        MAPF_PLAN_ORDERS_CASE(3, 2);
        MAPF_PLAN_ORDERS_CASE(3, 3);
        MAPF_PLAN_ORDERS_CASE(4, 3);
        MAPF_PLAN_ORDERS_CASE(4, 4);
    }
#undef MAPF_PLAN_ORDERS_CASE
    mapf_set_error("mapf_env_plan_prioritized_orders: unsupported map size");
    return MAPF_EINVAL;
}
