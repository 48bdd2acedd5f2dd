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
//
// Plan improvement (mapf_env_plan_lns, DESIGN.md §8 (f)6), large-neighbourhood search from a plan in the layout above: agent
// a < n follows p_0 = its position, p_t+1 = p_t + delta(actions[t, a]) for t < arrival[a], and parks on its goal from
// arrival[a] to H.  The input is checked once: a row of -1 (a failed plan) is left as it is with accepted -1; an action id
// > 4, a p_t off the l x l map or on an obstacle, p_arrival != goal, a move at t >= arrival, an arrival outside [0, H], a
// shared cell or a swap leave the environment as it is with accepted -2.  Iteration i draws k_a = word 0 of Philox of
// (g, PURPOSE_LNS | i << 8, a); the neighbourhood S is the min(k, n) agents of smallest (k_a, a), in that order.  The paths
// of the agents outside S are reserved as a planned path is committed, the agents of S are planned in order by the rules
// above, and the new paths are kept (accepted += 1) if every agent of S finds one and their arrivals sum to strictly less
// than before.  One warp runs all iterations of one environment with its tables kept across them; the path search,
// read-back and commit are the functions plan_body uses.
//
// Plan repair (mapf_env_plan_repair, DESIGN.md §8 (f)7), collision-based large-neighbourhood search (MAPF-LNS2) on the
// environments whose plan failed: vertex conflicts become soft, each costing 1, while obstacles and swaps stay hard.  The
// soft search keeps one frontier per collision count c = 0 .. C, F_c(t) the cells reached at t with exactly c vertex
// collisions and no fewer; a cell is in at most one layer, so the history stores a "reached" plane and the layer's four bits
// (5 tables instead of C + 1).  The agents are planned in index order with collisions allowed, then each iteration re-plans a
// group S (the agents with a collision first, in Philox order) against the others and keeps the new paths if their collision
// count (then their sum of costs) drops.  The tables are rebuilt from the current paths every iteration: in a colliding plan
// a bit can belong to two agents, so clearing one agent's bits is not undone by reserving it again.
#include <algorithm>
#include <climits>

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

struct RepairArgs {
    int I, K;                    // iterations, neighbourhood size
    uint2 key;                   // Philox key (seed)
    uint64_t env_offset;         // global index of environment 0
    int32_t *collisions;         // i32[B]: collisions left, -1 (no path), -2 (not a failed plan)
};

constexpr int kRepairTables = 10;  // Occ, SB_1 .. SB_4, the layer history: reached, the layer's bits 0 .. 3
static_assert(MAPF_PLAN_REPAIR_MAX_COLLISIONS >= 1 && MAPF_PLAN_REPAIR_MAX_COLLISIONS <= 15, "layers are stored in four bits");

struct LnsArgs {
    int I, K;                    // iterations, neighbourhood size
    uint32_t first;              // the first iteration's index
    uint2 key;                   // Philox key (seed)
    uint64_t env_offset;         // global index of environment 0
    int32_t *accepted;           // i32[B]: accepted iterations, -1 (failed plan), -2 (invalid plan)
};

// offsets of action k (environment.py:12): 0 stay, 1 x-1, 2 x+1, 3 y-1, 4 y+1
__device__ __forceinline__ int act_dx(int k) { return k == 1 ? -1 : (k == 2 ? 1 : 0); }
__device__ __forceinline__ int act_dy(int k) { return k == 3 ? -1 : (k == 4 ? 1 : 0); }

// A warp's tables: Occ at `occ`, SB_k at occ + k * tbl (k = 1 .. 4), the frontier history F at occ + 5 * tbl, one table =
// H + 1 time slices of WPT = 32 * RPL * RW words laid out [q][w][lane]; cell (x, y) is bit plan_bit(y) of word plan_cell(x, y).
// These two are plain inline, not __forceinline__: forced inlining happens before they are simplified and moves the address
// arithmetic of the planning kernels (more registers and instructions than with the local lambdas they replaced).
template <int RW, int RPL>
__device__ inline size_t plan_cell(int x, int y) { return (size_t)((x % RPL) * RW + ((y + 4) >> 5)) * 32 + x / RPL; }
__device__ inline uint32_t plan_bit(int y) { return 1u << ((y + 4) & 31); }

// The search of one agent from s to g against the reservations in the tables: last_busy(g), then the frontier F(0 .. t*),
// stored in the history.  Returns t*, or -1 where the agent finds no path within H.
template <int RW, int RPL>
__device__ __forceinline__ int plan_search(const uint32_t *const occ, const uint32_t *const sb, uint32_t *const fh, const size_t tbl,
                                           const int H, const int lane, const BfsFree<RW, RPL> &F, const uchar2 s, const uchar2 g)
{
    constexpr int WPT = 32 * RPL * RW;
    const size_t gi = plan_cell<RW, RPL>(g.x, g.y);
    const uint32_t gb = plan_bit(g.y);
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
            f[q][w] = (lane * RPL + q == s.x && ((s.y + 4) >> 5) == w) ? plan_bit(s.y) : 0u;
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
    return tstar;
}

// The path back from (g, t*) into path[0 .. t*] (x << 8 | y): lane k < 5 tests action k, the lowest admissible id wins
template <int RW, int RPL>
__device__ __forceinline__ void plan_read_back(const uint32_t *const sb, const uint32_t *const fh, const size_t tbl, const int L, const int lane,
                                               const uchar2 g, const int tstar, uint16_t *const path)
{
    constexpr int WPT = 32 * RPL * RW;
    int vx = g.x, vy = g.y;
    if (lane == 0) path[tstar] = (uint16_t)(vx << 8 | vy);
    for (int t = tstar; t >= 1; --t) {
        bool ok = false;
        if (lane < 5) {
            const int ux = vx - act_dx(lane), uy = vy - act_dy(lane);
            if (ux >= 0 && ux < L && uy >= 0 && uy < L) {
                ok = (__ldcg(fh + (size_t)(t - 1) * WPT + plan_cell<RW, RPL>(ux, uy)) & plan_bit(uy)) != 0;
                if (ok && lane > 0) ok = (__ldcg(sb + lane * tbl + (size_t)(t - 1) * WPT + plan_cell<RW, RPL>(vx, vy)) & plan_bit(vy)) == 0;
            }
        }
        const unsigned m = __ballot_sync(MAPF_FULL_MASK, ok);
        const int k = m ? __ffs(m) - 1 : 0;
        vx -= act_dx(k), vy -= act_dy(k);
        if (lane == 0) path[t - 1] = (uint16_t)(vx << 8 | vy);
    }
}

// commit: path[0 .. t*] into Occ(0 .. t*), the goal into Occ(t* .. H), each move's origin into SB_opposite(k); with ACTIONS,
// agent a's move ids into p.actions of environment e
template <int RW, int RPL, bool ACTIONS>
__device__ __forceinline__ void plan_commit(uint32_t *const occ, uint32_t *const sb, const size_t tbl, const int H, const int lane, const uchar2 g,
                                            const int tstar, const uint16_t *const path, const PlanArgs &p, const unsigned e, const int a)
{
    constexpr int WPT = 32 * RPL * RW;
    for (int t = lane; t <= H; t += 32) {
        const int c = t <= tstar ? path[t] : (g.x << 8 | g.y);
        const int x = c >> 8, y = c & 255;
        uint32_t *o = occ + (size_t)t * WPT + plan_cell<RW, RPL>(x, y);
        __stcg(o, __ldcg(o) | plan_bit(y));
        if (t < tstar) {
            const int x2 = path[t + 1] >> 8, y2 = path[t + 1] & 255;
            const int k = x2 < x ? 1 : (x2 > x ? 2 : (y2 < y ? 3 : (y2 > y ? 4 : 0)));
            if (k) {
                if constexpr (ACTIONS) p.actions[((size_t)t * p.d.B + e) * p.d.N + a] = (uint8_t)k;
                uint32_t *r = sb + (k & 1 ? k + 1 : k - 1) * tbl + (size_t)t * WPT + plan_cell<RW, RPL>(x, y);
                __stcg(r, __ldcg(r) | plan_bit(y));
            }
        }
    }
}

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
            const int tstar = plan_search<RW, RPL>(occ, sb, fh, tbl, H, lane, F, s, g);
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

            plan_read_back<RW, RPL>(sb, fh, tbl, d.L, lane, g, tstar, path);
            __syncwarp();
            plan_commit<RW, RPL, MODE != kPlanOrders>(occ, sb, tbl, H, lane, g, tstar, path, p, e, a);
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

// the action id of the move from cell c to cell c2 (x << 8 | y each), 0 for a wait
__device__ inline int plan_move(int c, int c2)
{
    const int x = c >> 8, y = c & 255, x2 = c2 >> 8, y2 = c2 & 255;
    return x2 < x ? 1 : (x2 > x ? 2 : (y2 < y ? 3 : (y2 > y ? 4 : 0)));
}

// Takes the path pth[0 .. H] (x << 8 | y, parked on the goal from its arrival) out of the tables (SET = false) or puts it back
// (SET = true): p_t in Occ(t), and p_t in SB_opposite(k)(t) for a move by action k.  In a valid plan every bit of the tables
// belongs to exactly one agent, so clearing a path's bits removes that agent and nobody else.
template <int RW, int RPL, bool SET>
__device__ __forceinline__ void plan_mark(uint32_t *const occ, const size_t tbl, const int H, const int lane, const uint16_t *const pth)
{
    constexpr int WPT = 32 * RPL * RW;
    for (int t = lane; t <= H; t += 32) {
        const int c = pth[t], x = c >> 8, y = c & 255;
        const uint32_t b = plan_bit(y);
        uint32_t *o = occ + (size_t)t * WPT + plan_cell<RW, RPL>(x, y);
        __stcg(o, SET ? (__ldcg(o) | b) : (__ldcg(o) & ~b));
        const int k = t < H ? plan_move(c, pth[t + 1]) : 0;
        if (k) {
            uint32_t *r = occ + (k & 1 ? k + 1 : k - 1) * tbl + (size_t)t * WPT + plan_cell<RW, RPL>(x, y);
            __stcg(r, SET ? (__ldcg(r) | b) : (__ldcg(r) & ~b));
        }
    }
}

// Plan improvement (mapf_env_plan_lns): one warp per environment, all I iterations on it.  The warp checks the input plan
// while it reserves every path in its tables, then per iteration takes the neighbourhood S out of the tables, re-plans S's
// agents one after the other with plan()'s search, read-back and commit, and keeps the new paths (already in the tables) if
// every agent of S found one and their arrivals sum to less than before; otherwise it clears them and puts the old paths back.
// The tables are kept across iterations; the current paths and the candidates live in the warp's scratch after its tables.
template <int RW, int RPL>
__global__ void __launch_bounds__(kPlanWarps * 32) plan_lns_kernel(const PlanArgs p, const LnsArgs z)
{
    __shared__ uint16_t s_path[kPlanWarps][MAPF_PLAN_MAX_HORIZON + 1];  // the agent being re-planned at t = 0 .. t*
    __shared__ uint8_t s_agent[kPlanWarps][MAPF_MAX_AGENTS];             // S in planning order
    __shared__ uint32_t s_key[kPlanWarps][MAPF_MAX_AGENTS];
    __shared__ int16_t s_arr[kPlanWarps][MAPF_MAX_AGENTS];               // each agent's current arrival
    __shared__ int16_t s_new[kPlanWarps][MAPF_MAX_AGENTS];               // the candidate arrival of S's j-th agent
    constexpr int WPT = 32 * RPL * RW;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const EnvDims &d = p.d;
    const int H = p.H;
    const size_t tbl = (size_t)(H + 1) * WPT;
    uint32_t *const occ = p.scratch + kPlanCounterWords + (size_t)(blockIdx.x * kPlanWarps + wid) * p.warp_words;
    uint32_t *const sb = occ;
    uint32_t *const fh = occ + 5 * tbl;
    uint16_t *const cur = reinterpret_cast<uint16_t *>(occ + kPlanTables * tbl);  // u16[N][H+1]: the current paths
    uint16_t *const cand = cur + (size_t)d.N * (H + 1);                            // u16[N][H+1]: S's j-th candidate in row j
    uint16_t *const path = s_path[wid];
    uint8_t *const agent = s_agent[wid];
    uint32_t *const key = s_key[wid];
    int16_t *const arr_now = s_arr[wid], *const arr_new = s_new[wid];

    for (;;) {
        unsigned e = 0;
        if (lane == 0) e = atomicAdd(p.scratch, 1u);
        e = __shfl_sync(MAPF_FULL_MASK, e, 0);
        if (e >= (unsigned)d.B) break;
        const int n = p.sz_n ? (int)__ldcg(p.sz_n + e) : d.N;
        const int l = p.sz_l ? (int)__ldcg(p.sz_l + e) : d.L;
        const uchar2 *const pos = reinterpret_cast<const uchar2 *>(p.pos) + (size_t)e * d.N;
        const uchar2 *const goal = reinterpret_cast<const uchar2 *>(p.goal) + (size_t)e * d.N;
        const uint32_t *const ob = p.obst + (size_t)e * d.obst_stride;
        int32_t *const arr = p.arrival + (size_t)e * d.N;

        // a failed plan (every present arrival -1) stays as it is
        bool failed = true;
        for (int a = lane; a < n; a += 32) failed &= __ldcg(arr + a) == -1;
        if (__all_sync(MAPF_FULL_MASK, failed)) {
            if (lane == 0) z.accepted[e] = -1;
            continue;
        }

        // clean tables, then every path reserved while it is checked: lane l walks agents l, l + 32, .. over t = 0 .. H
        {
            uint4 *zr = reinterpret_cast<uint4 *>(occ);
            const size_t n4 = 5 * tbl / 4;
            for (size_t i = lane; i < n4; i += 32) __stcg(zr + i, make_uint4(0u, 0u, 0u, 0u));
        }
        __syncwarp();
        bool bad = false;
        for (int a = lane; a < n && !bad; a += 32) {
            const int ar = __ldcg(arr + a);
            arr_now[a] = (int16_t)ar;
            if (ar < 0 || ar > H) {
                bad = true;
                break;
            }
            const uchar2 s = __ldcg(pos + a), g = __ldcg(goal + a);
            uint16_t *const pa = cur + (size_t)a * (H + 1);
            int x = s.x, y = s.y;
            for (int t = 0;; ++t) {
                // off the l x l map or on an obstacle; a vertex conflict (the bit is somebody else's); not on the goal at arrival
                if (x < 0 || x >= l || y < 0 || y >= l || (__ldcg(ob + (x + 4) * d.RWS + ((y + 4) >> 5)) & plan_bit(y)) ||
                    (atomicOr(occ + (size_t)t * WPT + plan_cell<RW, RPL>(x, y), plan_bit(y)) & plan_bit(y)) ||
                    (t == ar && (x != g.x || y != g.y))) {
                    bad = true;
                    break;
                }
                pa[t] = (uint16_t)(x << 8 | y);
                if (t == H) break;
                const int k = p.actions[((size_t)t * d.B + e) * d.N + a];
                if (k > 4 || (k && t >= ar)) {  // an unknown action, a move after arrival
                    bad = true;
                    break;
                }
                if (k) {
                    atomicOr(sb + (k & 1 ? k + 1 : k - 1) * tbl + (size_t)t * WPT + plan_cell<RW, RPL>(x, y), plan_bit(y));
                    x += act_dx(k), y += act_dy(k);
                }
            }
        }
        bad = __any_sync(MAPF_FULL_MASK, bad);
        __syncwarp();
        if (!bad) {
            // a swap: agent a's move u -> v by action k meets another agent's move v -> u, which put v into SB_k(t)
            for (int a = lane; a < n; a += 32) {
                const uint16_t *const pa = cur + (size_t)a * (H + 1);
                for (int t = 0; t < arr_now[a]; ++t) {
                    const int k = plan_move(pa[t], pa[t + 1]), x = pa[t + 1] >> 8, y = pa[t + 1] & 255;
                    if (k && (__ldcg(sb + k * tbl + (size_t)t * WPT + plan_cell<RW, RPL>(x, y)) & plan_bit(y))) bad = true;
                }
            }
            bad = __any_sync(MAPF_FULL_MASK, bad);
        }
        if (bad) {
            if (lane == 0) z.accepted[e] = -2;
            continue;
        }

        EnvDims df = d;  // the free cells: l_e x l_e on a sized handle
        df.L = l;
        BfsFree<RW, RPL> F;
        bfs_load_free<RW, RPL, 1>(df, ob, F);
        const int m = min(z.K, n);
        const uint64_t ge = z.env_offset + e;  // the environment's global index
        int acc = 0;
        for (uint32_t i = z.first; i < z.first + (uint32_t)z.I; ++i) {
            // S: the m agents of smallest (k_a, a), in that order
            for (int a = lane; a < n; a += 32)
                key[a] = philox4x32_10(make_uint4((uint32_t)ge, (uint32_t)(ge >> 32), PURPOSE_LNS | (i << 8), (uint32_t)a), z.key).x;
            __syncwarp();
            for (int a = lane; a < n; a += 32) {
                const uint32_t ka = key[a];
                int r = 0;
                for (int b = 0; b < n; ++b) r += key[b] < ka || (key[b] == ka && b < a);
                if (r < m) agent[r] = (uint8_t)a;
            }
            __syncwarp();
            int old = 0;
            for (int j = 0; j < m; ++j) {
                const int a = agent[j];
                plan_mark<RW, RPL, false>(occ, tbl, H, lane, cur + (size_t)a * (H + 1));
                old += arr_now[a];
                __syncwarp();
            }
            int j = 0, soc = 0;
            for (; j < m; ++j) {
                const int a = agent[j];
                const uchar2 s = __ldcg(pos + a), g = __ldcg(goal + a);
                const int tstar = plan_search<RW, RPL>(occ, sb, fh, tbl, H, lane, F, s, g);
                __syncwarp();
                if (tstar < 0) break;
                plan_read_back<RW, RPL>(sb, fh, tbl, d.L, lane, g, tstar, path);
                __syncwarp();
                plan_commit<RW, RPL, false>(occ, sb, tbl, H, lane, g, tstar, path, p, e, a);
                uint16_t *const pc = cand + (size_t)j * (H + 1);
                for (int t = lane; t <= H; t += 32) pc[t] = t <= tstar ? path[t] : (uint16_t)(g.x << 8 | g.y);
                if (lane == 0) arr_new[j] = (int16_t)tstar;
                soc += tstar;
                __syncwarp();
            }
            if (j == m && soc < old) {  // accepted: the candidates are in the tables already
                for (int q = 0; q < m; ++q) {
                    const int a = agent[q];
                    const uint16_t *const pc = cand + (size_t)q * (H + 1);
                    uint16_t *const pa = cur + (size_t)a * (H + 1);
                    for (int t = lane; t <= H; t += 32) pa[t] = pc[t];
                    if (lane == 0) arr_now[a] = arr_new[q];
                }
                ++acc;
            } else {  // rejected: the candidates planned so far out of the tables, the old paths back in
                for (int q = 0; q < j; ++q) {
                    plan_mark<RW, RPL, false>(occ, tbl, H, lane, cand + (size_t)q * (H + 1));
                    __syncwarp();
                }
                for (int q = 0; q < m; ++q) {
                    plan_mark<RW, RPL, true>(occ, tbl, H, lane, cur + (size_t)agent[q] * (H + 1));
                    __syncwarp();
                }
            }
            __syncwarp();
        }

        if (acc > 0) {  // the final paths: arrivals, and the actions that follow them (0 from the arrival on)
            for (int a = lane; a < n; a += 32) arr[a] = arr_now[a];
            for (int t = 0; t < H; ++t)
                for (int a = lane; a < n; a += 32) {
                    const uint16_t *const pa = cur + (size_t)a * (H + 1);
                    p.actions[((size_t)t * d.B + e) * d.N + a] = (uint8_t)plan_move(pa[t], pa[t + 1]);
                }
        }
        if (lane == 0) z.accepted[e] = acc;
        __syncwarp();
    }
}

// The soft search of one agent from s to g against the reservations in the tables (mapf_env_plan_repair): the layers
// F_c(0 .. t*) go into the history as a reached plane at lh and the layer's bit j at lh + (1 + j) * tbl.  Returns t*, the
// earliest t of least c(t) + park(t), and its cost and c(t*) in cost / cstar, or -1 where the goal is in no layer up to H.
// Layers below the lowest and above the highest non-empty one are skipped.  The search stops once t >= last_busy(g) and the
// best cost is at most the lowest non-empty layer: that layer never decreases with t and park(t) = 0 from last_busy(g) on,
// so no later t is cheaper.  The current slice's planes are read back from the history, so that no instantiation spills.
template <int RW, int RPL>
__device__ __forceinline__ int repair_search(const uint32_t *const occ, uint32_t *const lh, const size_t tbl, const int H, const int lane,
                                             const BfsFree<RW, RPL> &F, const uchar2 s, const uchar2 g, int &cost, int &cstar)
{
    constexpr int WPT = 32 * RPL * RW;
    constexpr int C = MAPF_PLAN_REPAIR_MAX_COLLISIONS;
    const uint32_t *const sb = occ;
    const size_t gi = plan_cell<RW, RPL>(g.x, g.y);
    const uint32_t gb = plan_bit(g.y);
    const int gl = g.x / RPL, gq = g.x % RPL, gw = (g.y + 4) >> 5;
    // last_busy(goal), and the count of t with the goal in Occ(t): park(t) = nb - seen(t), seen(t) = #{t' <= t : busy}
    int lb = -1;
    unsigned nb = 0;
#pragma unroll 4
    for (int t = lane; t <= H; t += 32)
        if (__ldcg(occ + (size_t)t * WPT + gi) & gb) lb = t, ++nb;
    lb = __reduce_max_sync(MAPF_FULL_MASK, lb);
    nb = __reduce_add_sync(MAPF_FULL_MASK, nb);
    int seen = (__ldcg(occ + gi) & gb) ? 1 : 0;

#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            const size_t o = (q * RW + w) * 32 + lane;
            __stcg(lh + o, (lane * RPL + q == s.x && ((s.y + 4) >> 5) == w) ? plan_bit(s.y) : 0u);
#pragma unroll
            for (int j = 1; j <= 4; ++j) __stcg(lh + j * tbl + o, 0u);
        }
    int best = INT_MAX, tstar = -1, cb = 0;
    if (s.x == g.x && s.y == g.y) best = (int)nb - seen, tstar = 0;
    int low = 0, top = 0;  // the lowest and the highest non-empty layer at t
    for (int t = 0; t < H && !(t >= lb && best <= low); ++t) {
        const size_t ot = (size_t)t * WPT;
        uint32_t on[RPL][RW], nr[RPL][RW], nbit[4][RPL][RW], rp[RPL][RW];  // Occ(t+1), reached at t+1, its bits, R_c-1(t)
#pragma unroll
        for (int q = 0; q < RPL; ++q)
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                on[q][w] = __ldcg(occ + ot + WPT + (q * RW + w) * 32 + lane);
                nr[q][w] = rp[q][w] = 0u;
#pragma unroll
                for (int j = 0; j < 4; ++j) nbit[j][q][w] = 0u;
            }
        int nlow = -1, ntop = -1;
        const int chi = min(top + 1, C);
#pragma unroll 1
        for (int c = low; c <= chi; ++c) {
            uint32_t fc[RPL][RW];  // F_c(t)
#pragma unroll
            for (int q = 0; q < RPL; ++q)
#pragma unroll
                for (int w = 0; w < RW; ++w) {
                    const size_t o = ot + (q * RW + w) * 32 + lane;
                    uint32_t x = 0u;
                    if (c <= top) {
                        x = __ldcg(lh + o);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint32_t b = __ldcg(lh + (1 + j) * tbl + o);
                            x &= (c >> j & 1) ? b : ~b;
                        }
                    }
                    fc[q][w] = x;
                }
            uint32_t any = 0;
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                uint32_t above, below;
                bfs_rows_around<RW, RPL, 32, false>(fc, w, lane, above, below);
#pragma unroll
                for (int q = 0; q < RPL; ++q) {
                    const size_t o = ot + (q * RW + w) * 32 + lane;
                    const uint32_t x = fc[q][w];
                    const uint32_t from_dn = q < RPL - 1 ? fc[q < RPL - 1 ? q + 1 : q][w] : below;  // action 1 (x-1)
                    const uint32_t from_up = q > 0 ? fc[q > 0 ? q - 1 : 0][w] : above;              // action 2 (x+1)
                    const uint32_t from_rt = w < RW - 1 ? __funnelshift_r(x, fc[q][w < RW - 1 ? w + 1 : w], 1) : x >> 1;  // 3
                    const uint32_t from_lt = w > 0 ? __funnelshift_l(fc[q][w > 0 ? w - 1 : 0], x, 1) : x << 1;            // 4
                    const uint32_t r = (x | (from_dn & ~__ldcg(sb + tbl + o)) | (from_up & ~__ldcg(sb + 2 * tbl + o)) |
                                        (from_rt & ~__ldcg(sb + 3 * tbl + o)) | (from_lt & ~__ldcg(sb + 4 * tbl + o))) & F.v[q][w];
                    const uint32_t nf = ((r & ~on[q][w]) | (rp[q][w] & on[q][w])) & ~nr[q][w];  // F_c(t+1)
                    rp[q][w] = r;
                    nr[q][w] |= nf;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (c >> j & 1) nbit[j][q][w] |= nf;
                    any |= nf;
                }
            }
            if (__any_sync(MAPF_FULL_MASK, any != 0)) {
                ntop = c;
                if (nlow < 0) nlow = c;
            }
        }
        uint32_t xr = 0, xo = 0;
        int xc = 0;
#pragma unroll
        for (int q = 0; q < RPL; ++q)
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                const size_t o = ot + WPT + (q * RW + w) * 32 + lane;
                __stcg(lh + o, nr[q][w]);
#pragma unroll
                for (int j = 0; j < 4; ++j) __stcg(lh + (1 + j) * tbl + o, nbit[j][q][w]);
                if (q == gq && w == gw) {
                    xr = nr[q][w], xo = on[q][w];
#pragma unroll
                    for (int j = 0; j < 4; ++j) xc |= (nbit[j][q][w] & gb) ? 1 << j : 0;
                }
            }
        low = nlow, top = ntop;
        if (top < 0) break;  // nothing reachable at t + 1
        seen += __any_sync(MAPF_FULL_MASK, lane == gl && (xo & gb)) ? 1 : 0;
        const int cg = __shfl_sync(MAPF_FULL_MASK, (xr & gb) ? xc : -1, gl);  // c(t+1)
        if (cg >= 0 && cg + (int)nb - seen < best) best = cg + (int)nb - seen, tstar = t + 1, cb = cg;
    }
    cost = best, cstar = cb;
    return tstar;
}

// The path back from (g, t*, c(t*)) into path[0 .. t*] (x << 8 | y): at (v, t, c) the layer c' = c - [v in Occ(t)], and lane
// k < 5 tests action k, whose predecessor must be in F_c'(t-1); the lowest admissible id wins
template <int RW, int RPL>
__device__ __forceinline__ void repair_read_back(const uint32_t *const occ, const uint32_t *const lh, const size_t tbl, const int L,
                                                 const int lane, const uchar2 g, const int tstar, int c, uint16_t *const path)
{
    constexpr int WPT = 32 * RPL * RW;
    const uint32_t *const sb = occ;
    int vx = g.x, vy = g.y;
    if (lane == 0) path[tstar] = (uint16_t)(vx << 8 | vy);
    for (int t = tstar; t >= 1; --t) {
        c -= (__ldcg(occ + (size_t)t * WPT + plan_cell<RW, RPL>(vx, vy)) & plan_bit(vy)) != 0;
        bool ok = false;
        if (lane < 5) {
            const int ux = vx - act_dx(lane), uy = vy - act_dy(lane);
            if (ux >= 0 && ux < L && uy >= 0 && uy < L) {
                const size_t o = (size_t)(t - 1) * WPT + plan_cell<RW, RPL>(ux, uy);
                const uint32_t b = plan_bit(uy);
                ok = (__ldcg(lh + o) & b) != 0;
                for (int j = 0; j < 4; ++j) ok &= ((__ldcg(lh + (1 + j) * tbl + o) & b) != 0) == ((c >> j & 1) != 0);
                if (ok && lane > 0) ok = (__ldcg(sb + lane * tbl + (size_t)(t - 1) * WPT + plan_cell<RW, RPL>(vx, vy)) & plan_bit(vy)) == 0;
            }
        }
        const unsigned m = __ballot_sync(MAPF_FULL_MASK, ok);
        const int k = m ? __ffs(m) - 1 : 0;
        vx -= act_dx(k), vy -= act_dy(k);
        if (lane == 0) path[t - 1] = (uint16_t)(vx << 8 | vy);
    }
}

// Clean tables (Occ, SB_1 .. SB_4, and with DUP the plane at occ + 5 * tbl), then the current paths cur[a][0 .. H] of the
// agents with skip[a] == 0 reserved; lane l owns the time slices l, l + 32, ..  Returns on every lane the reservations that
// found their Occ bit set already, the vertex excess of those agents whatever their order.  With DUP such a cell is set in
// the plane at occ + 5 * tbl.
template <int RW, int RPL, bool DUP>
__device__ __forceinline__ int repair_reserve(uint32_t *const occ, const size_t tbl, const int H, const int lane, const int n,
                                              const uint16_t *const cur, const uint8_t *const skip)
{
    constexpr int WPT = 32 * RPL * RW;
    {
        uint4 *zr = reinterpret_cast<uint4 *>(occ);
        const size_t n4 = (DUP ? 6 : 5) * tbl / 4;
        for (size_t i = lane; i < n4; i += 32) __stcg(zr + i, make_uint4(0u, 0u, 0u, 0u));
    }
    __syncwarp();
    unsigned hits = 0;
    for (int t = lane; t <= H; t += 32)
        for (int a = 0; a < n; ++a) {
            if (skip[a]) continue;
            const uint16_t *const pa = cur + (size_t)a * (H + 1);
            const int c = pa[t], x = c >> 8, y = c & 255;
            const size_t o = (size_t)t * WPT + plan_cell<RW, RPL>(x, y);
            const uint32_t b = plan_bit(y), old = __ldcg(occ + o);
            if (old & b) {
                ++hits;
                if constexpr (DUP) __stcg(occ + 5 * tbl + o, __ldcg(occ + 5 * tbl + o) | b);
            } else {
                __stcg(occ + o, old | b);
            }
            const int k = t < H ? plan_move(c, pa[t + 1]) : 0;
            if (k) {
                uint32_t *r = occ + (k & 1 ? k + 1 : k - 1) * tbl + o;
                __stcg(r, __ldcg(r) | b);
            }
        }
    __syncwarp();
    return (int)__reduce_add_sync(MAPF_FULL_MASK, hits);
}

// Plan repair (mapf_env_plan_repair): one warp per environment, the initial soft plan and all I iterations on it.  Per
// iteration the tables are built twice from the current paths: once with every agent, which marks the cells of more than one
// agent and so K, and once with the agents outside S, which gives G(X); S is then planned into them.
template <int RW, int RPL>
__global__ void __launch_bounds__(kPlanWarps * 32, RW * RPL <= 4 ? 3 : 1) plan_repair_kernel(const PlanArgs p, const RepairArgs z)
{
    __shared__ uint16_t s_path[kPlanWarps][MAPF_PLAN_MAX_HORIZON + 1];  // the agent being planned at t = 0 .. t*
    __shared__ uint8_t s_agent[kPlanWarps][MAPF_MAX_AGENTS];             // S in planning order
    __shared__ uint8_t s_ink[kPlanWarps][MAPF_MAX_AGENTS];               // a in K
    __shared__ uint8_t s_ins[kPlanWarps][MAPF_MAX_AGENTS];               // a in S
    __shared__ uint32_t s_key[kPlanWarps][MAPF_MAX_AGENTS];
    __shared__ int16_t s_arr[kPlanWarps][MAPF_MAX_AGENTS];               // each agent's current arrival
    __shared__ int16_t s_new[kPlanWarps][MAPF_MAX_AGENTS];               // the candidate arrival of S's j-th agent
    constexpr int WPT = 32 * RPL * RW;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const EnvDims &d = p.d;
    const int H = p.H;
    const size_t tbl = (size_t)(H + 1) * WPT;
    uint32_t *const occ = p.scratch + kPlanCounterWords + (size_t)(blockIdx.x * kPlanWarps + wid) * p.warp_words;
    uint32_t *const sb = occ;
    uint32_t *const lh = occ + 5 * tbl;                                            // the layer history, 5 tables
    uint16_t *const cur = reinterpret_cast<uint16_t *>(occ + kRepairTables * tbl);  // u16[N][H+1]: the current paths
    uint16_t *const cand = cur + (size_t)d.N * (H + 1);                            // u16[N][H+1]: S's j-th candidate in row j
    uint16_t *const path = s_path[wid];
    uint8_t *const agent = s_agent[wid], *const in_k = s_ink[wid], *const in_s = s_ins[wid];
    uint32_t *const key = s_key[wid];
    int16_t *const arr_now = s_arr[wid], *const arr_new = s_new[wid];

    for (;;) {
        unsigned e = 0;
        if (lane == 0) e = atomicAdd(p.scratch, 1u);
        e = __shfl_sync(MAPF_FULL_MASK, e, 0);
        if (e >= (unsigned)d.B) break;
        const int n = p.sz_n ? (int)__ldcg(p.sz_n + e) : d.N;
        const uchar2 *const pos = reinterpret_cast<const uchar2 *>(p.pos) + (size_t)e * d.N;
        const uchar2 *const goal = reinterpret_cast<const uchar2 *>(p.goal) + (size_t)e * d.N;
        int32_t *const arr = p.arrival + (size_t)e * d.N;

        // only a failed plan (every present arrival -1) is repaired
        bool failed = true;
        for (int a = lane; a < n; a += 32) failed &= __ldcg(arr + a) == -1;
        if (!__all_sync(MAPF_FULL_MASK, failed)) {
            if (lane == 0) z.collisions[e] = -2;
            continue;
        }

        {
            uint4 *zr = reinterpret_cast<uint4 *>(occ);
            const size_t n4 = 5 * tbl / 4;
            for (size_t i = lane; i < n4; i += 32) __stcg(zr + i, make_uint4(0u, 0u, 0u, 0u));
        }
        EnvDims df = d;  // the free cells: l_e x l_e on a sized handle
        if (p.sz_l) df.L = (int)__ldcg(p.sz_l + e);
        BfsFree<RW, RPL> F;
        bfs_load_free<RW, RPL, 1>(df, p.obst + (size_t)e * d.obst_stride, F);
        __syncwarp();

        // the initial plan: every agent in index order against the agents before it
        int G = 0, res = 0;
        for (int a = 0; a < n; ++a) {
            const uchar2 s = __ldcg(pos + a), g = __ldcg(goal + a);
            int cost, c;
            const int tstar = repair_search<RW, RPL>(occ, lh, tbl, H, lane, F, s, g, cost, c);
            __syncwarp();
            if (tstar < 0) {
                res = -1;
                break;
            }
            repair_read_back<RW, RPL>(occ, lh, tbl, d.L, lane, g, tstar, c, path);
            __syncwarp();
            plan_commit<RW, RPL, false>(occ, sb, tbl, H, lane, g, tstar, path, p, e, a);
            uint16_t *const pa = cur + (size_t)a * (H + 1);
            for (int t = lane; t <= H; t += 32) pa[t] = t <= tstar ? path[t] : (uint16_t)(g.x << 8 | g.y);
            if (lane == 0) arr_now[a] = (int16_t)tstar;
            G += cost;
            __syncwarp();
        }

        if (res == 0) {
            const int m = min(z.K, n);
            const uint64_t ge = z.env_offset + e;  // the environment's global index
            for (uint32_t i = 0; i < (uint32_t)z.I && G > 0; ++i) {
                // K: the agents on a cell of more than one agent at some t
                for (int a = lane; a < n; a += 32) in_k[a] = 0, in_s[a] = 0;
                __syncwarp();
                repair_reserve<RW, RPL, true>(occ, tbl, H, lane, n, cur, in_s);
                for (int t = lane; t <= H; t += 32)
                    for (int a = 0; a < n; ++a) {
                        const int c = cur[(size_t)a * (H + 1) + t], y = c & 255;
                        if (__ldcg(lh + (size_t)t * WPT + plan_cell<RW, RPL>(c >> 8, y)) & plan_bit(y)) in_k[a] = 1;
                    }
                for (int a = lane; a < n; a += 32)
                    key[a] = philox4x32_10(make_uint4((uint32_t)ge, (uint32_t)(ge >> 32), PURPOSE_REPAIR | (i << 8), (uint32_t)a), z.key).x;
                __syncwarp();
                // S: the first m agents by ([a not in K], k_a, a)
                for (int a = lane; a < n; a += 32) {
                    const uint64_t ka = (uint64_t)!in_k[a] << 32 | key[a];
                    int r = 0;
                    for (int b = 0; b < n; ++b) {
                        const uint64_t kb = (uint64_t)!in_k[b] << 32 | key[b];
                        r += kb < ka || (kb == ka && b < a);
                    }
                    if (r < m) agent[r] = (uint8_t)a, in_s[a] = 1;
                }
                __syncwarp();
                const int f_old = G - repair_reserve<RW, RPL, false>(occ, tbl, H, lane, n, cur, in_s);
                int old = 0;
                for (int j = 0; j < m; ++j) old += arr_now[agent[j]];
                int j = 0, f_new = 0, soc = 0;
                for (; j < m; ++j) {
                    const int a = agent[j];
                    const uchar2 s = __ldcg(pos + a), g = __ldcg(goal + a);
                    int cost, c;
                    const int tstar = repair_search<RW, RPL>(occ, lh, tbl, H, lane, F, s, g, cost, c);
                    __syncwarp();
                    if (tstar < 0) break;
                    repair_read_back<RW, RPL>(occ, lh, tbl, d.L, lane, g, tstar, c, path);
                    __syncwarp();
                    plan_commit<RW, RPL, false>(occ, sb, tbl, H, lane, g, tstar, path, p, e, a);
                    uint16_t *const pc = cand + (size_t)j * (H + 1);
                    for (int t = lane; t <= H; t += 32) pc[t] = t <= tstar ? path[t] : (uint16_t)(g.x << 8 | g.y);
                    if (lane == 0) arr_new[j] = (int16_t)tstar;
                    f_new += cost, soc += tstar;
                    __syncwarp();
                }
                if (j == m && (f_new < f_old || (f_new == f_old && soc < old))) {  // accepted
                    for (int q = 0; q < m; ++q) {
                        const uint16_t *const pc = cand + (size_t)q * (H + 1);
                        uint16_t *const pa = cur + (size_t)agent[q] * (H + 1);
                        for (int t = lane; t <= H; t += 32) pa[t] = pc[t];
                        if (lane == 0) arr_now[agent[q]] = arr_new[q];
                    }
                    G += f_new - f_old;
                }
                __syncwarp();
            }
            res = G;
        }

        // collision-free: the paths as plan() writes them; otherwise plan()'s failure form
        for (int a = lane; a < d.N; a += 32) arr[a] = res ? -1 : (a < n ? arr_now[a] : 0);
        for (int t = 0; t < H; ++t)
            for (int a = lane; a < d.N; a += 32) {
                const uint16_t *const pa = cur + (size_t)a * (H + 1);
                p.actions[((size_t)t * d.B + e) * d.N + a] = res || a >= n ? 0 : (uint8_t)plan_move(pa[t], pa[t + 1]);
            }
        if (lane == 0) z.collisions[e] = res;
        __syncwarp();
    }
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

template <int RW, int RPL>
int launch_plan_lns(mapf_env *env, int H, int I, int K, uint64_t seed, uint64_t env_offset, uint32_t first, uint8_t *d_actions,
                    int32_t *d_arrival, int32_t *d_accepted, cudaStream_t st)
{
    const EnvDims &d = env->d;
    // the six tables, then the current and the candidate paths (u16[N][H+1] each), rounded to 16 bytes
    const size_t warp_words = ((size_t)kPlanTables * (H + 1) * 32 * RPL * RW + (size_t)d.N * (H + 1) + 3) & ~(size_t)3;
    const int64_t block_bytes = (int64_t)kPlanWarps * warp_words * 4;
    int64_t blocks = 0;
    int rc = plan_blocks(env, plan_lns_kernel<RW, RPL>, d.B, block_bytes, blocks);
    if (rc != MAPF_OK) return rc;
    rc = reserve_plan_scratch(env, (int64_t)kPlanCounterWords * 4 + blocks * block_bytes, st, "mapf_env_plan_lns: scratch");
    if (rc != MAPF_OK) return rc;
    LnsArgs z;
    z.I = I, z.K = K, z.first = first;
    z.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    z.env_offset = env_offset;
    z.accepted = d_accepted;
    MAPF_CUDA(cudaMemsetAsync(env->pp_scratch, 0, 4, st));
    plan_lns_kernel<RW, RPL><<<(unsigned)blocks, kPlanWarps * 32, 0, st>>>(plan_args(env, H, warp_words, d_actions, d_arrival), z);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

template <int RW, int RPL>
int launch_plan_repair(mapf_env *env, int H, int I, int K, uint64_t seed, uint64_t env_offset, uint8_t *d_actions, int32_t *d_arrival,
                       int32_t *d_collisions, cudaStream_t st)
{
    const EnvDims &d = env->d;
    // the ten tables, then the current and the candidate paths (u16[N][H+1] each), rounded to 16 bytes
    const size_t warp_words = ((size_t)kRepairTables * (H + 1) * 32 * RPL * RW + (size_t)d.N * (H + 1) + 3) & ~(size_t)3;
    const int64_t block_bytes = (int64_t)kPlanWarps * warp_words * 4;
    int64_t blocks = 0;
    int rc = plan_blocks(env, plan_repair_kernel<RW, RPL>, d.B, block_bytes, blocks);
    if (rc != MAPF_OK) return rc;
    rc = reserve_plan_scratch(env, (int64_t)kPlanCounterWords * 4 + blocks * block_bytes, st, "mapf_env_plan_repair: scratch");
    if (rc != MAPF_OK) return rc;
    RepairArgs z;
    z.I = I, z.K = K;
    z.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    z.env_offset = env_offset;
    z.collisions = d_collisions;
    MAPF_CUDA(cudaMemsetAsync(env->pp_scratch, 0, 4, st));
    plan_repair_kernel<RW, RPL><<<(unsigned)blocks, kPlanWarps * 32, 0, st>>>(plan_args(env, H, warp_words, d_actions, d_arrival), z);
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

int mapf_launch_plan_lns(mapf_env *env, int H, int iterations, int neighborhood, uint64_t seed, uint64_t env_offset, uint32_t first_iteration,
                         uint8_t *d_actions, int32_t *d_arrival, int32_t *d_accepted, cudaStream_t st)
{
    const int rpl = (env->d.L + 31) / 32;
#define MAPF_PLAN_LNS_CASE(rw, r)                                                                                             \
    case rw * 8 + r:                                                                                                          \
        return launch_plan_lns<rw, r>(env, H, iterations, neighborhood, seed, env_offset, first_iteration, d_actions, d_arrival, \
                                      d_accepted, st)
    switch (env->d.RW * 8 + rpl) {
        MAPF_PLAN_LNS_CASE(1, 1);
        MAPF_PLAN_LNS_CASE(2, 1);
        MAPF_PLAN_LNS_CASE(2, 2);
        MAPF_PLAN_LNS_CASE(3, 2);
        MAPF_PLAN_LNS_CASE(3, 3);
        MAPF_PLAN_LNS_CASE(4, 3);
        MAPF_PLAN_LNS_CASE(4, 4);
    }
#undef MAPF_PLAN_LNS_CASE
    mapf_set_error("mapf_env_plan_lns: unsupported map size");
    return MAPF_EINVAL;
}

int mapf_launch_plan_repair(mapf_env *env, int H, int iterations, int neighborhood, uint64_t seed, uint64_t env_offset, uint8_t *d_actions,
                            int32_t *d_arrival, int32_t *d_collisions, cudaStream_t st)
{
    const int rpl = (env->d.L + 31) / 32;
#define MAPF_PLAN_REPAIR_CASE(rw, r) \
    case rw * 8 + r: return launch_plan_repair<rw, r>(env, H, iterations, neighborhood, seed, env_offset, d_actions, d_arrival, d_collisions, st)
    switch (env->d.RW * 8 + rpl) {
        MAPF_PLAN_REPAIR_CASE(1, 1);
        MAPF_PLAN_REPAIR_CASE(2, 1);
        MAPF_PLAN_REPAIR_CASE(2, 2);
        MAPF_PLAN_REPAIR_CASE(3, 2);
        MAPF_PLAN_REPAIR_CASE(3, 3);
        MAPF_PLAN_REPAIR_CASE(4, 3);
        MAPF_PLAN_REPAIR_CASE(4, 4);
    }
#undef MAPF_PLAN_REPAIR_CASE
    mapf_set_error("mapf_env_plan_repair: unsupported map size");
    return MAPF_EINVAL;
}
