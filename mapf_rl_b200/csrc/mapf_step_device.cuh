// mapf_step_device.cuh — device code shared by the step kernels (mapf_step_kernels.cu: one launch per step) and the
// persistent rollout kernel (mapf_rollout_kernels.cu): Environment.step (environment.py:278-430) fused with the observe()
// it ends in (environment.py:430, 433-467) for ONE environment handled by ONE warp, lane = agent (K = ceil(N/32) agents
// per lane).
//   1. all inputs of the env (positions, goals, actions, step counter, obstacle bitmap) are requested up front so their
//      DRAM/L2 latencies overlap;
//   2. conflict resolution runs in registers / shared memory (order-independent fixed point of the reference's
//      restart-on-change scans, SURVEY.md A.2);
//   3. every lane gathers its agent's 6 x 9 x 9 window as a 486-BIT stream (obstacle / agent bitmaps in shared memory,
//      heuristic bits from the agent's 16x16 navi tile) and streams it, word by word, into the env's dense bit stream in
//      shared memory;
//   4. the warp expands bits to bool bytes and writes the env's N*486-byte block with fully coalesced 128-bit stores.
#pragma once
#include <cstdlib>
#include <type_traits>

#include "mapf_common.cuh"

namespace {

enum : int {
    MAPF_STEPF_NAVI_KEEP = 1,      // heuristic-map loads carry an L2 evict_last policy
    MAPF_STEPF_OBS_POLICY = 2,     // observation stores carry an L2 evict_first policy (else st.global.cs)
    MAPF_STEPF_CHECK_UNIQUE = 16,  // post-step uniqueness check of the agents' cells (environment.py:424-428) -> MAPF_ERRBIT_UNIQUE
#ifdef MAPF_ENABLE_DIAG
    // diagnosis builds only (results are WRONG with these set; they bound the kernel from below)
    MAPF_STEPF_DIAG_NO_NAVI = 4,   // skip the heuristic-map loads
    MAPF_STEPF_DIAG_NO_STORE = 8,  // skip the observation stores
#endif
};

// reward codes (include/mapf_b200.h MAPF_RCODE_*): index into reward_fn; 5 = first observation of a re-generated
// environment (mapf_env_rollout with auto-reset), reward 0
enum : int { RC_MOVE = MAPF_RCODE_MOVE, RC_STAY_ON = MAPF_RCODE_STAY_ON, RC_STAY_OFF = MAPF_RCODE_STAY_OFF,
             RC_COLLISION = MAPF_RCODE_COLLISION, RC_FINISH = MAPF_RCODE_FINISH, RC_RESET = MAPF_RCODE_RESET };

// navi tile cache of the rollout kernel: one 16-row tile (128 B) per agent in shared memory, rows padded to this stride
constexpr int kTileStride = 18;  // u64 per agent slot: 144 B keeps every slot 16-byte aligned for cp.async

// 4 bits -> 4 bool bytes: bit b lands at bit 8b.  The four shifted copies of x (shifts 0,7,14,21)
// do not overlap for x < 16, so the multiply has no carries.
__device__ __forceinline__ uint32_t expand4(uint32_t x) { return (x * 0x00204081u) & 0x01010101u; }

__device__ __forceinline__ uint32_t smem_addr(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }

// reward_fn[c] without a dynamically indexed parameter array (that would push the whole struct to local memory)
__device__ __forceinline__ float reward_of(const StepParams &p, int c)
{
    float r = p.r[0];
    r = c == 1 ? p.r[1] : r;
    r = c == 2 ? p.r[2] : r;
    r = c == 3 ? p.r[3] : r;
    r = c == 4 ? p.r[4] : r;
    return c == 5 ? 0.0f : r;
}

__device__ __forceinline__ uint32_t window9(const uint32_t *row, int bitoff)
{
    const int w = bitoff >> 5;
    return __funnelshift_r(row[w], row[w + 1], bitoff & 31) & 0x1ffu;
}

__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint2 ldg_policy(const uint2 *ptr, uint64_t pol)
{
    uint2 v;
    asm("ld.global.nc.L2::cache_hint.v2.b32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ uint4 ldg_policy(const uint4 *ptr, uint64_t pol)
{
    uint4 v;
    asm("ld.global.nc.L2::cache_hint.v4.b32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ void stg_policy(uint4 *ptr, const uint4 &v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;"
                 :
                 : "l"(ptr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol)
                 : "memory");
}

// Compile-time walk over the 54 nine-bit fields (channel c = F / 9, window row u = F % 9) of one agent's
// observation bit stream.  A 64-bit accumulator collects fields; every completed 32-bit word is handed to
// `emit` immediately, so at most two stream words are live in registers at any time.  `mid` runs once, between the
// obstacle channel and the first heuristic channel (field 18).
template <int F>
struct FieldWalk {
    template <typename Val, typename Emit, typename Mid>
    __device__ __forceinline__ static void run(uint64_t acc, Val &&val, Emit &&emit, Mid &&mid)
    {
        constexpr int pos = 9 * F, m = pos >> 5, s = pos & 31;
        if constexpr (F == 18) mid();
        acc |= (uint64_t)val(std::integral_constant<int, F>{}) << s;
        if constexpr (s + 9 >= 32) {
            emit(std::integral_constant<int, m>{}, (uint32_t)acc);
            acc >>= 32;
        }
        if constexpr (F + 1 < 54) FieldWalk<F + 1>::run(acc, val, emit, mid);
        else emit(std::integral_constant<int, 15>{}, (uint32_t)acc);  // bits 480..485
    }
};

// Registers of one environment that outlive env_step_gather (final positions, to clear the agent bitmap).
template <int K>
struct EnvRegs {
    int px[K], py[K];
    bool valid[K];
    // carried from step to step by the persistent rollout kernel only:
    int gx[K], gy[K];  // goals
    int tile[K];       // navi tile (x >> 3) * NB + (y >> 3) held in the agent's shared-memory tile slot, -1 = none
    int act_next[K];   // the action of the NEXT step, requested one step ahead (the only global load of a resident step)
    int step;          // step counter
    bool finished;     // all agents stood on their goals after the last step (environment.py:415)
    int sel;           // navi_sel[e]: which heuristic-map buffer holds the live instance
};

// One warp, one environment: Environment.step (DO_STEP) and the observation BIT stream of all its agents.
// On return the env's N*486-bit stream sits in s_bits starting at bit `head` (every lane has passed a
// __syncwarp after its last write), positions / rewards / done / steps are stored, and the agent bitmap
// still holds this env's bits (clear_agent_bits undoes them).
// RESIDENT (persistent rollout kernel): the env's state is resident in the warp -- its obstacle bitmap sits in s_obst and
// positions, goals and the step counter arrive in `out` (loaded once per work item by the kernel), so a step starts with
// one load (the action); the heuristic rows come from the agent's tile slot in shared memory (`s_tiles`), refilled with
// cp.async only when the agent has moved to another tile (once in ~12 steps).  `reset_step`: the environment has just
// been re-generated -- nobody moves, rewards are 0, done is 0 and the step counter stays 0 (the call emits the new
// episode's first observation).  Actions are software-pipelined: out.act_next holds this step's actions (the kernel loads
// the first step's), `next_actions` (NULL on the last step of an item) is where the next step's are requested from.
// SIZED (sized handle, never RESIDENT): the environment has n_e = sz_n[e] agents on an l_e = sz_l[e] map
// inside the handle's N x L layout.  Agents a >= n_e are absent: their actions are never read, they hold no cell, their
// reward is 0 with code MAPF_RCODE_RESET and their 486-bit stream is zero.  A move outside l_e is a collision; the bitmap
// and the heuristic maps are zero outside l_e, so the gather itself needs no clipping.
// PACKED (never RESIDENT): agent a's stream starts at bit 512 a (MAPF_OBS_PACKED_BYTES_PER_AGENT) and `head` is 0, so every
// agent owns its 16 words: bits 486..511 are written as 0 and no word is shared with a neighbour.
template <int RW, int K, bool DO_STEP, bool DO_OBS = true, bool RESIDENT = false, bool SIZED = false, bool PACKED = false>
__device__ __forceinline__ void env_step_gather(const StepParams &p, const int e, const int lane, uint32_t *s_obst,
                                                uint32_t *s_agent, uint32_t *s_bits, uint16_t *s_tgt, uint16_t *s_cell,
                                                const int head, const uint64_t pol_keep, EnvRegs<K> &out,
                                                const uint8_t *s_act = nullptr, uint64_t *s_tiles = nullptr,
                                                const bool reset_step = false, const uint8_t *next_actions = nullptr,
                                                const uint8_t *sz_n = nullptr, const uint8_t *sz_l = nullptr)
{
    constexpr int RWS = RW + 1;
    const EnvDims &d = p.d;
    const int N = d.N, L = d.L;
    int NA = N, LB = L;  // agents present, bounds of a move
    if constexpr (SIZED) NA = __ldg(sz_n + e), LB = __ldg(sz_l + e);
    // The cell -> agent grid of the step phase lives in the bit-stream buffer (the two are never live at
    // the same time).  It is never cleared: an entry is trusted only if it round-trips through s_cell.
    uint8_t *s_occ = reinterpret_cast<uint8_t *>(s_bits);
    // RANKED (maps wider than 88 cells): L*L bytes of grid would be by far the largest buffer of the warp (14.4 KB at 120x120
    // against 7.8 KB of bit stream for 128 agents), so "who stands on cell c" is answered from the agent BITMAP of the old
    // positions instead: the occupant of a set bit is the agent whose cell has the same RANK among the set bits (row prefix
    // of popcounts + popcount of the bits below inside the row), looked up in a rank -> agent table of N bytes that is
    // rebuilt every step.  Claims of lower slots (K > 1) and the 'unique' check only need one bit per cell.
    //   s_bits: [0, claim_words) claim bitmap (bit = cell index) | u8 s_pref[R] rank of a row's first bit | u8 s_r2a[N]
    // Measured at 80x80 / 64 agents (RW = 3; profiles/r2_c4_ranked_lookup.jsonl): the ranked form lifts the whole-batch step
    // kernel from 20 to 32 resident warps per SM and changes nothing (42.1 us against 41.0-41.7: the ~100 extra instructions
    // per step cost what the occupancy gives; the rollout kernel loses 2 %), so the byte grid stays where it fits.  At 120x120 /
    // 128 agents x 4096 environments (RW = 4) the ranked form is 12 % faster in the rollout kernel (67.2 against 76.4 us per step)
    // and 14 % in the host-buffer step; with 1024 environments (7 warps per SM either way) the two are equal.
    constexpr bool RANKED = MAPF_RANKED_LOOKUP(RW);
    [[maybe_unused]] const int claim_words = ((L * L + 127) >> 7) << 2;
    [[maybe_unused]] uint8_t *s_pref = reinterpret_cast<uint8_t *>(s_bits + claim_words);
    [[maybe_unused]] uint8_t *s_r2a = s_pref + ((d.R + 3) & ~3);
    [[maybe_unused]] auto rank_of = [&](const int X, const int Y) {  // padded coordinates; set bits below (X, Y)
        const uint32_t *row = s_agent + X * RWS;
        int rk = s_pref[X];
        const int wq = Y >> 5;
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            const uint32_t m = w < wq ? 0xffffffffu : (w == wq ? ((1u << (Y & 31)) - 1u) : 0u);
            rk += __popc(row[w] & m);
        }
        return rk;
    };
    const bool navi_keep = p.flags & MAPF_STEPF_NAVI_KEEP;
    // the buffer that holds the slot's live heuristic maps (mapf_common.cuh)
    [[maybe_unused]] const uint32_t *navi_live = p.navi;
    if constexpr (DO_OBS) {
        if constexpr (RESIDENT) navi_live = out.sel ? p.navi_alt : p.navi;
        else if (p.navi_alt && __ldg(p.navi_sel + e)) navi_live = p.navi_alt;
    }
    {
        // ---- request every input of this env up front ----
        if constexpr (!RESIDENT) {
            // obstacle bitmap: global -> shared without passing through registers (LDGSTS), so nothing below
            // waits for it until the cp.async.wait_all in front of the first __syncwarp
            const uint4 *src = reinterpret_cast<const uint4 *>(p.obst + (size_t)e * d.obst_stride);
            const uint32_t dst = smem_addr(s_obst);
            for (int w = lane; w < (p.obst_words >> 2); w += 32)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * w), "l"(src + w) : "memory");
        }
        int px[K], py[K];
        bool valid[K];
        [[maybe_unused]] int gx[K], gy[K], act[K];
        [[maybe_unused]] int step_now = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int a = k * 32 + lane;
            valid[k] = a < NA;
            px[k] = py[k] = 0;
            if constexpr (DO_STEP) gx[k] = gy[k] = act[k] = 0;
            if constexpr (RESIDENT) {
                px[k] = out.px[k];
                py[k] = out.py[k];
                if constexpr (DO_STEP) {
                    gx[k] = out.gx[k];
                    gy[k] = out.gy[k];
                    // this step's action was requested during the previous step (the load's ~1 us of latency used to be the
                    // first thing every step waited for: 9 % of the kernel's stall samples); request the next one now
                    if (!reset_step) act[k] = out.act_next[k];
                    if (valid[k] && next_actions) out.act_next[k] = __ldg(next_actions + (size_t)e * N + a);
                }
            } else if (valid[k]) {
                const uchar2 pp = reinterpret_cast<const uchar2 *>(p.pos)[(size_t)e * N + a];
                px[k] = pp.x;
                py[k] = pp.y;
                if constexpr (DO_STEP) {
                    const uchar2 gg = __ldg(reinterpret_cast<const uchar2 *>(p.goal) + (size_t)e * N + a);
                    gx[k] = gg.x;
                    gy[k] = gg.y;
                    act[k] = s_act ? s_act[a] : __ldg(p.actions + (size_t)e * N + a);
                }
            }
        }
        if constexpr (DO_STEP)
            if (lane == 0) step_now = RESIDENT ? out.step : p.steps[e];
        [[maybe_unused]] bool finished = false;
        if constexpr (DO_STEP) {
            int tx[K], ty[K], tcell[K], mycell[K], occ_j[K];
            int code[K];
            bool mover[K], occ_ok[K], fail[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int a = k * 32 + lane;
                if (act[k] > 4) {  // environment.py:289-290 raises; we latch and treat as stay
                    atomicOr(p.err, MAPF_ERRBIT_ACTION);
                    act[k] = 0;
                }
                mycell[k] = px[k] * L + py[k];
                if constexpr (RANKED) {
                    // bitmap of the OLD positions (s_agent is all zero between environments / steps)
                    if (valid[k]) atomicOr(&s_agent[(px[k] + 4) * RWS + ((py[k] + 4) >> 5)], 1u << ((py[k] + 4) & 31));
                } else {
                    s_cell[a] = valid[k] ? (uint16_t)mycell[k] : (uint16_t)0xffff;
                    if (valid[k]) s_occ[mycell[k]] = (uint8_t)a;
                }
            }
            if constexpr (RANKED && K > 1) {  // claim bitmap: the last bit stream is still in there
                for (int w = lane; w < (claim_words >> 2); w += 32) reinterpret_cast<uint4 *>(s_bits)[w] = make_uint4(0, 0, 0, 0);
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();  // staged obstacle bitmap, s_cell and s_occ (the old-position bitmap) visible to every lane
            if constexpr (RANKED) {
                // rank of every row's first bit: lane owns rows RW*lane .. RW*lane + RW - 1 (R <= 32 RW)
                int cnt[RW], tot = 0;
#pragma unroll
                for (int i = 0; i < RW; ++i) {
                    const int row = lane * RW + i;
                    int c = 0;
                    if (row < d.R) {
#pragma unroll
                        for (int w = 0; w < RW; ++w) c += __popc(s_agent[row * RWS + w]);
                    }
                    cnt[i] = c;
                    tot += c;
                }
                int incl = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(MAPF_FULL_MASK, incl, o);
                    if (lane >= o) incl += v;
                }
                int run = incl - tot;
#pragma unroll
                for (int i = 0; i < RW; ++i) {
                    const int row = lane * RW + i;
                    if (row < d.R) s_pref[row] = (uint8_t)run;
                    run += cnt[i];
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                // stay / move pass, environment.py:298-311
                const bool on_goal = px[k] == gx[k] && py[k] == gy[k];
                code[k] = act[k] == 0 ? (on_goal ? RC_STAY_ON : RC_STAY_OFF) : RC_MOVE;
                mover[k] = valid[k] && act[k] != 0;
                // action table environment.py:12
                tx[k] = px[k] + (act[k] == 2) - (act[k] == 1);
                ty[k] = py[k] + (act[k] == 4) - (act[k] == 3);
                tcell[k] = tx[k] * L + ty[k];
                if (mover[k]) {
                    // round 1: out of range / obstacle, environment.py:320-332
                    bool bad = tx[k] < 0 || ty[k] < 0 || tx[k] >= LB || ty[k] >= LB;
                    if (!bad) bad = (s_obst[(tx[k] + 4) * RWS + ((ty[k] + 4) >> 5)] >> ((ty[k] + 4) & 31)) & 1u;
                    if (bad) {
                        code[k] = RC_COLLISION;
                        mover[k] = false;
                    }
                }
                s_tgt[k * 32 + lane] = mover[k] ? (uint16_t)tcell[k] : (uint16_t)0xffff;
            }
            __syncwarp();
            if constexpr (RANKED) {
#pragma unroll
                for (int k = 0; k < K; ++k)
                    if (valid[k]) s_r2a[rank_of(px[k] + 4, py[k] + 4)] = (uint8_t)(k * 32 + lane);
                __syncwarp();
            }
            // round 2: swap, environment.py:335-365 (order-independent form: both partners revert)
            bool swapped[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                occ_j[k] = 0xff;
                occ_ok[k] = false;
                swapped[k] = false;
                if (mover[k]) {
                    if constexpr (RANKED) {
                        const int X = tx[k] + 4, Y = ty[k] + 4;
                        if ((s_agent[X * RWS + (Y >> 5)] >> (Y & 31)) & 1u) {
                            occ_ok[k] = true;
                            occ_j[k] = s_r2a[rank_of(X, Y)];
                            swapped[k] = s_tgt[occ_j[k]] == (uint16_t)mycell[k];
                        }
                    } else {
                        const int j = s_occ[tcell[k]];
                        occ_ok[k] = j < N && s_cell[j] == (uint16_t)tcell[k];
                        occ_j[k] = j;
                        swapped[k] = occ_ok[k] && s_tgt[j] == (uint16_t)mycell[k];
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (swapped[k]) {
                    s_tgt[k * 32 + lane] = 0xffff;
                    mover[k] = false;
                    code[k] = RC_COLLISION;
                }
                if constexpr (RANKED) {  // every lookup is done: take the old positions out of the bitmap again
                    if (valid[k]) s_agent[(px[k] + 4) * RWS + ((py[k] + 4) >> 5)] = 0;
                }
            }
            __syncwarp();
            // round 3: vertex conflicts, environment.py:369-406, as the greatest fixed point:
            //   fail if the target's occupant is not a live mover,
            //   fail if not the lowest id among live movers with the same target (:389-394),
            //   fail if the target's occupant is a live mover that fails (propagates backwards).
#pragma unroll
            for (int k = 0; k < K; ++k) {
                fail[k] = mover[k] && occ_ok[k] && s_tgt[occ_j[k]] == 0xffff;
                bool lower_claim = false;
                if (K > 1 && k > 0 && mover[k]) {
                    if constexpr (RANKED) {
                        lower_claim = (s_bits[tcell[k] >> 5] >> (tcell[k] & 31)) & 1u;  // only live movers of lower slots set bits
                    } else {
                        const int c = s_occ[tcell[k]];  // claim left by a lower slot (verified, never cleared)
                        lower_claim = c < N && (c >> 5) < k && s_tgt[c] == (uint16_t)tcell[k];
                    }
                }
                const unsigned mcode = mover[k] ? (unsigned)tcell[k] : (0x10000u | lane);
                const unsigned m = __match_any_sync(MAPF_FULL_MASK, mcode);
                const bool first = (__ffs(m) - 1) == lane;
                if (mover[k] && (!first || lower_claim)) fail[k] = true;
                if (K > 1 && k + 1 < K) {
                    __syncwarp();
                    if (mover[k]) {
                        if constexpr (RANKED) atomicOr(&s_bits[tcell[k] >> 5], 1u << (tcell[k] & 31));
                        else s_occ[tcell[k]] = (uint8_t)(k * 32 + lane);
                    }
                    __syncwarp();
                }
            }
            for (;;) {
                unsigned fm[K];
#pragma unroll
                for (int k = 0; k < K; ++k) fm[k] = __ballot_sync(MAPF_FULL_MASK, fail[k]);
                bool changed = false;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    if (mover[k] && !fail[k] && occ_ok[k]) {
                        const int j = occ_j[k];
                        unsigned mj = fm[0];
#pragma unroll
                        for (int q = 1; q < K; ++q)
                            if ((j >> 5) == q) mj = fm[q];
                        if ((mj >> (j & 31)) & 1u) {
                            fail[k] = true;
                            changed = true;
                        }
                    }
                }
                if (!__any_sync(MAPF_FULL_MASK, changed)) break;
            }
            // commit, environment.py:410-421
            bool all_goal = true;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (mover[k]) {
                    if (fail[k]) code[k] = RC_COLLISION;
                    else {
                        px[k] = tx[k];
                        py[k] = ty[k];
                    }
                }
                all_goal = all_goal && (!valid[k] || (px[k] == gx[k] && py[k] == gy[k]));
            }
            finished = __all_sync(MAPF_FULL_MASK, all_goal);
            const bool done = finished && !reset_step;
            if (p.flags & MAPF_STEPF_CHECK_UNIQUE) {
                // environment.py:424-428: every agent must stand on a cell of its own (cannot fail after a correct step
                // from a valid state; catches states injected through set_state / load)
                __syncwarp();
                bool dup = false;
                if constexpr (RANKED) {
                    for (int w = lane; w < (claim_words >> 2); w += 32) reinterpret_cast<uint4 *>(s_bits)[w] = make_uint4(0, 0, 0, 0);
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (valid[k]) {
                            const int c = px[k] * L + py[k];
                            if ((atomicOr(&s_bits[c >> 5], 1u << (c & 31)) >> (c & 31)) & 1u) dup = true;
                        }
                } else {
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (valid[k]) s_occ[px[k] * L + py[k]] = (uint8_t)(k * 32 + lane);
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (valid[k] && s_occ[px[k] * L + py[k]] != (uint8_t)(k * 32 + lane)) dup = true;
                }
                if (__any_sync(MAPF_FULL_MASK, dup) && lane == 0) atomicOr(p.err, MAPF_ERRBIT_UNIQUE);
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int a = k * 32 + lane;
                if (valid[k]) {
                    const uchar2 np = make_uchar2((unsigned char)px[k], (unsigned char)py[k]);
                    reinterpret_cast<uchar2 *>(p.pos)[(size_t)e * N + a] = np;
                    if constexpr (!DO_OBS)
                        if (p.pos_out) reinterpret_cast<uchar2 *>(p.pos_out)[(size_t)e * N + a] = np;  // snapshot for a later observe
                    const int c = reset_step ? RC_RESET : (done ? RC_FINISH : code[k]);
                    if (p.rewards) p.rewards[(size_t)e * N + a] = reward_of(p, c);
                    if (p.codes) p.codes[(size_t)e * N + a] = (uint8_t)c;
                } else if constexpr (SIZED) {
                    if (a < N) {
                        if (p.rewards) p.rewards[(size_t)e * N + a] = 0.0f;
                        if (p.codes) p.codes[(size_t)e * N + a] = (uint8_t)RC_RESET;
                    }
                }
            }
            if (lane == 0) {
                const int st = reset_step ? 0 : step_now + 1;
                step_now = st - 1;
                p.steps[e] = st;
                if (p.steps_out) p.steps_out[e] = st;
                p.done[e] = done ? 1 : 0;
            }
        } else {
            if (p.pos_out) {
#pragma unroll
                for (int k = 0; k < K; ++k)
                    if (valid[k])
                        reinterpret_cast<uchar2 *>(p.pos_out)[(size_t)e * N + k * 32 + lane] =
                            make_uchar2((unsigned char)px[k], (unsigned char)py[k]);
                    else if constexpr (SIZED) {
                        if (k * 32 + lane < N) reinterpret_cast<uchar2 *>(p.pos_out)[(size_t)e * N + k * 32 + lane] = make_uchar2(255, 255);
                    }
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();  // s_obst visible
        }

        if constexpr (DO_OBS) {
        // ---------------- observe, environment.py:433-467 ----------------
        [[maybe_unused]] int tile[K];
        if constexpr (RESIDENT) {
            // tile slots: an agent that has moved to another 16x16 navi tile fetches its 128-byte line into its own slot
            // (global -> shared, no registers); the copy runs under the agent-bitmap and obstacle channels below
#pragma unroll
            for (int k = 0; k < K; ++k) {
                tile[k] = out.tile[k];
                const int a = k * 32 + lane;
                const int tid = (px[k] >> 3) * d.NB + (py[k] >> 3);
                if (valid[k] && tid != tile[k]) {
                    const uint4 *src = reinterpret_cast<const uint4 *>(navi_live + ((size_t)e * N + a) * d.navi_agent_stride) + ((size_t)tid << 3);
                    const uint32_t dst = smem_addr(s_tiles + (size_t)a * kTileStride);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * j), "l"(src + j) : "memory");
                    tile[k] = tid;
                }
            }
        }
        // agent bitmap (environment.py:449-451): one shared-memory atomic per agent
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (valid[k]) atomicOr(&s_agent[(px[k] + 4) * RWS + ((py[k] + 4) >> 5)], 1u << ((py[k] + 4) & 31));
        __syncwarp();  // also orders the last s_occ reads before the bit stream overwrites that buffer

#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int a = k * 32 + lane;
            // this agent's 486 bits start at stream bit (head + 486 a) = word f, bit o  (512 a when PACKED)
            const int gbit = PACKED ? 8 * MAPF_OBS_PACKED_BYTES_PER_AGENT * a : head + MAPF_OBS_BYTES_PER_AGENT * a;
            const int o = gbit & 31;
            uint32_t *S = s_bits + (gbit >> 5);
            uint32_t x0 = 0;
            if (valid[k]) {
                const int x = px[k], y = py[k];
                // window rows x-4..x+4 are padded rows x..x+8; columns y-4..y+4 are padded bits y..y+8: all inside
                // navi tile (x >> 3, y >> 3), rows (x & 7) .. (x & 7) + 8 of one 128-byte line
                uint2 wr[9];
                if constexpr (!RESIDENT) {
                    const uint2 *nb = reinterpret_cast<const uint2 *>(navi_live + ((size_t)e * N + a) * d.navi_agent_stride) +
                                      ((size_t)((x >> 3) * d.NB + (y >> 3)) << 4) + (x & 7);
#ifdef MAPF_ENABLE_DIAG
                    if (p.flags & MAPF_STEPF_DIAG_NO_NAVI) {
#pragma unroll
                        for (int u = 0; u < 9; ++u) wr[u] = make_uint2(x + u, y);
                    } else
#endif
                    {
                        // the nine rows as FIVE aligned 16-byte loads (ten rows from the even row at or below the first):
                        // every lane reads another line, so a warp-wide load costs 32 L1 wavefronts whatever its width --
                        // 160 per agent slot instead of 288 with nine 8-byte loads (whole-batch step at C2 35.8 -> 35.0 us,
                        // host-buffer step 5.7 -> 6.1 G agent-steps/s; profiles/r2_navi_row_loads.jsonl)
                        const uint4 *nq = reinterpret_cast<const uint4 *>(nb - (x & 1));
                        uint4 q[5];
                        if (navi_keep) {
#pragma unroll
                            for (int u = 0; u < 5; ++u) q[u] = ldg_policy(nq + u, pol_keep);
                        } else {
#pragma unroll
                            for (int u = 0; u < 5; ++u) q[u] = __ldg(nq + u);
                        }
                        const bool odd = x & 1;
#pragma unroll
                        for (int u = 0; u < 9; ++u) {
                            // row u of the window is loaded row u + odd; loaded row r = halves of q[r / 2]
                            const uint2 ev = (u & 1) ? make_uint2(q[u / 2].z, q[u / 2].w) : make_uint2(q[u / 2].x, q[u / 2].y);
                            const uint2 od = ((u + 1) & 1) ? make_uint2(q[(u + 1) / 2].z, q[(u + 1) / 2].w)
                                                           : make_uint2(q[(u + 1) / 2].x, q[(u + 1) / 2].y);
                            wr[u] = odd ? od : ev;
                        }
                    }
                }
                auto mid = [&]() {
                    if constexpr (RESIDENT) {
                        // the tile line(s) requested above have landed in this lane's own slot(s)
                        asm volatile("cp.async.wait_all;" ::: "memory");
                        const uint2 *rows = reinterpret_cast<const uint2 *>(s_tiles + (size_t)a * kTileStride) + (x & 7);
#pragma unroll
                        for (int u = 0; u < 9; ++u) wr[u] = rows[u];
                    }
                };
                const int sh = y & 7;
                const uint32_t *ag_row = s_agent + x * RWS, *ob_row = s_obst + x * RWS;
                uint32_t prev = 0;
                auto val = [&](auto fc) -> uint32_t {
                    constexpr int f = decltype(fc)::value, c = f / 9, u = f % 9;
                    if constexpr (c == 0) {
                        uint32_t v = window9(ag_row + u * RWS, y);
                        if constexpr (u == 4) v &= ~0x10u;  // own centre cleared, environment.py:461
                        return v;
                    } else if constexpr (c == 1) {
                        return window9(ob_row + u * RWS, y);
                    } else {
                        // direction dd = c - 2: 16 column bits at bit 16 dd of the tile row
                        constexpr int dd = c - 2;
                        const uint32_t half = dd < 2 ? wr[u].x : wr[u].y;
                        return (half >> (sh + 16 * (dd & 1))) & 0x1ffu;
                    }
                };
                auto emit = [&](auto mc, uint32_t w) {
                    constexpr int m = decltype(mc)::value;
                    if constexpr (m == 0) x0 = w << o;
                    else S[m] = __funnelshift_l(prev, w, o);
                    prev = w;
                };
                FieldWalk<0>::run(0ull, val, emit, mid);
                if (((o + 485) >> 5) == 16) S[16] = __funnelshift_l(prev, 0u, o);
            } else if constexpr (SIZED) {
                // an absent agent's 486 bits are zero (words it shares with its neighbours: see below)
                if (a < N) {
#pragma unroll
                    for (int m = PACKED ? 0 : 1; m < 16; ++m) S[m] = 0;
                    if (!PACKED && ((o + 485) >> 5) == 16) S[16] = 0;
                }
            }
            __syncwarp();
            // first word: shared with the previous agent's last word unless this agent starts a word
            bool streams = valid[k];
            if constexpr (SIZED && !PACKED) streams = a < N;
            if (streams) {
                if (PACKED || o == 0 || a == 0) S[0] = x0;
                else S[0] |= x0;
            }
            __syncwarp();
        }
        if constexpr (RESIDENT) {
#pragma unroll
            for (int k = 0; k < K; ++k) out.tile[k] = tile[k];
        }
        }  // DO_OBS

#pragma unroll
        for (int k = 0; k < K; ++k) {
            out.px[k] = px[k];
            out.py[k] = py[k];
            out.valid[k] = valid[k];
        }
        if constexpr (RESIDENT && DO_STEP) {
            out.step = step_now + 1;
            out.finished = finished;
        }
    }
}

template <int RW, int K>
__device__ __forceinline__ void clear_agent_bits(uint32_t *s_agent, const EnvRegs<K> &r)
{
    constexpr int RWS = RW + 1;
#pragma unroll
    for (int k = 0; k < K; ++k)
        if (r.valid[k]) s_agent[(r.px[k] + 4) * RWS + ((r.py[k] + 4) >> 5)] = 0;
    __syncwarp();
}

// Expand the env's bit stream (1 bit -> 1 bool byte) and write its N*486-byte observation block: 16 bytes per lane per
// store, fully coalesced streaming stores; `head` = bytes between the 16-byte boundary below obs_env and obs_env.
__device__ __forceinline__ void expand_store_block(const StepParams &p, uint8_t *obs_env, const int head, const size_t env_bytes,
                                                   const uint32_t *s_bits, const int lane, const bool obs_policy,
                                                   const uint64_t pol_stream)
{
    const int total = head + (int)env_bytes;
    const int c_lo = (head + 15) >> 4, c_hi = total >> 4;  // chunks [c_lo, c_hi) are whole
    uint8_t *obase = obs_env - head;                       // 16-byte aligned
    const uint16_t *S16 = reinterpret_cast<const uint16_t *>(s_bits);
#pragma unroll 4
    for (int c = c_lo + lane; c < c_hi; c += 32) {
        const uint32_t s = S16[c];
        uint4 v;
        v.x = expand4(s & 0xfu);
        v.y = expand4((s >> 4) & 0xfu);
        v.z = expand4((s >> 8) & 0xfu);
        v.w = expand4(s >> 12);
        uint4 *dst = reinterpret_cast<uint4 *>(obase + (c << 4));
#ifdef MAPF_ENABLE_DIAG
        if (p.flags & MAPF_STEPF_DIAG_NO_STORE) {
            if (v.x == 0xdeadbeefu) __stcs(dst, v);  // never true: keeps the expansion alive
        } else
#endif
        if (obs_policy) stg_policy(dst, v, pol_stream);
        else __stcs(dst, v);
    }
    // ragged first / last chunk of an unaligned observation block
    if ((head != 0 && lane == 0) || ((total & 15) != 0 && lane == 1)) {
        const int c = lane == 0 ? 0 : c_hi;
        const uint32_t s = S16[c];
        for (int b = 0; b < 16; ++b) {
            const int g = (c << 4) + b;
            if (g >= head && g < total) obase[g] = (uint8_t)((s >> b) & 1u);
        }
    }
}

// Store the env's packed frame (N * 64 bytes, already in stream order) with 16-byte streaming stores; obs_env is 16-byte
// aligned.
__device__ __forceinline__ void store_packed_block(uint8_t *obs_env, const int n_chunks, const uint32_t *s_bits, const int lane,
                                                   const bool obs_policy, const uint64_t pol_stream)
{
    const uint4 *src = reinterpret_cast<const uint4 *>(s_bits);
    uint4 *dst = reinterpret_cast<uint4 *>(obs_env);
#pragma unroll 4
    for (int c = lane; c < n_chunks; c += 32) {
        if (obs_policy) stg_policy(dst + c, src[c], pol_stream);
        else __stcs(dst + c, src[c]);
    }
}

}  // namespace
