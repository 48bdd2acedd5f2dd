// mapf_reset_device.cuh — device-side instance generation for ONE environment by ONE warp: Environment.reset / __init__
// without the host (environment.py:100-138 == :156-192, map_partition :21-70).  Called by reset_kernel
// (mapf_reset_kernels.cu) and by the persistent rollout kernel when an episode ends inside the launch
// (mapf_rollout_kernels.cu, worker.py:390,422-428).
//
// Lane = map row (rows lane + 32 q, RPL rows per lane), each row RW words of padded column bits -- the same bit-parallel
// representation the BFS uses, so nothing but registers and shuffles is needed:
//   * obstacle map: iid Bernoulli(density) per cell; density < 0 draws triangular(0, 0.33, 0.5) once per
//     environment (environment.py:100,156)
//   * components with >= 2 cells (map_partition keeps only those, :65-67) = free cells that have a free
//     4-neighbour; the map is redrawn while there are none (:107-110)
//   * agent i: start = uniform over all cells of components that still have >= 2 unused cells (the
//     reference picks a component with probability proportional to its remaining size and then a uniform
//     cell in it, :120-131 -- the same distribution), goal = uniform over the unused cells of the same
//     component (:133-135); a component left with < 2 unused cells is dropped (:137).  The component of
//     a start cell is found by a bit-parallel flood fill, cached between agents (almost every start
//     falls in the giant component).
// Randomness is counter-based (Philox4x32-10): the instance with global index g uses key (seed) and counters
// (g, purpose, index), so any sharding of a batch over GPUs draws the instances a single GPU would.  The RNG stream of the
// reference (numpy / random globals) is NOT reproduced: parity with the reference goes through Environment.load; this
// generator is tested distributionally against the reference, and instance by instance against a host restatement of the
// rules above (tests/generator_ref.py).
#pragma once
#include "mapf_common.cuh"

namespace {


__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// PURPOSE_LEVEL: the setting a sized handle's reset draws for the slot (reset_levels_kernel), counter (g, 3, 0)
// PURPOSE_ORDER: agent a's key in priority order r of the planner (plan_orders_kernel), counter (g, 4 | r << 8, a)
// PURPOSE_LNS: agent a's key in iteration i of plan improvement (plan_lns_kernel), counter (g, 5 | i << 8, a)
// PURPOSE_REPAIR: agent a's key in iteration i of plan repair (plan_repair_kernel), counter (g, 6 | i << 8, a)
enum : uint32_t {
    PURPOSE_DENSITY = 0, PURPOSE_MAP = 1, PURPOSE_AGENT = 2, PURPOSE_LEVEL = 3, PURPOSE_ORDER = 4, PURPOSE_LNS = 5, PURPOSE_REPAIR = 6
};

#ifdef MAPF_ENABLE_DIAG
// diagnosis build: cycles of the generator's phases for environment 0 (profiles/tools/r2_generator_phases.py); accumulated in
// registers and written once at the end (a global read-modify-write per tick would be what gets measured)
__device__ unsigned long long g_reset_cycles[8];
#define MAPF_RESET_TICK(slot)                 \
    do {                                      \
        const long long _now = clock64();     \
        _acc[slot] += _now - _t0;             \
        _t0 = _now;                           \
    } while (0)
#else
#define MAPF_RESET_TICK(slot) do {} while (0)
#endif

template <int RW, int RPL>
struct Bits {
    uint32_t v[RPL][RW];
};

// 4-neighbour dilation of a row-per-lane bitmap (the wave step of the BFS kernel)
template <int RW, int RPL>
__device__ __forceinline__ void dilate(const Bits<RW, RPL> &f, Bits<RW, RPL> &out, int lane)
{
#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            const uint32_t x = f.v[q][w];
            uint32_t fl = x << 1, fr = x >> 1;
            if (w > 0) fl |= f.v[q][w > 0 ? w - 1 : 0] >> 31;
            if (w < RW - 1) fr |= f.v[q][w < RW - 1 ? w + 1 : w] << 31;
            uint32_t up = __shfl_up_sync(MAPF_FULL_MASK, x, 1);
            uint32_t dn = __shfl_down_sync(MAPF_FULL_MASK, x, 1);
            uint32_t wrap_up = 0, wrap_dn = 0;
            if (q > 0) wrap_up = __shfl_sync(MAPF_FULL_MASK, f.v[q > 0 ? q - 1 : 0][w], 31);
            if (q < RPL - 1) wrap_dn = __shfl_sync(MAPF_FULL_MASK, f.v[q < RPL - 1 ? q + 1 : q][w], 0);
            if (lane == 0) up = wrap_up;
            if (lane == 31) dn = wrap_dn;
            out.v[q][w] = fl | fr | up | dn;
        }
}

template <int RW, int RPL>
__device__ __forceinline__ int count_bits(const Bits<RW, RPL> &m)
{
    int c = 0;
#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w) c += __popc(m.v[q][w]);
    return c;
}

// position of the n-th (0-based) set bit of m (n < popc(m)): five halving steps (__fns is a ~100-instruction sequence)
__device__ __forceinline__ int nth_set_bit(uint32_t m, int n)
{
    int pos = 0;
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const int c = __popc(m & ((1u << half) - 1u));
        if (n >= c) {
            n -= c;
            pos += half;
            m >>= half;
        }
    }
    return pos;
}

// Uniform pick among the set bits of a warp-wide bitmap: returns (row << 8) | padded column, or -1 if the
// bitmap is empty.  `total_out` receives the number of set bits.  The pick is the r-th set bit in (lane, q, w, bit) order,
// r = floor(rnd * total / 2^32).  Written for LATENCY -- an in-launch re-generation runs two picks per agent on one warp, and
// they were two thirds of the generator's 54 us (profiles/r2_generator_phases.jsonl): the exclusive prefix of the per-lane
// counts comes from bit-sliced ballots (independent votes instead of a five-step shuffle scan), the bit inside the owning
// word from nth_set_bit, and the owner's answer reaches the warp through one OR-reduction.
template <int RW, int RPL>
__device__ __forceinline__ int pick_bit(const Bits<RW, RPL> &m, uint32_t rnd, int lane, int &total_out)
{
    constexpr int kMax = 32 * RW * RPL;                                    // a lane's count is at most this
    constexpr int kBits = kMax >= 512 ? 10 : (kMax >= 256 ? 9 : (kMax >= 128 ? 8 : (kMax >= 64 ? 7 : 6)));
    const int c = count_bits(m);
    const uint32_t lt = (1u << lane) - 1u;
    int excl = 0, total = 0;
#pragma unroll
    for (int k = 0; k < kBits; ++k) {
        const uint32_t b = __ballot_sync(MAPF_FULL_MASK, (c >> k) & 1);
        excl += __popc(b & lt) << k;
        total += __popc(b) << k;
    }
    total_out = total;
    if (total == 0) return -1;
    const int r = (int)__umulhi(rnd, (uint32_t)total);
    int local = r - excl;
    uint32_t code = 0;
    if (local >= 0 && local < c) {
        bool found = false;
#pragma unroll
        for (int q = 0; q < RPL; ++q)
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                const int pc = __popc(m.v[q][w]);
                if (!found && local < pc) {
                    code = (uint32_t)((((lane + 32 * q) << 8) | (32 * w + nth_set_bit(m.v[q][w], local))) + 1);
                    found = true;
                }
                if (!found) local -= pc;
            }
    }
    return (int)__reduce_or_sync(MAPF_FULL_MASK, code) - 1;  // exactly one lane owns the r-th bit
}

template <int RW, int RPL>
__device__ __forceinline__ void clear_cell(Bits<RW, RPL> &m, int code, int lane)
{
    const int row = code >> 8, col = code & 0xff;
#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w)
            if (lane + 32 * q == row && (col >> 5) == w) m.v[q][w] &= ~(1u << (col & 31));
}

template <int RW, int RPL>
__device__ __forceinline__ bool test_cell(const Bits<RW, RPL> &m, int code, int lane)
{
    const int row = code >> 8, col = code & 0xff;
    bool hit = false;
#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w)
            if (lane + 32 * q == row && (col >> 5) == w) hit = (m.v[q][w] >> (col & 31)) & 1u;
    return __any_sync(MAPF_FULL_MASK, hit);
}

// All 32 lanes of the warp call together.  Writes obst / pos / goal of environment e and steps[e] = 0.
// The instance has N <= d.N agents on an L <= d.L map (a sized handle's slot; rows N.. of pos / goal are not written).  The
// draw does not depend on the template's capacity: the map is keyed by row and quad, and the picks run in lane-major row
// order, in which rows past L are empty.
template <int RW, int RPL>
__device__ __forceinline__ void reset_env_warp(const EnvDims &d, const int e, const uint64_t seed, const uint64_t g,
                                               const float density, uint32_t *__restrict__ obst, uint8_t *__restrict__ pos,
                                               uint8_t *__restrict__ goal, int32_t *__restrict__ steps, int32_t *__restrict__ err,
                                               const int L, const int N)
{
    const int lane = threadIdx.x & 31;
    const int NS = d.N;  // row stride of pos / goal
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t g_lo = (uint32_t)g, g_hi = (uint32_t)(g >> 32);

    // environment.py:100 / :156 — one density per environment
    float dens = density;
    if (density < 0.f) {
        const uint4 r = philox4x32_10(make_uint4(g_lo, g_hi, PURPOSE_DENSITY, 0u), key);
        const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);  // [0, 1)
        // inverse CDF of triangular(a = 0, c = 0.33, b = 0.5): F(c) = (c - a) / (b - a) = 0.66
        dens = u < 0.66f ? sqrtf(u * 0.5f * 0.33f) : 0.5f - sqrtf((1.0f - u) * 0.5f * 0.17f);
    }
    const uint32_t thresh = dens <= 0.f ? 0u : (dens >= 1.f ? 0xffffffffu : (uint32_t)((double)dens * 4294967296.0));

    // `comp` caches the component of the last start cell, `big` the largest component filled so far: almost every start falls
    // into the giant component, but every start that does not used to evict it from the (single) cache and the next agent
    // paid for another ~70-iteration flood fill of the giant component -- half of the generator's instructions at density 0.3
    Bits<RW, RPL> fre, elig, comp, big;
    int big_n = 0;
#ifdef MAPF_ENABLE_DIAG
    long long _t0 = clock64();
    long long _acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
    for (uint32_t attempt = 0;; ++attempt) {
        if (attempt >= 256) {  // practically unreachable: e.g. density ~1 or more agents than usable cells
            if (lane == 0) atomicOr(err, MAPF_ERRBIT_RESET);
            break;
        }
        // ---- obstacle map: one Philox call per 4 cells ----
#pragma unroll
        for (int q = 0; q < RPL; ++q) {
            const int row = lane + 32 * q;
#pragma unroll
            for (int w = 0; w < RW; ++w) fre.v[q][w] = 0;
            if (row < L) {
                for (int y4 = 0; y4 < L; y4 += 4) {
                    const uint4 r = philox4x32_10(make_uint4(g_lo, g_hi, PURPOSE_MAP | (attempt << 8), (uint32_t)(row * 64 + (y4 >> 2))), key);
                    // the four cells as one nibble at padded column y4 + 4 (a multiple of 4: it never straddles two words)
                    uint32_t nib = (r.x >= thresh ? 1u : 0u) | (r.y >= thresh ? 2u : 0u) | (r.z >= thresh ? 4u : 0u) | (r.w >= thresh ? 8u : 0u);
                    if (y4 + 4 > L) nib &= (1u << (L - y4)) - 1u;
                    const int p = y4 + 4;
#pragma unroll
                    for (int w = 0; w < RW; ++w)
                        if ((p >> 5) == w) fre.v[q][w] |= nib << (p & 31);
                }
            }
        }
        MAPF_RESET_TICK(0);  // map
        // ---- cells of components with >= 2 cells: free with a free neighbour ----
        dilate(fre, elig, lane);
#pragma unroll
        for (int q = 0; q < RPL; ++q)
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                elig.v[q][w] &= fre.v[q][w];
                comp.v[q][w] = 0;
                big.v[q][w] = 0;
            }
        big_n = 0;
        // ---- agents ----
        bool ok = true;
        MAPF_RESET_TICK(1);  // eligibility
        // the agents' draws, all at once: lane l holds those of agents l, l + 32, ... (the loop below is one dependent chain per
        // agent; ten Philox rounds at its head were 200 cycles of it)
        uint32_t draw_x[MAPF_MAX_AGENTS / 32], draw_y[MAPF_MAX_AGENTS / 32];
#pragma unroll
        for (int k = 0; k < MAPF_MAX_AGENTS / 32; ++k) {
            draw_x[k] = draw_y[k] = 0;
            if (k * 32 < N) {
                const uint4 r = philox4x32_10(make_uint4(g_lo, g_hi, PURPOSE_AGENT | (attempt << 8), (uint32_t)(k * 32 + lane)), key);
                draw_x[k] = r.x, draw_y[k] = r.y;
            }
        }
        for (int i = 0; i < N; ++i) {
            uint2 r = make_uint2(0u, 0u);
#pragma unroll
            for (int k = 0; k < MAPF_MAX_AGENTS / 32; ++k)
                if ((i >> 5) == k) r = make_uint2(__shfl_sync(MAPF_FULL_MASK, draw_x[k], i & 31), __shfl_sync(MAPF_FULL_MASK, draw_y[k], i & 31));
            MAPF_RESET_TICK(2);  // agent draw
            int total;
            const int s = pick_bit(elig, r.x, lane, total);
            MAPF_RESET_TICK(3);  // first pick
            if (s < 0) {  // the reference regenerates the map (:107-110) / would raise mid-way; we redraw
                ok = false;
                break;
            }
            if (!test_cell(comp, s, lane) && big_n > 0 && test_cell(big, s, lane)) {
#pragma unroll
                for (int q = 0; q < RPL; ++q)
#pragma unroll
                    for (int w = 0; w < RW; ++w) comp.v[q][w] = big.v[q][w];
            } else if (!test_cell(comp, s, lane)) {
                // flood fill the component of s over the full free map
#pragma unroll
                for (int q = 0; q < RPL; ++q)
#pragma unroll
                    for (int w = 0; w < RW; ++w) comp.v[q][w] = 0;
                {
                    const int row = s >> 8, col = s & 0xff;
#pragma unroll
                    for (int q = 0; q < RPL; ++q)
#pragma unroll
                        for (int w = 0; w < RW; ++w)
                            if (lane + 32 * q == row && (col >> 5) == w) comp.v[q][w] = 1u << (col & 31);
                }
                for (;;) {
                    // four dilations per vote (a converged fill is a fixed point: the extra ones change nothing)
                    uint32_t grew = 0;
#pragma unroll
                    for (int rep = 0; rep < 4; ++rep) {
                        Bits<RW, RPL> nb;
                        dilate(comp, nb, lane);
                        grew = 0;
#pragma unroll
                        for (int q = 0; q < RPL; ++q)
#pragma unroll
                            for (int w = 0; w < RW; ++w) {
                                const uint32_t add = nb.v[q][w] & fre.v[q][w] & ~comp.v[q][w];
                                comp.v[q][w] |= add;
                                grew |= add;
                            }
                    }
                    if (!__any_sync(MAPF_FULL_MASK, grew != 0)) break;
                }
                const int n = __reduce_add_sync(MAPF_FULL_MASK, count_bits(comp));
                if (n > big_n) {
                    big_n = n;
#pragma unroll
                    for (int q = 0; q < RPL; ++q)
#pragma unroll
                        for (int w = 0; w < RW; ++w) big.v[q][w] = comp.v[q][w];
                }
            }
            MAPF_RESET_TICK(4);  // component (cache test / flood fill)
            clear_cell(elig, s, lane);
            Bits<RW, RPL> cand;
#pragma unroll
            for (int q = 0; q < RPL; ++q)
#pragma unroll
                for (int w = 0; w < RW; ++w) cand.v[q][w] = elig.v[q][w] & comp.v[q][w];
            int cnt;
            const int t = pick_bit(cand, r.y, lane, cnt);  // cnt >= 1: the component was eligible
            clear_cell(elig, t, lane);
            if (cnt - 1 < 2) {  // environment.py:137
#pragma unroll
                for (int q = 0; q < RPL; ++q)
#pragma unroll
                    for (int w = 0; w < RW; ++w) elig.v[q][w] &= ~comp.v[q][w];
            }
            MAPF_RESET_TICK(5);  // second pick + bookkeeping
            if (lane == 0) {
                const size_t o = ((size_t)e * NS + i) * 2;
                pos[o] = (uint8_t)(s >> 8);
                pos[o + 1] = (uint8_t)((s & 0xff) - 4);
                goal[o] = (uint8_t)(t >> 8);
                goal[o + 1] = (uint8_t)((t & 0xff) - 4);
            }
            MAPF_RESET_TICK(6);  // stores
        }
        if (ok) break;
    }

    // ---- store the padded obstacle bitmap (border rows / spare word zero), steps = 0 ----
    uint32_t *ob = obst + (size_t)e * d.obst_stride;
    for (int w = lane; w < d.obst_stride; w += 32) {
        const int prow = w / d.RWS;
        if (prow < 4 || prow >= L + 4 || w - prow * d.RWS >= RW) ob[w] = 0;
    }
#pragma unroll
    for (int q = 0; q < RPL; ++q) {
        const int row = lane + 32 * q;
        if (row < L) {
#pragma unroll
            for (int w = 0; w < RW; ++w) {
                const int lo = max(4 - 32 * w, 0), hi = min(L + 4 - 32 * w, 32);
                uint32_t cm = 0;
                if (hi > lo) cm = (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
                ob[(row + 4) * d.RWS + w] = ~fre.v[q][w] & cm;
            }
        }
    }
    if (lane == 0) steps[e] = 0;
#ifdef MAPF_ENABLE_DIAG
    MAPF_RESET_TICK(7);  // bitmap store
    if (e == 0 && lane == 0)
        for (int i = 0; i < 8; ++i) g_reset_cycles[i] = (unsigned long long)_acc[i];
#endif
}

template <int RW, int RPL>
__device__ __forceinline__ void reset_env_warp(const EnvDims &d, const int e, const uint64_t seed, const uint64_t g,
                                               const float density, uint32_t *__restrict__ obst, uint8_t *__restrict__ pos,
                                               uint8_t *__restrict__ goal, int32_t *__restrict__ steps, int32_t *__restrict__ err)
{
    reset_env_warp<RW, RPL>(d, e, seed, g, density, obst, pos, goal, steps, err, d.L, d.N);
}

}  // namespace
