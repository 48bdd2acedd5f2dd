// mapf_bfs_device.cuh — K3 as a warp-level device function: Environment.get_navi_map (environment.py:217-276) for the
// APW agents of one warp.  Called by bfs_navi_kernel (mapf_env_kernels.cu: load / reset) and by the persistent rollout
// kernel when an environment is re-generated inside the launch (mapf_rollout_kernels.cu).
//
// Lane l of an agent's group owns the RPL consecutive map rows RPL*l .. RPL*l + RPL - 1 (blocked, so that only the first and
// the last of them need a neighbour lane: two shuffles per word and wave whatever RPL is), each row RW words
// of padded column bits.  One wave:
//   new = (frontier shifted to the four neighbours) & free-and-unvisited
// Adjacent reachable cells of a 4-connected grid differ by exactly one in distance, so the heuristic bit "neighbour in
// direction d is strictly closer" (environment.py:260-274) is "its distance mod 3 is mine minus one": the loop only
// records which residue a cell's wave had and the four direction planes are derived once after the last wave.
// APW agents share a warp (LW = 32 / APW lanes each): maps of up to 48 rows fit 16 lanes x 3 rows, so two agents' waves
// run in one instruction stream; the warp iterates until both are done.
// All 32 lanes must call together; `alive` = this lane's group has an agent (a, of environment e; i = its index in
// dist_out's leading dimension).  Obstacle rows and goals are read with ld.global.cg: inside the rollout kernel they were
// written by this very launch.
#pragma once
#include <type_traits>

#include "mapf_common.cuh"

namespace {

#ifdef MAPF_ENABLE_DIAG
// diagnosis build: cycles of a search's phases, summed over the searches of environment 0 ([0] init, [1] waves, [2] emit,
// [3] searches, [4] wave triples); one atomic per search
__device__ unsigned long long g_bfs_cycles[8];
#endif

// state of one agent's search in its lanes' registers
template <int RW, int RPL>
struct BfsState {
    uint32_t unv[RPL][RW];  // free and not yet visited
    uint32_t fro[RPL][RW];  // frontier of the previous wave
    uint32_t m1[RPL][RW];   // cells whose wave number is 1 mod 3
    uint32_t m2[RPL][RW];   // ... 2 mod 3 (reached cells in neither: 0 mod 3)
};

// in-map column mask of word w: padded bits [4, L + 4)
__device__ __forceinline__ uint32_t bfs_column_mask(int L, int w)
{
    const int lo = max(4 - 32 * w, 0), hi = min(L + 4 - 32 * w, 32);
    if (hi <= lo) return 0u;
    return (hi - lo == 32) ? 0xffffffffu : (((1u << (hi - lo)) - 1u) << lo);
}

// free cells of this lane's map rows: the same for every agent of the environment (a caller that searches for one agent
// after the other loads them once)
template <int RW, int RPL>
struct BfsFree {
    uint32_t v[RPL][RW];
};

template <int RW, int RPL, int APW>
__device__ __forceinline__ void bfs_load_free(const EnvDims &d, const uint32_t *ob, BfsFree<RW, RPL> &F)
{
    constexpr int LW = 32 / APW;
    const int lane = (threadIdx.x & 31) % LW;    // lane within the agent's group
#pragma unroll
    for (int q = 0; q < RPL; ++q) {
        const int row = lane * RPL + q;
#pragma unroll
        for (int w = 0; w < RW; ++w)
            F.v[q][w] = (row < d.L) ? (~__ldcg(ob + (row + 4) * d.RWS + w) & bfs_column_mask(d.L, w)) : 0u;
    }
}

template <int RW, int RPL, int APW>
__device__ __forceinline__ void bfs_init(const EnvDims &d, const BfsFree<RW, RPL> &F, const int gx, const int gy, const bool alive,
                                         BfsState<RW, RPL> &S)
{
    constexpr int LW = 32 / APW;
    const int lane = (threadIdx.x & 31) % LW;
#pragma unroll
    for (int q = 0; q < RPL; ++q) {
        const int row = lane * RPL + q;
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            const uint32_t fre = alive ? F.v[q][w] : 0u;  // a group without an agent owns no rows
            const int p = gy + 4;
            S.fro[q][w] = (row == gx && (p >> 5) == w) ? ((1u << (p & 31)) & fre) : 0u;
            S.unv[q][w] = fre & ~S.fro[q][w];
            S.m1[q][w] = S.m2[q][w] = 0;
        }
    }
}

// Word w of the rows of the neighbouring lanes that touch this lane's block: the last row of the lane above and the first
// row of the lane below, 0 past the group's ends.
// WRAP: the group's last row is past the map (L < LW * RPL), so the neighbour rows can come from a rotating shuffle with
// nothing to zero at the group's ends -- the first lane receives the last lane's (empty) last row, and what the last lane
// receives lands on that empty row, where free-and-unvisited is 0.
template <int RW, int RPL, int LW, bool WRAP>
__device__ __forceinline__ void bfs_rows_around(const uint32_t (&f)[RPL][RW], const int w, const int lane, uint32_t &above,
                                                uint32_t &below)
{
    if constexpr (WRAP) {
        above = __shfl_sync(MAPF_FULL_MASK, f[RPL - 1][w], (lane + LW - 1) & (LW - 1), LW);
        below = __shfl_sync(MAPF_FULL_MASK, f[0][w], (lane + 1) & (LW - 1), LW);
    } else {
        above = __shfl_up_sync(MAPF_FULL_MASK, f[RPL - 1][w], 1, LW);
        below = __shfl_down_sync(MAPF_FULL_MASK, f[0][w], 1, LW);
        if (lane == 0) above = 0;
        if (lane == LW - 1) below = 0;
    }
}

// One wave: nw = (frontier shifted to the four neighbours) & free-and-unvisited; returns the OR of this lane's words.
template <int RW, int RPL, int APW, bool WRAP>
__device__ __forceinline__ uint32_t bfs_wave(const BfsState<RW, RPL> &S, uint32_t (&nw)[RPL][RW])
{
    constexpr int LW = 32 / APW;
    const int lane = (threadIdx.x & 31) % LW;
    uint32_t any = 0;
#pragma unroll
    for (int w = 0; w < RW; ++w) {
        uint32_t above, below;
        bfs_rows_around<RW, RPL, LW, WRAP>(S.fro, w, lane, above, below);
#pragma unroll
        for (int q = 0; q < RPL; ++q) {
            const uint32_t f = S.fro[q][w];
            const uint32_t fl = w > 0 ? __funnelshift_l(S.fro[q][w > 0 ? w - 1 : 0], f, 1) : f << 1;
            const uint32_t fr = w < RW - 1 ? __funnelshift_r(f, S.fro[q][w < RW - 1 ? w + 1 : w], 1) : f >> 1;
            const uint32_t up = q > 0 ? S.fro[q > 0 ? q - 1 : 0][w] : above;
            const uint32_t dn = q < RPL - 1 ? S.fro[q < RPL - 1 ? q + 1 : q][w] : below;
            const uint32_t x = (fl | fr | up | dn) & S.unv[q][w];
            nw[q][w] = x;
            any |= x;
        }
    }
    return any;
}

template <int RW, int RPL, int SEL>
__device__ __forceinline__ void bfs_apply(BfsState<RW, RPL> &S, const uint32_t (&nw)[RPL][RW])
{
#pragma unroll
    for (int q = 0; q < RPL; ++q)
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            // nw is a subset of unv and disjoint from the residue planes: clearing / setting its bits is a subtraction / an
            // addition, which the compiler can place on the FMA pipe (IMAD.IADD) -- the search is bound by the ALU pipe
            // (LOP3 / SHF at half rate: ncu math-pipe throttle), the FMA pipe is idle
            S.unv[q][w] -= nw[q][w];
            S.fro[q][w] = nw[q][w];
            if constexpr (SEL == 1) S.m1[q][w] += nw[q][w];
            if constexpr (SEL == 2) S.m2[q][w] += nw[q][w];
        }
}

// The four heuristic planes from the residues -- with z = reached cells of residue 0, "neighbour n is closer" holds at a
// cell c iff (c in m1, n in z) or (c in m2, n in m1) or (c in z, n in m2) -- emitted as the overlapping 16x16 tiles
// (mapf_common.cuh): a map row is padded row pr = row + 4, which is row pr & 7 of tile row-block pr >> 3 and row
// (pr & 7) + 8 of the block above.
// KEEP: the caller's free rows are still live (one agent after the other with the rows loaded once); else they are read
// again here, which keeps them out of the wave loop's register budget (the 64-register load / reset kernels).
template <int RW, int RPL, int APW, bool KEEP>
__device__ __forceinline__ void bfs_emit(const EnvDims &d, const uint32_t *ob, const BfsFree<RW, RPL> &F, const int e, const int a,
                                         const bool alive, const BfsState<RW, RPL> &S, uint32_t *__restrict__ navi)
{
    constexpr int LW = 32 / APW;
    const int lane = (threadIdx.x & 31) % LW;
    uint32_t pl[4][RPL][RW];
    uint32_t z[RPL][RW];
#pragma unroll
    for (int q = 0; q < RPL; ++q) {
        const int row = alive ? lane * RPL + q : d.L;
#pragma unroll
        for (int w = 0; w < RW; ++w) {
            uint32_t fre;
            if constexpr (KEEP) fre = alive ? F.v[q][w] : 0u;
            else fre = (row < d.L) ? (~__ldcg(ob + (row + 4) * d.RWS + w) & bfs_column_mask(d.L, w)) : 0u;
            z[q][w] = fre & ~S.unv[q][w] & ~S.m1[q][w] & ~S.m2[q][w];
        }
    }
    auto closer = [](uint32_t c1, uint32_t c2, uint32_t cz, uint32_t n1, uint32_t n2, uint32_t nz) -> uint32_t {
        return (c1 & nz) | (c2 & n1) | (cz & n2);
    };
#pragma unroll
    for (int w = 0; w < RW; ++w) {
        // residue rows of the neighbouring lanes that touch this lane's block
        uint32_t a1 = __shfl_up_sync(MAPF_FULL_MASK, S.m1[RPL - 1][w], 1, LW), b1 = __shfl_down_sync(MAPF_FULL_MASK, S.m1[0][w], 1, LW);
        uint32_t a2 = __shfl_up_sync(MAPF_FULL_MASK, S.m2[RPL - 1][w], 1, LW), b2 = __shfl_down_sync(MAPF_FULL_MASK, S.m2[0][w], 1, LW);
        uint32_t az = __shfl_up_sync(MAPF_FULL_MASK, z[RPL - 1][w], 1, LW), bz = __shfl_down_sync(MAPF_FULL_MASK, z[0][w], 1, LW);
        if (lane == 0) a1 = a2 = az = 0;
        if (lane == LW - 1) b1 = b2 = bz = 0;
#pragma unroll
        for (int q = 0; q < RPL; ++q) {
            auto left = [&](const uint32_t(&m)[RPL][RW]) {  // bit y <- bit y-1
                return w > 0 ? __funnelshift_l(m[q][w > 0 ? w - 1 : 0], m[q][w], 1) : m[q][w] << 1;
            };
            auto right = [&](const uint32_t(&m)[RPL][RW]) {  // bit y <- bit y+1
                return w < RW - 1 ? __funnelshift_r(m[q][w], m[q][w < RW - 1 ? w + 1 : w], 1) : m[q][w] >> 1;
            };
            const uint32_t c1 = S.m1[q][w], c2 = S.m2[q][w], cz = z[q][w];
            const uint32_t u1 = q > 0 ? S.m1[q > 0 ? q - 1 : 0][w] : a1, u2 = q > 0 ? S.m2[q > 0 ? q - 1 : 0][w] : a2,
                           uz = q > 0 ? z[q > 0 ? q - 1 : 0][w] : az;
            const uint32_t d1 = q < RPL - 1 ? S.m1[q < RPL - 1 ? q + 1 : q][w] : b1, d2 = q < RPL - 1 ? S.m2[q < RPL - 1 ? q + 1 : q][w] : b2,
                           dz = q < RPL - 1 ? z[q < RPL - 1 ? q + 1 : q][w] : bz;
            pl[0][q][w] = closer(c1, c2, cz, u1, u2, uz);                             // neighbour x-1   environment.py:260
            pl[1][q][w] = closer(c1, c2, cz, d1, d2, dz);                             // neighbour x+1   environment.py:264
            pl[2][q][w] = closer(c1, c2, cz, left(S.m1), left(S.m2), left(z));        // neighbour y-1   environment.py:268
            pl[3][q][w] = closer(c1, c2, cz, right(S.m1), right(S.m2), right(z));     // neighbour y+1   environment.py:272
        }
    }
    uint2 *nv = reinterpret_cast<uint2 *>(navi + ((size_t)e * d.N + a) * d.navi_agent_stride);
#pragma unroll
    for (int q = 0; q < RPL; ++q) {
        const int row = lane * RPL + q;
        if (row >= d.L || !alive) continue;
        const int pr = row + 4, bx1 = pr >> 3, r1 = pr & 7;
#pragma unroll
        for (int by = 0; by < 4 * RW; ++by) {
            if (by >= d.NB) continue;
            constexpr int kLast = RW - 1;
            const int w = by >> 2;          // compile-time after unrolling
            const int s = (by & 3) * 8;
            uint32_t f[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                f[k] = __funnelshift_r(pl[k][q][w], w < kLast ? pl[k][q][w < kLast ? w + 1 : kLast] : 0u, s) & 0xffffu;
            const uint2 v = make_uint2(f[0] | (f[1] << 16), f[2] | (f[3] << 16));
            if (bx1 < d.NB) nv[((size_t)(bx1 * d.NB + by) << 4) + r1] = v;
            if (bx1 > 0) nv[((size_t)((bx1 - 1) * d.NB + by) << 4) + r1 + 8] = v;
        }
    }
}

// One search per agent group of the warp.  The waves run three at a time (one per residue) and the warp votes on the third
// only: a wave that finds nothing is followed by waves that find nothing, so at most two idle waves are run at the end.
// DIST: int32 distances are emitted too (parity with search.compute_heuristics) -- a separate instantiation, so the common
// loop carries none of it.
template <int RW, int RPL, int APW, bool WRAP, bool DIST, bool KEEP>
__device__ __forceinline__ void bfs_navi_search(const EnvDims &d, const int e, const int a, const int i, const bool alive,
                                                const uint32_t *__restrict__ ob, const BfsFree<RW, RPL> &F, const int gx, const int gy,
                                                uint32_t *__restrict__ navi, int32_t *__restrict__ dist_out)
{
    constexpr int LW = 32 / APW;
    const int lane = (threadIdx.x & 31) % LW;
#ifdef MAPF_ENABLE_DIAG
    const long long tb0 = clock64();
    long long triples = 0;
#endif
    BfsState<RW, RPL> S;
    bfs_init<RW, RPL, APW>(d, F, gx, gy, alive, S);
#ifdef MAPF_ENABLE_DIAG
    const long long tb1 = clock64();
#endif

    int32_t *dist = nullptr;
    if constexpr (DIST) {
        dist = alive ? dist_out + ((size_t)i * d.N + a) * d.L * d.L : nullptr;
        for (int q = 0; q < RPL; ++q) {
            const int row = lane * RPL + q;
            if (dist && row < d.L)
                for (int y = 0; y < d.L; ++y) dist[row * d.L + y] = MAPF_DIST_UNREACHABLE;
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < RPL; ++q)
#pragma unroll
            for (int w = 0; w < RW; ++w)
                if (dist && S.fro[q][w]) dist[gx * d.L + gy] = 0;
    }

    auto wave = [&](auto selc, const int t) -> uint32_t {
        constexpr int sel = decltype(selc)::value;  // t mod 3
        uint32_t nw[RPL][RW];
        const uint32_t any = bfs_wave<RW, RPL, APW, WRAP>(S, nw);
        bfs_apply<RW, RPL, sel>(S, nw);
        if constexpr (DIST) {
#pragma unroll
            for (int q = 0; q < RPL; ++q)
#pragma unroll
                for (int w = 0; w < RW; ++w) {
                    uint32_t x = dist ? nw[q][w] : 0u;
                    while (x) {
                        int b = __ffs(x) - 1;
                        x &= x - 1;
                        dist[(lane * RPL + q) * d.L + (32 * w + b - 4)] = t;
                    }
                }
        }
        return any;
    };
    for (int t = 1;; t += 3) {
        wave(std::integral_constant<int, 1>{}, t);
        wave(std::integral_constant<int, 2>{}, t + 1);
        const uint32_t any = wave(std::integral_constant<int, 0>{}, t + 2);
#ifdef MAPF_ENABLE_DIAG
        ++triples;
#endif
        if (!__any_sync(MAPF_FULL_MASK, any != 0)) break;
    }
#ifdef MAPF_ENABLE_DIAG
    const long long tb2 = clock64();
#endif
    bfs_emit<RW, RPL, APW, KEEP>(d, ob, F, e, a, alive, S, navi);
#ifdef MAPF_ENABLE_DIAG
    if (e == 0 && (threadIdx.x & 31) == 0) {
        const long long tb3 = clock64();
        atomicAdd(&g_bfs_cycles[0], (unsigned long long)(tb1 - tb0));
        atomicAdd(&g_bfs_cycles[1], (unsigned long long)(tb2 - tb1));
        atomicAdd(&g_bfs_cycles[2], (unsigned long long)(tb3 - tb2));
        atomicAdd(&g_bfs_cycles[3], 1ull);
        atomicAdd(&g_bfs_cycles[4], (unsigned long long)triples);
    }
#endif
}

// All 32 lanes call together; picks the instantiation (uniform branches: L and dist_out are launch-wide).
template <int RW, int RPL, int APW>
__device__ __forceinline__ void bfs_navi_warp(const EnvDims &d, const int e, const int a, const int i, const bool alive,
                                              const uint32_t *__restrict__ obst, const uint8_t *__restrict__ goal,
                                              uint32_t *__restrict__ navi, int32_t *__restrict__ dist_out)
{
    constexpr int LW = 32 / APW;
    const uint32_t *ob = obst + (size_t)e * d.obst_stride;
    const uchar2 gg = __ldcg(reinterpret_cast<const uchar2 *>(goal) + (size_t)e * d.N + a);
    BfsFree<RW, RPL> F;
    bfs_load_free<RW, RPL, APW>(d, ob, F);
    if (dist_out) bfs_navi_search<RW, RPL, APW, false, true, false>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, dist_out);
    else if (d.L < LW * RPL) bfs_navi_search<RW, RPL, APW, true, false, false>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, nullptr);
    else bfs_navi_search<RW, RPL, APW, false, false, false>(d, e, a, i, alive, ob, F, gg.x, gg.y, navi, nullptr);
}

// The same for a caller that searches for the agents of ONE environment one group after the other (in-launch re-generation):
// the free rows and the goal arrive in registers, loaded once per environment instead of once (twice: emit) per group.
template <int RW, int RPL, int APW>
__device__ __forceinline__ void bfs_navi_warp_pre(const EnvDims &d, const int e, const int a, const bool alive, const uint32_t *__restrict__ ob,
                                                  const BfsFree<RW, RPL> &F, const int gx, const int gy, uint32_t *__restrict__ navi)
{
    constexpr int LW = 32 / APW;
    if (d.L < LW * RPL) bfs_navi_search<RW, RPL, APW, true, false, true>(d, e, a, 0, alive, ob, F, gx, gy, navi, nullptr);
    else bfs_navi_search<RW, RPL, APW, false, false, true>(d, e, a, 0, alive, ob, F, gx, gy, navi, nullptr);
}

}  // namespace
