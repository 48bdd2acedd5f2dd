// mapf_per_kernels.cu — K4: prioritized-replay sum tree (buffer.py:16-105) and the TD-error /
// priority arithmetic around it (buffer.py:170-177, worker.py:186-203, 300-308), sm_100a.
//
// The tree is an fp64 array heap of 2*capacity-1 nodes exactly like SumTree.tree (buffer.py:25), so
// results are bit-comparable with numpy: every parent is recomputed as left + right (order-free),
// duplicate leaf indices resolve "last in batch order wins" (numpy fancy assignment, buffer.py:97),
// and the sampling descent uses the reference's comparisons (buffer.py:66-70) with FMA contraction
// disabled.  The whole tree (8 MiB at the reference's 2^19 leaves) lives in L2; the kernels are
// latency-bound (layer-1 dependent levels), not bandwidth-bound, so one CTA handles a batch and the
// fused learner tail (TD -> priority -> leaf write -> ancestor refresh) is a single launch.
//
// What the latency is made of, and how the batch-sized paths avoid it (a level of the straightforward form -- read both
// children from L2, add, write, barrier -- is one L2 round trip, and there are layer-1 = 19 of them):
//   * update (n <= 256, thread k = entry k, leaf indices non-decreasing -- what the stratified sampler returns and what an
//     episode insert is; anything else takes the straightforward form): a path node's new value is its child's new value
//     + the SIBLING's value.
//       - The top 11 levels of the tree (2047 nodes, 16 KB) are copied to shared memory as a dense block and updated in
//         place there: a level is  v += top[j ^ 1]; j >>= 1; top[j] = v  (threads that share a node write the same bits).
//       - Below them every sibling of every leaf-to-root path is known from the leaf index alone: all of them are
//         requested at once (one round trip).  A sibling the batch touches as well must be taken at its NEW value: with
//         sorted leaves the threads of one node are contiguous, and the sibling's threads -- if there are any -- are
//         the group right after (even node) or right before (odd node) one's own: each thread keeps the two neighbour
//         groups' positions and, when two groups merge one level up, hops once (the pointers are published in shared
//         memory next to the nodes and values).  No hash table, no atomics: measured, a level through an open-addressing
//         table in shared memory (atomicCAS inserts) cost ~2000 cycles, twice the L2 round trip it was meant to save
//         (profiles/r2_per_phases.jsonl).
//       - New node values leave as fire-and-forget stores.  Duplicate leaves: the last LIVE entry of a group of equal
//         leaves provides the value (numpy's "last one wins"); masked / out-of-range entries ride along in the group of
//         their left neighbour and never provide one.
//   * sample: the descent runs on the shared-memory copy of the top 11 levels (in the fused cycle kernel: the copy the
//     update has just refreshed), then fetches the whole 3-level subtree under the current node (14 independent loads)
//     per round trip: 1 + 3 round trips at 2^19 leaves instead of 19 + 1; the leaf value stays in a register for the
//     importance weight.
#include <cmath>
#include <mutex>
#include <set>
#include <utility>

#include "mapf_common.cuh"

namespace {

constexpr int kPerThreads = 256;
constexpr int kFastUpdateMax = 256;   // batch entries handled by the shared-memory update path (one per thread)
constexpr int kTopLevels = 11;        // levels of the tree kept as a dense copy in shared memory (2^11 - 1 nodes, 16 KB)

// profiles/tools/per_phase_probe.cu compiles this file with MAPF_PER_TIMING: thread 0 leaves clock64 stamps at the phase
// boundaries (the barriers keep the CTA's warps within a phase of each other)
#ifdef MAPF_PER_TIMING
__device__ unsigned long long g_per_stamps[96];
#define PER_STAMP(i)                                         \
    do {                                                     \
        if (threadIdx.x == 0) g_per_stamps[i] = clock64();   \
    } while (0)
#else
#define PER_STAMP(i)
#endif

__host__ __device__ inline int per_top_levels(int layer) { return layer < kTopLevels ? layer : kTopLevels; }
// dynamic shared memory: double top[2^tc] (1-based heap index) | update only: double sib[layer - tc][npad] | double v[npad] |
// u32 node[npad] | int nxt[npad] | int prv[npad] | u8 live[npad]
__host__ __device__ inline size_t per_sample_smem(int layer) { return ((size_t)1 << per_top_levels(layer)) * 8; }
__host__ __device__ inline size_t per_update_smem(int64_t n, int layer)
{
    if (n > kFastUpdateMax) return 0;
    const size_t npad = (size_t)((n + 31) & ~(int64_t)31);
    return per_sample_smem(layer) + (size_t)(layer - per_top_levels(layer)) * npad * 8 + npad * (8 + 4 + 4 + 4 + 1);
}

__device__ __forceinline__ unsigned long long stamp_of(unsigned long long epoch, int64_t k)
{
    return (epoch << 32) | (unsigned long long)(k + 1);
}

// Leaf writes with numpy's duplicate rule, then the level-by-level ancestor refresh.  Single CTA.
// `active[k]` (optional) masks entries out (stale indices, worker.py:192-201).  An index outside [0, capacity) -- numpy
// raises IndexError -- is skipped and latched in *err (mapf_per_status).
__device__ void tree_update_cta(double *tree, unsigned long long *stamps, unsigned long long epoch, int64_t capacity,
                                int layer, const int64_t *idx, const double *prio_in, const float *prio32, double alpha,
                                const uint8_t *active, int64_t n, int32_t *err)
{
    auto live = [&](int64_t k) -> bool {
        if (active && !active[k]) return false;
        const int64_t i = idx[k];
        return i >= 0 && i < capacity;
    };
    // phase 1: the highest batch position claims each leaf
    for (int64_t k = threadIdx.x; k < n; k += blockDim.x) {
        if (live(k)) atomicMax(&stamps[idx[k]], stamp_of(epoch, k));
        else if (!active || active[k]) atomicOr(err, MAPF_ERRBIT_INDEX);
    }
    __syncthreads();
    // phase 2: winners store the leaf
    for (int64_t k = threadIdx.x; k < n; k += blockDim.x) {
        if (!live(k)) continue;
        if (stamps[idx[k]] == stamp_of(epoch, k)) {
            double v = prio_in ? prio_in[k] : pow((double)prio32[k], alpha);
            tree[capacity - 1 + idx[k]] = v;
        }
    }
    __syncthreads();
    // phase 3: ancestors, buffer.py:99-102 (np.unique only removes redundant work; recomputing a parent
    // twice from final children gives the same bits)
    for (int l = 1; l < layer; ++l) {
        for (int64_t k = threadIdx.x; k < n; k += blockDim.x) {
            if (!live(k)) continue;
            int64_t node = ((capacity - 1 + idx[k] + 1) >> l) - 1;  // l-th ancestor in the array heap
            tree[node] = __dadd_rn(tree[2 * node + 1], tree[2 * node + 2]);
        }
        __syncthreads();
    }
}

constexpr int kMaxLow = 20;  // levels below the dense top that the sorted update path handles (capacity <= 2^30)

// The same update for a sorted batch of n <= kFastUpdateMax entries (thread k = entry k) with the level loop in shared
// memory (file header).  Nodes are named by their 1-based heap index j (root 1, parent j >> 1, sibling j ^ 1, array index
// j - 1); a node of depth d has j in [2^d, 2^(d+1)).  Returns false, having written nothing, when the live leaf indices are
// not non-decreasing (the caller takes the straightforward form); on a true return s_top holds the refreshed top of the tree.
__device__ bool tree_update_sorted(double *tree, int64_t capacity, int layer, const int64_t *idx, const double *prio_in,
                                   const float *prio32, double alpha, const uint8_t *active, int n, int32_t *err, unsigned char *smem)
{
    const int k = threadIdx.x;
    const int npad = (n + 31) & ~31;
    const int tc = per_top_levels(layer);             // depths 0 .. tc-1 are dense
    const int nlow = layer - tc;                       // depths tc .. layer-1: neighbour groups
    double *s_top = reinterpret_cast<double *>(smem);                 // [2^tc]
    double *s_sib = s_top + ((size_t)1 << tc);                        // [nlow][npad] old value of the path's low siblings
    double *s_v = s_sib + (size_t)nlow * npad;                        // [npad] value of the entry's current node
    uint32_t *s_node = reinterpret_cast<uint32_t *>(s_v + npad);      // [npad] the entry's current node
    int *s_nxt = reinterpret_cast<int *>(s_node + npad);              // [npad] first entry of the next group
    int *s_prv = s_nxt + npad;                                        // [npad] last entry of the previous group
    uint8_t *s_live = reinterpret_cast<uint8_t *>(s_prv + npad);      // [npad]
    PER_STAMP(0);
    // the dense top, old values: eight coalesced loads per thread (2^tc - 1 <= 8 x 256), in flight under the index load
    const int ntop = (1 << tc) - 1;
    double top_r[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int i = q * (int)blockDim.x + k;
        if (i < ntop) top_r[q] = tree[i];
    }
    bool lv = false;
    uint32_t j = 0;
    if (k < n) {
        const bool act = !active || active[k];
        const int64_t i = idx[k];
        lv = act && i >= 0 && i < capacity;
        if (act && !lv) atomicOr(err, MAPF_ERRBIT_INDEX);
        if (lv) j = (uint32_t)(capacity + i);
        s_node[k] = j;
        s_live[k] = lv ? 1 : 0;
    }
    PER_STAMP(1);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int i = q * (int)blockDim.x + k;
        if (i < ntop) s_top[i + 1] = top_r[q];
    }
    __syncthreads();
    // entries that are not live ride along in the group of the nearest live entry to the left (to the right at the front)
    if (k < n && !lv) {
        int q = k - 1;
        while (q >= 0 && !s_live[q]) --q;
        if (q < 0) {
            q = k + 1;
            while (q < n && !s_live[q]) ++q;
        }
        j = q < n ? s_node[q] : 0u;
    }
    if (!__syncthreads_or(lv)) return true;  // nothing to write
    if (k < n) s_node[k] = j;
    double sib[kMaxLow];
    if (k < n) {  // every low sibling of the path: one round trip, in flight while the groups are found
        uint32_t c = j;
#pragma unroll
        for (int l = 0; l < kMaxLow; ++l)
            if (l < nlow) {
                sib[l] = tree[(c ^ 1u) - 1u];
                c >>= 1;
            }
    }
    __syncthreads();
    const bool sorted = k == 0 || k >= n || s_node[k] >= s_node[k - 1];
    if (!__syncthreads_and(sorted)) return false;
    PER_STAMP(2);
    // groups of equal leaves; the last live entry of a group provides the value (buffer.py:97: the last duplicate wins)
    int nxt = n, prv = -1;
    double v = 0.0;
    if (k < n) {
        nxt = k + 1;
        while (nxt < n && s_node[nxt] == j) ++nxt;
        prv = k - 1;
        while (prv >= 0 && s_node[prv] == j) --prv;
        if (lv) s_v[k] = prio_in ? prio_in[k] : pow((double)prio32[k], alpha);
    }
    __syncthreads();
    if (k < n) {
        int w = nxt - 1;
        while (!s_live[w]) --w;
        v = s_v[w];
        if (w == k) tree[j - 1] = v;
        if (nlow == 0) s_top[j] = v;  // a tree that is dense down to its leaves
#pragma unroll
        for (int l = 0; l < kMaxLow; ++l)
            if (l < nlow) s_sib[(size_t)l * npad + k] = sib[l];
    }
    __syncthreads();
    if (k < n) {
        s_v[k] = v;
        s_nxt[k] = nxt;
        s_prv[k] = prv;
    }
    __syncthreads();
    PER_STAMP(3);
    for (int d = layer - 1; d > 0; --d) {  // node j of depth d -> its parent; buffer.py:99-102
        if (k < n) {
            double sv;
            if (d >= tc) {
                const int nb = (j & 1u) ? prv : nxt;  // where the sibling's entries are, if the batch has any
                if (nb >= 0 && nb < n && s_node[nb] == (j ^ 1u)) sv = s_v[nb];
                else sv = s_sib[(size_t)(layer - 1 - d) * npad + k];
            } else {
                sv = s_top[j ^ 1u];
            }
            v = __dadd_rn(v, sv);  // left + right; the order does not matter to the bits
            j >>= 1;
            if (k == prv + 1) tree[j - 1] = v;  // one store per child group (the sibling group stores the same bits)
            if (d - 1 < tc) s_top[j] = v;  // sharers of the node write the same bits
        }
        if (d - 1 >= tc) {
            __syncthreads();  // this level's nodes / values have been read
            if (k < n) {
                s_node[k] = j;
                s_v[k] = v;
                s_nxt[k] = nxt;
                s_prv[k] = prv;
            }
            __syncthreads();
            if (k < n) {  // two sibling groups have become one: hop over the other half
                if (nxt < n && s_node[nxt] == j) nxt = s_nxt[nxt];
                if (prv >= 0 && s_node[prv] == j) prv = s_prv[prv];
            }
        } else {
            __syncthreads();
        }
        PER_STAMP(4 + (layer - 1 - d));
    }
    return true;
}

__device__ __forceinline__ bool fast_update_ok(int64_t n, int64_t capacity)
{
    return n <= kFastUpdateMax && n <= (int64_t)blockDim.x && blockDim.x * 8 >= (1u << kTopLevels) - 1 && capacity <= ((int64_t)1 << 30);  // (layer - top levels <= kMaxLow)
}

__global__ void __launch_bounds__(kPerThreads)
per_update_kernel(double *tree, unsigned long long *stamps, unsigned long long epoch, int64_t capacity, int layer,
                  const int64_t *idx, const double *prio, int64_t n, int32_t *err)
{
    extern __shared__ __align__(16) unsigned char per_smem[];
    if (!(fast_update_ok(n, capacity) && tree_update_sorted(tree, capacity, layer, idx, prio, nullptr, 0.0, nullptr, (int)n, err, per_smem)))
        tree_update_cta(tree, stamps, epoch, capacity, layer, idx, prio, nullptr, 0.0, nullptr, n, err);
}

// multi-CTA variants for batches larger than one CTA handles comfortably
__global__ void per_claim_kernel(unsigned long long *stamps, unsigned long long epoch, int64_t capacity, const int64_t *idx, int64_t n,
                                 int32_t *err)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (idx[k] >= 0 && idx[k] < capacity) atomicMax(&stamps[idx[k]], stamp_of(epoch, k));
    else atomicOr(err, MAPF_ERRBIT_INDEX);
}
__global__ void per_leaf_kernel(double *tree, const unsigned long long *stamps, unsigned long long epoch, int64_t capacity,
                                const int64_t *idx, const double *prio, int64_t n)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n && idx[k] >= 0 && idx[k] < capacity && stamps[idx[k]] == stamp_of(epoch, k)) tree[capacity - 1 + idx[k]] = prio[k];
}
__global__ void per_level_kernel(double *tree, int64_t capacity, int l, const int64_t *idx, int64_t n)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n && idx[k] >= 0 && idx[k] < capacity) {
        int64_t node = ((capacity - 1 + idx[k] + 1) >> l) - 1;
        tree[node] = __dadd_rn(tree[2 * node + 1], tree[2 * node + 2]);
    }
}

// one step of the descent, buffer.py:66-70; returns true when it went right
__device__ __forceinline__ bool descend(double &p, const double left)
{
    bool right = false;
    if (!(p <= left)) {
        right = true;
        p = __dsub_rn(p, left);
    }
    if (p == 0.0) p = 1e-5;
    return right;
}

// SumTree.batch_sample, buffer.py:56-78.  One thread per sample; the top of the tree comes from shared memory (`top_ready`:
// the update has just left its refreshed copy there), the rest in round trips of three levels (file header).  `tree` may have
// been written by this CTA just before (a barrier lies between; plain loads: ld.global.cg compiles to LDG.STRONG.GPU, which
// measured ~2.5x the latency of a weak load here).  Nodes by 1-based heap index j (children 2j, 2j + 1).  A sampled leaf
// whose priority is not > 0 -- the reference asserts (buffer.py:74) -- is returned as the reference's descent finds it and
// latched in *err (mapf_per_status).
__device__ void sample_cta(const double *tree, int64_t capacity, int layer, const double *__restrict__ uniforms,
                           int64_t batch, int64_t *__restrict__ idx_out, double *__restrict__ prio_out,
                           float *__restrict__ weight_out, double beta, unsigned char *smem, const bool top_ready, int32_t *err)
{
    __shared__ double s_min[32];
    double *s_top = reinterpret_cast<double *>(smem);
    const int tc = per_top_levels(layer);   // cached depths 0 .. tc-1
    PER_STAMP(40);
    const double u0 = threadIdx.x < batch ? uniforms[threadIdx.x] : 0.0;  // in flight while the top arrives
    if (!top_ready) {
        const int ntop = (1 << tc) - 1, k = threadIdx.x;
        for (int base = 0; base < ntop; base += 8 * (int)blockDim.x) {  // eight coalesced loads in flight per thread
            double r[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int i = base + q * (int)blockDim.x + k;
                if (i < ntop) r[q] = tree[i];
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int i = base + q * (int)blockDim.x + k;
                if (i < ntop) s_top[i + 1] = r[q];
            }
        }
        __syncthreads();
    }
    PER_STAMP(41);
    const double sum = s_top[1];
    const double interval = __ddiv_rn(sum, (double)batch);  // :58
    double local_min = 1.0e300;
    double pr_first = 0.0;  // the value of this thread's first sample (batch <= blockDim: its only one)
    for (int64_t i = threadIdx.x; i < batch; i += blockDim.x) {
        // :60  np.arange(0,sum,interval)[i] + np.random.uniform(0,interval)[i]; no FMA contraction
        const double u = i == (int64_t)threadIdx.x ? u0 : uniforms[i];
        double p = __dadd_rn(__dmul_rn((double)i, interval), __dmul_rn(u, interval));
        if (i == 0 && p == 0.0) p = 1e-5;  // :61-62
        int64_t j = 1;
        int l = 0;
        for (; l < tc - 1; ++l)  // :66-70 on the cached levels
            j = 2 * j + (descend(p, s_top[2 * j]) ? 1 : 0);
        double pr = s_top[j];  // the leaf, when the whole tree is cached
        PER_STAMP(42);
        while (l < layer - 1) {
            // the subtree under j: its descendants at depth g are the 2^g nodes from j << g
            const int g = layer - 1 - l < 3 ? layer - 1 - l : 3;
            const double *a = tree + ((j << 1) - 1);
            const double *b = tree + ((j << 2) - 1);
            const double *c = tree + ((j << 3) - 1);
            // a step only looks at LEFT children; the right ones matter at the last level of the last group, where the
            // node the descent ends on (the leaf) gives the priority.  One SM retires about one scattered request per
            // cycle, so at 192 samples a request costs as much as 1/700 of a round trip: 7 loads per group, not 14.
            const bool fin = l + g == layer - 1;
            double a0 = a[0], a1 = 0;
            double b0 = 0, b1 = 0, b2 = 0, b3 = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0, c5 = 0, c6 = 0, c7 = 0;
            if (g >= 2) b0 = b[0], b2 = b[2];
            if (g >= 3) c0 = c[0], c2 = c[2], c4 = c[4], c6 = c[6];
            if (fin) {
                if (g == 1) a1 = a[1];
                if (g == 2) b1 = b[1], b3 = b[3];
                if (g == 3) c1 = c[1], c3 = c[3], c5 = c[5], c7 = c[7];
            }
            const bool r1 = descend(p, a0);
            int rel = r1 ? 1 : 0;
            pr = r1 ? a1 : a0;
            if (g >= 2) {
                const bool r2 = descend(p, r1 ? b2 : b0);
                rel = 2 * rel + (r2 ? 1 : 0);
                pr = r1 ? (r2 ? b3 : b2) : (r2 ? b1 : b0);
            }
            if (g >= 3) {
                const double lval = rel == 0 ? c0 : (rel == 1 ? c2 : (rel == 2 ? c4 : c6));
                const double rval = rel == 0 ? c1 : (rel == 1 ? c3 : (rel == 2 ? c5 : c7));
                const bool r3 = descend(p, lval);
                rel = 2 * rel + (r3 ? 1 : 0);
                pr = r3 ? rval : lval;
            }
            j = (j << g) + rel;
            l += g;  // pr = the value of the node the group ended on (the leaf, after the last group)
            PER_STAMP(43 + (l - tc) / 3);
        }
        const int64_t node = j - 1;
        if (i == (int64_t)threadIdx.x) pr_first = pr;
        prio_out[i] = pr;                     // :72
        idx_out[i] = node - (capacity - 1);   // :73
        if (!(pr > 0.0)) atomicOr(err, MAPF_ERRBIT_PRIORITY);  // :74 asserts priorities > 0; the batch's weights are then undefined
        local_min = fmin(local_min, pr);
    }
    PER_STAMP(46);
    if (weight_out) {  // worker.py:165-166
        for (int o = 16; o > 0; o >>= 1) local_min = fmin(local_min, __shfl_xor_sync(MAPF_FULL_MASK, local_min, o));
        if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = local_min;
        __syncthreads();
        double m = s_min[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmin(m, s_min[w]);
        for (int64_t i = threadIdx.x; i < batch; i += blockDim.x)
            weight_out[i] = powf((float)((i == (int64_t)threadIdx.x ? pr_first : prio_out[i]) / m), -(float)beta);  // fp32: 1e-6 relative
    }
    PER_STAMP(47);
}

__global__ void __launch_bounds__(kPerThreads)
per_sample_kernel(const double *__restrict__ tree, int64_t capacity, int layer, const double *__restrict__ uniforms,
                  int64_t batch, int64_t *__restrict__ idx_out, double *__restrict__ prio_out,
                  float *__restrict__ weight_out, double beta, int32_t *err)
{
    extern __shared__ __align__(16) unsigned char per_smem[];
    sample_cta(tree, capacity, layer, uniforms, batch, idx_out, prio_out, weight_out, beta, per_smem, false, err);
}

// Learner TD error -> priority -> stale mask (worker.py:300-308, 192-201), one thread per transition
__device__ void td_cta(const float *__restrict__ q_online, const float *__restrict__ q_target_next,
                       const float *__restrict__ q_online_next, const int64_t *__restrict__ action,
                       const float *__restrict__ reward, const float *__restrict__ done, const float *__restrict__ steps,
                       const int64_t *__restrict__ idx, int64_t n, float gamma, int64_t old_ptr, int64_t ptr,
                       int64_t slot_steps, float *__restrict__ td_out, float *__restrict__ prio_out, float *prio_scratch,
                       uint8_t *active)
{
    for (int64_t k = threadIdx.x; k < n; k += blockDim.x) {
        const float *qt = q_target_next + k * 5;
        float boot;
        if (q_online_next) {  // double-Q option: online argmax, target value
            const float *qn = q_online_next + k * 5;
            int best = 0;
            for (int a = 1; a < 5; ++a)
                if (qn[a] > qn[best]) best = a;
            boot = qt[best];
        } else {  // worker.py:302 target-network max
            boot = qt[0];
            for (int a = 1; a < 5; ++a) boot = fmaxf(boot, qt[a]);
        }
        const float q_ = __fmul_rn(1.0f - done[k], boot);                                      // :302
        const float disc = powf(gamma, steps[k]);                                              // :306
        const float target = __fadd_rn(reward[k], __fmul_rn(disc, q_));
        const float td = __fsub_rn(q_online[k * 5 + action[k]], target);                       // :306
        const float pr = fmaxf(fabsf(td), 1e-6f);                                              // :308
        if (td_out) td_out[k] = td;
        if (prio_out) prio_out[k] = pr;
        prio_scratch[k] = pr;
        // worker.py:192-201 discard samples whose episode slot was rewritten since sampling
        bool keep = true;
        const int64_t lo = old_ptr * slot_steps, hi = ptr * slot_steps;
        if (ptr > old_ptr) keep = (idx[k] < lo) || (idx[k] >= hi);
        else if (ptr < old_ptr) keep = (idx[k] < lo) && (idx[k] >= hi);
        active[k] = keep ? 1 : 0;
    }
    __syncthreads();
}

// Fused learner tail: TD error -> priority -> stale mask -> leaf = prio^alpha -> ancestor refresh.
__global__ void __launch_bounds__(kPerThreads)
per_td_update_kernel(double *tree, unsigned long long *stamps, unsigned long long epoch, int64_t capacity, int layer,
                     const float *__restrict__ q_online, const float *__restrict__ q_target_next,
                     const float *__restrict__ q_online_next, const int64_t *__restrict__ action,
                     const float *__restrict__ reward, const float *__restrict__ done, const float *__restrict__ steps,
                     const int64_t *__restrict__ idx, int64_t n, float gamma, double alpha, int64_t old_ptr, int64_t ptr,
                     int64_t slot_steps, float *__restrict__ td_out, float *__restrict__ prio_out, float *prio_scratch,
                     uint8_t *active, int32_t *err)
{
    extern __shared__ __align__(16) unsigned char per_smem[];
    td_cta(q_online, q_target_next, q_online_next, action, reward, done, steps, idx, n, gamma, old_ptr, ptr, slot_steps, td_out,
           prio_out, prio_scratch, active);
    if (!(fast_update_ok(n, capacity) && tree_update_sorted(tree, capacity, layer, idx, nullptr, prio_scratch, alpha, active, (int)n, err, per_smem)))
        tree_update_cta(tree, stamps, epoch, capacity, layer, idx, nullptr, prio_scratch, alpha, active, n, err);
}

// One learner cycle in ONE launch (north star (4)): the priorities of the batch that has just been through the two Q
// forwards go into the tree (TD -> priority -> stale mask -> leaf -> ancestors), then the NEXT batch is drawn from the
// refreshed tree with its importance-sampling weights (worker.py:300-308, 186-203, 106-116, 165-166).  Either half may be
// empty (n == 0).
__global__ void __launch_bounds__(kPerThreads)
per_cycle_kernel(double *tree, unsigned long long *stamps, unsigned long long epoch, int64_t capacity, int layer,
                 const mapf_per_cycle_args a, float *prio_scratch, uint8_t *active, int32_t *err)
{
    extern __shared__ __align__(16) unsigned char per_smem[];
    bool top_ready = false;
    if (a.n_update > 0) {
        td_cta(a.d_q_online, a.d_q_target_next, a.d_q_online_next, a.d_action, a.d_reward, a.d_done, a.d_steps, a.d_idx, a.n_update,
               a.gamma, a.old_ptr, a.ptr, a.slot_steps, a.d_td_out, a.d_prio_out, prio_scratch, active);
        top_ready = fast_update_ok(a.n_update, capacity) &&
                    tree_update_sorted(tree, capacity, layer, a.d_idx, nullptr, prio_scratch, a.alpha, active, (int)a.n_update, err, per_smem);
        if (!top_ready) tree_update_cta(tree, stamps, epoch, capacity, layer, a.d_idx, nullptr, prio_scratch, a.alpha, active, a.n_update, err);
        __syncthreads();  // the update's stores are visible to the CTA
    }
    if (a.n_sample > 0)
        sample_cta(tree, capacity, layer, a.d_uniforms, a.n_sample, a.d_sample_idx_out, a.d_sample_prio_out, a.d_sample_weight_out,
                   a.beta, per_smem, top_ready, err);
}

// LocalBuffer.finish, buffer.py:170-177: |sum_j gamma^j r[t+j] + max_a q[t,a] - q[t,a_t]| over j < forward_steps (rewards past
// the episode end are 0); `gpow[j]` = gamma^j as Python evaluates 0.99**j (fp64, computed on the host)
struct ActorTdPowers {
    double g[8];
};
__global__ void actor_td_kernel(const float *__restrict__ rew, const float *__restrict__ q, const uint8_t *__restrict__ act,
                                const int32_t *__restrict__ size, int episodes, int capacity, int forward_steps,
                                const ActorTdPowers gpow, double *__restrict__ td)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (int64_t)episodes * capacity) return;
    const int ep = (int)(g / capacity), t = (int)(g - (int64_t)ep * capacity);
    const int sz = size[ep];
    double out = 0.0;
    if (t < sz) {
        const float *qq = q + g * 5;
        float qmax = qq[0];
        for (int a = 1; a < 5; ++a) qmax = fmaxf(qmax, qq[a]);
        // np.convolve(ret, [gamma^(n-1), ..., gamma, 1.0], 'valid')[t]: accumulated from j = 0 upwards
        double conv = __dmul_rn((double)rew[g], 1.0);
        for (int j = 1; j < forward_steps; ++j) {
            const double rj = (t + j < sz) ? (double)rew[g + j] : 0.0;
            conv = __dadd_rn(conv, __dmul_rn(rj, gpow.g[j]));
        }
        const double target = __dadd_rn(conv, (double)qmax);
        out = fabs(__dsub_rn(target, (double)qq[act[g]]));
    }
    td[g] = out;
}

}  // namespace

// the fast paths' shared memory goes past the 48 KB a kernel gets without asking (per device, idempotent, host-only call)
static cudaError_t per_smem_optin(const void *kernel, size_t smem)
{
    if (smem <= 48 * 1024) return cudaSuccess;
    static std::mutex mu;
    static std::set<std::pair<int, const void *>> done;  // (device, kernel) pairs that have been raised
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    if (done.count({dev, kernel})) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess) done.insert({dev, kernel});
    return e;
}

int mapf_launch_per_update(mapf_per *t, PerScratch *s, const int64_t *d_idx, const double *d_prio, int64_t n, cudaStream_t st)
{
    if (n <= 0) return MAPF_OK;
    const unsigned long long epoch = ++s->epoch;
    if (n <= 4096) {
        const size_t smem = per_update_smem(n, t->layer);
        MAPF_CUDA(per_smem_optin((const void *)per_update_kernel, smem));
        per_update_kernel<<<1, kPerThreads, smem, st>>>(t->tree, s->stamps, epoch, t->capacity, t->layer, d_idx, d_prio, n, s->err);
    } else {
        const int tb = 256;
        const unsigned grid = (unsigned)((n + tb - 1) / tb);
        per_claim_kernel<<<grid, tb, 0, st>>>(s->stamps, epoch, t->capacity, d_idx, n, s->err);
        per_leaf_kernel<<<grid, tb, 0, st>>>(t->tree, s->stamps, epoch, t->capacity, d_idx, d_prio, n);
        for (int l = 1; l < t->layer; ++l) per_level_kernel<<<grid, tb, 0, st>>>(t->tree, t->capacity, l, d_idx, n);
    }
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_per_sample(mapf_per *t, const double *d_uniforms, int64_t batch, int64_t *d_idx_out, double *d_prio_out,
                           float *d_weight_out, double beta, cudaStream_t st)
{
    if (batch <= 0) return MAPF_OK;
    const size_t smem = per_sample_smem(t->layer);
    MAPF_CUDA(per_smem_optin((const void *)per_sample_kernel, smem));
    per_sample_kernel<<<1, kPerThreads, smem, st>>>(t->tree, t->capacity, t->layer, d_uniforms, batch, d_idx_out, d_prio_out,
                                                    d_weight_out, beta, t->scratch.err);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_per_td_update(mapf_per *t, PerScratch *s, const float *q_online, const float *q_target_next,
                              const float *q_online_next, const int64_t *action, const float *reward, const float *done,
                              const float *steps, const int64_t *idx, int64_t n, float gamma, double alpha, int64_t old_ptr,
                              int64_t ptr, int64_t slot_steps, float *td_out, float *prio_out, cudaStream_t st)
{
    if (n <= 0) return MAPF_OK;
    const unsigned long long epoch = ++s->epoch;
    const size_t smem = per_update_smem(n, t->layer);
    MAPF_CUDA(per_smem_optin((const void *)per_td_update_kernel, smem));
    per_td_update_kernel<<<1, kPerThreads, smem, st>>>(t->tree, s->stamps, epoch, t->capacity, t->layer, q_online, q_target_next,
                                                    q_online_next, action, reward, done, steps, idx, n, gamma, alpha, old_ptr,
                                                    ptr, slot_steps, td_out, prio_out, s->prio32, s->active, s->err);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_per_cycle(mapf_per *t, PerScratch *s, const mapf_per_cycle_args *a, cudaStream_t st)
{
    if (a->n_update <= 0 && a->n_sample <= 0) return MAPF_OK;
    const unsigned long long epoch = ++s->epoch;
    size_t smem = a->n_update > 0 ? per_update_smem(a->n_update, t->layer) : 0;
    if (a->n_sample > 0 && per_sample_smem(t->layer) > smem) smem = per_sample_smem(t->layer);
    MAPF_CUDA(per_smem_optin((const void *)per_cycle_kernel, smem));
    per_cycle_kernel<<<1, kPerThreads, smem, st>>>(t->tree, s->stamps, epoch, t->capacity, t->layer, *a, s->prio32, s->active, s->err);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_actor_td(const float *d_rew, const float *d_q, const uint8_t *d_act, const int32_t *d_size, int episodes,
                         int capacity, int forward_steps, double gamma, double *d_td_out, cudaStream_t st)
{
    const int64_t total = (int64_t)episodes * capacity;
    if (total <= 0) return MAPF_OK;
    ActorTdPowers gp{};
    for (int j = 0; j < 8; ++j) gp.g[j] = j == 0 ? 1.0 : (j == 1 ? gamma : std::pow(gamma, (double)j));
    actor_td_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_rew, d_q, d_act, d_size, episodes, capacity, forward_steps, gp,
                                                                     d_td_out);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}
