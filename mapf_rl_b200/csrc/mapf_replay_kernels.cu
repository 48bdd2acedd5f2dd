// mapf_replay_kernels.cu — K5: the sampled-window gather of the replay store, the data format on the
// learner side of the hot path (GlobalBuffer.sample_batch, worker.py:106-184), sm_100a.
//
// The store keeps the reference's logical layout on the device (worker.py:36-42): episode slot g holds
// max_steps + 1 observation / comm-mask frames at rows g * (max_steps + 1) + f and max_steps action /
// reward / hidden rows at g * max_steps + t; tree leaf idx = g * max_steps + t.  Observations stay bool
// bytes exactly as the step kernel writes them.  For every sampled leaf the kernel gathers the
// bt_steps + forward_steps frame window (zero padded), converts bool -> fp16 on the fly
// (np.stack(b_obs).astype(np.float16), worker.py:169), gathers the comm masks and the stored hidden
// state, and emits the per-sample scalars — one launch, HBM-bound: per sample it reads at most
// W * N * 486 bytes and writes W * N * 972 (W = bt_steps + forward_steps).
#include <cuda_fp16.h>

#include "mapf_common.cuh"

namespace {

// parameters of the (W + 1, batch) grid kernels over a dense or a compact store
template <typename View>
struct GatherParams {
    View v;
    mapf_replay_batch o;
    const int64_t *idx;
    int32_t *err;
};

// two bool bytes (b0 at bits 0-7, b1 at bits 16-23) -> two fp16 (1.0 = 0x3C00)
__device__ __forceinline__ uint32_t bools_to_half2(uint32_t spread) { return spread * 0x3C00u; }

// the sampled window of one leaf (worker.py:115-137)
struct Window {
    int64_t idx, g;  // leaf and its episode slot (worker.py:115)
    int t, size;     // step of the leaf in the episode (:116) and the episode's size
    int steps;       // forward steps, min(forward_steps, size - t) (:122)
    int f0, len;     // the window starts at the episode start until bt_steps frames of history exist (:124-137);
                     // frames j >= len are zero padding (:139-142)
    int64_t row0;    // store row of window frame 0
    __device__ __forceinline__ int64_t row(const int j) const { return row0 + j; }
    // leaf of the stored hidden state, t - bt_steps (:137); -1 (zeros) while t < bt_steps (:127,:132)
    __device__ __forceinline__ int64_t hidden_leaf(const int bt_steps) const { return t >= bt_steps ? idx - bt_steps : -1; }
};

// dense and compact views share these fields
template <typename View>
__device__ __forceinline__ Window leaf_window(const View &v, const int64_t idx)
{
    Window w;
    w.idx = idx;
    w.g = idx / v.max_steps;
    w.t = (int)(idx - w.g * v.max_steps);
    w.size = v.size_buf[w.g];
    w.steps = min(v.forward_steps, w.size - w.t);
    w.f0 = max(0, w.t + 1 - v.bt_steps);
    w.len = w.t + 1 + w.steps - w.f0;
    w.row0 = w.g * (v.max_steps + 1) + w.f0;
    return w;
}

// the per-sample scalars of a gathered window
template <typename View>
__device__ __forceinline__ void gather_scalars(const View &v, const mapf_replay_batch &o, int32_t *err, const int64_t b,
                                               const Window &w)
{
    if (w.t >= w.size && err) atomicOr(err, 1);  // the reference asserts local_idx < size (worker.py:120)
    o.action[b] = v.act_buf[w.idx];                                             // :143
    o.reward[b] = v.rew_buf[w.idx];                                             // :144
    const bool done = (w.t == w.size - 1) && v.done_buf[w.g] != 0;              // :145-148
    o.done[b] = done ? 0x3C00 : 0;
    o.steps[b] = __half_as_ushort(__int2half_rn(w.steps));                      // :171 HalfTensor(b_steps)
    o.bt_steps[b] = min(w.t + 1, v.bt_steps);                                   // :150
}

__global__ void __launch_bounds__(256)
replay_gather_kernel(const GatherParams<mapf_replay_view> p)
{
    const mapf_replay_view &v = p.v;
    const int W = v.bt_steps + v.forward_steps;
    const int j = blockIdx.x;  // frame of the window, or W = the hidden-state / scalar block
    const int64_t b = blockIdx.y;
    const Window w = leaf_window(v, p.idx[b]);
    const int N = v.num_agents;

    if (j == W) {
        // the window's stored hidden state, zeros while t < bt_steps
        const int HB = N * v.latent_dim;  // halfs
        uint16_t *dst = p.o.hidden + (size_t)b * HB;
        const int64_t hid = w.hidden_leaf(v.bt_steps);
        const uint16_t *src = hid >= 0 ? v.hid_buf + (size_t)hid * HB : nullptr;
        if ((HB & 7) == 0) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
            uint4 *d4 = reinterpret_cast<uint4 *>(dst);
            for (int k = threadIdx.x; k < (HB >> 3); k += blockDim.x) d4[k] = src ? __ldg(s4 + k) : make_uint4(0, 0, 0, 0);
        } else {
            for (int k = threadIdx.x; k < HB; k += blockDim.x) dst[k] = src ? src[k] : (uint16_t)0;
        }
        if (threadIdx.x == 0) gather_scalars(v, p.o, p.err, b, w);
        return;
    }

    const bool live = j < w.len;
    const int64_t row = w.row(j);
    // ---- observation frame: N * 486 bool bytes -> fp16 ----
    {
        const int FB = N * MAPF_OBS_BYTES_PER_AGENT;
        const uint8_t *src = v.obs_buf + (size_t)row * FB;
        uint16_t *dst = p.o.obs + ((size_t)b * W + j) * FB;
        if ((FB & 15) == 0) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
            uint4 *d4 = reinterpret_cast<uint4 *>(dst);
            for (int k = threadIdx.x; k < (FB >> 4); k += blockDim.x) {
                uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
                if (live) {
                    const uint4 x = __ldg(s4 + k);
                    lo.x = bools_to_half2(__byte_perm(x.x, 0, 0x4140));
                    lo.y = bools_to_half2(__byte_perm(x.x, 0, 0x4342));
                    lo.z = bools_to_half2(__byte_perm(x.y, 0, 0x4140));
                    lo.w = bools_to_half2(__byte_perm(x.y, 0, 0x4342));
                    hi.x = bools_to_half2(__byte_perm(x.z, 0, 0x4140));
                    hi.y = bools_to_half2(__byte_perm(x.z, 0, 0x4342));
                    hi.z = bools_to_half2(__byte_perm(x.w, 0, 0x4140));
                    hi.w = bools_to_half2(__byte_perm(x.w, 0, 0x4342));
                }
                __stcs(d4 + 2 * k, lo);
                __stcs(d4 + 2 * k + 1, hi);
            }
        } else {  // N not a multiple of 8: 2 bools -> one 32-bit store (N * 486 is always even)
            const uint16_t *s2 = reinterpret_cast<const uint16_t *>(src);
            uint32_t *d2 = reinterpret_cast<uint32_t *>(dst);
            for (int k = threadIdx.x; k < (FB >> 1); k += blockDim.x) {
                uint32_t out = 0;
                if (live) {
                    const uint32_t x = s2[k];
                    out = bools_to_half2(__byte_perm(x, 0, 0x4140));
                }
                d2[k] = out;
            }
        }
    }
    // ---- communication mask frame: N * N bool bytes ----
    {
        const int CBytes = N * N;
        const uint8_t *src = v.comm_buf + (size_t)row * CBytes;
        uint8_t *dst = p.o.comm_mask + ((size_t)b * W + j) * CBytes;
        for (int k = threadIdx.x; k < CBytes; k += blockDim.x) dst[k] = live ? src[k] : (uint8_t)0;
    }
}

// ---- packed observation frames (include/mapf_b200.h: 64-byte agent rows, element k = bit k) -> dense elements ----

// one packed frame (N * 64 bytes, 16-byte aligned) into shared memory
__device__ __forceinline__ void load_frame(uint8_t *s_frame, const uint8_t *src, const int N)
{
    for (int k = threadIdx.x; k < N * (MAPF_OBS_PACKED_BYTES_PER_AGENT / 16); k += blockDim.x)
        reinterpret_cast<uint4 *>(s_frame)[k] = __ldg(reinterpret_cast<const uint4 *>(src) + k);
}

// elements e0 .. e0+7 of the frame's N * 486 (element e0 at bit 0); a group may run from one agent's row into the next
__device__ __forceinline__ uint32_t frame_bits8(const uint8_t *s_frame, const int N, const int e0)
{
    const int a = e0 / MAPF_OBS_BYTES_PER_AGENT, k0 = e0 - a * MAPF_OBS_BYTES_PER_AGENT;
    const uint8_t *r = s_frame + a * MAPF_OBS_PACKED_BYTES_PER_AGENT + (k0 >> 3);  // k0 <= 485: r[1] is byte 61 at most
    uint32_t w = ((uint32_t)r[0] | ((uint32_t)r[1] << 8)) >> (k0 & 7);
    const int n1 = MAPF_OBS_BYTES_PER_AGENT - k0;
    if (n1 < 8) {
        w &= (1u << n1) - 1u;  // the row's pad bits are no elements
        if (a + 1 < N) w |= (uint32_t)s_frame[(a + 1) * MAPF_OBS_PACKED_BYTES_PER_AGENT] << n1;
    }
    return w & 0xffu;
}

// 4 bits -> 4 bool bytes (as the step kernel's expansion)
__device__ __forceinline__ uint32_t expand4(uint32_t x) { return (x * 0x00204081u) & 0x01010101u; }

// two bits (element 2q at bit 0) -> two 16-bit values ONE / 0, or two bytes 1 / 0 (ONE = 1)
template <uint32_t ONE>
__device__ __forceinline__ uint32_t bits2_to_pair(const uint32_t x)
{
    return ONE == 1 ? ((x & 1u) | ((x & 2u) << 7)) : ((x & 1u) | ((x & 2u) << 15)) * ONE;
}

// Expand a frame in shared memory (live) or zeros (!live) into FB = N * 486 consecutive output elements at dst.  ONE = 1:
// u8 elements, else 16-bit elements whose 1.0 is ONE (fp16 0x3C00, bf16 0x3F80).  vec: dst is aligned for 8 elements per
// store (FB % 8 == 0 and a 16-byte aligned base); else one store of two elements each (FB is even, an even element pair
// never straddles two agents).
template <uint32_t ONE>
__device__ __forceinline__ void expand_frame(const uint8_t *s_frame, const int N, const bool live, void *dst, const bool vec)
{
    const int FB = N * MAPF_OBS_BYTES_PER_AGENT;
    if (vec) {
        for (int q = threadIdx.x; q < (FB >> 3); q += blockDim.x) {
            const uint32_t w = live ? frame_bits8(s_frame, N, q << 3) : 0u;
            if constexpr (ONE == 1) {
                __stcs(reinterpret_cast<uint2 *>(dst) + q, make_uint2(expand4(w & 0xfu), expand4(w >> 4)));
            } else {
                __stcs(reinterpret_cast<uint4 *>(dst) + q, make_uint4(bits2_to_pair<ONE>(w), bits2_to_pair<ONE>(w >> 2),
                                                                    bits2_to_pair<ONE>(w >> 4), bits2_to_pair<ONE>(w >> 6)));
            }
        }
    } else {
        for (int q = threadIdx.x; q < (FB >> 1); q += blockDim.x) {
            uint32_t x = 0;
            if (live) {
                const int e0 = q << 1, a = e0 / MAPF_OBS_BYTES_PER_AGENT, k0 = e0 - a * MAPF_OBS_BYTES_PER_AGENT;
                x = (s_frame[a * MAPF_OBS_PACKED_BYTES_PER_AGENT + (k0 >> 3)] >> (k0 & 7)) & 3u;
            }
            if constexpr (ONE == 1) reinterpret_cast<uint16_t *>(dst)[q] = (uint16_t)bits2_to_pair<1>(x);
            else reinterpret_cast<uint32_t *>(dst)[q] = bits2_to_pair<ONE>(x);
        }
    }
}

template <uint32_t ONE>
__global__ void __launch_bounds__(256)
obs_unpack_kernel(const uint8_t *__restrict__ bits, const int64_t *__restrict__ rows, const int N, void *__restrict__ out)
{
    __shared__ __align__(16) uint8_t s_frame[MAPF_MAX_AGENTS * MAPF_OBS_PACKED_BYTES_PER_AGENT];
    const int64_t f = blockIdx.x;
    const int FB = N * MAPF_OBS_BYTES_PER_AGENT;
    load_frame(s_frame, bits + (size_t)(rows ? rows[f] : f) * N * MAPF_OBS_PACKED_BYTES_PER_AGENT, N);
    __syncthreads();
    uint8_t *dst = reinterpret_cast<uint8_t *>(out) + (size_t)f * FB * (ONE == 1 ? 1 : 2);
    expand_frame<ONE>(s_frame, N, true, dst, (FB & 7) == 0);
}

// comm mask frame `row` of a compact store: packed rows (N rows of ceil(N / 8) bytes) -> N * N bool bytes, zeros if !live
__device__ __forceinline__ void expand_comm_frame(const uint8_t *comm_bits, const int64_t row, const int N, const bool live,
                                                  uint8_t *dst)
{
    const int CW = (N + 7) >> 3;
    const uint8_t *src = comm_bits + (size_t)row * N * CW;
    for (int k = threadIdx.x; k < N * N; k += blockDim.x) {
        const int i = k / N, c = k - i * N;
        dst[k] = live ? (uint8_t)((__ldg(src + i * CW + (c >> 3)) >> (c & 7)) & 1u) : (uint8_t)0;
    }
}

// replay_gather_kernel over a compact store: the same window, padding and scalars; the observation frame is expanded from
// bits to fp16 (eight halves per 16-byte store), the comm mask from bits to bytes, and the one stored hidden vector of the
// sample is written into each of its N rows
__global__ void __launch_bounds__(256)
replay_gather_compact_kernel(const GatherParams<mapf_replay_view_compact> p)
{
    __shared__ __align__(16) uint8_t s_frame[MAPF_MAX_AGENTS * MAPF_OBS_PACKED_BYTES_PER_AGENT];
    const mapf_replay_view_compact &v = p.v;
    const int W = v.bt_steps + v.forward_steps;
    const int j = blockIdx.x;
    const int64_t b = blockIdx.y;
    const Window w = leaf_window(v, p.idx[b]);
    const int N = v.num_agents;

    if (j == W) {
        // the window's stored hidden vector in every agent's row, zeros while t < bt_steps
        const int D = v.latent_dim;
        uint16_t *dst = p.o.hidden + (size_t)b * N * D;
        const int64_t hid = w.hidden_leaf(v.bt_steps);
        const uint16_t *src = hid >= 0 ? v.hid_buf + (size_t)hid * D : nullptr;
        if ((D & 7) == 0) {
            const int D8 = D >> 3;
            const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
            uint4 *d4 = reinterpret_cast<uint4 *>(dst);
            for (int k = threadIdx.x; k < N * D8; k += blockDim.x) d4[k] = src ? __ldg(s4 + k % D8) : make_uint4(0, 0, 0, 0);
        } else {
            for (int k = threadIdx.x; k < N * D; k += blockDim.x) dst[k] = src ? src[k % D] : (uint16_t)0;
        }
        if (threadIdx.x == 0) gather_scalars(v, p.o, p.err, b, w);
        return;
    }

    const bool live = j < w.len;
    const int64_t row = w.row(j);
    const int FB = N * MAPF_OBS_BYTES_PER_AGENT;
    if (live) load_frame(s_frame, v.obs_bits + (size_t)row * N * MAPF_OBS_PACKED_BYTES_PER_AGENT, N);
    __syncthreads();
    expand_frame<0x3C00u>(s_frame, N, live, p.o.obs + ((size_t)b * W + j) * FB, (FB & 7) == 0);
    expand_comm_frame(v.comm_bits, row, N, live, p.o.comm_mask + ((size_t)b * W + j) * N * N);
}

// ---- present-agent rows (mapf_rl_b200/present.py): output row first[f] + a holds agent a < min(n[f], N) of frame f; first is
// nondecreasing with first[f] + min(n[f], N) <= first[f + 1]; every other row up to out_rows is zeros ----

// frame f of output row m (-1 if m lies before first[0]): the last f with first[f] <= m
__device__ __forceinline__ int present_frame(const int32_t *__restrict__ first, const int count, const int64_t m)
{
    int lo = 0, hi = count;  // invariant: first[f] <= m for f < lo, first[f] > m for f >= hi
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(first + mid) <= m) lo = mid + 1;
        else hi = mid;
    }
    return lo - 1;
}

// Output rows are 486 elements, so one row does not start on a 16-byte boundary, but eight consecutive rows do (8 * 486
// elements, u8 or 16-bit).  A CTA therefore owns a run of rows (a multiple of 8), stages their packed 64-byte rows in shared
// memory -- laid out like one frame of that many agents, so frame_bits8 reads across row ends -- and writes 16-byte streaming
// stores that straddle rows.  Only the last run may be cut short by out_rows; its tail past the last whole 16 bytes is
// written element by element.
template <uint32_t ONE>
__device__ __forceinline__ void expand_run(const uint8_t *s_rows, const int nrows, const int64_t elems, void *dst)
{
    constexpr int G = ONE == 1 ? 16 : 8;  // elements per 16-byte store
    const int64_t groups = elems / G;
    for (int64_t q = threadIdx.x; q < groups; q += blockDim.x) {
        const int e0 = (int)q * G;
        const uint32_t w = frame_bits8(s_rows, nrows, e0);
        if constexpr (ONE == 1) {
            const uint32_t w2 = frame_bits8(s_rows, nrows, e0 + 8);
            __stcs(reinterpret_cast<uint4 *>(dst) + q,
                   make_uint4(expand4(w & 0xfu), expand4(w >> 4), expand4(w2 & 0xfu), expand4(w2 >> 4)));
        } else {
            __stcs(reinterpret_cast<uint4 *>(dst) + q, make_uint4(bits2_to_pair<ONE>(w), bits2_to_pair<ONE>(w >> 2),
                                                                bits2_to_pair<ONE>(w >> 4), bits2_to_pair<ONE>(w >> 6)));
        }
    }
    if (threadIdx.x == 0) {
        for (int64_t e = groups * G; e < elems; ++e) {
            const int a = (int)(e / MAPF_OBS_BYTES_PER_AGENT), k = (int)(e - (int64_t)a * MAPF_OBS_BYTES_PER_AGENT);
            const uint32_t bit = (s_rows[a * MAPF_OBS_PACKED_BYTES_PER_AGENT + (k >> 3)] >> (k & 7)) & 1u;
            if constexpr (ONE == 1) reinterpret_cast<uint8_t *>(dst)[e] = (uint8_t)bit;
            else reinterpret_cast<uint16_t *>(dst)[e] = (uint16_t)(bit * ONE);
        }
    }
}

constexpr int kUnpackRunRows = 32;  // output rows per CTA of obs_unpack_present_kernel

template <uint32_t ONE>
__global__ void __launch_bounds__(256)
obs_unpack_present_kernel(const uint8_t *__restrict__ bits, const int64_t *__restrict__ rows, const uint8_t *__restrict__ n,
                          const int32_t *__restrict__ first, const int count, const int N, const int64_t out_rows,
                          void *__restrict__ out)
{
    __shared__ __align__(16) uint8_t s_rows[kUnpackRunRows * MAPF_OBS_PACKED_BYTES_PER_AGENT];
    const int64_t r0 = (int64_t)blockIdx.x * kUnpackRunRows;
    const int nrows = (int)min((int64_t)kUnpackRunRows, out_rows - r0);
    // four threads per row, one 16-byte quarter each
    for (int k = threadIdx.x; k < kUnpackRunRows * 4; k += blockDim.x) {
        const int i = k >> 2;
        uint4 x = make_uint4(0, 0, 0, 0);
        if (i < nrows) {
            const int64_t m = r0 + i;
            const int f = present_frame(first, count, m);
            if (f >= 0) {
                const int64_t a = m - first[f];
                if (a < min((int)n[f], N))
                    x = __ldg(reinterpret_cast<const uint4 *>(bits + ((size_t)rows[f] * N + a) * MAPF_OBS_PACKED_BYTES_PER_AGENT) + (k & 3));
            }
        }
        reinterpret_cast<uint4 *>(s_rows)[k] = x;
    }
    __syncthreads();
    uint8_t *dst = reinterpret_cast<uint8_t *>(out) + (size_t)r0 * MAPF_OBS_BYTES_PER_AGENT * (ONE == 1 ? 1 : 2);
    expand_run<ONE>(s_rows, kUnpackRunRows, (int64_t)nrows * MAPF_OBS_BYTES_PER_AGENT, dst);
}

constexpr int kGatherRunRows = 8;  // output rows per observation CTA of replay_gather_present_kernel
constexpr int kGatherMaxW = 64;    // window frames the staging buffer holds (bt_steps + forward_steps, checked on the host)

struct PresentGatherParams {
    mapf_replay_view_compact v;
    mapf_replay_batch o;  // obs [out_rows, W, 6, 9, 9] and hidden [out_rows, latent] in present rows
    const uint8_t *agents;
    const int64_t *idx;
    const int32_t *first;
    int32_t *err;
    int batch;
    int64_t out_rows;
    int runs;  // CTAs [0, runs) write observation and hidden rows, CTA runs + b the comm mask and scalars of sample b
};

// replay_gather_compact_kernel's window, padding, error latch and scalars, with observations and hidden vectors in present
// rows: row first[b] + a is agent a < n_b of sample b, n_b = agents[slot of b] (clamped to N)
__global__ void __launch_bounds__(256)
replay_gather_present_kernel(const PresentGatherParams p)
{
    __shared__ __align__(16) uint8_t s_rows[kGatherRunRows * kGatherMaxW * MAPF_OBS_PACKED_BYTES_PER_AGENT];
    __shared__ int64_t s_obs[kGatherRunRows];  // packed row of the row's agent in window frame 0
    __shared__ int64_t s_hid[kGatherRunRows];  // leaf of the row's hidden vector, -1: zeros
    __shared__ int s_len[kGatherRunRows];      // live window frames, 0 in zero rows
    const mapf_replay_view_compact &v = p.v;
    const int W = v.bt_steps + v.forward_steps;
    const int N = v.num_agents;

    if ((int)blockIdx.x >= p.runs) {
        const int64_t b = blockIdx.x - p.runs;
        const Window w = leaf_window(v, p.idx[b]);
        if (threadIdx.x == 0) gather_scalars(v, p.o, p.err, b, w);
        for (int j = 0; j < W; ++j)
            expand_comm_frame(v.comm_bits, w.row(j), N, j < w.len, p.o.comm_mask + ((size_t)b * W + j) * N * N);
        return;
    }

    const int64_t r0 = (int64_t)blockIdx.x * kGatherRunRows;
    const int nrows = (int)min((int64_t)kGatherRunRows, p.out_rows - r0);
    if (threadIdx.x < kGatherRunRows) {
        const int i = threadIdx.x;
        int64_t obs = 0, hid = -1;
        int len = 0;
        if (i < nrows) {
            const int64_t m = r0 + i;
            const int b = present_frame(p.first, p.batch, m);
            if (b >= 0) {
                const int64_t idx = p.idx[b];
                const int a = (int)(m - p.first[b]);
                if (a < min((int)p.agents[idx / v.max_steps], N)) {
                    const Window w = leaf_window(v, idx);
                    obs = w.row(0) * N + a;
                    hid = w.hidden_leaf(v.bt_steps);
                    len = w.len;
                }
            }
        }
        s_obs[i] = obs;
        s_hid[i] = hid;
        s_len[i] = len;
    }
    __syncthreads();
    // packed rows [row][frame][64], four threads per 64 bytes
    for (int k = threadIdx.x; k < kGatherRunRows * W * 4; k += blockDim.x) {
        const int i = k / (W * 4), j = (k >> 2) - i * W;
        uint4 x = make_uint4(0, 0, 0, 0);
        if (j < s_len[i]) {
            const uint8_t *src = v.obs_bits + (size_t)(s_obs[i] + (int64_t)j * N) * MAPF_OBS_PACKED_BYTES_PER_AGENT;
            x = __ldg(reinterpret_cast<const uint4 *>(src) + (k & 3));
        }
        reinterpret_cast<uint4 *>(s_rows)[k] = x;
    }
    __syncthreads();
    expand_run<0x3C00u>(s_rows, kGatherRunRows * W, (int64_t)nrows * W * MAPF_OBS_BYTES_PER_AGENT,
                        p.o.obs + (size_t)r0 * W * MAPF_OBS_BYTES_PER_AGENT);
    // hidden: the sample's stored vector, zeros while t < bt_steps and in zero rows
    const int D = v.latent_dim;
    for (int k = threadIdx.x; k < nrows * D; k += blockDim.x) {
        const int i = k / D, c = k - i * D;
        const int64_t hid = s_hid[i];
        p.o.hidden[(size_t)(r0 + i) * D + c] = hid >= 0 ? v.hid_buf[(size_t)hid * D + c] : (uint16_t)0;
    }
}

// the (W + 1, batch) grid: CTA (j, b) writes window frame j of sample b, CTA (W, b) its hidden rows and scalars
template <typename View>
int launch_window_gather(void (*kernel)(GatherParams<View>), const View *view, const int64_t *d_idx, int64_t batch,
                         const mapf_replay_batch *out, int32_t *d_err, cudaStream_t st)
{
    const GatherParams<View> p{*view, *out, d_idx, d_err};
    const int W = view->bt_steps + view->forward_steps;
    kernel<<<dim3((unsigned)(W + 1), (unsigned)batch), 256, 0, st>>>(p);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

}  // namespace

int mapf_launch_obs_unpack_present(const uint8_t *d_bits, const int64_t *d_rows, const uint8_t *d_n, const int32_t *d_first,
                                   int64_t count, int N, int64_t out_rows, int dtype, void *d_out, cudaStream_t st)
{
    const unsigned grid = (unsigned)((out_rows + kUnpackRunRows - 1) / kUnpackRunRows);
    const int c = (int)count;
    switch (dtype) {
        case MAPF_DTYPE_U8: obs_unpack_present_kernel<1u><<<grid, 256, 0, st>>>(d_bits, d_rows, d_n, d_first, c, N, out_rows, d_out); break;
        case MAPF_DTYPE_F16:
            obs_unpack_present_kernel<0x3C00u><<<grid, 256, 0, st>>>(d_bits, d_rows, d_n, d_first, c, N, out_rows, d_out);
            break;
        default: obs_unpack_present_kernel<0x3F80u><<<grid, 256, 0, st>>>(d_bits, d_rows, d_n, d_first, c, N, out_rows, d_out); break;
    }
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_replay_gather_present(const mapf_replay_view_compact *view, const uint8_t *d_agents, const int64_t *d_idx,
                                      const int32_t *d_first, int64_t batch, int64_t out_rows, const mapf_replay_batch *out,
                                      int32_t *d_err, cudaStream_t st)
{
    PresentGatherParams p;
    p.v = *view;
    p.o = *out;
    p.agents = d_agents;
    p.idx = d_idx;
    p.first = d_first;
    p.err = d_err;
    p.batch = (int)batch;
    p.out_rows = out_rows;
    p.runs = (int)((out_rows + kGatherRunRows - 1) / kGatherRunRows);
    replay_gather_present_kernel<<<(unsigned)(p.runs + batch), 256, 0, st>>>(p);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_obs_unpack(const uint8_t *d_bits, const int64_t *d_rows, int64_t count, int N, int dtype, void *d_out,
                           cudaStream_t st)
{
    switch (dtype) {
        case MAPF_DTYPE_U8: obs_unpack_kernel<1u><<<(unsigned)count, 256, 0, st>>>(d_bits, d_rows, N, d_out); break;
        case MAPF_DTYPE_F16: obs_unpack_kernel<0x3C00u><<<(unsigned)count, 256, 0, st>>>(d_bits, d_rows, N, d_out); break;
        default: obs_unpack_kernel<0x3F80u><<<(unsigned)count, 256, 0, st>>>(d_bits, d_rows, N, d_out); break;
    }
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

int mapf_launch_replay_gather_compact(const mapf_replay_view_compact *view, const int64_t *d_idx, int64_t batch,
                                      const mapf_replay_batch *out, int32_t *d_err, cudaStream_t st)
{
    return launch_window_gather(replay_gather_compact_kernel, view, d_idx, batch, out, d_err, st);
}

int mapf_launch_replay_gather(const mapf_replay_view *view, const int64_t *d_idx, int64_t batch, const mapf_replay_batch *out,
                              int32_t *d_err, cudaStream_t st)
{
    return launch_window_gather(replay_gather_kernel, view, d_idx, batch, out, d_err, st);
}
