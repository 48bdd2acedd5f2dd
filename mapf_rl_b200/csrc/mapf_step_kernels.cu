// mapf_step_kernels.cu — K1 + K2: Environment.step (environment.py:278-430) fused with the observe()
// it ends in (environment.py:430, 433-467), hand-written for sm_100a.
//
// One warp per environment, lane = agent (K = ceil(N/32) agents per lane).  Per environment:
//   1. all inputs of the env (positions, goals, actions, step counter, obstacle bitmap) are requested
//      up front so their DRAM/L2 latencies overlap;
//   2. conflict resolution runs in registers / shared memory (order-independent fixed point of the
//      reference's restart-on-change scans, SURVEY.md A.2);
//   3. every lane gathers its agent's 6 x 9 x 9 window as a 486-BIT stream (obstacle / agent bitmaps in
//      shared memory, heuristic bits straight from the nibble-planar navi array) and streams it, word
//      by word, into the env's dense bit stream in shared memory;
//   4. the warp expands bits to bool bytes and writes the env's N*486-byte block with fully coalesced
//      128-bit stores.
// HBM-bound (486 B written per agent-step); nothing here is a dense contraction, so no tensor cores.
#include "mapf_step_device.cuh"

namespace {

// ---- K1+K2: every warp steps an env, then expands and stores its own observation block.
// (threadIdx.x is read by the kernel: the range its launch bounds give it is what lets the compiler form e with an OR)
// PACKED: the env's frame is N * 64 bytes of bits (MAPF_OBS_PACKED_BYTES_PER_AGENT), stored as it sits in shared memory.
template <int RW, int K, bool DO_STEP, int WARPS, bool SIZED, bool PACKED = false>
__device__ __forceinline__ void step_observe_body(const StepParams &p, uint32_t *smem, const int tid, const uint8_t *sz_n = nullptr,
                                                  const uint8_t *sz_l = nullptr)
{
    const EnvDims &d = p.d;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int N = d.N;

    uint32_t *s_obst = smem + (size_t)warp * p.warp_smem_words;
    uint32_t *s_agent = s_obst + p.obst_words;
    uint32_t *s_bits = s_agent + p.obst_words;
    uint16_t *s_tgt = reinterpret_cast<uint16_t *>(s_bits + p.bits_words);
    uint16_t *s_cell = s_tgt + 32 * K;

    const uint64_t pol_keep = l2_policy_evict_last();
    const uint64_t pol_stream = l2_policy_evict_first();
    const bool obs_policy = p.flags & MAPF_STEPF_OBS_POLICY;

    // the agent bitmap must start all-zero; afterwards each env clears the bits it set
    for (int w = lane; w < p.obst_words; w += 32) s_agent[w] = 0;
    __syncwarp();

    for (int e = p.env_begin + blockIdx.x * WARPS + warp; e < p.env_end; e += gridDim.x * WARPS) {
        const size_t env_bytes = (size_t)N * (PACKED ? MAPF_OBS_PACKED_BYTES_PER_AGENT : MAPF_OBS_BYTES_PER_AGENT);
        uint8_t *obs_env = p.obs + (size_t)(p.obs_rows ? p.obs_rows[e] : (int64_t)e) * env_bytes;
        const int head = PACKED ? 0 : (int)(reinterpret_cast<uintptr_t>(obs_env) & 15);  // bytes before the 16-B boundary
        EnvRegs<K> r;
        env_step_gather<RW, K, DO_STEP, true, false, SIZED, PACKED>(p, e, lane, s_obst, s_agent, s_bits, s_tgt, s_cell, head, pol_keep,
                                                                    r, nullptr, nullptr, false, nullptr, sz_n, sz_l);
        if constexpr (PACKED) store_packed_block(obs_env, N * (MAPF_OBS_PACKED_BYTES_PER_AGENT / 16), s_bits, lane, obs_policy, pol_stream);
        else expand_store_block(p, obs_env, head, env_bytes, s_bits, lane, obs_policy, pol_stream);
        __syncwarp();
        clear_agent_bits<RW, K>(s_agent, r);  // the agent bits this env set
    }
}

template <int RW, int K, bool DO_STEP, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
step_observe_kernel(const StepParams p)
{
    extern __shared__ __align__(16) uint32_t smem[];
    step_observe_body<RW, K, DO_STEP, WARPS, false>(p, smem, threadIdx.x);
}

// the same for a sized handle (per-environment agent count and side, mapf_env_enable_sizes): a separate instantiation, so
// the uniform kernels above carry none of it
template <int RW, int K, bool DO_STEP>
__global__ void __launch_bounds__(128)
step_observe_sized_kernel(const StepParams p, const uint8_t *__restrict__ sz_n, const uint8_t *__restrict__ sz_l)
{
    extern __shared__ __align__(16) uint32_t smem[];
    step_observe_body<RW, K, DO_STEP, 4, true>(p, smem, threadIdx.x, sz_n, sz_l);
}

// the same writing packed frames (mapf_env_step_observe_packed / mapf_env_observe_packed), uniform and sized: separate
// instantiations again, so the dense kernels above are unchanged
template <int RW, int K, bool DO_STEP, int WARPS, int MINB, bool SIZED>
__global__ void __launch_bounds__(WARPS * 32, MINB)
step_observe_packed_kernel(const StepParams p, const uint8_t *__restrict__ sz_n, const uint8_t *__restrict__ sz_l)
{
    extern __shared__ __align__(16) uint32_t smem[];
    step_observe_body<RW, K, DO_STEP, WARPS, SIZED, true>(p, smem, threadIdx.x, sz_n, sz_l);
}

// ---- K1 alone: Environment.step without the observation.  The host-buffer steps launch it ahead of the observe kernel so
// that the device-to-host copies of the results run WHILE the observation is being written; with p.pos_out it also leaves a
// snapshot of the new positions for that observe kernel, so the NEXT step may overwrite the positions meanwhile.
template <int RW, int K>
__global__ void __launch_bounds__(128)
step_only_kernel(const StepParams p)
{
    extern __shared__ __align__(16) uint32_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    uint32_t *s_obst = smem + (size_t)warp * p.warp_smem_words;
    uint32_t *s_agent = s_obst + p.obst_words;
    uint32_t *s_bits = s_agent + p.obst_words;
    uint16_t *s_tgt = reinterpret_cast<uint16_t *>(s_bits + p.bits_words);
    uint16_t *s_cell = s_tgt + 32 * K;
    const int e = blockIdx.x * 4 + warp;
    // The CTA's four action rows are contiguous (4 N bytes): fetched as 16-byte words, they are a few 128-byte requests per
    // CTA instead of one 32-byte request per warp -- mapf_env_step_host points `actions` at page-locked HOST memory and the
    // kernel's time is the PCIe round trips of this load.
    __shared__ __align__(16) uint8_t s_actions[4 * MAPF_MAX_AGENTS];
    const int N = p.d.N;
    const uint8_t *rows = p.actions + (size_t)blockIdx.x * 4 * N;
    const int nbytes = min(4, p.d.B - (int)blockIdx.x * 4) * N;
    const bool staged = ((reinterpret_cast<uintptr_t>(rows) | (uintptr_t)nbytes) & 15) == 0;
    if constexpr (MAPF_RANKED_LOOKUP(RW)) {  // the ranked occupant lookup builds the old positions' bitmap in s_agent: it must start all-zero
        for (int w = lane; w < p.obst_words; w += 32) s_agent[w] = 0;
    }
    if (staged) {
        for (int w = threadIdx.x; w < (nbytes >> 4); w += blockDim.x)
            reinterpret_cast<uint4 *>(s_actions)[w] = __ldg(reinterpret_cast<const uint4 *>(rows) + w);
    }
    __syncthreads();
    if (e >= p.d.B) return;
    EnvRegs<K> r;
    env_step_gather<RW, K, true, false>(p, e, lane, s_obst, s_agent, s_bits, s_tgt, s_cell, 0, 0ull, r,
                                        staged ? s_actions + warp * N : nullptr);
}

// ---- launch plumbing ---------------------------------------------------------------------------
struct StepTuning {
    int variant;       // CTA shape / register cap of the (RW = 2, K = 1) instantiation, see launch_step_rwk
    int flags;
    int ctas_per_sm;   // > 0: persistent grid of that many CTAs per SM, each warp strides over environments
};

StepTuning &tuning()
{
    static StepTuning t = [] {
        StepTuning r{1, MAPF_STEPF_NAVI_KEEP, 0};
        if (const char *s = std::getenv("MAPF_STEP_VARIANT")) r.variant = std::atoi(s);
        if (const char *s = std::getenv("MAPF_STEP_FLAGS")) r.flags = std::atoi(s);
        if (const char *s = std::getenv("MAPF_STEP_CTAS_PER_SM")) r.ctas_per_sm = std::atoi(s);
        return r;
    }();
    return t;
}

template <int RW, int K, bool DO_STEP, int WARPS, int MINB>
int launch_step_cfg(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    auto kern = step_observe_kernel<RW, K, DO_STEP, WARPS, MINB>;
    const size_t smem = (size_t)p.warp_smem_words * 4 * WARPS;
    if (smem > 227 * 1024) {
        mapf_set_error("map too large for the step kernel's shared memory");
        return MAPF_EINVAL;
    }
    if (smem > 48 * 1024)  // per-device attribute; cheap enough to set on every large-smem launch
        MAPF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = (p.env_end - p.env_begin + WARPS - 1) / WARPS;
    if (tuning().ctas_per_sm > 0) {
        const int cap = env->num_sms * tuning().ctas_per_sm;
        if (grid > cap) grid = cap;
    }
    kern<<<grid, WARPS * 32, smem, st>>>(p);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

template <int RW, int K, bool DO_STEP>
int launch_step_rwk(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    if constexpr (RW == 2 && K == 1) {
        // CTA shape / register budget of the hot geometry (40x40, <= 32 agents), measured at 8192 x 32 (profiles/
        // r1_rollout_cta_shapes.log; us per step as one whole-batch launch / as 8 rollout chains):
        //   0: 8 warps, 48 regs, 40 warps/SM   33.3 / 24.9        7: 8 warps, 64 regs, 32 warps/SM   34.8 / 24.2
        //   4: 4 warps, 40 regs, 48 warps/SM   34.3 / 25.7        8: 4 warps, 64 regs, 32 warps/SM   34.6 / 24.4
        // 1 (default) picks 0 for a launch over the whole batch and 7 for a sub-batch launch of the chained rollout, whose
        // concurrent chains supply the parallelism that the extra resident warps otherwise would.
        int v = tuning().variant;
        if (v == 1) v = (p.env_end - p.env_begin < env->d.B) ? 7 : 0;
        switch (v) {
            case 0: return launch_step_cfg<RW, K, DO_STEP, 8, 5>(env, p, st);
            case 7: return launch_step_cfg<RW, K, DO_STEP, 8, 4>(env, p, st);
            case 8: return launch_step_cfg<RW, K, DO_STEP, 4, 8>(env, p, st);
            default: break;  // 4: the general shape below
        }
    }
    if constexpr (K == 2 && DO_STEP && RW <= 2) {  // (at 80x80 shared memory holds 20 warps per SM and the cap costs 1.4 %)
        // two agents per lane (33..64 agents): the general shape below runs at 80 registers / 24 warps per SM.  Capped at
        // 64 registers (32 warps per SM, no spills) a whole-batch launch of 8192 x 64 agents takes 69.2 instead of 72.7 us;
        // the rollout's sub-batch launches are no faster (52.8 vs 52.4 us per step; profiles/r1_rollout_cta_shapes.log)
        int v = tuning().variant;
        if (v == 1) v = (p.env_end - p.env_begin < env->d.B) ? 4 : 9;
        if (v == 9) return launch_step_cfg<RW, K, DO_STEP, 4, 8>(env, p, st);
    }
    return launch_step_cfg<RW, K, DO_STEP, 4, (K == 1 ? 12 : 1)>(env, p, st);
}

template <int RW, int K, bool DO_STEP>
int launch_step_sized(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    auto kern = step_observe_sized_kernel<RW, K, DO_STEP>;
    const size_t smem = (size_t)p.warp_smem_words * 4 * 4;
    if (smem > 227 * 1024) {
        mapf_set_error("map too large for the step kernel's shared memory");
        return MAPF_EINVAL;
    }
    if (smem > 48 * 1024) MAPF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(p.env_end - p.env_begin + 3) / 4, 128, smem, st>>>(p, env->sz_n, env->sz_l);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

template <int RW, bool DO_STEP>
int launch_step_rw(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    if (env->sz_n) {
        switch (env->d.K) {
            case 1: return launch_step_sized<RW, 1, DO_STEP>(env, p, st);
            case 2: return launch_step_sized<RW, 2, DO_STEP>(env, p, st);
            case 3: return launch_step_sized<RW, 3, DO_STEP>(env, p, st);
            case 4: return launch_step_sized<RW, 4, DO_STEP>(env, p, st);
        }
    }
    switch (env->d.K) {
        case 1: return launch_step_rwk<RW, 1, DO_STEP>(env, p, st);
        case 2: return launch_step_rwk<RW, 2, DO_STEP>(env, p, st);
        case 3: return launch_step_rwk<RW, 3, DO_STEP>(env, p, st);
        case 4: return launch_step_rwk<RW, 4, DO_STEP>(env, p, st);
    }
    mapf_set_error("unsupported agent count");
    return MAPF_EINVAL;
}

// Packed frames take the CTA shape the dense whole-batch launch takes for the same geometry (launch_step_rwk), so the two
// compare at equal occupancy; a sized handle takes the shape of step_observe_sized_kernel.
template <int RW, int K, bool DO_STEP, bool SIZED>
int launch_packed_rwk(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    constexpr bool hot1 = !SIZED && RW == 2 && K == 1, hot2 = !SIZED && K == 2 && DO_STEP && RW <= 2;
    constexpr int WARPS = hot1 ? 8 : 4;
    constexpr int MINB = hot1 ? 5 : (hot2 ? 8 : (SIZED || K > 1 ? 1 : 12));
    auto kern = step_observe_packed_kernel<RW, K, DO_STEP, WARPS, MINB, SIZED>;
    const size_t smem = (size_t)p.warp_smem_words * 4 * WARPS;
    if (smem > 227 * 1024) {
        mapf_set_error("map too large for the step kernel's shared memory");
        return MAPF_EINVAL;
    }
    if (smem > 48 * 1024) MAPF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(p.env_end - p.env_begin + WARPS - 1) / WARPS, WARPS * 32, smem, st>>>(p, env->sz_n, env->sz_l);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

template <int RW, bool DO_STEP, bool SIZED>
int launch_packed_rw(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    switch (env->d.K) {
        case 1: return launch_packed_rwk<RW, 1, DO_STEP, SIZED>(env, p, st);
        case 2: return launch_packed_rwk<RW, 2, DO_STEP, SIZED>(env, p, st);
        case 3: return launch_packed_rwk<RW, 3, DO_STEP, SIZED>(env, p, st);
        case 4: return launch_packed_rwk<RW, 4, DO_STEP, SIZED>(env, p, st);
    }
    mapf_set_error("unsupported agent count");
    return MAPF_EINVAL;
}

template <bool DO_STEP, bool SIZED>
int launch_packed_sz(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    switch (env->d.RW) {
        case 1: return launch_packed_rw<1, DO_STEP, SIZED>(env, p, st);
        case 2: return launch_packed_rw<2, DO_STEP, SIZED>(env, p, st);
        case 3: return launch_packed_rw<3, DO_STEP, SIZED>(env, p, st);
        case 4: return launch_packed_rw<4, DO_STEP, SIZED>(env, p, st);
    }
    mapf_set_error("unsupported map size");
    return MAPF_EINVAL;
}

template <bool DO_STEP>
int launch_packed(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    return env->sz_n ? launch_packed_sz<DO_STEP, true>(env, p, st) : launch_packed_sz<DO_STEP, false>(env, p, st);
}

template <bool DO_STEP>
int launch_step(const mapf_env *env, StepParams &p, cudaStream_t st)
{
    switch (env->d.RW) {
        case 1: return launch_step_rw<1, DO_STEP>(env, p, st);
        case 2: return launch_step_rw<2, DO_STEP>(env, p, st);
        case 3: return launch_step_rw<3, DO_STEP>(env, p, st);
        case 4: return launch_step_rw<4, DO_STEP>(env, p, st);
    }
    mapf_set_error("unsupported map size");
    return MAPF_EINVAL;
}

}  // namespace

static int g_tuning_generation = 0;
int mapf_step_tuning_generation() { return g_tuning_generation; }  // captured launches are stale once this moves

int mapf_step_flags() { return tuning().flags | 0; }

// Everything of StepParams that does not depend on the call: geometry, arena pointers, rewards, shared-memory layout.
StepParams mapf_make_step_params(const mapf_env *env, bool packed)
{
    StepParams p{};
    const EnvDims &d = env->d;
    p.d = d;
    p.obst = env->obst;
    p.pos = env->pos;
    p.goal = env->goal;
    p.navi = env->navi;
    p.navi_alt = env->navi_alt;
    p.navi_sel = env->navi_sel;
    p.steps = env->steps;
    p.err = env->err;
    for (int i = 0; i < 5; ++i) p.r[i] = env->reward[i];
    p.obst_words = d.obst_stride;
    // stream words: 15 head bits max + N*486 bits, +2 words of slack for the u16 tail read (packed: 16 words per agent); the
    // same buffer holds the L*L-byte occupancy grid of the step phase
    const int stream_words = packed ? d.N * (MAPF_OBS_PACKED_BYTES_PER_AGENT / 4) : ((15 + d.N * MAPF_OBS_BYTES_PER_AGENT + 31) >> 5) + 2;
    // step-phase scratch in the same buffer: the L*L-byte occupancy grid, or (`RANKED` in mapf_step_device.cuh) the claim
    // bitmap + row ranks + rank -> agent table
    const int occ_words = MAPF_RANKED_LOOKUP(d.RW) ? ((((d.L * d.L + 127) >> 7) << 2) + ((d.R + 3) >> 2) + ((d.N + 3) >> 2)) : ((d.L * d.L + 3) >> 2);
    p.bits_words = stream_words > occ_words ? stream_words : occ_words;
    const int words = 2 * p.obst_words + p.bits_words + (32 * d.K) /* s_tgt + s_cell, u16 each */;
    p.warp_smem_words = (words + 3) & ~3;
    p.flags = tuning().flags | (env->check_unique ? MAPF_STEPF_CHECK_UNIQUE : 0);
    p.env_begin = 0;
    p.env_end = d.B;
    return p;
}

void mapf_set_step_tuning(int variant, int flags, int ctas_per_sm)
{
    ++g_tuning_generation;
    StepTuning &t = tuning();
    if (variant >= 0) t.variant = variant;
    if (flags >= 0) t.flags = flags;
    if (ctas_per_sm >= 0) t.ctas_per_sm = ctas_per_sm;
}

static void fill_out(StepParams &p, const StepOut &o)
{
    p.rewards = o.rewards;
    p.codes = o.codes;
    p.done = o.done;
    p.steps_out = o.steps;
}

int mapf_launch_step(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs, const int64_t *d_obs_rows, const StepOut &out,
                     cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env);
    p.actions = d_actions;
    p.obs = d_obs;
    p.obs_rows = d_obs_rows;
    fill_out(p, out);
    return launch_step<true>(env, p, st);
}

template <int RW, int K>
static int launch_step_only_cfg(mapf_env *env, const StepParams &p, cudaStream_t st)
{
    auto kern = step_only_kernel<RW, K>;
    const size_t smem = (size_t)p.warp_smem_words * 4 * 4;
    if (smem > 227 * 1024) {
        mapf_set_error("map too large for the step kernel's shared memory");
        return MAPF_EINVAL;
    }
    if (smem > 48 * 1024) MAPF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(env->d.B + 3) / 4, 128, smem, st>>>(p);
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

// One step of the sub-batch [e0, e1) only (chained rollout: independent chains of launches over disjoint env ranges);
// all pointers are those of the whole batch.
int mapf_launch_step_range(mapf_env *env, int e0, int e1, const uint8_t *d_actions, uint8_t *d_obs, const StepOut &out,
                           cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env);
    p.actions = d_actions;
    p.obs = d_obs;
    fill_out(p, out);
    p.env_begin = e0;
    p.env_end = e1;
    return launch_step<true>(env, p, st);
}

int mapf_launch_step_only(mapf_env *env, const uint8_t *d_actions, const StepOut &out, uint8_t *d_pos_snapshot, cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env);
    p.actions = d_actions;
    p.pos_out = d_pos_snapshot;
    fill_out(p, out);
    switch (env->d.RW * 10 + env->d.K) {
        case 11: return launch_step_only_cfg<1, 1>(env, p, st);
        case 12: return launch_step_only_cfg<1, 2>(env, p, st);
        case 13: return launch_step_only_cfg<1, 3>(env, p, st);
        case 14: return launch_step_only_cfg<1, 4>(env, p, st);
        case 21: return launch_step_only_cfg<2, 1>(env, p, st);
        case 22: return launch_step_only_cfg<2, 2>(env, p, st);
        case 23: return launch_step_only_cfg<2, 3>(env, p, st);
        case 24: return launch_step_only_cfg<2, 4>(env, p, st);
        case 31: return launch_step_only_cfg<3, 1>(env, p, st);
        case 32: return launch_step_only_cfg<3, 2>(env, p, st);
        case 33: return launch_step_only_cfg<3, 3>(env, p, st);
        case 34: return launch_step_only_cfg<3, 4>(env, p, st);
        case 41: return launch_step_only_cfg<4, 1>(env, p, st);
        case 42: return launch_step_only_cfg<4, 2>(env, p, st);
        case 43: return launch_step_only_cfg<4, 3>(env, p, st);
        case 44: return launch_step_only_cfg<4, 4>(env, p, st);
    }
    mapf_set_error("unsupported geometry");
    return MAPF_EINVAL;
}

// d_pos_src (optional): observe THESE positions (a snapshot left by mapf_launch_step_only) instead of the handle's
int mapf_launch_observe(mapf_env *env, uint8_t *d_obs, const int64_t *d_obs_rows, uint8_t *d_pos, const uint8_t *d_pos_src,
                        cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env);
    if (d_pos_src) p.pos = const_cast<uint8_t *>(d_pos_src);
    p.obs = d_obs;
    p.obs_rows = d_obs_rows;
    p.pos_out = d_pos;
    return launch_step<false>(env, p, st);
}

// packed frames (mapf_env_step_observe_packed / mapf_env_observe_packed): d_bits_base is 16-byte aligned, rows optional
int mapf_launch_step_packed(mapf_env *env, const uint8_t *d_actions, uint8_t *d_bits, const int64_t *d_rows, const StepOut &out,
                            cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env, true);
    p.actions = d_actions;
    p.obs = d_bits;
    p.obs_rows = d_rows;
    fill_out(p, out);
    return launch_packed<true>(env, p, st);
}

int mapf_launch_observe_packed(mapf_env *env, uint8_t *d_bits, const int64_t *d_rows, uint8_t *d_pos, cudaStream_t st)
{
    StepParams p = mapf_make_step_params(env, true);
    p.obs = d_bits;
    p.obs_rows = d_rows;
    p.pos_out = d_pos;
    return launch_packed<false>(env, p, st);
}
