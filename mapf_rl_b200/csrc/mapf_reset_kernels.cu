// mapf_reset_kernels.cu — device-side instance generation: Environment.reset / __init__ without the
// host (environment.py:100-138 == :156-192, map_partition :21-70), sm_100a.
//
// One warp per environment (mapf_reset_device.cuh), followed by a masked BFS launch.
#include "mapf_reset_device.cuh"

namespace {

template <int RW, int RPL>
__global__ void __launch_bounds__(128)
reset_kernel(EnvDims d, const uint8_t *__restrict__ mask, uint64_t seed, uint64_t env_offset, float density,
             uint32_t *__restrict__ obst, uint8_t *__restrict__ pos, uint8_t *__restrict__ goal,
             int32_t *__restrict__ steps, int32_t *__restrict__ err)
{
    const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (e >= d.B) return;
    if (mask && !mask[e]) return;
    reset_env_warp<RW, RPL>(d, e, seed, env_offset + (uint64_t)e, density, obst, pos, goal, steps, err);
}

// Sized handle: every slot being reset draws its setting uniformly from the K levels (n, l) -- index (w K) >> 32 with w the
// first word of Philox counter (g, PURPOSE_LEVEL, 0) of its own stream g = env_offset + e, so the draw does not depend on how
// the batch is sharded -- and generates instance g at that setting: what reset() of a uniform (n, l) handle draws for g.
// Absent agent rows read 255.
template <int RW, int RPL>
__global__ void __launch_bounds__(128)
reset_levels_kernel(EnvDims d, const uint8_t *__restrict__ mask, uint64_t seed, uint64_t env_offset, float density,
                    const uint8_t *__restrict__ levels, int num_levels, uint32_t *__restrict__ obst, uint8_t *__restrict__ pos,
                    uint8_t *__restrict__ goal, int32_t *__restrict__ steps, int32_t *__restrict__ err, uint8_t *__restrict__ sz_n,
                    uint8_t *__restrict__ sz_l)
{
    const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (e >= d.B) return;
    if (mask && !mask[e]) return;
    const int lane = threadIdx.x & 31;
    const uint64_t g = env_offset + (uint64_t)e;
    const uint4 r = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), PURPOSE_LEVEL, 0u),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const int k = (int)(((uint64_t)r.x * (uint64_t)num_levels) >> 32);
    const int n = levels[2 * k], l = levels[2 * k + 1];
    reset_env_warp<RW, RPL>(d, e, seed, g, density, obst, pos, goal, steps, err, l, n);
    for (int a = n + lane; a < d.N; a += 32) {
        reinterpret_cast<uchar2 *>(pos)[(size_t)e * d.N + a] = make_uchar2(255, 255);
        reinterpret_cast<uchar2 *>(goal)[(size_t)e * d.N + a] = make_uchar2(255, 255);
    }
    if (lane == 0) sz_n[e] = (uint8_t)n, sz_l[e] = (uint8_t)l;
}

// The NEXT instance of every listed slot (the slots whose episode ends inside the coming rollout launch) into the staging
// arrays: instance number episode[e] + 1 of slot e, i.e. what the rollout kernel would generate in place at the episode's
// end.  The list's length is only known on the device: a fixed grid claims list entries from a counter.
template <int RW, int RPL>
__global__ void __launch_bounds__(128)
pregen_reset_kernel(EnvDims d, const uint32_t *__restrict__ list, int min_count, unsigned long long *__restrict__ counter, uint64_t seed,
                    uint64_t env_offset, uint64_t stride, float density, const uint32_t *__restrict__ episode,
                    uint32_t *__restrict__ pg_obst, uint8_t *__restrict__ pg_pos, uint8_t *__restrict__ pg_goal,
                    int32_t *__restrict__ pg_steps, uint32_t *__restrict__ pg_n, int32_t *__restrict__ err)
{
    const int lane = threadIdx.x & 31;
    const unsigned long long count = list[0];
    if (count < (unsigned long long)min_count) return;  // few: the rollout kernel re-generates them itself
    for (;;) {
        unsigned long long it = 0;
        if (lane == 0) it = atomicAdd(counter, 1ull);
        it = __shfl_sync(MAPF_FULL_MASK, it, 0);
        if (it >= count) break;
        const int e = (int)list[1 + it];
        // (__ldcg: beside a running rollout kernel the slot's episode count may just have moved on -- a done-triggered episode
        // end -- and the instance staged here is then simply never adopted)
        const uint32_t n = __ldcg(episode + e) + 1u;
        const uint64_t g = env_offset + (uint64_t)n * stride + (uint64_t)e;
        reset_env_warp<RW, RPL>(d, e, seed, g, density, pg_obst, pg_pos, pg_goal, pg_steps, err);
        if (lane == 0) pg_n[e] = n;
    }
}

template <int RW>
int launch_reset_rw(mapf_env *env, const uint8_t *mask, uint64_t seed, uint64_t off, float density, int pregen_min, cudaStream_t st,
                    const uint8_t *levels = nullptr, int num_levels = 0)
{
    const EnvDims &d = env->d;
    const int rpl = (d.L + 31) / 32;
    const int warps = 4;
    const bool pregen = pregen_min >= 0;
    const int grid = pregen ? env->num_sms * 4 : (d.B + warps - 1) / warps;
#define MAPF_RESET_LAUNCH(RPL)                                                                                                   \
    do {                                                                                                                         \
        if (levels)                                                                                                              \
            reset_levels_kernel<RW, RPL><<<grid, warps * 32, 0, st>>>(d, mask, seed, off, density, levels, num_levels, env->obst,    \
                                                                      env->pos, env->goal, env->steps, env->err, env->sz_n,      \
                                                                      env->sz_l);                                                \
        else if (pregen)                                                                                                         \
            pregen_reset_kernel<RW, RPL><<<grid, warps * 32, 0, st>>>(d, env->ro_prio, pregen_min, env->ro_work + 2, env->ar_seed, \
                                                                      env->ar_offset, env->ar_stride, env->ar_density,           \
                                                                      env->ro_episode, env->pg_obst, env->pg_pos, env->pg_goal,  \
                                                                      env->pg_steps, env->pg_n, env->err);                       \
        else                                                                                                                     \
            reset_kernel<RW, RPL><<<grid, warps * 32, 0, st>>>(d, mask, seed, off, density, env->obst, env->pos, env->goal,      \
                                                                env->steps, env->err);                                           \
    } while (0)
    switch (rpl) {
        case 1: MAPF_RESET_LAUNCH(1); break;
        case 2: MAPF_RESET_LAUNCH(2); break;
        case 3: MAPF_RESET_LAUNCH(3); break;
        case 4: MAPF_RESET_LAUNCH(4); break;
        default: mapf_set_error("unsupported map size"); return MAPF_EINVAL;
    }
#undef MAPF_RESET_LAUNCH
    MAPF_CUDA(cudaGetLastError());
    return MAPF_OK;
}

}  // namespace

int mapf_launch_bfs_masked(mapf_env *env, const uint8_t *d_mask, cudaStream_t st);
int mapf_launch_pregen_bfs(mapf_env *env, int min_count, cudaStream_t st);

static int launch_reset(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density, int pregen_min,
                        cudaStream_t st, const uint8_t *levels = nullptr, int num_levels = 0)
{
    switch (env->d.RW) {
        case 1: return launch_reset_rw<1>(env, d_mask, seed, env_offset, density, pregen_min, st, levels, num_levels);
        case 2: return launch_reset_rw<2>(env, d_mask, seed, env_offset, density, pregen_min, st, levels, num_levels);
        case 3: return launch_reset_rw<3>(env, d_mask, seed, env_offset, density, pregen_min, st, levels, num_levels);
        case 4: return launch_reset_rw<4>(env, d_mask, seed, env_offset, density, pregen_min, st, levels, num_levels);
    }
    mapf_set_error("unsupported map size");
    return MAPF_EINVAL;
}

int mapf_launch_reset(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density,
                      cudaStream_t st)
{
    const int rc = launch_reset(env, d_mask, seed, env_offset, density, -1, st);
    if (rc != MAPF_OK) return rc;
    return mapf_launch_bfs_masked(env, d_mask, st);  // get_navi_map, environment.py:195
}

// sized handle: d_levels u8[K, 2] (checked by the caller), then the masked BFS of the slots it re-generated
int mapf_launch_reset_levels(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density,
                             const uint8_t *d_levels, int num_levels, cudaStream_t st)
{
    const int rc = launch_reset(env, d_mask, seed, env_offset, density, -1, st, d_levels, num_levels);
    if (rc != MAPF_OK) return rc;
    return mapf_launch_bfs_masked(env, d_mask, st);
}

// Episode handling of mapf_env_rollout: the next instance of every slot listed in env->ro_prio (rollout_prio_kernel), generator
// + heuristic maps at the full occupancy of the dedicated kernels, staged for the rollout kernel to adopt (mapf_common.cuh).
int mapf_launch_pregen(mapf_env *env, int min_count, cudaStream_t st)
{
    const int rc = launch_reset(env, nullptr, 0, 0, 0.f, min_count < 0 ? 0 : min_count, st);
    if (rc != MAPF_OK) return rc;
    return mapf_launch_pregen_bfs(env, min_count, st);
}

#ifdef MAPF_ENABLE_DIAG
// diagnosis build only: cycles per generator phase of environment 0 in the last reset_kernel launch
extern "C" int mapf_diag_reset_cycles(unsigned long long *out8)
{
    return cudaMemcpyFromSymbol(out8, g_reset_cycles, sizeof(unsigned long long) * 8) == cudaSuccess ? 0 : -1;
}
#endif
