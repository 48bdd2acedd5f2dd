// mapf_abi.cu — extern "C" entry points of libmapf_b200.so (declared in include/mapf_b200.h).
// Argument validation, arena ownership and stream plumbing only; the kernels live in
// mapf_env_kernels.cu / mapf_reset_kernels.cu / mapf_per_kernels.cu.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <type_traits>

#include "mapf_common.cuh"

// launchers (other translation units)
int mapf_launch_pack_load(mapf_env *, const int32_t *, int, const uint8_t *, const uint8_t *, const uint8_t *, cudaStream_t);
int mapf_launch_pack_load_sized(mapf_env *, const int32_t *, int, const uint8_t *, const uint8_t *, const uint8_t *, const uint8_t *,
                                const uint8_t *, cudaStream_t);
int mapf_launch_reset_levels(mapf_env *, const uint8_t *, uint64_t, uint64_t, float, const uint8_t *, int, cudaStream_t);
int mapf_launch_validate_state(mapf_env *, const int32_t *, int, cudaStream_t);
int mapf_launch_bfs(mapf_env *, const int32_t *, int, int32_t *, cudaStream_t);
int mapf_launch_plan(mapf_env *, int, uint8_t *, int32_t *, cudaStream_t);
int mapf_launch_plan_orders(mapf_env *, int, int, uint64_t, uint64_t, uint8_t *, int32_t *, int32_t *, uint8_t *, cudaStream_t);
int mapf_launch_step(mapf_env *, const uint8_t *, uint8_t *, const int64_t *, const StepOut &, cudaStream_t);
int mapf_launch_observe(mapf_env *, uint8_t *, const int64_t *, uint8_t *, const uint8_t *, cudaStream_t);
int mapf_launch_step_only(mapf_env *, const uint8_t *, const StepOut &, uint8_t *, cudaStream_t);
int mapf_launch_step_range(mapf_env *, int, int, const uint8_t *, uint8_t *, const StepOut &, cudaStream_t);
int mapf_launch_rollout(mapf_env *, int, int, int, const uint8_t *, int, uint8_t *, int, const StepOut &, int, cudaStream_t);
bool mapf_rollout_supported(const mapf_env *);
void mapf_set_rollout_tuning(int, int, int, int);
void mapf_set_rollout_pregen(int);
int &rollout_pregen_ref();
void mapf_set_rollout_tasks(int);
int &rollout_tasks_ref();
void mapf_set_step_tuning(int, int, int);
int mapf_step_tuning_generation();
int mapf_launch_unpack(mapf_env *, uint8_t *, uint8_t *, cudaStream_t);
int mapf_launch_comm_mask(mapf_env *, int, uint8_t *, cudaStream_t);
int mapf_launch_reset(mapf_env *, const uint8_t *, uint64_t, uint64_t, float, cudaStream_t);
int mapf_launch_per_update(mapf_per *, PerScratch *, const int64_t *, const double *, int64_t, cudaStream_t);
int mapf_launch_per_sample(mapf_per *, const double *, int64_t, int64_t *, double *, float *, double, cudaStream_t);
int mapf_launch_per_td_update(mapf_per *, PerScratch *, const float *, const float *, const float *, const int64_t *,
                              const float *, const float *, const float *, const int64_t *, int64_t, float, double, int64_t,
                              int64_t, int64_t, float *, float *, cudaStream_t);
int mapf_launch_per_cycle(mapf_per *, PerScratch *, const mapf_per_cycle_args *, cudaStream_t);
int mapf_launch_actor_td(const float *, const float *, const uint8_t *, const int32_t *, int, int, int, double, double *, cudaStream_t);
int mapf_launch_replay_gather(const mapf_replay_view *, const int64_t *, int64_t, const mapf_replay_batch *, int32_t *, cudaStream_t);
int mapf_launch_step_packed(mapf_env *, const uint8_t *, uint8_t *, const int64_t *, const StepOut &, cudaStream_t);
int mapf_launch_observe_packed(mapf_env *, uint8_t *, const int64_t *, uint8_t *, cudaStream_t);
int mapf_launch_comm_mask_packed(mapf_env *, int, uint8_t *, uint8_t *, const int64_t *, cudaStream_t);
int mapf_launch_obs_unpack(const uint8_t *, const int64_t *, int64_t, int, int, void *, cudaStream_t);
int mapf_launch_replay_gather_compact(const mapf_replay_view_compact *, const int64_t *, int64_t, const mapf_replay_batch *, int32_t *,
                                      cudaStream_t);
int mapf_launch_obs_unpack_present(const uint8_t *, const int64_t *, const uint8_t *, const int32_t *, int64_t, int, int64_t, int,
                                   void *, cudaStream_t);
int mapf_launch_replay_gather_present(const mapf_replay_view_compact *, const uint8_t *, const int64_t *, const int32_t *, int64_t,
                                      int64_t, const mapf_replay_batch *, int32_t *, cudaStream_t);

static thread_local std::string g_last_error;

void mapf_set_error(const std::string &msg) { g_last_error = msg; }

int mapf_cuda_fail(cudaError_t e, const char *what)
{
    g_last_error = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return MAPF_ECUDA;
}

namespace {
struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard()
    {
        if (ok && prev >= 0) cudaSetDevice(prev);
    }
};

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// MAPF_ECUDA with `fn`'s message when the process sees no device
int require_device(const char *fn)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        mapf_set_error(std::string(fn) + ": no CUDA device (this library has no CPU fallback)");
        return MAPF_ECUDA;
    }
    return MAPF_OK;
}

// the arguments only mapf_replay_gather_present takes
struct PresentRowArgs {
    const uint8_t *agents;
    const int32_t *first;
    int64_t out_rows;
};

// The checks of the three window gathers, every MAPF_EINVAL before MAPF_ECUDA.  A compact store's obs_bits must be 16-byte
// aligned (the gathers load packed frames 16 bytes at a time); the present gather (pr != nullptr) stages at most 64 window
// frames and writes its observations 16 bytes at a time.
template <typename View>
int check_window_gather(const char *fn, const View *view, const int64_t *d_idx, int64_t batch, const mapf_replay_batch *out,
                        const PresentRowArgs *pr = nullptr)
{
    constexpr bool compact = std::is_same_v<View, mapf_replay_view_compact>;
    if (!view || !out || batch < 0 || (batch > 0 && !d_idx) ||
        (pr && (pr->out_rows < 0 || (batch > 0 && (!pr->first || !pr->agents))))) {
        mapf_set_error(std::string(fn) + ": NULL argument");
        return MAPF_EINVAL;
    }
    if (view->num_agents < 1 || view->num_agents > MAPF_MAX_AGENTS || view->max_steps < 1 || view->bt_steps < 1 ||
        view->forward_steps < 1 || view->latent_dim < 1 || batch > 65535 ||
        (pr && ((int64_t)view->bt_steps + view->forward_steps > 64 || pr->out_rows > 0x7fffffff))) {
        mapf_set_error(std::string(fn) + (pr ? ": bad dimensions (bt_steps + forward_steps <= 64, batch <= 65535)"
                                             : ": bad dimensions (batch <= 65535)"));
        return MAPF_EINVAL;
    }
    const void *obs, *comm;
    if constexpr (compact) obs = view->obs_bits, comm = view->comm_bits;
    else obs = view->obs_buf, comm = view->comm_buf;
    if (!obs || !comm || !view->hid_buf || !view->act_buf || !view->rew_buf || !view->done_buf || !view->size_buf || !out->obs ||
        !out->comm_mask || !out->hidden || !out->action || !out->reward || !out->done || !out->steps || !out->bt_steps ||
        (compact && !aligned16(obs)) || (pr && !aligned16(out->obs))) {
        mapf_set_error(std::string(fn) + (pr        ? ": NULL buffer, or obs_bits or the obs output not 16-byte aligned"
                                          : compact ? ": NULL buffer or obs_bits not 16-byte aligned"
                                                    : ": NULL buffer"));
        return MAPF_EINVAL;
    }
    return require_device(fn);
}

bool host_is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();  // clear: an unregistered pointer is not an error for us
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// Device-side alias of a page-locked, mapped host buffer (cudaHostAlloc / torch pin_memory under UVA), or
// nullptr when the buffer cannot be addressed by a kernel.
template <typename T>
T *host_device_alias(T *p)
{
    void *dptr = nullptr;
    if (!p || cudaHostGetDevicePointer(&dptr, const_cast<void *>(static_cast<const void *>(p)), 0) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return static_cast<T *>(dptr);
}

// what a host pointer is RIGHT NOW (never cached: a page-locked buffer may have been freed and a pageable one mapped at the
// same address since the last call); two driver queries of well under a microsecond each
template <typename T>
T *pinned_alias(T *p)
{
    if (!p || !host_is_pinned(p)) return nullptr;
    return host_device_alias(p);
}

// MAPF_STEP_HOST_MODE: forms of mapf_env_step_host (fp32 rewards; measured on 8192 x 32 agents in round 1, profiles/):
//   < 4  step kernel, then the observe kernel while the results are copied on a side stream, issued call by call   88 us
//   4    the same sequence captured once per buffer set and replayed with one cudaGraphLaunch (default)           58-62 us
// (dropped in round 2: DMA copies either side of the fused kernel 109 us; the fused kernel storing 1 MB of fp32 rewards
// straight into host memory 87-97 us.)  The throughput form is mapf_env_step_host_codes: one fused kernel, u8 reward codes
// published zero-copy, the call returns when the results -- not the observation stores -- are done.
int &step_host_mode_ref()
{
    static int m = [] {
        const char *s = std::getenv("MAPF_STEP_HOST_MODE");
        return s ? std::atoi(s) : 4;
    }();
    return m;
}
int step_host_mode() { return step_host_mode_ref(); }
template <typename T>
int dev_alloc(T **p, size_t count, int64_t *total)
{
    size_t bytes = count * sizeof(T);
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), bytes);
    if (e != cudaSuccess) {
        mapf_cuda_fail(e, "cudaMalloc");
        return MAPF_ENOMEM;
    }
    *total += (int64_t)bytes;
    return MAPF_OK;
}
}  // namespace

extern "C" {

int mapf_abi_version(void) { return MAPF_ABI_VERSION; }

const char *mapf_last_error(void) { return g_last_error.c_str(); }

int mapf_env_create(const mapf_env_config *cfg, mapf_env **out)
{
    if (!cfg || !out) {
        mapf_set_error("mapf_env_create: NULL argument");
        return MAPF_EINVAL;
    }
    *out = nullptr;
    if (cfg->num_envs < 1 || cfg->num_agents < 1 || cfg->num_agents > MAPF_MAX_AGENTS || cfg->map_length < 2 ||
        cfg->map_length > MAPF_MAX_MAP_SIDE) {
        mapf_set_error("mapf_env_create: num_envs >= 1, 1 <= num_agents <= 128, 2 <= map_length <= 120 required");
        return MAPF_EINVAL;
    }
    if (cfg->obs_radius != MAPF_OBS_RADIUS) {
        mapf_set_error("mapf_env_create: only obs_radius = 4 is supported (config.py:14)");
        return MAPF_EINVAL;
    }
    if ((int64_t)cfg->num_agents > (int64_t)cfg->map_length * cfg->map_length) {
        mapf_set_error("mapf_env_create: more agents than cells");
        return MAPF_EINVAL;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        mapf_set_error("mapf_env_create: no CUDA device (this library has no CPU fallback)");
        return MAPF_ECUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) {
        mapf_set_error("mapf_env_create: bad device ordinal");
        return MAPF_EINVAL;
    }
    DeviceGuard guard(cfg->device);
    if (!guard.ok) {
        mapf_set_error("mapf_env_create: cudaSetDevice failed");
        return MAPF_ECUDA;
    }
    mapf_env *env = new (std::nothrow) mapf_env();
    if (!env) return MAPF_ENOMEM;
    std::memset(env, 0, sizeof(*env));
    EnvDims &d = env->d;
    d.B = cfg->num_envs;
    d.N = cfg->num_agents;
    d.L = cfg->map_length;
    d.R = d.L + 8;
    d.RW = (d.L + 8 + 31) / 32;
    d.RWS = d.RW + 1;
    d.NB = (d.L + 7) / 8;
    d.K = (d.N + 31) / 32;
    d.obst_stride = (d.R * d.RWS + 3) & ~3;
    d.navi_agent_stride = d.NB * d.NB * 32;
    {
        // MAPF_BFS_APW4=0: two agents per warp at every size (A/B runs)
        static const int apw4 = [] { const char *v = std::getenv("MAPF_BFS_APW4"); return v ? std::atoi(v) : 1; }();
        d.bfs_apw = (apw4 && d.RW == 2 && d.L <= 40) ? 4 : (d.RW <= 3 ? 2 : 1);
    }
    env->device = cfg->device;
    env->num_sms = 148;
    cudaDeviceGetAttribute(&env->num_sms, cudaDevAttrMultiProcessorCount, cfg->device);
    for (int i = 0; i < 5; ++i) env->reward[i] = cfg->reward_fn[i];

    int rc = MAPF_OK;
    int64_t total = 0;
    const size_t BN = (size_t)d.B * d.N;
    if (rc == MAPF_OK) rc = dev_alloc(&env->obst, (size_t)d.B * d.obst_stride, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->pos, BN * 2, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->goal, BN * 2, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->navi, BN * d.navi_agent_stride, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->steps, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->err, 1, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->navi_sel, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->pg_epi, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->pg_n, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->pg_cnt, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_work, 4, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_progress, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_episode, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_prio, (size_t)d.B + 1, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_prio_flag, (size_t)d.B, &total);
    env->ro_tq_cap = d.B + 32;  // >= one re-generation in flight per slot
    if (rc == MAPF_OK) rc = dev_alloc(&env->ro_tq, (size_t)env->ro_tq_cap * 4 + 4, &total);
    if (rc == MAPF_OK) {
        cudaError_t e2 = cudaMemset(env->obst, 0, (size_t)d.B * d.obst_stride * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->ro_work, 0, 32);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->ro_tq, 0x80, ((size_t)env->ro_tq_cap * 4 + 4) * 4);  // every entry free
        if (e2 == cudaSuccess) e2 = cudaMemset(env->ro_tq, 0, 16);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->navi_sel, 0, (size_t)d.B);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->pg_epi, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->pg_n, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->pg_cnt, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->ro_progress, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->ro_episode, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->pos, 0, BN * 2);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->goal, 0, BN * 2);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->navi, 0, BN * d.navi_agent_stride * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->steps, 0, (size_t)d.B * 4);
        if (e2 == cudaSuccess) e2 = cudaMemset(env->err, 0, 4);
        if (e2 == cudaSuccess) e2 = cudaDeviceSynchronize();
        if (e2 != cudaSuccess) rc = mapf_cuda_fail(e2, "cudaMemset(arena)");
    }
    env->arena_bytes = total;
    if (rc != MAPF_OK) {
        mapf_env_destroy(env);
        return rc;
    }
    *out = env;
    return MAPF_OK;
}

int mapf_env_destroy(mapf_env *env)
{
    if (!env) return MAPF_OK;
    DeviceGuard guard(env->device);
    cudaFree(env->obst);
    cudaFree(env->pos);
    cudaFree(env->goal);
    cudaFree(env->navi);
    cudaFree(env->navi_alt);
    cudaFree(env->navi_sel);
    cudaFree(env->pg_obst);
    cudaFree(env->pg_pos);
    cudaFree(env->pg_goal);
    cudaFree(env->pg_steps);
    cudaFree(env->pg_epi);
    cudaFree(env->pg_n);
    cudaFree(env->pg_cnt);
    if (env->pg_stream) cudaStreamDestroy(env->pg_stream);
    if (env->pg_fork) cudaEventDestroy(env->pg_fork);
    if (env->pg_join) cudaEventDestroy(env->pg_join);
    cudaFree(env->steps);
    cudaFree(env->err);
    cudaFree(env->sz_n);
    cudaFree(env->sz_l);
    cudaFree(env->sz_full);
    cudaFree(env->pp_scratch);
    cudaFree(env->ro_work);
    cudaFree(env->ro_progress);
    cudaFree(env->ro_episode);
    cudaFree(env->hp_pos[0]);
    cudaFree(env->hp_pos[1]);
    cudaFree(env->hp_results);
    if (env->hp_stream) cudaStreamDestroy(env->hp_stream);
    for (int i = 0; i < 2; ++i) {
        if (env->hp_step[i]) cudaEventDestroy(env->hp_step[i]);
        if (env->hp_obs[i]) cudaEventDestroy(env->hp_obs[i]);
    }
    if (env->hp_in) cudaEventDestroy(env->hp_in);
    if (env->hp_stepped) cudaEventDestroy(env->hp_stepped);
    cudaFree(env->ro_prio);
    cudaFree(env->ro_prio_flag);
    cudaFree(env->ro_tq);
    cudaFree(env->d_actions);
    cudaFree(env->d_obs);
    cudaFree(env->d_rewards);
    cudaFree(env->d_done);
    cudaFree(env->d_steps_out);
    if (env->h_pinned) cudaFreeHost(env->h_pinned);
    for (auto &c : env->hg)
        if (c.exec) cudaGraphExecDestroy(c.exec);
    if (env->cap_stream) cudaStreamDestroy(env->cap_stream);
    for (int j = 0; j < MAPF_MAX_CHAINS; ++j) {
        if (env->chain_stream[j]) cudaStreamDestroy(env->chain_stream[j]);
        if (env->chain_done[j]) cudaEventDestroy(env->chain_done[j]);
    }
    if (env->chain_fork) cudaEventDestroy(env->chain_fork);
    for (auto &g : env->rg)
        for (auto &x : g.exec)
            if (x) cudaGraphExecDestroy(x);
    if (env->side_stream) cudaStreamDestroy(env->side_stream);
    if (env->ev_stepped) cudaEventDestroy(env->ev_stepped);
    if (env->ev_copied) cudaEventDestroy(env->ev_copied);
    delete env;
    return MAPF_OK;
}

int64_t mapf_env_arena_bytes(const mapf_env *env) { return env ? env->arena_bytes : 0; }

#define REQUIRE_ENV(env)                          \
    if (!(env)) {                                 \
        mapf_set_error("NULL environment handle"); \
        return MAPF_EINVAL;                       \
    }                                             \
    DeviceGuard guard((env)->device);             \
    if (!guard.ok) {                              \
        mapf_set_error("cudaSetDevice failed");   \
        return MAPF_ECUDA;                        \
    }

// Other entry points call this first: what the host-step pipeline still has in flight (step kernel on its internal stream,
// observe kernel on the stream of the last call) is ordered before whatever they queue on `st`.
static int hp_drain(mapf_env *env, cudaStream_t st)
{
    if (!env->hp_active) return MAPF_OK;
    for (int i = 0; i < 2; ++i) {
        MAPF_CUDA(cudaStreamWaitEvent(st, env->hp_step[i], 0));
        MAPF_CUDA(cudaStreamWaitEvent(st, env->hp_obs[i], 0));
    }
    env->hp_active = 0;
    return MAPF_OK;
}
#define MAPF_DRAIN(env, st)                         \
    do {                                            \
        const int _rc = hp_drain((env), (st));      \
        if (_rc != MAPF_OK) return _rc;             \
    } while (0)

// entry points a sized handle (mapf_env_enable_sizes) does not serve
#define MAPF_REFUSE_SIZED(env, what)                                                              \
    if ((env)->sz_n) {                                                                            \
        mapf_set_error(what ": not available on a sized handle (per-environment agent count and map side)"); \
        return MAPF_EINVAL;                                                                       \
    }

// (n, l) pairs of a sized handle's levels / sizes, read to the host: 1 <= n <= N, 2 <= l <= L, n <= l * l
static int check_sizes(const mapf_env *env, const uint8_t *d_n, const uint8_t *d_l, size_t stride, int count, cudaStream_t st,
                       const char *what)
{
    const size_t bytes = (size_t)(count - 1) * stride + 1;  // element i at i * stride
    std::string h(2 * bytes, '\0');
    uint8_t *hn = reinterpret_cast<uint8_t *>(&h[0]), *hl = hn + bytes;
    MAPF_CUDA(cudaMemcpyAsync(hn, d_n, bytes, cudaMemcpyDeviceToHost, st));
    MAPF_CUDA(cudaMemcpyAsync(hl, d_l, bytes, cudaMemcpyDeviceToHost, st));
    MAPF_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < count; ++i) {
        const int n = hn[(size_t)i * stride], l = hl[(size_t)i * stride];
        if (n < 1 || n > env->d.N || l < 2 || l > env->d.L || n > l * l) {
            mapf_set_error(std::string(what) + ": agent count " + std::to_string(n) + " / map side " + std::to_string(l) +
                           " outside 1 <= n <= " + std::to_string(env->d.N) + ", 2 <= l <= " + std::to_string(env->d.L) + ", n <= l * l");
            return MAPF_EINVAL;
        }
    }
    return MAPF_OK;
}

int mapf_env_load(mapf_env *env, const int32_t *d_env_ids, int32_t n, const uint8_t *d_maps, const uint8_t *d_agents,
                  const uint8_t *d_goals, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (n < 0 || n > env->d.B || !d_maps || !d_agents || !d_goals) {
        mapf_set_error("mapf_env_load: bad arguments");
        return MAPF_EINVAL;
    }
    if (n == 0) return MAPF_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // a sized handle records (N, L) for the loaded slots
    int rc = env->sz_n ? mapf_launch_pack_load_sized(env, d_env_ids, n, d_maps, d_agents, d_goals, nullptr, nullptr, st)
                       : mapf_launch_pack_load(env, d_env_ids, n, d_maps, d_agents, d_goals, st);
    if (rc != MAPF_OK) return rc;
    rc = mapf_launch_validate_state(env, d_env_ids, n, st);  // coordinates inside the map, one agent per cell
    if (rc != MAPF_OK) return rc;
    return mapf_launch_bfs(env, d_env_ids, n, nullptr, st);
}

int mapf_env_enable_sizes(mapf_env *env)
{
    REQUIRE_ENV(env);
    if (env->sz_n) return MAPF_OK;
    if (env->ar_max_steps > 0 || env->hp_stream || env->d_actions) {
        mapf_set_error("mapf_env_enable_sizes: the handle already uses episode handling or the host-buffer steps");
        return MAPF_EINVAL;
    }
    const EnvDims &d = env->d;
    int64_t total = env->arena_bytes;
    int rc = dev_alloc(&env->sz_n, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->sz_l, (size_t)d.B, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&env->sz_full, 2, &total);
    if (rc == MAPF_OK) {
        const uint8_t full[2] = {(uint8_t)d.N, (uint8_t)d.L};
        cudaError_t e = cudaMemset(env->sz_n, d.N, (size_t)d.B);
        if (e == cudaSuccess) e = cudaMemset(env->sz_l, d.L, (size_t)d.B);
        if (e == cudaSuccess) e = cudaMemcpy(env->sz_full, full, 2, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) rc = mapf_cuda_fail(e, "mapf_env_enable_sizes");
    }
    if (rc != MAPF_OK) {
        cudaFree(env->sz_n), cudaFree(env->sz_l), cudaFree(env->sz_full);
        env->sz_n = env->sz_l = env->sz_full = nullptr;
        return rc;
    }
    env->arena_bytes = total;
    return MAPF_OK;
}

int mapf_env_load_sized(mapf_env *env, const int32_t *d_env_ids, int32_t n, const uint8_t *d_maps, const uint8_t *d_agents,
                        const uint8_t *d_goals, const uint8_t *d_num_agents, const uint8_t *d_map_length, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!env->sz_n) {
        mapf_set_error("mapf_env_load_sized: the handle is not sized (mapf_env_enable_sizes)");
        return MAPF_EINVAL;
    }
    if (n < 0 || n > env->d.B || !d_maps || !d_agents || !d_goals || !d_num_agents || !d_map_length) {
        mapf_set_error("mapf_env_load_sized: bad arguments");
        return MAPF_EINVAL;
    }
    if (n == 0) return MAPF_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = check_sizes(env, d_num_agents, d_map_length, 1, n, st, "mapf_env_load_sized");
    if (rc != MAPF_OK) return rc;
    rc = mapf_launch_pack_load_sized(env, d_env_ids, n, d_maps, d_agents, d_goals, d_num_agents, d_map_length, st);
    if (rc != MAPF_OK) return rc;
    rc = mapf_launch_validate_state(env, d_env_ids, n, st);  // coordinates inside the slot's map, one agent per cell
    if (rc != MAPF_OK) return rc;
    return mapf_launch_bfs(env, d_env_ids, n, nullptr, st);
}

int mapf_env_reset_levels(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density,
                          const uint8_t *d_levels, int32_t num_levels, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!env->sz_n) {
        mapf_set_error("mapf_env_reset_levels: the handle is not sized (mapf_env_enable_sizes)");
        return MAPF_EINVAL;
    }
    if (density >= 1.0f || !d_levels || num_levels < 1) {
        mapf_set_error("mapf_env_reset_levels: density < 1 and at least one level required");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rc = check_sizes(env, d_levels, d_levels + 1, 2, num_levels, st, "mapf_env_reset_levels");
    if (rc != MAPF_OK) return rc;
    return mapf_launch_reset_levels(env, d_mask, seed, env_offset, density, d_levels, num_levels, st);
}

int mapf_env_get_sizes(mapf_env *env, uint8_t *d_num_agents_out, uint8_t *d_map_length_out, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!env->sz_n) {
        mapf_set_error("mapf_env_get_sizes: the handle is not sized (mapf_env_enable_sizes)");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (d_num_agents_out) MAPF_CUDA(cudaMemcpyAsync(d_num_agents_out, env->sz_n, (size_t)env->d.B, cudaMemcpyDeviceToDevice, st));
    if (d_map_length_out) MAPF_CUDA(cudaMemcpyAsync(d_map_length_out, env->sz_l, (size_t)env->d.B, cudaMemcpyDeviceToDevice, st));
    return MAPF_OK;
}

int mapf_env_bfs_navi(mapf_env *env, const int32_t *d_env_ids, int32_t n, int32_t *d_dist_out, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_env_ids) n = env->d.B;
    if (n < 0 || n > env->d.B) {
        mapf_set_error("mapf_env_bfs_navi: bad n");
        return MAPF_EINVAL;
    }
    if (n == 0) return MAPF_OK;
    return mapf_launch_bfs(env, d_env_ids, n, d_dist_out, static_cast<cudaStream_t>(stream));
}

int mapf_env_plan_prioritized(mapf_env *env, int32_t horizon, uint8_t *d_actions, int32_t *d_arrival, void *stream)
{
    REQUIRE_ENV(env);
    if (horizon < 1 || horizon > MAPF_PLAN_MAX_HORIZON || !d_actions || !d_arrival) {
        mapf_set_error("mapf_env_plan_prioritized: 1 <= horizon <= 1024 and non-NULL d_actions, d_arrival required");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MAPF_DRAIN(env, st);
    return mapf_launch_plan(env, horizon, d_actions, d_arrival, st);
}

int mapf_env_plan_prioritized_orders(mapf_env *env, int32_t horizon, int32_t orders, uint64_t seed, uint64_t env_offset,
                                     uint8_t *d_actions, int32_t *d_arrival, int32_t *d_order, uint8_t *d_rank, void *stream)
{
    REQUIRE_ENV(env);
    if (horizon < 1 || horizon > MAPF_PLAN_MAX_HORIZON || orders < 1 || orders > MAPF_PLAN_MAX_ORDERS || !d_actions || !d_arrival ||
        !d_order || !d_rank) {
        mapf_set_error("mapf_env_plan_prioritized_orders: 1 <= horizon <= 1024, 1 <= orders <= 256 and non-NULL d_actions, "
                       "d_arrival, d_order, d_rank required");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MAPF_DRAIN(env, st);
    return mapf_launch_plan_orders(env, horizon, orders, seed, env_offset, d_actions, d_arrival, d_order, d_rank, st);
}

int mapf_env_plan_lns(mapf_env *env, int32_t horizon, int32_t iterations, int32_t neighborhood, uint64_t seed, uint64_t env_offset,
                      uint32_t first_iteration, uint8_t *d_actions, int32_t *d_arrival, int32_t *d_accepted, void *stream)
{
    REQUIRE_ENV(env);
    if (horizon < 1 || horizon > MAPF_PLAN_MAX_HORIZON || iterations < 0 || neighborhood < 1 || neighborhood > env->d.N ||
        (uint64_t)first_iteration + (uint64_t)iterations > MAPF_PLAN_LNS_MAX_ITERATION || !d_actions || !d_arrival || !d_accepted) {
        mapf_set_error("mapf_env_plan_lns: 1 <= horizon <= 1024, iterations >= 0, 1 <= neighborhood <= N, first_iteration + "
                       "iterations <= 2^24 and non-NULL d_actions, d_arrival, d_accepted required");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MAPF_DRAIN(env, st);
    return mapf_launch_plan_lns(env, horizon, iterations, neighborhood, seed, env_offset, first_iteration, d_actions, d_arrival, d_accepted,
                                st);
}

int mapf_env_plan_repair(mapf_env *env, int32_t horizon, int32_t iterations, int32_t neighborhood, uint64_t seed, uint64_t env_offset,
                         uint8_t *d_actions, int32_t *d_arrival, int32_t *d_collisions, void *stream)
{
    REQUIRE_ENV(env);
    if (horizon < 1 || horizon > MAPF_PLAN_MAX_HORIZON || iterations < 0 || iterations > MAPF_PLAN_REPAIR_MAX_ITERATIONS || neighborhood < 1 ||
        neighborhood > env->d.N || !d_actions || !d_arrival || !d_collisions) {
        mapf_set_error("mapf_env_plan_repair: 1 <= horizon <= 1024, 0 <= iterations <= 2^24, 1 <= neighborhood <= N and non-NULL "
                       "d_actions, d_arrival, d_collisions required");
        return MAPF_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MAPF_DRAIN(env, st);
    return mapf_launch_plan_repair(env, horizon, iterations, neighborhood, seed, env_offset, d_actions, d_arrival, d_collisions, st);
}

int mapf_env_step_observe_ex(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs, const int64_t *d_obs_rows, float *d_rewards,
                             uint8_t *d_codes, uint8_t *d_done, int32_t *d_steps, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_actions || !d_obs || !d_done) {
        mapf_set_error("mapf_env_step_observe: NULL buffer");
        return MAPF_EINVAL;
    }
    StepOut out;
    out.rewards = d_rewards, out.codes = d_codes, out.done = d_done, out.steps = d_steps;
    return mapf_launch_step(env, d_actions, d_obs, d_obs_rows, out, static_cast<cudaStream_t>(stream));
}

int mapf_env_step_observe(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs, float *d_rewards, uint8_t *d_done,
                          int32_t *d_steps, void *stream)
{
    if (!d_rewards) {
        mapf_set_error("mapf_env_step_observe: NULL buffer");
        return MAPF_EINVAL;
    }
    return mapf_env_step_observe_ex(env, d_actions, d_obs, nullptr, d_rewards, nullptr, d_done, d_steps, stream);
}

int mapf_env_step_observe_rows(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs_base, const int64_t *d_obs_rows,
                               float *d_rewards, uint8_t *d_done, int32_t *d_steps, void *stream)
{
    if (!d_obs_rows || !d_rewards) {
        mapf_set_error("mapf_env_step_observe_rows: NULL buffer");
        return MAPF_EINVAL;
    }
    return mapf_env_step_observe_ex(env, d_actions, d_obs_base, d_obs_rows, d_rewards, nullptr, d_done, d_steps, stream);
}

int mapf_env_observe_rows(mapf_env *env, uint8_t *d_obs_base, const int64_t *d_obs_rows, uint8_t *d_pos, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_obs_base || !d_obs_rows) {
        mapf_set_error("mapf_env_observe_rows: NULL buffer");
        return MAPF_EINVAL;
    }
    return mapf_launch_observe(env, d_obs_base, d_obs_rows, d_pos, nullptr, static_cast<cudaStream_t>(stream));
}

int mapf_env_observe(mapf_env *env, uint8_t *d_obs, uint8_t *d_pos, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_obs) {
        mapf_set_error("mapf_env_observe: NULL buffer");
        return MAPF_EINVAL;
    }
    return mapf_launch_observe(env, d_obs, nullptr, d_pos, nullptr, static_cast<cudaStream_t>(stream));
}

int mapf_env_step_observe_packed(mapf_env *env, const uint8_t *d_actions, uint8_t *d_bits_base, const int64_t *d_bits_rows,
                                 float *d_rewards, uint8_t *d_codes, uint8_t *d_done, int32_t *d_steps, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_actions || !d_bits_base || !d_done || !aligned16(d_bits_base)) {
        mapf_set_error("mapf_env_step_observe_packed: NULL buffer or d_bits_base not 16-byte aligned");
        return MAPF_EINVAL;
    }
    StepOut out;
    out.rewards = d_rewards, out.codes = d_codes, out.done = d_done, out.steps = d_steps;
    return mapf_launch_step_packed(env, d_actions, d_bits_base, d_bits_rows, out, static_cast<cudaStream_t>(stream));
}

int mapf_env_observe_packed(mapf_env *env, uint8_t *d_bits_base, const int64_t *d_bits_rows, uint8_t *d_pos, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_bits_base || !aligned16(d_bits_base)) {
        mapf_set_error("mapf_env_observe_packed: NULL buffer or d_bits_base not 16-byte aligned");
        return MAPF_EINVAL;
    }
    return mapf_launch_observe_packed(env, d_bits_base, d_bits_rows, d_pos, static_cast<cudaStream_t>(stream));
}

namespace {
// How the chained form of mapf_env_rollout runs T steps: S chains of `per` environments each; P > 0 when whole slot periods
// of P steps are replayed from per-chain captured graphs.
struct RolloutPlan {
    int S, per, P;
    bool graphs;
};
// MAPF_ROLLOUT_PERSISTENT=0: never use the persistent kernel (chains of launches instead); the kernel's own knobs live in
// mapf_rollout_kernels.cu (mapf_debug_rollout_tuning)
int &rollout_persistent_ref()
{
    static int v = [] {
        const char *s = std::getenv("MAPF_ROLLOUT_PERSISTENT");
        return s ? std::atoi(s) : 1;
    }();
    return v;
}
// the persistent kernel serves the default request (chains = 0) for up to 64 agents; episode handling needs it
bool rollout_uses_persistent(const mapf_env *env, int chains)
{
    if (!mapf_rollout_supported(env)) return false;
    if (env->ar_max_steps > 0) return true;
    return rollout_persistent_ref() != 0 && chains == 0;
}

RolloutPlan rollout_plan(const EnvDims &d, int T, int action_slots, int obs_slots, int out_slots, int chains, bool capturing)
{
    auto gcd = [](int a, int b) { while (b) { int r = a % b; a = b; b = r; } return a; };
    auto lcm_cap = [&](int a, int b) { const long long l = (long long)a / gcd(a, b) * b; return l > 64 ? 65 : (int)l; };
    RolloutPlan pl;
    pl.P = lcm_cap(lcm_cap(action_slots, obs_slots), out_slots);
    pl.graphs = pl.P <= 64 && T >= 4 * pl.P && d.B >= 2048 && chains != 1 && !capturing;
    // sub-batches are multiples of 4 environments (one CTA of the step kernel serves 4)
    pl.S = chains ? chains : (d.B >= 2048 ? (pl.graphs ? 8 : 4) : 1);
    pl.per = (((d.B + pl.S - 1) / pl.S) + 3) & ~3;
    pl.S = (d.B + pl.per - 1) / pl.per;
    if (pl.S == 1) pl.graphs = false;
    return pl;
}
}  // namespace

int mapf_env_rollout_plan(mapf_env *env, int32_t T, int32_t action_slots, int32_t obs_slots, int32_t out_slots, int32_t chains,
                          int32_t *chains_out, int32_t *envs_per_chain_out, int32_t *graph_period_out)
{
    REQUIRE_ENV(env);
    if (T < 0 || action_slots < 1 || obs_slots < 1 || out_slots < 1 || chains < 0 || chains > MAPF_MAX_CHAINS) {
        mapf_set_error("mapf_env_rollout_plan: T >= 0, slot counts >= 1 and 0 <= chains <= 16 required");
        return MAPF_EINVAL;
    }
    if (rollout_uses_persistent(env, chains)) {  // one launch for the whole rollout
        if (chains_out) *chains_out = 0;
        if (envs_per_chain_out) *envs_per_chain_out = env->d.B;
        if (graph_period_out) *graph_period_out = 0;
        return MAPF_OK;
    }
    const RolloutPlan pl = rollout_plan(env->d, T, action_slots, obs_slots, out_slots, chains, false);
    if (chains_out) *chains_out = pl.S;
    if (envs_per_chain_out) *envs_per_chain_out = pl.per;
    if (graph_period_out) *graph_period_out = pl.graphs ? pl.P : 0;
    return MAPF_OK;
}

int mapf_env_rollout_ex(mapf_env *env, const mapf_rollout_io *io, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_REFUSE_SIZED(env, "mapf_env_rollout");
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!io || !io->d_actions || !io->d_obs || !io->d_done) {
        mapf_set_error("mapf_env_rollout: NULL buffer");
        return MAPF_EINVAL;
    }
    const int T = io->T, action_slots = io->action_slots, obs_slots = io->obs_slots, out_slots = io->out_slots, chains = io->chains;
    if (T < 0 || action_slots < 1 || obs_slots < 1 || out_slots < 1 || chains < 0 || chains > MAPF_MAX_CHAINS) {
        mapf_set_error("mapf_env_rollout: T >= 0, slot counts >= 1 and 0 <= chains <= 16 required");
        return MAPF_EINVAL;
    }
    if (T == 0) return MAPF_OK;
    const EnvDims &d = env->d;
    const size_t BN = (size_t)d.B * d.N;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const uint8_t *d_actions = io->d_actions;
    uint8_t *d_obs = io->d_obs;
    StepOut ring;
    ring.rewards = io->d_rewards, ring.codes = io->d_codes, ring.done = io->d_done, ring.steps = io->d_steps;
    if (rollout_uses_persistent(env, chains)) {
        const int rc = mapf_launch_rollout(env, 0, d.B, T, d_actions, action_slots, d_obs, obs_slots, ring, out_slots, st);
        if (rc != MAPF_EINVAL) return rc;
    }
    if (env->ar_max_steps > 0) {
        mapf_set_error("mapf_env_rollout: episode handling (mapf_env_set_autoreset) is served by the persistent kernel only "
                       "(up to 64 agents, per-warp state within shared memory)");
        return MAPF_EINVAL;
    }
    // Chained form.  The launches of a long rollout repeat with period P = lcm(slot counts): those are captured once per chain
    // into a graph of P kernel nodes and replayed (one cudaGraphLaunch per chain and period instead of P launches of ~4 us of
    // host time each, which bound 8 chains at 32 us per step); short rollouts and the tail are launched directly.
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    MAPF_CUDA(cudaStreamIsCapturing(st, &cap));
    const RolloutPlan pl = rollout_plan(d, T, action_slots, obs_slots, out_slots, chains, cap != cudaStreamCaptureStatusNone);
    const int S = pl.S, per = pl.per, P = pl.P;
    const bool graphs = pl.graphs;
    auto step_t = [&](int t, int e0, int e1, cudaStream_t q) -> int {
        const size_t sa = (size_t)(t % action_slots), so = (size_t)(t % obs_slots), sr = (size_t)(t % out_slots);
        StepOut o;
        o.rewards = ring.rewards ? ring.rewards + sr * BN : nullptr;
        o.codes = ring.codes ? ring.codes + sr * BN : nullptr;
        o.done = ring.done + sr * d.B;
        o.steps = ring.steps ? ring.steps + sr * d.B : nullptr;
        return mapf_launch_step_range(env, e0, e1, d_actions + sa * BN, d_obs + so * BN * MAPF_OBS_BYTES_PER_AGENT, o, q);
    };
    if (S == 1) {
        for (int t = 0; t < T; ++t) {
            const int rc = step_t(t, 0, d.B, st);
            if (rc != MAPF_OK) return rc;
        }
        return MAPF_OK;
    }
    if (!env->chain_fork) MAPF_CUDA(cudaEventCreateWithFlags(&env->chain_fork, cudaEventDisableTiming));
    for (int j = 0; j < S; ++j) {
        if (!env->chain_stream[j]) {
            MAPF_CUDA(cudaStreamCreateWithFlags(&env->chain_stream[j], cudaStreamNonBlocking));
            MAPF_CUDA(cudaEventCreateWithFlags(&env->chain_done[j], cudaEventDisableTiming));
        }
    }
    // fork: every chain starts after what the caller queued on `stream` (actions ready, earlier readers of the buffers done)
    MAPF_CUDA(cudaEventRecord(env->chain_fork, st));
    for (int j = 0; j < S; ++j) MAPF_CUDA(cudaStreamWaitEvent(env->chain_stream[j], env->chain_fork, 0));
    int rc = MAPF_OK;
    int t_begin = 0;
    if (graphs) {
        mapf_env::RolloutGraph *g = nullptr;
        const int gen = mapf_step_tuning_generation();
        for (auto &c : env->rg)
            if (c.exec[0] && c.act == d_actions && c.obs == d_obs && c.rew == ring.rewards && c.codes == ring.codes && c.done == ring.done &&
                c.steps == ring.steps && c.action_slots == action_slots && c.obs_slots == obs_slots && c.out_slots == out_slots && c.S == S &&
                c.P == P && c.tuning_gen == gen)
                g = &c;
        if (!g) {
            g = &env->rg[env->rg_next];
            env->rg_next = (env->rg_next + 1) % 2;
            for (auto &x : g->exec)
                if (x) {
                    cudaGraphExecDestroy(x);
                    x = nullptr;
                }
            if (!env->cap_stream) MAPF_CUDA(cudaStreamCreateWithFlags(&env->cap_stream, cudaStreamNonBlocking));
            for (int j = 0; j < S && rc == MAPF_OK; ++j) {
                const int e0 = j * per, e1 = e0 + per < d.B ? e0 + per : d.B;
                cudaGraph_t graph = nullptr;
                MAPF_CUDA(cudaStreamBeginCapture(env->cap_stream, cudaStreamCaptureModeThreadLocal));
                for (int t = 0; t < P && rc == MAPF_OK; ++t) rc = step_t(t, e0, e1, env->cap_stream);
                cudaError_t ce = cudaStreamEndCapture(env->cap_stream, &graph);
                if (rc == MAPF_OK && ce != cudaSuccess) rc = mapf_cuda_fail(ce, "cudaStreamEndCapture");
                if (rc == MAPF_OK) {
                    ce = cudaGraphInstantiate(&g->exec[j], graph, 0);
                    if (ce != cudaSuccess) rc = mapf_cuda_fail(ce, "cudaGraphInstantiate");
                }
                if (graph) cudaGraphDestroy(graph);
            }
            if (rc != MAPF_OK) {
                for (auto &x : g->exec)
                    if (x) {
                        cudaGraphExecDestroy(x);
                        x = nullptr;
                    }
            } else {
                g->act = d_actions, g->obs = d_obs, g->rew = ring.rewards, g->codes = ring.codes, g->done = ring.done, g->steps = ring.steps;
                g->action_slots = action_slots, g->obs_slots = obs_slots, g->out_slots = out_slots, g->S = S, g->P = P, g->tuning_gen = gen;
            }
        }
        // period-major issue order: every chain has a period of work queued before any gets its second one
        for (; rc == MAPF_OK && t_begin + P <= T; t_begin += P)
            for (int j = 0; j < S && rc == MAPF_OK; ++j) {
                const cudaError_t ce = cudaGraphLaunch(g->exec[j], env->chain_stream[j]);
                if (ce != cudaSuccess) rc = mapf_cuda_fail(ce, "cudaGraphLaunch");
            }
    }
    // step-major issue order, so that every chain has work queued from the start; chain j's launch t+1 follows its
    // launch t by stream order and nothing else
    for (int t = t_begin; t < T && rc == MAPF_OK; ++t)
        for (int j = 0; j < S && rc == MAPF_OK; ++j) {
            const int e0 = j * per, e1 = e0 + per < d.B ? e0 + per : d.B;
            rc = step_t(t, e0, e1, env->chain_stream[j]);
        }
    // join (also after a failed launch: the caller's stream must not run ahead of what was queued)
    for (int j = 0; j < S; ++j) {
        cudaError_t e = cudaEventRecord(env->chain_done[j], env->chain_stream[j]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, env->chain_done[j], 0);
        if (e != cudaSuccess && rc == MAPF_OK) rc = mapf_cuda_fail(e, "mapf_env_rollout join");
    }
    return rc;
}

int mapf_env_rollout(mapf_env *env, int32_t T, const uint8_t *d_actions, int32_t action_slots, uint8_t *d_obs, int32_t obs_slots,
                     float *d_rewards, uint8_t *d_done, int32_t *d_steps, int32_t out_slots, int32_t chains, void *stream)
{
    if (!d_rewards) {
        mapf_set_error("mapf_env_rollout: NULL buffer");
        return MAPF_EINVAL;
    }
    mapf_rollout_io io{};
    io.T = T, io.d_actions = d_actions, io.action_slots = action_slots, io.d_obs = d_obs, io.obs_slots = obs_slots;
    io.d_rewards = d_rewards, io.d_codes = nullptr, io.d_done = d_done, io.d_steps = d_steps, io.out_slots = out_slots, io.chains = chains;
    return mapf_env_rollout_ex(env, &io, stream);
}

int mapf_env_set_autoreset(mapf_env *env, int32_t max_steps, uint64_t seed, uint64_t env_offset, uint64_t stride, float density,
                           void *stream)
{
    REQUIRE_ENV(env);
    MAPF_REFUSE_SIZED(env, "mapf_env_set_autoreset");
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (max_steps < 0 || density >= 1.0f) {
        mapf_set_error("mapf_env_set_autoreset: max_steps >= 0 and density < 1 required");
        return MAPF_EINVAL;
    }
    if (max_steps > 0 && !mapf_rollout_supported(env)) {
        mapf_set_error("mapf_env_set_autoreset: episode handling is served by the persistent kernel only (up to 64 agents)");
        return MAPF_EINVAL;
    }
    env->ar_max_steps = max_steps;
    env->ar_seed = seed, env->ar_offset = env_offset, env->ar_stride = stride ? stride : (uint64_t)env->d.B;
    env->ar_density = density;
    MAPF_CUDA(cudaMemsetAsync(env->ro_episode, 0, (size_t)env->d.B * 4, static_cast<cudaStream_t>(stream)));
    MAPF_CUDA(cudaMemsetAsync(env->pg_epi, 0, (size_t)env->d.B * 4, static_cast<cudaStream_t>(stream)));
    if (max_steps > 0 && !env->navi_alt) {
        // the second heuristic-map buffer and the staging of pre-generated instances (mapf_common.cuh).  Without the memory
        // for them episodes are still handled, by re-generating inside the rollout kernel.
        const EnvDims &d = env->d;
        const size_t BN = (size_t)d.B * d.N;
        int64_t total = 0;
        int rc = dev_alloc(&env->navi_alt, BN * d.navi_agent_stride, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->pg_obst, (size_t)d.B * d.obst_stride, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->pg_pos, BN * 2, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->pg_goal, BN * 2, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->pg_steps, (size_t)d.B, &total);
        if (rc == MAPF_OK) {
            // border rows / columns of a staged bitmap are zero like the live one's (the generator writes map rows only)
            MAPF_CUDA(cudaMemsetAsync(env->pg_obst, 0, (size_t)d.B * d.obst_stride * 4, static_cast<cudaStream_t>(stream)));
            MAPF_CUDA(cudaMemsetAsync(env->navi_alt, 0, BN * d.navi_agent_stride * 4, static_cast<cudaStream_t>(stream)));
            env->arena_bytes += total;
        } else {
            cudaGetLastError();
            cudaFree(env->navi_alt), cudaFree(env->pg_obst), cudaFree(env->pg_pos), cudaFree(env->pg_goal), cudaFree(env->pg_steps);
            env->navi_alt = nullptr, env->pg_obst = nullptr, env->pg_pos = env->pg_goal = nullptr, env->pg_steps = nullptr;
        }
    }
    return MAPF_OK;
}

int mapf_env_episode_counts(mapf_env *env, uint32_t *d_counts_out, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_counts_out) {
        mapf_set_error("mapf_env_episode_counts: NULL buffer");
        return MAPF_EINVAL;
    }
    MAPF_CUDA(cudaMemcpyAsync(d_counts_out, env->ro_episode, (size_t)env->d.B * 4, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    return MAPF_OK;
}

int mapf_env_set_checks(mapf_env *env, int32_t check_unique)
{
    REQUIRE_ENV(env);
    env->check_unique = check_unique != 0;
    env->checks_gen++;  // captured step_host graphs carry the old flag
    return MAPF_OK;
}

int mapf_env_step_host(mapf_env *env, const uint8_t *h_actions, uint8_t *h_obs, float *h_rewards, uint8_t *h_done,
                       int32_t *h_steps, uint8_t *d_obs_opt, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_REFUSE_SIZED(env, "mapf_env_step_host");
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!h_actions || !h_rewards || !h_done) {
        mapf_set_error("mapf_env_step_host: NULL buffer");
        return MAPF_EINVAL;
    }
    const EnvDims &d = env->d;
    const size_t BN = (size_t)d.B * d.N;
    int64_t total = env->arena_bytes;
    int rc = MAPF_OK;
    if (!env->d_actions) {
        if (rc == MAPF_OK) rc = dev_alloc(&env->d_actions, BN, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->d_rewards, BN, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->d_done, (size_t)d.B, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->d_steps_out, (size_t)d.B, &total);
    }
    if (rc == MAPF_OK && !env->h_pinned) {
        cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&env->h_pinned), BN + BN * 4 + (size_t)d.B * 5 + 128);
        if (e != cudaSuccess) rc = mapf_cuda_fail(e, "cudaMallocHost");
    }
    if (rc == MAPF_OK && !d_obs_opt && !env->d_obs) rc = dev_alloc(&env->d_obs, BN * MAPF_OBS_BYTES_PER_AGENT, &total);
    env->arena_bytes = total;
    if (rc != MAPF_OK) return rc;

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t *obs_dev = d_obs_opt ? d_obs_opt : env->d_obs;
    // pinned layout: actions u8[BN] | pad to 16 | rewards f32[BN] | steps i32[B] | done u8[B]
    uint8_t *pin_act = env->h_pinned;
    float *pin_rew = reinterpret_cast<float *>(env->h_pinned + ((BN + 15) & ~(size_t)15));
    int32_t *pin_steps = reinterpret_cast<int32_t *>(pin_rew + BN);
    uint8_t *pin_done = reinterpret_cast<uint8_t *>(pin_steps + d.B);
    // page-locked caller buffers are used in place; pageable ones go through the handle's pinned staging area (one extra
    // host memcpy each way)
    const uint8_t *act_alias = pinned_alias(h_actions);
    const bool out_direct = host_is_pinned(h_rewards) && host_is_pinned(h_done) && (!h_steps || host_is_pinned(h_steps));
    const uint8_t *src_act = h_actions;
    if (!act_alias) {
        std::memcpy(pin_act, h_actions, BN);
        src_act = pin_act;
        act_alias = host_device_alias(pin_act);
    }
    float *dst_rew = out_direct ? h_rewards : pin_rew;
    uint8_t *dst_done = out_direct ? h_done : pin_done;
    int32_t *dst_steps = h_steps ? (out_direct ? h_steps : pin_steps) : nullptr;
    // split: step kernel -> {observe kernel on `st`  ||  result copies on the side stream} -> join
    if (!env->side_stream) {
        MAPF_CUDA(cudaStreamCreateWithFlags(&env->side_stream, cudaStreamNonBlocking));
        MAPF_CUDA(cudaEventCreateWithFlags(&env->ev_stepped, cudaEventDisableTiming));
        MAPF_CUDA(cudaEventCreateWithFlags(&env->ev_copied, cudaEventDisableTiming));
    }
    // issues the whole sequence on `q` (forking to the side stream and joining back)
    auto enqueue = [&](cudaStream_t q) -> int {
        const uint8_t *a = act_alias;  // read in place over PCIe
        if (!a) {
            MAPF_CUDA(cudaMemcpyAsync(env->d_actions, src_act, BN, cudaMemcpyHostToDevice, q));
            a = env->d_actions;
        }
        StepOut o;
        o.rewards = env->d_rewards, o.done = env->d_done, o.steps = env->d_steps_out;
        int r = mapf_launch_step_only(env, a, o, nullptr, q);
        if (r != MAPF_OK) return r;
        MAPF_CUDA(cudaEventRecord(env->ev_stepped, q));
        MAPF_CUDA(cudaStreamWaitEvent(env->side_stream, env->ev_stepped, 0));
        MAPF_CUDA(cudaMemcpyAsync(dst_rew, env->d_rewards, BN * 4, cudaMemcpyDeviceToHost, env->side_stream));
        if (dst_steps)
            MAPF_CUDA(cudaMemcpyAsync(dst_steps, env->d_steps_out, (size_t)d.B * 4, cudaMemcpyDeviceToHost, env->side_stream));
        MAPF_CUDA(cudaMemcpyAsync(dst_done, env->d_done, (size_t)d.B, cudaMemcpyDeviceToHost, env->side_stream));
        MAPF_CUDA(cudaEventRecord(env->ev_copied, env->side_stream));
        r = mapf_launch_observe(env, obs_dev, nullptr, nullptr, nullptr, q);
        if (r != MAPF_OK) return r;
        if (h_obs) MAPF_CUDA(cudaMemcpyAsync(h_obs, obs_dev, BN * MAPF_OBS_BYTES_PER_AGENT, cudaMemcpyDeviceToHost, q));
        MAPF_CUDA(cudaStreamWaitEvent(q, env->ev_copied, 0));
        return MAPF_OK;
    };
    if (step_host_mode() >= 4) {
        // one cudaGraphLaunch instead of nine stream calls: the sequence is captured per buffer set
        const int gen = mapf_step_tuning_generation() * 65536 + env->checks_gen;
        mapf_env::HostGraph *g = nullptr;
        for (auto &c : env->hg)
            if (c.exec && c.act == (const void *)act_alias && c.rew == dst_rew && c.done == dst_done && c.steps == dst_steps && c.hobs == h_obs &&
                c.obs_dev == obs_dev && c.gen == gen)
                g = &c;
        if (!g) {
            if (!env->cap_stream) MAPF_CUDA(cudaStreamCreateWithFlags(&env->cap_stream, cudaStreamNonBlocking));
            g = &env->hg[env->hg_next];
            env->hg_next = (env->hg_next + 1) % 32;
            if (g->exec) {
                cudaGraphExecDestroy(g->exec);
                g->exec = nullptr;
            }
            cudaGraph_t graph = nullptr;
            MAPF_CUDA(cudaStreamBeginCapture(env->cap_stream, cudaStreamCaptureModeThreadLocal));
            rc = enqueue(env->cap_stream);
            cudaError_t ce = cudaStreamEndCapture(env->cap_stream, &graph);
            if (rc != MAPF_OK) {
                if (graph) cudaGraphDestroy(graph);
                return rc;
            }
            if (ce != cudaSuccess) return mapf_cuda_fail(ce, "cudaStreamEndCapture");
            ce = cudaGraphInstantiate(&g->exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ce != cudaSuccess) return mapf_cuda_fail(ce, "cudaGraphInstantiate");
            g->act = act_alias, g->rew = dst_rew, g->done = dst_done, g->steps = dst_steps, g->hobs = h_obs, g->obs_dev = obs_dev, g->gen = gen;
        }
        MAPF_CUDA(cudaGraphLaunch(g->exec, st));
    } else {
        rc = enqueue(st);
        if (rc != MAPF_OK) return rc;
    }
    MAPF_CUDA(cudaStreamSynchronize(st));
    if (!out_direct) {
        std::memcpy(h_rewards, pin_rew, BN * 4);
        std::memcpy(h_done, pin_done, (size_t)d.B);
        if (h_steps) std::memcpy(h_steps, pin_steps, (size_t)d.B * 4);
    }
    return MAPF_OK;
}

int mapf_env_step_host_codes(mapf_env *env, const uint8_t *h_actions, uint8_t *h_codes, uint8_t *h_done, int32_t *h_steps,
                             uint8_t *d_obs, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_REFUSE_SIZED(env, "mapf_env_step_host_codes");
    if (!h_actions || !h_codes || !h_done || !d_obs) {
        mapf_set_error("mapf_env_step_host_codes: NULL buffer");
        return MAPF_EINVAL;
    }
    const EnvDims &d = env->d;
    const size_t BN = (size_t)d.B * d.N;
    const size_t off_steps = (BN + 15) & ~(size_t)15, off_done = off_steps + (size_t)d.B * 4;
    const size_t res_bytes = off_done + d.B;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!env->hp_stream) {
        int64_t total = env->arena_bytes;
        int rc = dev_alloc(&env->hp_pos[0], BN * 2, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->hp_pos[1], BN * 2, &total);
        if (rc == MAPF_OK) rc = dev_alloc(&env->hp_results, res_bytes + 16, &total);
        env->arena_bytes = total;
        if (rc != MAPF_OK) return rc;
        MAPF_CUDA(cudaStreamCreateWithFlags(&env->hp_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            MAPF_CUDA(cudaEventCreateWithFlags(&env->hp_step[i], cudaEventDisableTiming));
            MAPF_CUDA(cudaEventCreateWithFlags(&env->hp_obs[i], cudaEventDisableTiming));
        }
        MAPF_CUDA(cudaEventCreateWithFlags(&env->hp_in, cudaEventDisableTiming));
        MAPF_CUDA(cudaEventCreateWithFlags(&env->hp_stepped, cudaEventDisableTiming));
    }
    if (!env->h_pinned) {
        cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&env->h_pinned), BN + BN * 4 + (size_t)d.B * 5 + 128);
        if (e != cudaSuccess) return mapf_cuda_fail(e, "cudaMallocHost");
    }
    // pinned staging for pageable caller buffers: actions u8[BN] | pad | results (codes | steps | done, as on the device)
    uint8_t *pin_act = env->h_pinned;
    uint8_t *pin_res = env->h_pinned + ((BN + 15) & ~(size_t)15);
    // MAPF_HOSTCODES_MODE: 1 (default) = device staging + DMA copies (ONE contiguous copy when the caller's three buffers are
    // laid out like the staging: codes | pad to 16 | steps | done), 0 = the step kernel stores its results straight into
    // page-locked host memory (measured: 56 us against 42 us latency per call, the scattered 32-byte PCIe writes cost more
    // than the one DMA; profiles/r2_e2e_probe.jsonl)
    static const int copy_mode = [] { const char *v = std::getenv("MAPF_HOSTCODES_MODE"); return v ? std::atoi(v) : 1; }();
    const uint8_t *act_alias = pinned_alias(h_actions);   // the only query on the critical path: the kernel launch follows
    const bool act_direct = act_alias != nullptr;
    if (!act_direct) {
        std::memcpy(pin_act, h_actions, BN);
        act_alias = host_device_alias(pin_act);
    }
    // a new run of the pipeline: the step stream starts after what the caller has queued on `st` (a reset, a load, ...)
    if (!env->hp_active) {
        MAPF_CUDA(cudaEventRecord(env->hp_in, st));
        MAPF_CUDA(cudaStreamWaitEvent(env->hp_stream, env->hp_in, 0));
        env->hp_t = 0;
        env->hp_active = 1;
    }
    const int slot = (int)(env->hp_t & 1);
    // the observe kernel of two calls ago has read the snapshot this step overwrites
    if (env->hp_t >= 2) MAPF_CUDA(cudaStreamWaitEvent(env->hp_stream, env->hp_obs[slot], 0));
    // where the kernel writes its results: the device staging block (default), or -- MAPF_HOSTCODES_MODE=0 -- the caller's
    // page-locked buffers / the pinned staging area in place
    uint8_t *codes_alias = nullptr, *done_alias = nullptr;
    int32_t *steps_alias = nullptr;
    bool out_direct = false;
    if (copy_mode == 0) {
        codes_alias = pinned_alias(h_codes), done_alias = pinned_alias(h_done);
        steps_alias = h_steps ? pinned_alias(h_steps) : nullptr;
        out_direct = codes_alias && done_alias && (!h_steps || steps_alias);
        if (!out_direct) {
            codes_alias = host_device_alias(pin_res), done_alias = host_device_alias(pin_res + off_done);
            steps_alias = reinterpret_cast<int32_t *>(host_device_alias(pin_res + off_steps));
        }
    }
    const bool zero_copy = copy_mode == 0 && codes_alias && done_alias && (steps_alias || (out_direct && !h_steps));
    StepOut o;
    if (zero_copy) {
        o.codes = codes_alias, o.done = done_alias, o.steps = h_steps || !out_direct ? steps_alias : nullptr;
    } else {
        o.codes = env->hp_results;
        o.steps = reinterpret_cast<int32_t *>(env->hp_results + off_steps);
        o.done = env->hp_results + off_done;
    }
    int rc;
    if (act_alias) {
        rc = mapf_launch_step_only(env, act_alias, o, env->hp_pos[slot], env->hp_stream);  // reads the actions in place over PCIe
    } else {
        if (!env->d_actions) {
            int64_t total = env->arena_bytes;
            rc = dev_alloc(&env->d_actions, BN, &total);
            env->arena_bytes = total;
            if (rc != MAPF_OK) return rc;
        }
        MAPF_CUDA(cudaMemcpyAsync(env->d_actions, act_direct ? h_actions : pin_act, BN, cudaMemcpyHostToDevice, env->hp_stream));
        rc = mapf_launch_step_only(env, env->d_actions, o, env->hp_pos[slot], env->hp_stream);
    }
    if (rc != MAPF_OK) return rc;
    // stage 2 on the caller's stream starts as soon as the step kernel is done (the result copies run next to it): the
    // observation of the snapshot, ordered before anything queued on `st` afterwards
    MAPF_CUDA(cudaEventRecord(env->hp_stepped, env->hp_stream));
    MAPF_CUDA(cudaStreamWaitEvent(st, env->hp_stepped, 0));
    rc = mapf_launch_observe(env, d_obs, nullptr, nullptr, env->hp_pos[slot], st);
    if (rc != MAPF_OK) return rc;
    MAPF_CUDA(cudaEventRecord(env->hp_obs[slot], st));
    if (!zero_copy) {
        // (queried while the step kernel is already running: off the critical path)
        out_direct = host_is_pinned(h_codes) && host_is_pinned(h_done) && (!h_steps || host_is_pinned(h_steps));
        const bool contiguous = out_direct && h_steps && reinterpret_cast<uint8_t *>(h_steps) == h_codes + off_steps && h_done == h_codes + off_done;
        if (contiguous) {
            MAPF_CUDA(cudaMemcpyAsync(h_codes, env->hp_results, res_bytes, cudaMemcpyDeviceToHost, env->hp_stream));
        } else if (out_direct) {
            MAPF_CUDA(cudaMemcpyAsync(h_codes, env->hp_results, BN, cudaMemcpyDeviceToHost, env->hp_stream));
            if (h_steps) MAPF_CUDA(cudaMemcpyAsync(h_steps, env->hp_results + off_steps, (size_t)d.B * 4, cudaMemcpyDeviceToHost, env->hp_stream));
            MAPF_CUDA(cudaMemcpyAsync(h_done, env->hp_results + off_done, (size_t)d.B, cudaMemcpyDeviceToHost, env->hp_stream));
        } else {
            MAPF_CUDA(cudaMemcpyAsync(pin_res, env->hp_results, res_bytes, cudaMemcpyDeviceToHost, env->hp_stream));
        }
    }
    MAPF_CUDA(cudaEventRecord(env->hp_step[slot], env->hp_stream));
    env->hp_t++;
    // the results are on the host when stage 1 is done; the observe kernel keeps running
    MAPF_CUDA(cudaEventSynchronize(env->hp_step[slot]));
    if (!out_direct) {
        std::memcpy(h_codes, pin_res, BN);
        std::memcpy(h_done, pin_res + off_done, (size_t)d.B);
        if (h_steps) std::memcpy(h_steps, pin_res + off_steps, (size_t)d.B * 4);
    }
    return MAPF_OK;
}

int mapf_debug_step_tuning(int32_t variant, int32_t flags, int32_t ctas_per_sm)
{
    mapf_set_step_tuning(variant, flags, ctas_per_sm);
    return MAPF_OK;
}

int mapf_debug_rollout_tuning(int32_t persistent, int32_t warps_per_sm, int32_t chunk, int32_t store_mode, int32_t stagger_ns)
{
    if (persistent >= 0) rollout_persistent_ref() = persistent;
    mapf_set_rollout_tuning(warps_per_sm, chunk, store_mode, stagger_ns);
    return MAPF_OK;
}

int mapf_debug_rollout_pregen(int32_t on)
{
    if (on >= 0) mapf_set_rollout_pregen(on);
    return rollout_pregen_ref();
}

int mapf_debug_rollout_tasks(int32_t on)
{
    if (on >= 0) mapf_set_rollout_tasks(on);
    return rollout_tasks_ref();
}

int mapf_debug_step_host_mode(int32_t mode)
{
    if (mode >= 0) step_host_mode_ref() = mode;
    return step_host_mode_ref();
}

int mapf_env_comm_mask(mapf_env *env, int32_t max_comm_agents, uint8_t *d_mask_out, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_mask_out || max_comm_agents < 1 || max_comm_agents > 3) {
        mapf_set_error("mapf_env_comm_mask: NULL buffer or max_comm_agents outside 1..3 (config.py:58)");
        return MAPF_EINVAL;
    }
    return mapf_launch_comm_mask(env, max_comm_agents, d_mask_out, static_cast<cudaStream_t>(stream));
}

int mapf_env_comm_mask_packed(mapf_env *env, int32_t max_comm_agents, uint8_t *d_mask_out, uint8_t *d_bits_base,
                              const int64_t *d_bits_rows, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (!d_bits_base || max_comm_agents < 1 || max_comm_agents > 3) {
        mapf_set_error("mapf_env_comm_mask_packed: NULL buffer or max_comm_agents outside 1..3 (config.py:58)");
        return MAPF_EINVAL;
    }
    return mapf_launch_comm_mask_packed(env, max_comm_agents, d_mask_out, d_bits_base, d_bits_rows, static_cast<cudaStream_t>(stream));
}

int mapf_env_get_state(mapf_env *env, uint8_t *d_map, uint8_t *d_pos, uint8_t *d_goals, int32_t *d_steps, uint8_t *d_navi,
                       void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t BN2 = (size_t)env->d.B * env->d.N * 2;
    if (d_pos) MAPF_CUDA(cudaMemcpyAsync(d_pos, env->pos, BN2, cudaMemcpyDeviceToDevice, st));
    if (d_goals) MAPF_CUDA(cudaMemcpyAsync(d_goals, env->goal, BN2, cudaMemcpyDeviceToDevice, st));
    if (d_steps) MAPF_CUDA(cudaMemcpyAsync(d_steps, env->steps, (size_t)env->d.B * 4, cudaMemcpyDeviceToDevice, st));
    return mapf_launch_unpack(env, d_map, d_navi, st);
}

int mapf_env_set_state(mapf_env *env, const uint8_t *d_pos, const int32_t *d_steps, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (d_pos) {
        MAPF_CUDA(cudaMemcpyAsync(env->pos, d_pos, (size_t)env->d.B * env->d.N * 2, cudaMemcpyDeviceToDevice, st));
        const int rc = mapf_launch_validate_state(env, nullptr, env->d.B, st);  // clamps + latches MAPF_ESTATE
        if (rc != MAPF_OK) return rc;
    }
    if (d_steps) MAPF_CUDA(cudaMemcpyAsync(env->steps, d_steps, (size_t)env->d.B * 4, cudaMemcpyDeviceToDevice, st));
    return MAPF_OK;
}

int mapf_env_status(mapf_env *env, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t bits = 0;
    MAPF_CUDA(cudaMemcpyAsync(&bits, env->err, 4, cudaMemcpyDeviceToHost, st));
    MAPF_CUDA(cudaStreamSynchronize(st));
    if (bits) {
        MAPF_CUDA(cudaMemsetAsync(env->err, 0, 4, st));
        MAPF_CUDA(cudaStreamSynchronize(st));
    }
    if (bits & MAPF_ERRBIT_STATE) {
        mapf_set_error("invalid state: coordinate outside the map or slot id outside the batch");
        return MAPF_ESTATE;
    }
    if (bits & MAPF_ERRBIT_ACTION) {
        mapf_set_error("action index out of range");
        return MAPF_EACTION;
    }
    if (bits & MAPF_ERRBIT_UNIQUE) {
        mapf_set_error("unique");
        return MAPF_EUNIQUE;
    }
    if (bits & MAPF_ERRBIT_RESET) {
        mapf_set_error("no empty position");  // environment.py:31
        return MAPF_ENOSPACE;
    }
    if (bits & MAPF_ERRBIT_INTERNAL) {
        mapf_set_error("rollout scheduler: a chunk hand-over never arrived");
        return MAPF_EINTERNAL;
    }
    return MAPF_OK;
}

int mapf_env_reset(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density, void *stream)
{
    REQUIRE_ENV(env);
    MAPF_DRAIN(env, static_cast<cudaStream_t>(stream));
    if (density >= 1.0f) {
        mapf_set_error("mapf_env_reset: density must be < 1");
        return MAPF_EINVAL;
    }
    if (env->sz_n)  // a sized handle draws at (N, L) and records it: the one-level form of mapf_env_reset_levels
        return mapf_launch_reset_levels(env, d_mask, seed, env_offset, density, env->sz_full, 1, static_cast<cudaStream_t>(stream));
    return mapf_launch_reset(env, d_mask, seed, env_offset, density, static_cast<cudaStream_t>(stream));
}

/* ---------------------------------------------------------------------------------------------- */

int mapf_per_create(int64_t capacity, int32_t device, mapf_per **out)
{
    if (!out || capacity < 1 || (capacity & (capacity - 1)) != 0) {
        mapf_set_error("buffer size only support power of 2 size");  // buffer.py:23
        return MAPF_EINVAL;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        mapf_set_error("mapf_per_create: no CUDA device (this library has no CPU fallback)");
        return MAPF_ECUDA;
    }
    if (device < 0 || device >= ndev) {
        mapf_set_error("mapf_per_create: bad device ordinal");
        return MAPF_EINVAL;
    }
    DeviceGuard guard(device);
    mapf_per *t = new (std::nothrow) mapf_per();
    if (!t) return MAPF_ENOMEM;
    std::memset(t, 0, sizeof(*t));
    t->capacity = capacity;
    t->device = device;
    int layer = 1;
    while ((int64_t(1) << (layer - 1)) < capacity) ++layer;  // buffer.py:20-22
    t->layer = layer;
    int64_t total = 0;
    const int64_t nodes = 2 * capacity - 1;
    t->scratch.cap_n = 1 << 16;
    int rc = dev_alloc(&t->tree, (size_t)nodes, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&t->scratch.stamps, (size_t)capacity, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&t->scratch.prio32, (size_t)t->scratch.cap_n, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&t->scratch.active, (size_t)t->scratch.cap_n, &total);
    if (rc == MAPF_OK) rc = dev_alloc(&t->scratch.err, 1, &total);
    if (rc == MAPF_OK) {
        cudaError_t e = cudaMemset(t->tree, 0, (size_t)nodes * 8);
        if (e == cudaSuccess) e = cudaMemset(t->scratch.err, 0, 4);
        if (e == cudaSuccess) e = cudaMemset(t->scratch.stamps, 0, (size_t)capacity * 8);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) rc = mapf_cuda_fail(e, "cudaMemset(tree)");
    }
    if (rc != MAPF_OK) {
        mapf_per_destroy(t);
        return rc;
    }
    *out = t;
    return MAPF_OK;
}

int mapf_per_destroy(mapf_per *t)
{
    if (!t) return MAPF_OK;
    DeviceGuard guard(t->device);
    cudaFree(t->tree);
    cudaFree(t->scratch.stamps);
    cudaFree(t->scratch.prio32);
    cudaFree(t->scratch.active);
    cudaFree(t->scratch.err);
    delete t;
    return MAPF_OK;
}

double *mapf_per_tree_ptr(mapf_per *t) { return t ? t->tree : nullptr; }

#define REQUIRE_PER(t)                          \
    if (!(t)) {                                 \
        mapf_set_error("NULL sum-tree handle"); \
        return MAPF_EINVAL;                     \
    }                                           \
    DeviceGuard guard((t)->device);             \
    if (!guard.ok) {                            \
        mapf_set_error("cudaSetDevice failed"); \
        return MAPF_ECUDA;                      \
    }

int mapf_per_update(mapf_per *t, const int64_t *d_idx, const double *d_prio, int64_t n, void *stream)
{
    REQUIRE_PER(t);
    if (n < 0 || (n > 0 && (!d_idx || !d_prio))) {
        mapf_set_error("mapf_per_update: bad arguments");
        return MAPF_EINVAL;
    }
    return mapf_launch_per_update(t, &t->scratch, d_idx, d_prio, n, static_cast<cudaStream_t>(stream));
}

int mapf_per_sample(mapf_per *t, const double *d_uniforms, int64_t batch, int64_t *d_idx_out, double *d_prio_out,
                    float *d_weight_out, double beta, void *stream)
{
    REQUIRE_PER(t);
    if (batch < 1 || !d_uniforms || !d_idx_out || !d_prio_out) {
        mapf_set_error("mapf_per_sample: bad arguments");
        return MAPF_EINVAL;
    }
    return mapf_launch_per_sample(t, d_uniforms, batch, d_idx_out, d_prio_out, d_weight_out, beta,
                                  static_cast<cudaStream_t>(stream));
}

int mapf_per_td_update(mapf_per *t, const float *d_q_online, const float *d_q_target_next, const float *d_q_online_next,
                       const int64_t *d_action, const float *d_reward, const float *d_done, const float *d_steps,
                       const int64_t *d_idx, int64_t n, float gamma, double alpha, int64_t old_ptr, int64_t ptr,
                       int64_t slot_steps, float *d_td_out, float *d_prio_out, void *stream)
{
    REQUIRE_PER(t);
    if (n < 0 || n > t->scratch.cap_n || (n > 0 && (!d_q_online || !d_q_target_next || !d_action || !d_reward || !d_done ||
                                                    !d_steps || !d_idx))) {
        mapf_set_error("mapf_per_td_update: bad arguments (n <= 65536)");
        return MAPF_EINVAL;
    }
    return mapf_launch_per_td_update(t, &t->scratch, d_q_online, d_q_target_next, d_q_online_next, d_action, d_reward, d_done,
                                     d_steps, d_idx, n, gamma, alpha, old_ptr, ptr, slot_steps, d_td_out, d_prio_out,
                                     static_cast<cudaStream_t>(stream));
}

int mapf_per_cycle(mapf_per *t, const mapf_per_cycle_args *a, void *stream)
{
    REQUIRE_PER(t);
    if (!a || a->n_update < 0 || a->n_sample < 0 || a->n_update > t->scratch.cap_n) {
        mapf_set_error("mapf_per_cycle: bad arguments (n_update <= 65536)");
        return MAPF_EINVAL;
    }
    if (a->n_update > 0 && (!a->d_q_online || !a->d_q_target_next || !a->d_action || !a->d_reward || !a->d_done || !a->d_steps || !a->d_idx)) {
        mapf_set_error("mapf_per_cycle: NULL buffer in the update half");
        return MAPF_EINVAL;
    }
    if (a->n_sample > 0 && (!a->d_uniforms || !a->d_sample_idx_out || !a->d_sample_prio_out)) {
        mapf_set_error("mapf_per_cycle: NULL buffer in the sample half");
        return MAPF_EINVAL;
    }
    return mapf_launch_per_cycle(t, &t->scratch, a, static_cast<cudaStream_t>(stream));
}

int mapf_per_status(mapf_per *t, void *stream)
{
    REQUIRE_PER(t);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t bits = 0;
    MAPF_CUDA(cudaMemcpyAsync(&bits, t->scratch.err, 4, cudaMemcpyDeviceToHost, st));
    MAPF_CUDA(cudaStreamSynchronize(st));
    // one condition per call, and only its bit is cleared: a second latched condition surfaces on the next call
    const int32_t bit = (bits & MAPF_ERRBIT_INDEX) ? MAPF_ERRBIT_INDEX : (bits & MAPF_ERRBIT_PRIORITY);
    if (!bit) return MAPF_OK;
    const int32_t rest = bits & ~bit;
    MAPF_CUDA(cudaMemcpyAsync(t->scratch.err, &rest, 4, cudaMemcpyHostToDevice, st));
    MAPF_CUDA(cudaStreamSynchronize(st));
    if (bit == MAPF_ERRBIT_INDEX) {
        mapf_set_error("sum tree: leaf index outside [0, capacity) (skipped)");
        return MAPF_EINDEX;
    }
    mapf_set_error("sum tree: a sampled leaf's priority is not > 0 (buffer.py:74 asserts priorities > 0)");
    return MAPF_EPRIORITY;
}

int mapf_actor_td_n(const float *d_rew, const float *d_q, const uint8_t *d_act, const int32_t *d_size, int32_t episodes,
                    int32_t capacity, int32_t forward_steps, double gamma, double *d_td_out, void *stream)
{
    if (episodes < 0 || capacity < 1 || forward_steps < 1 || forward_steps > 8 ||
        (episodes > 0 && (!d_rew || !d_q || !d_act || !d_size || !d_td_out))) {
        mapf_set_error("mapf_actor_td: bad arguments (1 <= forward_steps <= 8)");
        return MAPF_EINVAL;
    }
    return mapf_launch_actor_td(d_rew, d_q, d_act, d_size, episodes, capacity, forward_steps, gamma, d_td_out,
                                static_cast<cudaStream_t>(stream));
}

int mapf_actor_td(const float *d_rew, const float *d_q, const uint8_t *d_act, const int32_t *d_size, int32_t episodes,
                  int32_t capacity, double *d_td_out, void *stream)
{
    return mapf_actor_td_n(d_rew, d_q, d_act, d_size, episodes, capacity, 2, 0.99, d_td_out, stream);  // config.py:30, buffer.py:175
}

int mapf_replay_gather(const mapf_replay_view *view, const int64_t *d_idx, int64_t batch, const mapf_replay_batch *out,
                       int32_t *d_err, void *stream)
{
    const int rc = check_window_gather("mapf_replay_gather", view, d_idx, batch, out);
    if (rc != MAPF_OK || batch == 0) return rc;
    return mapf_launch_replay_gather(view, d_idx, batch, out, d_err, static_cast<cudaStream_t>(stream));
}

int mapf_obs_unpack(const uint8_t *d_bits_base, const int64_t *d_rows, int64_t count, int32_t num_agents, int32_t dtype,
                    void *d_out, void *stream)
{
    if (count < 0 || (count > 0 && (!d_bits_base || !d_out)) || !aligned16(d_bits_base) || !aligned16(d_out)) {
        mapf_set_error("mapf_obs_unpack: NULL buffer, negative count or a pointer not 16-byte aligned");
        return MAPF_EINVAL;
    }
    if (num_agents < 1 || num_agents > MAPF_MAX_AGENTS || dtype < MAPF_DTYPE_U8 || dtype > MAPF_DTYPE_BF16 || count > 0x7fffffff) {
        mapf_set_error("mapf_obs_unpack: num_agents outside 1..128, unknown dtype or count >= 2^31");
        return MAPF_EINVAL;
    }
    const int rc = require_device("mapf_obs_unpack");
    if (rc != MAPF_OK || count == 0) return rc;
    return mapf_launch_obs_unpack(d_bits_base, d_rows, count, num_agents, dtype, d_out, static_cast<cudaStream_t>(stream));
}

int mapf_replay_gather_compact(const mapf_replay_view_compact *view, const int64_t *d_idx, int64_t batch,
                               const mapf_replay_batch *out, int32_t *d_err, void *stream)
{
    const int rc = check_window_gather("mapf_replay_gather_compact", view, d_idx, batch, out);
    if (rc != MAPF_OK || batch == 0) return rc;
    return mapf_launch_replay_gather_compact(view, d_idx, batch, out, d_err, static_cast<cudaStream_t>(stream));
}

int mapf_obs_unpack_present(const uint8_t *d_bits_base, const int64_t *d_rows, const uint8_t *d_n, const int32_t *d_first,
                            int64_t count, int32_t num_agents, int64_t out_rows, int32_t dtype, void *d_out, void *stream)
{
    if (count < 0 || out_rows < 0 || (count > 0 && (!d_bits_base || !d_rows || !d_n || !d_first)) || (out_rows > 0 && !d_out) ||
        !aligned16(d_bits_base) || !aligned16(d_out)) {
        mapf_set_error("mapf_obs_unpack_present: NULL buffer, negative count or a pointer not 16-byte aligned");
        return MAPF_EINVAL;
    }
    if (num_agents < 1 || num_agents > MAPF_MAX_AGENTS || dtype < MAPF_DTYPE_U8 || dtype > MAPF_DTYPE_BF16 || count > 0x7fffffff ||
        out_rows > 0x7fffffff) {
        mapf_set_error("mapf_obs_unpack_present: num_agents outside 1..128, unknown dtype, or count or out_rows >= 2^31");
        return MAPF_EINVAL;
    }
    const int rc = require_device("mapf_obs_unpack_present");
    if (rc != MAPF_OK || out_rows == 0) return rc;
    return mapf_launch_obs_unpack_present(d_bits_base, d_rows, d_n, d_first, count, num_agents, out_rows, dtype, d_out,
                                          static_cast<cudaStream_t>(stream));
}

int mapf_replay_gather_present(const mapf_replay_view_compact *view, const uint8_t *d_agents, const int64_t *d_idx,
                               const int32_t *d_first, int64_t batch, int64_t out_rows, const mapf_replay_batch *out,
                               int32_t *d_err, void *stream)
{
    const PresentRowArgs pr{d_agents, d_first, out_rows};
    const int rc = check_window_gather("mapf_replay_gather_present", view, d_idx, batch, out, &pr);
    if (rc != MAPF_OK || (batch == 0 && out_rows == 0)) return rc;
    return mapf_launch_replay_gather_present(view, d_agents, d_idx, d_first, batch, out_rows, out, d_err,
                                             static_cast<cudaStream_t>(stream));
}

}  // extern "C"
