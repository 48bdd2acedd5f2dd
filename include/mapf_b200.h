/*
 * mapf_b200.h — C ABI of libmapf_b200.so: the B200-native (sm_100a) batched MAPF environment
 * hot path + prioritized-replay sum-tree / TD kernels.
 *
 * This is the drop-in boundary.  The reference (ZiyuanMa/MAPF_RL) is pure Python and has no FFI;
 * its boundary for this path is the duck-typed class `environment.Environment` and
 * `buffer.SumTree` / `buffer.LocalBuffer`.  Every entry point below names the reference interface
 * (file:line in /root/reference) it replaces.  The Python mirror of those classes
 * (mapf_rl_b200/environment.py, mapf_rl_b200/buffer.py) binds exactly these symbols through ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures.  `stream` is a cudaStream_t passed as
 *     void* (NULL = legacy default stream).
 *   - every pointer named d_* is DEVICE memory owned by the caller; h_* is HOST memory.
 *     The library never returns memory the caller must free; a handle owns only its state arena.
 *   - all functions return 0 on success, a negative MAPF_E* code otherwise; mapf_last_error()
 *     returns a thread-local message for the last failure.
 *   - functions are asynchronous on `stream` unless documented otherwise; one handle must not be
 *     used from two threads at once (the reference env is single-threaded, worker.py:355-361).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     MAPF_ECUDA.
 *
 * Coordinates follow the reference: position (x, y) = (row, col) of map[x, y]; actions
 * 0 stay, 1 up (x-1), 2 down (x+1), 3 left (y-1), 4 right (y+1)  (environment.py:12).
 */
#ifndef MAPF_B200_H
#define MAPF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAPF_ABI_VERSION 2

#define MAPF_OK 0
#define MAPF_EINVAL (-1)   /* bad argument (shape, NULL, unsupported size)          */
#define MAPF_ECUDA (-2)    /* CUDA runtime error / no device                         */
#define MAPF_EACTION (-3)  /* an action was outside 0..4 (environment.py:289-290)    */
#define MAPF_EUNIQUE (-4)  /* two agents share a cell (environment.py:424-428)       */
#define MAPF_ENOMEM (-5)
#define MAPF_ENOSPACE (-6) /* reset could not place the agents ('no empty position', environment.py:31) */
#define MAPF_ESTATE (-7)   /* load / set_state: coordinate outside the map or slot id outside the batch (the reference raises
                              IndexError on the same input; two agents on one cell latch MAPF_EUNIQUE) */
#define MAPF_EINTERNAL (-8) /* the rollout scheduler gave up waiting for a chunk hand-over (a bug, never expected) */
#define MAPF_EINDEX (-9)   /* sum tree: a leaf index outside [0, capacity) was skipped (numpy raises IndexError) */
#define MAPF_EPRIORITY (-10) /* sum tree: a sampled leaf has priority 0 (the reference asserts priorities > 0, buffer.py:74) */

/* Reward codes: the position of an agent's reward in reward_fn (config.py:8-12).  Every step entry point can emit these
 * u8 codes instead of / next to the fp32 rewards: a reward takes one of five values, so the host side of an actor reads
 * B*N bytes per step instead of 4*B*N and looks the value up in its 5-entry table. */
#define MAPF_RCODE_MOVE 0
#define MAPF_RCODE_STAY_ON_GOAL 1
#define MAPF_RCODE_STAY_OFF_GOAL 2
#define MAPF_RCODE_COLLISION 3
#define MAPF_RCODE_FINISH 4
#define MAPF_RCODE_RESET 5 /* reward 0: the step re-generated the environment (mapf_env_set_autoreset); on a sized
                              handle (mapf_env_enable_sizes) also the code of every absent agent slot a >= n_e */
#define MAPF_RCODE_STAY_ON MAPF_RCODE_STAY_ON_GOAL
#define MAPF_RCODE_STAY_OFF MAPF_RCODE_STAY_OFF_GOAL

#define MAPF_OBS_RADIUS 4  /* config.py:14 — the only radius any reference consumer uses */
#define MAPF_FOV 9
#define MAPF_OBS_CHANNELS 6
#define MAPF_OBS_BYTES_PER_AGENT 486 /* 6*9*9, config.py:7 obs_shape */
/* Packed observation (the compact replay store): one 64-byte row per agent.  Element k = c*81 + r*9 + col of the agent's
 * flattened 6x9x9 bool observation is bit (k & 7) of byte (k >> 3), LSB first -- np.packbits(obs.reshape(N, 486), axis=-1,
 * bitorder="little") padded to 64 bytes; bits 486..511 are always 0.  A frame is N*64 bytes.  This is the step kernel's own
 * bit stream with agent a at bit 512*a instead of 486*a, so every agent starts on a word boundary. */
#define MAPF_OBS_PACKED_BYTES_PER_AGENT 64
/* Packed communication mask: agent i's row is CW = ceil(N/8) bytes, bit j (LSB first) = mask[i][j]; a frame is N*CW bytes. */

/* element types of mapf_obs_unpack */
#define MAPF_DTYPE_U8 0
#define MAPF_DTYPE_F16 1
#define MAPF_DTYPE_BF16 2
#define MAPF_MAX_AGENTS 128
#define MAPF_MAX_MAP_SIDE 120
#define MAPF_DIST_UNREACHABLE 2147483647 /* environment.py:218 */

typedef struct mapf_env mapf_env; /* opaque: a lockstep batch of B independent environments */
typedef struct mapf_per mapf_per; /* opaque: one prioritized-replay sum tree               */

typedef struct mapf_env_config {
    int32_t num_envs;    /* B >= 1                                                          */
    int32_t num_agents;  /* N, 1..MAPF_MAX_AGENTS          (environment.py:75 num_agents)   */
    int32_t map_length;  /* L, 2..MAPF_MAX_MAP_SIDE, square (environment.py:75 map_length)  */
    int32_t obs_radius;  /* must be 4                       (environment.py:76)             */
    int32_t device;      /* CUDA device ordinal                                             */
    /* reward_fn in the order move, stay_on_goal, stay_off_goal, collision, finish
     * (config.py:8-12, environment.py:76,142) */
    float reward_fn[5];
} mapf_env_config;

/* ---- lifetime ---------------------------------------------------------------------------- */
int mapf_abi_version(void);
const char *mapf_last_error(void);

/* Environment.__init__ storage part (environment.py:75-144): allocates the device arena. */
int mapf_env_create(const mapf_env_config *cfg, mapf_env **out);
int mapf_env_destroy(mapf_env *env);
/* bytes of device memory held by the handle */
int64_t mapf_env_arena_bytes(const mapf_env *env);

/* ---- Environment.load (environment.py:198-215) -------------------------------------------- */
/* Loads `n` instances into the env slots listed in d_env_ids (NULL => slots 0..n-1), resets their
 * step counters to 0 and recomputes their heuristic maps (get_navi_map, environment.py:217-276).
 *   d_maps   u8[n, L, L]  0 = free, non-zero = obstacle
 *   d_agents u8[n, N, 2]  (x, y);   d_goals u8[n, N, 2]                                   */
int mapf_env_load(mapf_env *env, const int32_t *d_env_ids, int32_t n, const uint8_t *d_maps,
                  const uint8_t *d_agents, const uint8_t *d_goals, void *stream);

/* ---- Environment.get_navi_map (environment.py:217-276) / search.compute_heuristics
 *      (search.py:24-55) -------------------------------------------------------------------- */
/* Recomputes the per-agent BFS heuristic maps of the listed env slots (NULL => all B).
 * d_dist_out (optional) receives the distance maps, i32[n, N, L, L], 2147483647 where
 * unreachable / obstacle — the same numbers search.compute_heuristics returns where finite. */
int mapf_env_bfs_navi(mapf_env *env, const int32_t *d_env_ids, int32_t n, int32_t *d_dist_out, void *stream);

/* ---- Environment.step (environment.py:278-430), fused with the observe() it ends in (:430) -- */
/*   d_actions  u8[B, N]          in
 *   d_obs      u8[B, N, 6, 9, 9] out, bool bytes, layout of environment.py:444-465
 *   d_rewards  f32[B, N]         out (the reference's python numbers cast to fp32)
 *   d_done     u8[B]             out (environment.py:415-419)
 *   d_steps    i32[B]            out, optional: env.steps after the step (environment.py:412)
 * An action outside 0..4 is treated as "stay" and latches MAPF_EACTION (see mapf_env_status). */
int mapf_env_step_observe(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs, float *d_rewards,
                          uint8_t *d_done, int32_t *d_steps, void *stream);

/* The same step with every output optional but d_done: d_rewards f32[B, N] and / or d_codes u8[B, N] (MAPF_RCODE_*),
 * d_obs_rows (optional) as in mapf_env_step_observe_rows. */
int mapf_env_step_observe_ex(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs, const int64_t *d_obs_rows,
                             float *d_rewards, uint8_t *d_codes, uint8_t *d_done, int32_t *d_steps, void *stream);

/* Environment.observe (environment.py:433-467).  d_pos (optional) u8[B, N, 2]. */
int mapf_env_observe(mapf_env *env, uint8_t *d_obs, uint8_t *d_pos, void *stream);

/* Same two calls writing each environment's observation block at its own row of a replay store
 * (worker.py:96: obs_buf[slot*(max_steps+1) + t]): environment e writes N*486 bytes at
 * d_obs_base + d_obs_rows[e] * N*486.  d_obs_rows i64[B]. */
int mapf_env_step_observe_rows(mapf_env *env, const uint8_t *d_actions, uint8_t *d_obs_base, const int64_t *d_obs_rows,
                               float *d_rewards, uint8_t *d_done, int32_t *d_steps, void *stream);
int mapf_env_observe_rows(mapf_env *env, uint8_t *d_obs_base, const int64_t *d_obs_rows, uint8_t *d_pos, void *stream);

/* The same step and observe writing PACKED observations (MAPF_OBS_PACKED_BYTES_PER_AGENT): environment e writes its N*64-byte
 * frame at d_bits_base + d_bits_rows[e] * N*64 (d_bits_rows i64[B]; NULL = row e).  d_bits_base must be 16-byte aligned.
 * Positions, rewards, codes, done, steps and latched errors are those of mapf_env_step_observe_ex; the frame is
 * np.packbits of what the dense call writes, pad bits 0.  Uniform and sized handles (an absent agent's 64 bytes are 0). */
int mapf_env_step_observe_packed(mapf_env *env, const uint8_t *d_actions, uint8_t *d_bits_base, const int64_t *d_bits_rows,
                                 float *d_rewards, uint8_t *d_codes, uint8_t *d_done, int32_t *d_steps, void *stream);
int mapf_env_observe_packed(mapf_env *env, uint8_t *d_bits_base, const int64_t *d_bits_rows, uint8_t *d_pos, void *stream);

/* Packed observation frames -> dense [count, N, 6, 9, 9] elements of `dtype` (MAPF_DTYPE_U8 0 / 1, MAPF_DTYPE_F16 or
 * MAPF_DTYPE_BF16 0.0 / 1.0).  Frame i is read at d_bits_base + d_rows[i] * N*64 (d_rows i64[count]; NULL = row i).  Both
 * pointers must be 16-byte aligned. */
int mapf_obs_unpack(const uint8_t *d_bits_base, const int64_t *d_rows, int64_t count, int32_t num_agents, int32_t dtype,
                    void *d_out, void *stream);

/* Packed frames -> the observations of PRESENT agents only, one row each (mapf_rl_b200/present.py): output row d_first[f] + a
 * holds agent a < min(d_n[f], num_agents) of frame f (read at d_bits_base + d_rows[f] * N*64); every other row of
 * [0, out_rows) is zeros.  d_rows i64[count], d_n u8[count], d_first i32[count] nondecreasing with
 * d_first[f] + min(d_n[f], N) <= d_first[f + 1].  Output [out_rows, 6, 9, 9] of `dtype` as mapf_obs_unpack; d_bits_base and
 * d_out must be 16-byte aligned. */
int mapf_obs_unpack_present(const uint8_t *d_bits_base, const int64_t *d_rows, const uint8_t *d_n, const int32_t *d_first,
                            int64_t count, int32_t num_agents, int64_t out_rows, int32_t dtype, void *d_out, void *stream);

/* T lockstep steps with the actions already resident on the device: the loop `for t: obs, r, done, _ = env.step(a[t])`
 * of test.py:120-130 / worker.py:383-395 when the actions do not depend on the observations (replaying planner paths,
 * random-policy data generation, benchmarking).  Step t reads action slot t % action_slots, writes observation slot
 * t % obs_slots and rewards / done / steps slot t % out_slots; results equal T calls of mapf_env_step_observe.
 *   d_actions u8[action_slots, B, N]   d_obs u8[obs_slots, B, N, 6, 9, 9]
 *   d_rewards f32[out_slots, B, N]     d_done u8[out_slots, B]     d_steps i32[out_slots, B] (optional)
 * Environments are independent (no reference code path couples two Environment objects).  With chains = 0 and up to 64
 * agents the rollout is ONE launch of a persistent kernel (mapf_rollout_kernels.cu): the rollout is cut into work items
 * (environment, chunk of consecutive steps) that resident warps claim time-major from a global counter; a warp keeps the
 * environment's state in registers / shared memory for the steps of its item, each agent's current 16x16 heuristic tile is
 * cached in shared memory, warps drift out of phase on their own (one's observation stores overlap another's conflict
 * resolution) and nothing is launched between steps.  With chains >= 1 (or more than 64 agents) the batch runs as `chains`
 * contiguous sub-batches (1..MAPF_MAX_CHAINS), each an independent chain of T single-step launches on a stream of its own;
 * when T covers at least 4 periods P = lcm(slot counts) <= 64, whole periods are replayed from per-chain CUDA graphs.
 * The call forks from `stream` and joins back into it; it returns when everything is queued (asynchronous).
 * One handle runs one rollout at a time. */
#define MAPF_MAX_CHAINS 16
int mapf_env_rollout(mapf_env *env, int32_t T, const uint8_t *d_actions, int32_t action_slots, uint8_t *d_obs,
                     int32_t obs_slots, float *d_rewards, uint8_t *d_done, int32_t *d_steps, int32_t out_slots,
                     int32_t chains, void *stream);

/* mapf_env_rollout with every output ring optional but d_done, plus reward codes. */
typedef struct mapf_rollout_io {
    int32_t T;               /* steps                                                            */
    const uint8_t *d_actions; /* u8[action_slots, B, N]                                           */
    int32_t action_slots;
    uint8_t *d_obs;          /* u8[obs_slots, B, N, 6, 9, 9]                                     */
    int32_t obs_slots;
    float *d_rewards;        /* f32[out_slots, B, N] or NULL                                     */
    uint8_t *d_codes;        /* u8[out_slots, B, N] or NULL (MAPF_RCODE_*)                       */
    uint8_t *d_done;         /* u8[out_slots, B]                                                 */
    int32_t *d_steps;        /* i32[out_slots, B] or NULL                                        */
    int32_t out_slots;
    int32_t chains;          /* 0 = persistent kernel where it is served, else chains            */
} mapf_rollout_io;
int mapf_env_rollout_ex(mapf_env *env, const mapf_rollout_io *io, void *stream);

/* Episode handling inside mapf_env_rollout (the actor loop's `if done or env.steps >= max_steps: reset()`,
 * worker.py:390,422-428, config.py:29).  With max_steps > 0, a rollout step that finds its environment finished (all agents
 * on their goals after the previous step, or steps >= max_steps) does not move anybody: it draws a NEW instance for the
 * slot on the device (generator + heuristic maps, exactly what mapf_env_reset(mask = {e}, seed, env_offset + n * stride,
 * density) draws for the slot's n-th re-generation, n = 1, 2, ...), emits that instance's first observation, rewards 0
 * (MAPF_RCODE_RESET), done 0 and steps 0, and ignores the step's actions.  The step before it carries the terminal
 * observation / rewards / done / steps exactly as without episode handling.  `stride` = number of environments of the
 * whole job (all GPUs), so re-generated instances never collide with another slot's.  max_steps = 0 switches it off.
 * Only the persistent kernel serves it (up to 64 agents).  The call also zeroes the per-slot episode counters. */
int mapf_env_set_autoreset(mapf_env *env, int32_t max_steps, uint64_t seed, uint64_t env_offset, uint64_t stride,
                           float density, void *stream);

/* d_counts_out u32[B]: instances generated for each slot by the episode handling since mapf_env_set_autoreset. */
int mapf_env_episode_counts(mapf_env *env, uint32_t *d_counts_out, void *stream);

/* check_unique != 0: every step verifies that no two agents share a cell afterwards (environment.py:424-428) and latches
 * MAPF_EUNIQUE otherwise (read by mapf_env_status).  Off by default: a correct step from a valid state cannot violate it,
 * and load / set_state validate what they are given. */
int mapf_env_set_checks(mapf_env *env, int32_t check_unique);

/* How mapf_env_rollout would run these arguments: number of chains, environments per chain, and the number of steps per
 * replayed graph (0 = every step launched directly).  chains_out = 0 means the persistent kernel: one launch for the whole
 * rollout.  Outputs are optional. */
int mapf_env_rollout_plan(mapf_env *env, int32_t T, int32_t action_slots, int32_t obs_slots, int32_t out_slots,
                          int32_t chains, int32_t *chains_out, int32_t *envs_per_chain_out, int32_t *graph_period_out);

/* Host-buffer variant of step (what a per-process actor calls): actions in host memory in, rewards / done / steps (and
 * obs if h_obs != NULL) in host memory out, synchronous.  All h_* buffers are ordinary or page-locked host memory;
 * page-locked ones (cudaHostAlloc / cudaHostRegister / torch pin_memory) are used in place, pageable ones are staged
 * through the handle's own pinned area.  The call runs the step kernel (which reads page-locked actions in place over
 * PCIe), then the observe kernel WHILE rewards / done / steps are copied to the host on a side stream, captured once per
 * buffer set into a CUDA graph.  What a host pointer resolves to is re-validated on every call (a freed and re-used
 * address is detected).  d_obs_opt: if non-NULL the observation is written there (device replay tensor) instead of an
 * internal buffer. */
int mapf_env_step_host(mapf_env *env, const uint8_t *h_actions, uint8_t *h_obs, float *h_rewards,
                       uint8_t *h_done, int32_t *h_steps, uint8_t *d_obs_opt, void *stream);

/* The throughput form of the host-buffer step: reward CODES (u8[B, N], MAPF_RCODE_*) instead of fp32 rewards, run as a
 * two-stage pipeline.  Stage 1 (an internal stream): the step kernel reads the page-locked actions in place over PCIe and
 * leaves codes / steps / done in a device staging block plus a SNAPSHOT of the new positions; one DMA copy brings the
 * staging block back when h_steps == h_codes + align16(B*N) and h_done == h_steps + B (three copies otherwise).  Stage 2
 * (the caller's `stream`): the observe kernel writes the observation of that snapshot into d_obs (required, device memory).
 * The call returns when stage 1 is done -- h_codes / h_done / h_steps are final -- while stage 2 may still be running; it is
 * ordered before anything queued on `stream` afterwards, and the NEXT call's stage 1 overlaps it (it may overwrite the
 * positions, the snapshot is double-buffered).  Any other entry point on the handle first waits for the pipeline to drain.
 * Pageable host buffers are staged through the handle's own pinned area. */
int mapf_env_step_host_codes(mapf_env *env, const uint8_t *h_actions, uint8_t *h_codes, uint8_t *h_done, int32_t *h_steps,
                             uint8_t *d_obs, void *stream);

/* Tuning (process-wide; profiles/, tests): CTA shape of the single-launch step kernel.
 *   variant     1 (default) picks the CTA shape per launch, 0 / 7 / 8 / 4 / 9 force one (launch_step_rwk in
 *               mapf_step_kernels.cu);  < 0 leaves the current value
 *   flags       1 = L2 evict_last on heuristic-map loads, 2 = L2 evict_first policy on observation stores; < 0 keeps
 *   ctas_per_sm cap on resident CTAs per SM (0 = as many as fit); < 0 keeps
 * The same three values are read once from MAPF_STEP_VARIANT / MAPF_STEP_FLAGS / MAPF_STEP_CTAS_PER_SM. */
int mapf_debug_step_tuning(int32_t variant, int32_t flags, int32_t ctas_per_sm);
/* Knobs of the persistent kernel behind mapf_env_rollout (process-wide; < 0 keeps a value): persistent 0 = never use it,
 * warps_per_sm = resident warps per SM (0 = 16), chunk = steps per work item (0 = automatic), store_mode 0 = direct
 * 16-byte stores / 1 = bulk (TMA) stores from a shared-memory staging block, stagger_ns = spread of the warps' start.
 * Read once from MAPF_ROLLOUT_PERSISTENT / _WARPS_PER_SM / _CHUNK / _STORE_MODE / _STAGGER_NS. */
int mapf_debug_rollout_tuning(int32_t persistent, int32_t warps_per_sm, int32_t chunk, int32_t store_mode, int32_t stagger_ns);
/* Episode handling of mapf_env_rollout (mapf_env_set_autoreset).  The environments whose episode ends at the step cap inside
 * a launch are known before it, and their next instances can be generated ahead by the dedicated generator / BFS kernels and
 * adopted by the rollout kernel at the episode's end.  mode 1 (default) = automatic: BEFORE the launch when many are due
 * (the kernels run at full occupancy), BESIDE it on a second stream when few are (the kernels are latency-bound then);
 * 2 = always before; 3 = always beside; 0 = never: every episode end re-generates inside the rollout kernel (generator by the
 * environment's warp, the per-agent searches as tasks any warp takes), which is also what happens when a staged instance
 * is not ready in time and for a second episode end of an environment in one launch; < 0 only queries.  Read once from
 * MAPF_ROLLOUT_PREGEN.  Every form produces the same instances. */
int mapf_debug_rollout_pregen(int32_t on);
/* In-launch re-generations announce their per-agent searches as tasks any warp of the rollout kernel takes (1) or run them
 * all on the environment's own warp (0, default); < 0 only queries.  Read once from MAPF_ROLLOUT_TASKS.  Same instances. */
int mapf_debug_rollout_tasks(int32_t on);
/* Selects the form of mapf_env_step_host (0..4, see mapf_abi.cu; < 0 only queries); returns the mode in force. */
int mapf_debug_step_host_mode(int32_t mode);

/* ---- communication mask of Network.step (model.py:196-208), the actor-side glue next to observe() ------
 *   d_mask_out u8[B, N, N]: mask[i][j] = 1 iff agent j is inside agent i's 9x9 field of view (|dx| <= 4 and
 *   |dy| <= 4) AND j is one of the `max_comm_agents` (config.py:58, 1..3) nearest agents of i by Euclidean
 *   distance, i itself included.  torch.topk's order among equal distances is unspecified; ties go to
 *   the lower agent id here. */
int mapf_env_comm_mask(mapf_env *env, int32_t max_comm_agents, uint8_t *d_mask_out, void *stream);
/* The same mask in one launch as the dense u8[B, N, N] (d_mask_out, optional: what the Q-network consumes) AND as packed rows
 * (the comm-mask format above): environment e writes N*ceil(N/8) bytes at d_bits_base + d_bits_rows[e] * N*ceil(N/8)
 * (d_bits_rows i64[B]; NULL = row e).  Uniform and sized handles. */
int mapf_env_comm_mask_packed(mapf_env *env, int32_t max_comm_agents, uint8_t *d_mask_out, uint8_t *d_bits_base,
                              const int64_t *d_bits_rows, void *stream);

/* ---- state access (attributes read by worker.py:390,426 / test.py:46-48,130) --------------- */
/* Any output pointer may be NULL.  d_map u8[B,L,L]; d_pos/d_goals u8[B,N,2]; d_steps i32[B];
 * d_navi u8[B,N,4,L,L] = navi_map without the obs_radius padding (environment.py:253-276). */
int mapf_env_get_state(mapf_env *env, uint8_t *d_map, uint8_t *d_pos, uint8_t *d_goals, int32_t *d_steps,
                       uint8_t *d_navi, void *stream);
/* Overwrite agent positions / step counters (used to restore snapshots). Either may be NULL. */
int mapf_env_set_state(mapf_env *env, const uint8_t *d_pos, const int32_t *d_steps, void *stream);

/* Synchronous: returns the latched error (MAPF_OK, MAPF_EACTION, MAPF_EUNIQUE, MAPF_ENOSPACE, MAPF_ESTATE,
 * MAPF_EINTERNAL) and clears it. */
int mapf_env_status(mapf_env *env, void *stream);

/* ---- Environment.reset instance generation (environment.py:146-196), device side ----------- */
/* Draws new random instances for the slots whose d_mask byte is non-zero (NULL => all): obstacle map
 * iid Bernoulli(density) (density < 0 => one triangular(0, 0.33, 0.5) draw per env, :156), start and
 * goal of every agent in one 4-connected free component (:159-192), steps = 0, heuristic maps
 * recomputed.  Counter-based RNG: env slot e uses stream (seed, env_offset + e) so shards of a
 * multi-GPU job draw the instances a single GPU would.  Distributional parity only (SURVEY 8c). */
int mapf_env_reset(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density,
                   void *stream);

/* ---- per-environment agent count and map side (the reference's curriculum, worker.py:424-425) ---- */
/* A SIZED handle keeps, next to the maxima (N, L) it was created with, a setting (n_e, l_e), 1 <= n_e <= N,
 * 2 <= l_e <= L, per slot e.  Agents a < n_e on cells inside l_e x l_e get exactly what a handle created with (n_e, l_e)
 * gives for the same instance and actions.  Agents a >= n_e are absent: their actions are never read, they hold no cell
 * and take no part in conflicts, `done`, the 'unique' check or the comm mask (rows and columns 0); every step and observe
 * writes their 486 observation bytes as zeros, their reward as 0 with code MAPF_RCODE_RESET; positions and goals read 255,
 * distances MAPF_DIST_UNREACHABLE, heuristic bits 0.  Cells outside l_e are off the map: a move there is a collision, the
 * observation shows 0 on every channel, the map reads 0 and the BFS does not enter them.
 * mapf_env_load / mapf_env_reset on a sized handle give the loaded / reset slots (N, L).  A sized handle does not serve
 * mapf_env_rollout, mapf_env_rollout_ex, mapf_env_set_autoreset, mapf_env_step_host or mapf_env_step_host_codes
 * (MAPF_EINVAL). */

/* Opts the handle in (allocates u8 n[B], l[B], initialised to (N, L)).  A handle that never calls it runs the uniform
 * kernels.  MAPF_EINVAL once the handle has used episode handling or the host-buffer steps. */
int mapf_env_enable_sizes(mapf_env *env);
/* mapf_env_load with a setting per instance: d_num_agents u8[n], d_map_length u8[n].  Map cells outside l_e and agent
 * rows >= n_e of d_maps u8[n, L, L] / d_agents, d_goals u8[n, N, 2] are ignored.  A setting outside the maxima returns
 * MAPF_EINVAL before any launch; a coordinate >= l_e latches MAPF_ESTATE. */
int mapf_env_load_sized(mapf_env *env, const int32_t *d_env_ids, int32_t n, const uint8_t *d_maps, const uint8_t *d_agents,
                        const uint8_t *d_goals, const uint8_t *d_num_agents, const uint8_t *d_map_length, void *stream);
/* mapf_env_reset drawing each reset slot's setting uniformly from d_levels u8[K, 2] = (n, l) pairs: index (w * K) >> 32,
 * w = one Philox word of the slot's own stream (seed, env_offset + e) under a purpose of its own.  The slot's instance is
 * then the one a uniform (n, l) handle's mapf_env_reset draws for that stream, whatever the sharding.  K < 1 or a level
 * outside the maxima returns MAPF_EINVAL before any launch. */
int mapf_env_reset_levels(mapf_env *env, const uint8_t *d_mask, uint64_t seed, uint64_t env_offset, float density,
                          const uint8_t *d_levels, int32_t num_levels, void *stream);
/* The slots' settings: d_num_agents_out u8[B], d_map_length_out u8[B] (either may be NULL). */
int mapf_env_get_sizes(mapf_env *env, uint8_t *d_num_agents_out, uint8_t *d_map_length_out, void *stream);

/* ---- buffer.SumTree (buffer.py:16-105) ------------------------------------------------------ */
/* capacity must be a power of two (buffer.py:23).  Tree nodes are fp64 like the reference. */
int mapf_per_create(int64_t capacity, int32_t device, mapf_per **out);
int mapf_per_destroy(mapf_per *tree);
/* device pointer to the 2*capacity-1 fp64 nodes (SumTree.tree, buffer.py:25); leaves start at capacity-1 */
double *mapf_per_tree_ptr(mapf_per *tree);

/* SumTree.batch_update (buffer.py:95-105): leaf[d_idx[k]] = d_prio[k] (duplicates: last in batch order
 * wins, numpy fancy assignment), then every touched ancestor = left + right, level by level.
 * d_idx is NOT modified (the reference mutates it in place, buffer.py:96; the Python mirror
 * reproduces that).  Any order, any duplicates, any n; a batch of up to 256 non-decreasing indices -- what
 * mapf_per_sample returns and what an episode insert (worker.py:87-94) is -- runs its level loop in shared memory
 * (same bits, about half the time; DESIGN.md K4). */
int mapf_per_update(mapf_per *tree, const int64_t *d_idx, const double *d_prio, int64_t n, void *stream);

/* SumTree.batch_sample (buffer.py:56-78) with caller-supplied uniforms u in [0,1):
 * prefix_i = i*interval + u_i*interval.  d_weight_out (optional) = (p / min_batch p)^(-beta)
 * (worker.py:165-166; fp32 powf, 1e-6 relative).  d_idx_out is non-decreasing (stratified prefixes).  A sampled leaf
 * whose priority is not > 0 (buffer.py:74 asserts) is returned as the reference finds it and latches MAPF_EPRIORITY
 * (mapf_per_status). */
int mapf_per_sample(mapf_per *tree, const double *d_uniforms, int64_t batch, int64_t *d_idx_out,
                    double *d_prio_out, float *d_weight_out, double beta, void *stream);

/* Fused learner tail (worker.py:300-308 + 186-203 + buffer.py:95-105), one call after the two
 * Q-network forwards:
 *   td      = Q(s,a) - (r + gamma^steps * (1-done) * max_a' Qtgt(s',a'))        (worker.py:302-306)
 *             (d_q_online_next != NULL => double-Q: a* = argmax Q_online(s'), bootstrap Qtgt(s',a*))
 *   prio    = max(|td|, 1e-6)                                                  (worker.py:308)
 *   leaf    = prio^alpha for samples whose episode slot was not overwritten since sampling
 *             (window [old_ptr, ptr) in units of slot_steps leaves, wrap-aware, worker.py:192-201)
 *   then the ancestor refresh of batch_update.
 * All fp32 inputs; tree in fp64.  d_td_out / d_prio_out f32[n] (either may be NULL). */
int mapf_per_td_update(mapf_per *tree, const float *d_q_online, const float *d_q_target_next,
                       const float *d_q_online_next, const int64_t *d_action, const float *d_reward,
                       const float *d_done, const float *d_steps, const int64_t *d_idx, int64_t n, float gamma,
                       double alpha, int64_t old_ptr, int64_t ptr, int64_t slot_steps, float *d_td_out,
                       float *d_prio_out, void *stream);

/* One learner cycle in ONE launch (north star (4)): the priorities of the batch that has just been through the two Q
 * forwards go into the tree (the mapf_per_td_update half), then the NEXT batch is drawn from the refreshed tree with its
 * importance-sampling weights (the mapf_per_sample half).  Either half may be empty (n_update / n_sample = 0). */
typedef struct mapf_per_cycle_args {
    /* update half: arguments of mapf_per_td_update */
    const float *d_q_online, *d_q_target_next, *d_q_online_next;
    const int64_t *d_action;
    const float *d_reward, *d_done, *d_steps;
    const int64_t *d_idx;
    int64_t n_update;
    float gamma;
    double alpha;
    int64_t old_ptr, ptr, slot_steps;
    float *d_td_out, *d_prio_out;
    /* sample half: arguments of mapf_per_sample */
    const double *d_uniforms;
    int64_t n_sample;
    int64_t *d_sample_idx_out;
    double *d_sample_prio_out;
    float *d_sample_weight_out;
    double beta;
} mapf_per_cycle_args;
int mapf_per_cycle(mapf_per *tree, const mapf_per_cycle_args *args, void *stream);

/* Synchronous: MAPF_EINDEX if an update since the last call was handed a leaf index outside [0, capacity) (such entries
 * are skipped), MAPF_EPRIORITY if a sample (mapf_per_sample, mapf_per_cycle) returned a leaf whose priority is not > 0
 * (indices and priorities are still the reference's; the weights of that batch are undefined), else MAPF_OK.  Reports
 * one condition per call, MAPF_EINDEX first, and clears only its latch, so a second condition is reported by the next
 * call.  One tree handle is used from one stream at a time. */
int mapf_per_status(mapf_per *tree, void *stream);

/* LocalBuffer.finish TD (buffer.py:170-177) for `episodes` episodes of up to `capacity` steps:
 *   td[e,t] = | r[e,t] + 0.99*r[e,t+1] + max_a q[e,t,a] - q[e,t,act[e,t]] |,  0 for t >= size[e]
 *   d_rew f32[episodes, capacity] (already rounded through fp16 by the caller, buffer.py:122),
 *   d_q f32[episodes, capacity, 5], d_act u8[episodes, capacity], d_size i32[episodes],
 *   d_td_out f64[episodes, capacity]. */
int mapf_actor_td(const float *d_rew, const float *d_q, const uint8_t *d_act, const int32_t *d_size,
                  int32_t episodes, int32_t capacity, double *d_td_out, void *stream);
/* The same for config.forward_steps = n (1..8) and another discount: td = | sum_{j<n} gamma^j r[e,t+j] + max_a q - q[a_t] |
 * (buffer.py:174-175 builds the kernel [0.99^(n-1), ..., 1] from config.forward_steps; mapf_actor_td is n = 2, 0.99). */
int mapf_actor_td_n(const float *d_rew, const float *d_q, const uint8_t *d_act, const int32_t *d_size, int32_t episodes,
                    int32_t capacity, int32_t forward_steps, double gamma, double *d_td_out, void *stream);

/* ---- GlobalBuffer.sample_batch window gather (worker.py:106-184) -------------------------------- */
/* Device-resident replay store in the reference's logical layout (worker.py:36-42): episode slot g owns
 * observation / comm-mask rows g*(max_steps+1) + f (f = 0..max_steps) and action / reward / hidden rows
 * g*max_steps + t; sum-tree leaf idx = g*max_steps + t.  All pointers are device memory owned by the caller. */
typedef struct mapf_replay_view {
    const uint8_t *obs_buf;    /* u8 bool [(max_steps+1)*capacity, num_agents, 6, 9, 9]   worker.py:36 */
    const uint8_t *comm_buf;   /* u8 bool [(max_steps+1)*capacity, num_agents, num_agents] worker.py:42 */
    const uint16_t *hid_buf;   /* fp16 [max_steps*capacity, num_agents, latent_dim]       worker.py:39 */
    const uint8_t *act_buf;    /* u8  [max_steps*capacity]                                 worker.py:37 */
    const uint16_t *rew_buf;   /* fp16 [max_steps*capacity]                                worker.py:38 */
    const uint8_t *done_buf;   /* u8 bool [capacity]                                       worker.py:40 */
    const int32_t *size_buf;   /* i32 [capacity]                                           worker.py:41 */
    int32_t num_agents;        /* config.max_num_agetns                                                */
    int32_t max_steps;         /* config.max_steps (256)                                               */
    int32_t bt_steps;          /* config.bt_steps (16)                                                 */
    int32_t forward_steps;     /* config.forward_steps (2)                                             */
    int32_t latent_dim;        /* config.latent_dim (256)                                              */
} mapf_replay_view;

/* outputs for `batch` sampled leaves, W = bt_steps + forward_steps frames each (worker.py:168-182) */
typedef struct mapf_replay_batch {
    uint16_t *obs;        /* fp16 [batch, W, num_agents, 6, 9, 9], zero padded (worker.py:139-142,169)  */
    uint8_t *comm_mask;   /* u8 bool [batch, W, num_agents, num_agents]                  (worker.py:176)  */
    uint16_t *hidden;     /* fp16 [batch*num_agents, latent_dim], zeros while t < bt_steps (worker.py:175) */
    int64_t *action;      /* i64 [batch]                                                 (worker.py:170)  */
    uint16_t *reward;     /* fp16 [batch]                                                (worker.py:171)  */
    uint16_t *done;       /* fp16 [batch] 0 / 1                                          (worker.py:173)  */
    uint16_t *steps;      /* fp16 [batch] min(forward_steps, size - t)                   (worker.py:174)  */
    int64_t *bt_steps;    /* i64 [batch] min(t + 1, bt_steps)                            (worker.py:175)  */
} mapf_replay_batch;

/* d_idx i64[batch]: sampled leaves (from mapf_per_sample).  d_err (optional) i32[1]: bit 0 is set if a
 * leaf lies beyond its episode's size (the reference asserts, worker.py:120). */
int mapf_replay_gather(const mapf_replay_view *view, const int64_t *d_idx, int64_t batch, const mapf_replay_batch *out,
                       int32_t *d_err, void *stream);

/* The compact store: the same logical store with packed observations and comm masks (formats above) and ONE hidden vector per
 * transition (the reference writes agent 0's hidden state into every agent's row, buffer.py:148).  About 12x fewer bytes per
 * transition at 32 agents (DESIGN.md §3). */
typedef struct mapf_replay_view_compact {
    const uint8_t *obs_bits;   /* u8 [(max_steps+1)*capacity, num_agents, 64]                  */
    const uint8_t *comm_bits;  /* u8 [(max_steps+1)*capacity, num_agents, ceil(num_agents/8)]  */
    const uint16_t *hid_buf;   /* fp16 [max_steps*capacity, latent_dim]                        */
    const uint8_t *act_buf;    /* u8  [max_steps*capacity]                                      */
    const uint16_t *rew_buf;   /* fp16 [max_steps*capacity]                                     */
    const uint8_t *done_buf;   /* u8 bool [capacity]                                            */
    const int32_t *size_buf;   /* i32 [capacity]                                                */
    int32_t num_agents;
    int32_t max_steps;
    int32_t bt_steps;
    int32_t forward_steps;
    int32_t latent_dim;
} mapf_replay_view_compact;

/* mapf_replay_gather from a compact store: fills the same mapf_replay_batch with the same contents the dense gather gives
 * for the same logical store (fp16 observations, u8 comm masks, the sample's hidden vector in each of its N rows, scalars,
 * zero padding, d_err).  view->obs_bits must be 16-byte aligned. */
int mapf_replay_gather_compact(const mapf_replay_view_compact *view, const int64_t *d_idx, int64_t batch,
                               const mapf_replay_batch *out, int32_t *d_err, void *stream);

/* mapf_replay_gather_compact with observations and hidden vectors in PRESENT-agent rows (mapf_rl_b200/present.py): sample b
 * has n_b = min(d_agents[slot of b], num_agents) agents (d_agents u8[capacity], the store's per-slot agent count), and row
 * d_first[b] + a (d_first i32[batch] nondecreasing, d_first[b] + n_b <= d_first[b + 1]) holds its agent a:
 *   out->obs     fp16 [out_rows, W, 6, 9, 9]   the agent's window frames, zero padded as the compact gather pads them
 *   out->hidden  fp16 [out_rows, latent_dim]    the sample's stored vector, zeros while t < bt_steps
 * Rows of [0, out_rows) that hold no agent are zeros.  comm_mask, the scalars and d_err are those of
 * mapf_replay_gather_compact.  W = bt_steps + forward_steps <= 64; obs_bits and out->obs must be 16-byte aligned. */
int mapf_replay_gather_present(const mapf_replay_view_compact *view, const uint8_t *d_agents, const int64_t *d_idx,
                               const int32_t *d_first, int64_t batch, int64_t out_rows, const mapf_replay_batch *out,
                               int32_t *d_err, void *stream);

/* ---- prioritized planning on the device (DESIGN.md §8 (f)5) --------------------------------------------------------------
 * A collision-free plan for every environment of the batch from its current state (map, positions as starts, goals), in one
 * launch.  Agents a = 0 .. n_e - 1 (n_e = N on a uniform handle) are planned in index order; agent a takes the
 * earliest-arrival space-time path, waits included, that neither enters a cell a higher-priority agent occupies at that time
 * nor swaps cells with one, and then parks on its goal until the horizon.  Its arrival is the first t <= horizon at which it
 * stands on its goal and no higher-priority agent enters the goal at t or later.  Ties between paths go to the lowest action id
 * when the path is read back from the goal.
 *   d_actions  u8[horizon, B, N]  action ids of environment.py:12; 0 from an agent's arrival on, for absent agents and for a
 *                                 failed environment -- the [T, B, N] layout mapf_env_rollout replays
 *   d_arrival  i32[B, N]          each agent's arrival step; 0 for absent agents; the whole row -1 where some agent finds no
 *                                 path within the horizon (the agents after it are not planned)
 * MAPF_EINVAL for a horizon outside 1 .. MAPF_PLAN_MAX_HORIZON or a NULL buffer, MAPF_ENOMEM if the planner's scratch (per
 * resident warp: six bit tables of horizon + 1 map slices, added to mapf_env_arena_bytes) cannot be allocated.  Reads the
 * handle's state and writes nothing in it; asynchronous on `stream`. */
#define MAPF_PLAN_MAX_HORIZON 1024
int mapf_env_plan_prioritized(mapf_env *env, int32_t horizon, uint8_t *d_actions, int32_t *d_arrival, void *stream);

/* The best of `orders` priority orders per environment.  Order 0 is index order; order r >= 1 sorts the present agents a by
 * (k_a, a), k_a = word 0 of Philox4x32-10 with counter (g_lo, g_hi, 4 | r << 8, a) and key (seed_lo, seed_hi), where
 * g = env_offset + e is the environment's global index -- so a batch sharded over handles plans what one handle would.  Each
 * order is planned as mapf_env_plan_prioritized plans index order, with the agents taken in that order; the environment's
 * result is its solved order of smallest sum of costs, ties to the smallest r.
 *   d_actions  u8[horizon, B, N]  that order's actions, as mapf_env_plan_prioritized writes them
 *   d_arrival  i32[B, N]          that order's arrivals, indexed by agent; 0 for absent agents; the whole row -1 where every
 *                                 order fails (actions 0 there)
 *   d_order    i32[B]             the winning r, -1 where every order fails
 *   d_rank     u8[B, N]           agent a's position in the winning order; 255 for absent agents and failed environments
 * MAPF_EINVAL for a horizon outside 1 .. MAPF_PLAN_MAX_HORIZON, orders outside 1 .. MAPF_PLAN_MAX_ORDERS or a NULL buffer,
 * MAPF_ENOMEM if the planner's scratch (mapf_env_plan_prioritized's, plus 8 bytes per environment) cannot be allocated.
 * Every order is planned once, and the winning one once more to write its results.  Reads the handle's state and writes
 * nothing in it; asynchronous on `stream`. */
#define MAPF_PLAN_MAX_ORDERS 256
int mapf_env_plan_prioritized_orders(mapf_env *env, int32_t horizon, int32_t orders, uint64_t seed, uint64_t env_offset,
                                     uint8_t *d_actions, int32_t *d_arrival, int32_t *d_order, uint8_t *d_rank, void *stream);

/* ---- CBS expert / solvable-instance generator (search.py:58-442, test.py:23-79; SURVEY 8(f)4) -- HOST code ------------------
 * Conflict-based search over space-time A*: a collision-free set of paths of minimal sum of costs (search.py:17-21), as the
 * action script search.find_path returns (search.py:396-442).  All pointers are HOST memory; no kernel is launched.
 *   h_map     u8[L, L]   1 = obstacle                                  (CBSSolver(my_map, ...), search.py:277)
 *   h_starts, h_goals u8[N, 2] (x, y)                                  (env.agents_pos / env.goals_pos, :400-402)
 *   h_dist    i32[N, L, L] or NULL: per-agent distances to the goal, MAPF_DIST_UNREACHABLE where there is no path -- the
 *             optional output of mapf_env_bfs_navi copied to the host (== search.compute_heuristics, :24-55); NULL computes
 *             them here
 *   max_steps            config.max_steps (256): low-level nodes at that timestep are not expanded (search.py:186-187)
 *   time_limit_ms        wall-clock limit of the high-level search (the reference: 5000, search.py:320; 0 = none)
 *   node_limit           high-level nodes expanded at most (>= 1; makes a bounded search reproducible)
 *   h_actions_out u8[max_T, N] action ids of environment.py:12, one row per step, every path padded with stays
 *   T_out     steps of the script (the reference's `opt_steps`, test.py:58); -1: no solution within the limits (find_path
 *             returns None) or longer than max_T
 *   cost_out  (optional) sum of costs; expanded_out (optional) high-level nodes expanded
 * The sum of costs equals the reference's for every instance both solve (CBS is optimal whatever conflict it splits on); the
 * paths are one of several optimal sets: the reference draws the conflict and the constrained agent with random.choice and
 * stops on wall-clock time, here the search is deterministic (first conflict, standard split). */
int mapf_cbs_solve(const uint8_t *h_map, int32_t map_length, int32_t num_agents, const uint8_t *h_starts, const uint8_t *h_goals,
                   const int32_t *h_dist, int32_t max_steps, int32_t time_limit_ms, int64_t node_limit, uint8_t *h_actions_out,
                   int32_t max_T, int32_t *T_out, int32_t *cost_out, int64_t *expanded_out);
/* n instances of one geometry on `threads` host threads (0 = all): arrays as above with a leading dimension n
 * (create_test's loop, test.py:47-58, with the solver calls in parallel). */
int mapf_cbs_solve_batch(int32_t n, const uint8_t *h_maps, int32_t map_length, int32_t num_agents, const uint8_t *h_starts,
                         const uint8_t *h_goals, const int32_t *h_dist, int32_t max_steps, int32_t time_limit_ms, int64_t node_limit,
                         uint8_t *h_actions_out, int32_t max_T, int32_t *T_out, int32_t *cost_out, int64_t *expanded_out,
                         int32_t threads);

#ifdef __cplusplus
}
#endif
#endif /* MAPF_B200_H */
