/*
 * psk_craft.h — C ABI of the B200-native batched Craft environment + BFS teacher.
 *
 * The reference (khanhptnk/psketch) has no FFI: its boundary for this path is the duck-typed
 * Python object API of worlds/craft.py and the teachers/ package.  Every entry point below replaces
 * one reference method, applied to a whole batch of environments whose state lives in HBM as
 * structure-of-arrays tensors; psketch_b200/worlds/craft.py and psketch_b200/teachers/ are the
 * Python-side mirror that binds them (ctypes) and INTEGRATION.md shows the binding a reference
 * maintainer would add.
 *
 * Conventions: every function returns PSK_OK (0) or a PSK_ERR_* code and never throws; all
 * `uint8_t*`/`float*`/... arguments are DEVICE pointers unless the name starts with `host_`;
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); launches are
 * asynchronous on that stream.  Kernel-detected conditions that make the reference raise are
 * OR-ed into `*err_flags` (device int32, may be NULL) as PSK_FLAG_* bits.
 *
 * Domain: 1 <= width, height <= 64 (the agent record stores x and y as bytes; the teacher's boards
 * hold 64 rows of 64 cells), window_w and window_h odd from 1 to 9, 1 <= n_kinds <= 24.  Even windows
 * are outside it: the pooled window has ww^2 + 1 cells per axis, which the reference's block_reduce pads
 * and its features() then rejects by its own length check.  Five geometries have specialised kernels
 * (8x8 / 3, 10x10 / 5 and 16x16, 32x32, 64x64 with a 3x3 window, fused tick and rollout kernels up to
 * 128 cells); every other one runs the generic tier (psk_craft_generic.cu), which reads the geometry
 * from the tables at run time and serves the tick and rollout entry points as separate launches.
 * Same results either way.  Tables outside the domain: PSK_ERR_UNSUPPORTED.
 *
 * Device state layout (one env = one row in each array):
 *   grid  u8[n][cell_stride]   kind id per cell, 0 = free, cell (x, y) at x*height + y
 *                              (the reference's one-hot float64 grid[x, y, kind], craft.py:275-283);
 *                              cell_stride = width*height rounded up to a multiple of 64.
 *   agent u8[n][32]            bytes 0..23 inventory counts by kind id (reference: float64[K]),
 *                              24 x, 25 y, 26 dir, 27 task id, 28 timer, 29..31 reserved.
 */
#ifndef PSK_CRAFT_H
#define PSK_CRAFT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSK_OK 0
#define PSK_ERR_UNSUPPORTED 1 /* tables outside the domain below */
#define PSK_ERR_BADARG 2
#define PSK_ERR_CUDA 3

#define PSK_FLAG_BAD_ACTION 1   /* step(): "Unexpected action" exception, worlds/craft.py:415-416 */
#define PSK_FLAG_INV_OVERFLOW 2 /* an inventory count would exceed 255 (u8 storage) */
#define PSK_FLAG_BAD_LEAF 4     /* teacher: leaf is neither 'use' nor 'go', demonstration.py:18 */
#define PSK_FLAG_OFF_GRID 8     /* reserved, never raised: no kernel checks the agent position.  The
                                   Python entry points (VecCraft, HostCraft) reject positions outside
                                   the grid; a C caller must not pass one (rows would be indexed
                                   outside the env's grid row) */
#define PSK_FLAG_CHAIN_TIMEOUT 16 /* fused kernels: the previous launch on the same envs never finished
                                     (aborted launch / overwritten counters); the kernel went on instead
                                     of hanging, results of that call are not to be trusted */

#define PSK_AGENT_BYTES 32
#define PSK_AG_X 24
#define PSK_AG_Y 25
#define PSK_AG_DIR 26
#define PSK_AG_TASK 27
#define PSK_AG_TIMER 28

#define PSK_MAX_INV 24
#define PSK_MAX_KINDS 32
#define PSK_MAX_RECIPES 16
#define PSK_MAX_TASKS 32
#define PSK_MAX_TASK_NODES 16

#define PSK_ACT_DOWN 0
#define PSK_ACT_UP 1
#define PSK_ACT_LEFT 2
#define PSK_ACT_RIGHT 3
#define PSK_ACT_USE 4
#define PSK_ACT_STOP 5
#define PSK_ACT_INVALID 255 /* expert output where the reference asserts */

/* Domain tables (host struct, passed by pointer; the library keeps a device copy per GPU and
 * refreshes it when the content changes — do the first call with new tables outside a CUDA-graph
 * capture).
 * Replaces: Cookbook (worlds/cookbook.py:7-26), the kind sets of CraftWorld.__init__
 * (worlds/craft.py:101-107) and the hint tree of TaskManager (data/task.py:34-59).
 * Built by psketch_b200/tables.py:CraftTables. */
typedef struct psk_craft_tables {
    int32_t width, height, n_kinds, window_w, window_h;
    int32_t n_recipes, n_tasks;
    int32_t water_kind, stone_kind, bridge_kind, axe_kind;
    int32_t reserved;
    uint8_t kind_class[PSK_MAX_KINDS];                       /* 0 free,1 inert,2 workshop,3 water,4 stone,5 grabbable */
    uint8_t recipes[PSK_MAX_RECIPES][8];                     /* out, workshop, n_in, in0, cnt0, in1, cnt1, yield — firing order */
    uint8_t task_len[PSK_MAX_TASKS];                         /* nodes in the pre-order flattening of each task's hint tree */
    uint8_t task_nodes[PSK_MAX_TASKS][PSK_MAX_TASK_NODES][4]; /* sat class, arg kind, leaf kind, skip_to */
    uint16_t ws_recipes[PSK_MAX_KINDS];                      /* per kind id: bit r set = recipe r is made at this workshop
                                                                (derived from recipes[] by the library on every call — callers may leave it zero) */
} psk_craft_tables;

typedef struct psk_craft_state {
    uint8_t *grid;  /* [n][cell_stride] */
    uint8_t *agent; /* [n][PSK_AGENT_BYTES] */
    int64_t n;
    int32_t cell_stride;
    int32_t reserved;
} psk_craft_state;

/* Where a finished episode restarts from (CraftScenario.init, worlds/craft.py:270-273). */
typedef struct psk_craft_episodes {
    const uint8_t *scen_grid;  /* [n_scen][cell_stride] initial grids (shared between envs) */
    const int32_t *scen_idx;   /* [n] scenario of each env */
    const uint8_t *init_agent; /* [n][32] initial agent record (empty inventory, pos, dir, task, timer) */
} psk_craft_episodes;

/* library / build info: "psketch_b200 <version> sm_100a" */
const char *psk_version(void);
/* Run-time tuning knobs, for tests and same-box A/B runs: every kernel variant the dispatcher can
 * pick by batch size can also be forced.  value -1 = automatic (the default); each knob starts from
 * the environment variable PSK_<KEY IN UPPER CASE>.  Keys:
 *   rollout_variant  CTA shape of craft_rollout_kernel: 0 = 64 env threads + 2 feature warps,
 *                    2 = 32 + 2, 3 = 16 + 2, 4 = 16 + 1
 *   rollout_tma      0 = 128-bit vector stores, 1 = TMA bulk stores (cp.async.bulk)
 *   tile_chain       0 = consecutive fused launches wait for the whole previous grid
 *                    (griddepcontrol.wait); default: per-tile ticket counters (psk_common.cuh)
 *   tick_variant     CTA shape of craft_tick_kernel: 0 = 64+2, 1 = 128+4, 2 = 32+1, 3 = 64+4, 4 = 32+2
 *   tick_tma, tick_persist, feat_persist, tick_pdl,
 *   step_variant     0 = tables staged in shared memory (default), 1 = read-only path, 2 = 1 + row preload
 *   generic          1 = the five built geometries take the generic tier too (no fused tick / rollout)
 * Unknown keys return PSK_ERR_BADARG.  Results never depend on a knob: tests/test_fused_states_gpu.py
 * forces tick_variant, tick_tma, tick_persist, feat_persist, tick_pdl and rollout_variant /
 * rollout_tma on the reference's exported states; tests/test_craft_gpu.py covers step_variant,
 * tile_chain and the rollout variants on dataset rollouts. */
int psk_set_tuning(const char *key, int32_t value);
int psk_get_tuning(const char *key, int32_t *value);

/* number of features of one row (2 * window_w * window_h * n_kinds + n_kinds + 5), or -1 when the
 * tables are outside the domain; psk_craft_supported: 1 inside the domain, else 0 */
int psk_craft_n_features(const psk_craft_tables *t);
int psk_craft_supported(const psk_craft_tables *t);

/* CraftState.step (worlds/craft.py:332-424), in place.  reward (may be NULL) receives 0.0 per
 * env; active (may be NULL) masks envs that must not move (the trainers' `if not done[i]`,
 * trainers/imitation.py:68-72). */
int psk_craft_step(const psk_craft_tables *t, psk_craft_state s, const uint8_t *action,
                   const uint8_t *active, float *reward, int32_t *err_flags, void *stream);

/* CraftState.features (worlds/craft.py:296-330) as float32 (students/imitation.py:72-73):
 * out f32[n][n_features].  impl: 0 = default, 1 = shared-memory tile + 128-bit vector stores,
 * 2 = shared-memory tile + TMA bulk stores (cp.async.bulk). */
int psk_craft_features(const psk_craft_tables *t, psk_craft_state s, float *out, int impl,
                       void *stream);

/* The same feature rows as bytes, u8[n][n_features]: every feature is an exact integer <= 255 (0/1
 * indicators and the u8 inventory counts), so `(float)out[i][j]` IS the reference's value.  A
 * quarter of the f32 frame, for consumers on the far side of PCIe. */
int psk_craft_features_u8(const psk_craft_tables *t, psk_craft_state s, uint8_t *out, void *stream);

/* CraftState.satisfies (worlds/craft.py:285-294): out[i] = 1 True, 0 False, 2 None.
 * task (may be NULL) overrides the task id stored in the agent record. */
int psk_craft_satisfies(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                        uint8_t *out, void *stream);

/* DemonstrationTeacher.__call__ (teachers/demonstration.py:9-30, teachers/base.py:10-87):
 * action u8[n]; dist (may be NULL) i16[n] = BFS path length when a go[...] leaf was searched,
 * else -1. */
int psk_craft_expert(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                     uint8_t *action, int16_t *dist, int32_t *err_flags, void *stream);

/* BaseTeacher.find_closest_resources (teachers/base.py:27-34) for kind[i] (u8[n]):
 * goal u8[n][2] (255,255 if the kind is absent), length i16[n] (-1 = unreachable/None),
 * seq (may be NULL) u8[n][seq_cap] the action sequence padded with 255. */
int psk_craft_find_closest(const psk_craft_tables *t, psk_craft_state s, const uint8_t *kind,
                           uint8_t *goal, int16_t *length, uint8_t *seq, int32_t seq_cap,
                           void *stream);

/* CraftWorld.init_state for every env (worlds/craft.py:258-259): working state <- episode start. */
int psk_craft_reset(psk_craft_state s, psk_craft_episodes ep, const uint8_t *mask, void *stream);

/* One rollout tick for every env — the body of trainers/imitation.py:42-73:
 *     ref = teacher(task, s); f = s.features(); a = action_in ? action_in[i] : ref
 *     timer -= 1; done = (a == STOP) or timer <= 0
 *     done  -> success = s.satisfies(task); s <- episode start (auto-reset)
 *     !done -> s = s.step(a)
 * features_out f32[n][n_features] (may be NULL), expert_out u8[n], done_out/success_out u8[n]
 * (may be NULL), stats u64[4] device accumulators {episodes, successes, env_steps, reserved}
 * (may be NULL).  fused: 0 = three-kernel pipeline, PSK_TICK_FUSED = the single fused kernel,
 * PSK_TICK_ADVANCE_FIRST = the fused kernel in "step, then observe" order — what a policy in the
 * loop needs (students/imitation.py:71-84 reads features, THEN the trainer steps):
 *     action_in ? { timer -= 1; done/success/auto-reset or s = s.step(action_in[i]) } : nothing
 *     ref = teacher(task, s); f = s.features()          <- of the state AFTER the step
 * so one launch per timestep serves  a_t = policy(f_t); tick(a_t) -> f_{t+1}, ref_{t+1}, done_t.
 * In that order done_out / success_out describe the step just applied (0 when action_in is NULL).
 * PSK_TICK_STEP_FIRST = "step, then observe" WITHOUT the episode rules — what the language trainers
 * need (trainers/primitive_language.py:47-70, 93-113: every action of a running env is executed, STOP
 * is a no-op step, a finished env keeps its state for describe / satisfies):
 *     action_in ? s = s.step(action_in[i]) : nothing      <- CraftState.step only
 *     ref = teacher(task, s); f = s.features()          <- of the state AFTER the step
 * The timer byte and stats are not touched; done_out / success_out (may be NULL) are written as 0.
 * A bad action byte raises PSK_FLAG_BAD_ACTION and leaves the env as it was (as psk_craft_step). */
#define PSK_TICK_PIPELINE 0
#define PSK_TICK_FUSED 1
#define PSK_TICK_ADVANCE_FIRST 2
#define PSK_TICK_STEP_FIRST 3
int psk_craft_tick(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                   const uint8_t *action_in, float *features_out, uint8_t *expert_out,
                   uint8_t *done_out, uint8_t *success_out, unsigned long long *stats,
                   int32_t *err_flags, int fused, void *stream);

/* Testing hook (fault injection for PSK_FLAG_CHAIN_TIMEOUT): takes one ticket of the chaining group
 * that owns env `env` of this batch and never finishes it, like an aborted launch would.  The next
 * fused launch on these envs raises PSK_FLAG_CHAIN_TIMEOUT after a few seconds instead of hanging;
 * the one after that runs normally.  PSK_ERR_UNSUPPORTED if the batch does not chain. */
int psk_debug_chain_skip_ticket(psk_craft_state s, int64_t env, void *stream);

/* psk_craft_tick with the feature rows as bytes (features_out u8[n][n_features], see
 * psk_craft_features_u8) — same fused kernel, a quarter of the output traffic; order =
 * PSK_TICK_FUSED, PSK_TICK_ADVANCE_FIRST or PSK_TICK_STEP_FIRST. */
int psk_craft_tick_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                      const uint8_t *action_in, uint8_t *features_out, uint8_t *expert_out,
                      uint8_t *done_out, uint8_t *success_out, unsigned long long *stats,
                      int32_t *err_flags, int order, void *stream);

/* `ticks` consecutive rollout ticks in ONE launch (same per-tick semantics as psk_craft_tick):
 * every CTA keeps its envs' state in shared memory across the ticks, so HBM sees one state read,
 * one state write and `ticks` output frames.  For rollouts whose actions do not depend on
 * anything outside the kernel: teacher-driven (action_in NULL) or replay of action_in u8[ticks][n].
 * expert_out u8[ticks][n]; done_out / success_out u8[ticks][n] (may be NULL); features_out
 * f32[feat_ring][n][n_features] (may be NULL), tick t writes slot t % feat_ring. */
int psk_craft_rollout(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                      int32_t ticks, const uint8_t *action_in, float *features_out,
                      int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                      uint8_t *success_out, unsigned long long *stats, int32_t *err_flags,
                      void *stream);

/* psk_craft_rollout with byte frames: features_out u8[feat_ring][n][n_features]. */
int psk_craft_rollout_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                         int32_t ticks, const uint8_t *action_in, uint8_t *features_out,
                         int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                         uint8_t *success_out, unsigned long long *stats, int32_t *err_flags,
                         void *stream);

/* The Philox streams of the three sampler entry points below.  Generator: Philox4x32-10 (Salmon
 * et al., SC'11).  Stream (seed, s) at counter start c has key = (seed lo, seed hi) and counter words
 * (c lo, c hi, s lo, s hi); word 0 is incremented after each 4-word block, carrying into word 1 (not
 * into the stream words).  A block's words are consumed out[3], out[2], out[1], out[0], and a draw
 * below n is (u64(word) * n) >> 32.  random_free draws x, then y, and rejects an occupied cell.
 * Every output depends only on (seed, stream, counter), never on the launch geometry or the GPU;
 * oracle/sampler_oracle.c restates all of it and the tests compare it byte for byte.
 *
 * Shared blocks: the random actions of env e at clock t are the first word of block t of stream
 * (seed, e), which is the block of scenario e's (t+1)-th refill (offset 0).  With equal seeds (both
 * default to 123) the two sources are therefore correlated; generate_dataset separates its start
 * cells from its scenarios by XOR-ing the seed. */

/* Scenario sampling (make_data.py:74-144, `random_free` / `sample_scenario`): boundary ring, then
 * place_kinds[0..n_place) in order, then the agent, each at a uniformly random free cell that keeps
 * all free cells connected (reachable from the lowest-index free cell) and every occupied interior
 * cell next to a free cell, 4,096 draws at most.  Kind ids must be 1..n_kinds-1.
 * scen_grid u8[n][cell_stride] (cell x * H + y, the tail past W * H zeroed), init_pos u8[n][2].
 * A scenario that runs out of draws keeps the items placed so far, gets init_pos (0, 0) and counts
 * in *fail_count (device, may be NULL).  Scenario i uses stream (seed, i + offset), counter start 0. */
int psk_craft_sample_scenarios(const psk_craft_tables *t, uint8_t *scen_grid, uint8_t *init_pos,
                               const uint8_t *place_kinds, int32_t n_place, int32_t boundary_kind,
                               uint64_t seed, uint64_t offset, int64_t n, int32_t cell_stride,
                               int32_t *fail_count, void *stream);

/* Uniform random actions for off-policy rollouts: out[e] in [0, n_actions) (1..255 actions) is the
 * first draw of stream (seed, e) at counter start t + *t_dev (mod 2^64): counter words 0-1 hold the
 * clock, words 2-3 the env.  t_dev (device, may be NULL) lets a counter that lives on the device
 * (e.g. stats[2], the env-step count) advance the clock under CUDA-graph replay. */
int psk_random_actions(uint8_t *out, int64_t n, int32_t n_actions, uint64_t seed, uint64_t t,
                       const unsigned long long *t_dev, void *stream);
/* The same for `ticks` consecutive clocks at once: out u8[ticks][n], row k = the actions of clock
 * t + k — the action_in block of a psk_craft_rollout launch (off-policy rollouts, `ticks` per launch). */
int psk_random_actions_block(uint8_t *out, int64_t n, int32_t ticks, int32_t n_actions, uint64_t seed,
                             uint64_t t, const unsigned long long *t_dev, void *stream);

/* Dataset instance positions (make_data.py:203-208): per group, `per_group` distinct uniformly
 * random free cells of scenario group_scen[g] (a row index the caller guarantees is in range);
 * out_pos u8[n_groups][per_group][2].  Group g uses stream (seed, g + offset), counter start 1,
 * 65,536 draws at most per slot; a slot that runs out is 255/255 and counts in *fail_count, and the
 * next slot continues from the same generator state.  cell_stride >= W * H. */
int psk_craft_sample_positions(const psk_craft_tables *t, const uint8_t *scen_grid,
                               const int32_t *group_scen, int32_t per_group, uint8_t *out_pos,
                               uint64_t seed, uint64_t offset, int64_t n_groups,
                               int32_t cell_stride, int32_t *fail_count, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Host-buffer entry points: the caller keeps its environments in HOST memory, as the reference
 * does (every CraftState is a CPU object).  All pointers below are HOST pointers; pass pinned
 * memory (psk_host_alloc) so that the copies overlap with the kernels.  Chunks of the batch are
 * pipelined over several streams:  H2D(state) -> fused tick -> D2H(features, actions, state). */
typedef struct psk_craft_host_ctx psk_craft_host_ctx;

void *psk_host_alloc(size_t bytes); /* pinned host memory, NULL on failure */
void psk_host_free(void *p);

int psk_craft_host_create(const psk_craft_tables *t, int64_t max_envs, int64_t chunk_envs,
                          psk_craft_host_ctx **out);
void psk_craft_host_destroy(psk_craft_host_ctx *ctx);

/* Episode starts (same meaning as psk_craft_episodes), uploaded once and kept on the device. */
int psk_craft_host_set_episodes(psk_craft_host_ctx *ctx, const uint8_t *host_scen_grid,
                                int64_t n_scen, const int32_t *host_scen_idx,
                                const uint8_t *host_init_agent, int64_t n);

/* psk_craft_tick over host arrays: host_grid u8[n][cell_stride] and host_agent u8[n][32] are
 * read and overwritten with the new state; host_features f32[n][n_features] (may be NULL),
 * host_expert u8[n], host_done / host_success u8[n] (may be NULL), host_action_in u8[n] (may be
 * NULL = follow the teacher), host_stats u64[4] and host_err_flags (may be NULL) receive the
 * running episode statistics and the PSK_FLAG_* bits.  Returns after everything has landed. */
int psk_craft_host_tick(psk_craft_host_ctx *ctx, uint8_t *host_grid, uint8_t *host_agent,
                        const uint8_t *host_action_in, float *host_features,
                        uint8_t *host_expert, uint8_t *host_done, uint8_t *host_success,
                        int64_t n, unsigned long long *host_stats, int32_t *host_err_flags);

/* Resident mode of the host-buffer path.  A rollout's caller (trainers/imitation.py:42-77) only
 * consumes features, teacher actions and the done / success flags, and only produces actions: the
 * environments themselves can stay in HBM between ticks.  psk_craft_host_reset puts every env at its
 * episode start (world.init_state for the batch, trainers/imitation.py:26); put/get_state move
 * whole states when the caller wants them (state.pos / state.inventory for describe(),
 * teachers/primitive_language.py:60-66).  psk_craft_host_tick_resident = psk_craft_host_tick
 * without the state copies: H2D host_action_in u8[n] (NULL = follow the teacher), D2H the feature
 * frame in `feature_format` (host_features f32[n][nf] or u8[n][nf], NULL/NONE = no features), the
 * teacher actions and flags.  advance_first != 0: "step, then observe" (PSK_TICK_ADVANCE_FIRST) — the
 * host-in-the-loop form: the actions the host chose from the previous call's features go up, the
 * step is applied, and the features / teacher actions of the NEW states come down. */
#define PSK_FEATURES_NONE 0
#define PSK_FEATURES_F32 1
#define PSK_FEATURES_U8 2
/* host_features is f32[n][nf] exactly as with PSK_FEATURES_F32, but PCIe carries the u8 frame: it
 * lands in a pinned buffer the context owns and host threads (env PSK_HOST_THREADS, default
 * min(8, cores / 2) including the caller) widen each chunk into host_features while the next chunk
 * is in flight.  host_features need not be pinned.  psk_craft_host_set_threads: the number of
 * widening threads, the caller included (>= 1; several contexts on one box should share the cores);
 * psk_craft_host_threads: threads in use (0 before the first such call).  A host context is not
 * thread-safe: one thread at a time may call into it.
 * Split frame: when host_features IS pinned, the last d of a call's chunks cross PCIe as f32, straight
 * into host_features, while the host threads are still widening the byte chunks before them — the
 * copy engine's spare time is worth that many chunks of host work.  d follows the two measured rates
 * from call to call (d* = chunks (w - p) / (w + 3 p), w / p = widening / wire time per byte chunk;
 * 0 on hosts that widen faster than PCIe delivers).  psk_craft_host_set_wire_direct: fix d (>= 0),
 * or -1 = adaptive again (the default; env PSK_WIRE_DIRECT sets the initial choice);
 * psk_craft_host_wire_direct: the d the next call will use.  The host frame is the same either way.
 * psk_host_widen_u8_f32: the widening alone (dst[i] = src[i]) for callers that keep
 * PSK_FEATURES_U8 frames; no CUDA call. */
#define PSK_FEATURES_F32_WIRE_U8 3
int psk_craft_host_threads(const psk_craft_host_ctx *ctx);
int psk_craft_host_set_threads(psk_craft_host_ctx *ctx, int32_t threads);
/* Small batches (n <= max_envs, default 2048, env PSK_HOST_ZEROCOPY_MAX; 0 = never): when every buffer
 * of a psk_craft_host_tick_resident call is pinned, the fused kernel reads the actions from and writes
 * features / teacher actions / flags into the caller's memory itself (unified addressing): one launch and
 * one synchronize per call instead of a copy per buffer — the reference's own batch size is 32
 * (configs/experiments/imitation.yaml:17); measured 44 -> 31 us per call at 32 envs, 108 -> 91 at 2,048
 * (profiles/bench_runs/r2_host_small_batch_probe.json).  Same results; pageable buffers take the copy
 * route. */
int psk_craft_host_set_zerocopy_max(psk_craft_host_ctx *ctx, int64_t max_envs);
int psk_craft_host_wire_direct(const psk_craft_host_ctx *ctx);
/* Testing hook: the split rule on its own (no CUDA call).  Given a call of `chunks` chunks that sent d
 * as f32, whose last byte landed t_pcie_us and whose widening ended t_widen_us after its start, returns the
 * d of the next call; *p_us / *w_us hold the smoothed per-chunk rates between calls (start them at 0). */
int psk_debug_wire_split_next(int chunks, int d, double t_pcie_us, double t_widen_us, double *p_us,
                              double *w_us);
int psk_craft_host_set_wire_direct(psk_craft_host_ctx *ctx, int32_t chunks);
int psk_host_widen_u8_f32(const uint8_t *src, float *dst, size_t n, int threads);
int psk_craft_host_reset(psk_craft_host_ctx *ctx, int64_t n);
int psk_craft_host_put_state(psk_craft_host_ctx *ctx, const uint8_t *host_grid,
                             const uint8_t *host_agent, int64_t n);
int psk_craft_host_get_state(psk_craft_host_ctx *ctx, uint8_t *host_grid, uint8_t *host_agent,
                             int64_t n);
int psk_craft_host_tick_resident(psk_craft_host_ctx *ctx, const uint8_t *host_action_in,
                                 void *host_features, int32_t feature_format, int32_t advance_first,
                                 uint8_t *host_expert, uint8_t *host_done, uint8_t *host_success,
                                 int64_t n, unsigned long long *host_stats, int32_t *host_err_flags);

#ifdef __cplusplus
}
#endif
#endif /* PSK_CRAFT_H */
