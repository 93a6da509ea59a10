/*
 * psk_light.h — C ABI of the batched Light world (rooms / doors / keys), worlds/light.py.
 *
 * Replaces, for N environments per launch: LightState.step (worlds/light.py:212-235),
 * LightState.features (:191-204), LightState.satisfies (:208-210) and LightScenario.init
 * (:175-180).  The reference has no teacher for this world; psk_light_expert is specified here
 * (shortest action sequence over (position, remaining keys) to the goal room, ties broken by
 * the smallest action index) and validated against a brute-force search, not against psketch.
 *
 * Same conventions as psk_craft.h: DEVICE pointers, void* cudaStream_t, int status codes.
 * Scenario tables are shared between environments (scen_idx selects one per env).
 */
#ifndef PSK_LIGHT_H
#define PSK_LIGHT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSK_LIGHT_MAX_BOARD 32
#define PSK_LIGHT_MAX_DOORS 8
#define PSK_LIGHT_MAX_KEYS 8
#define PSK_LIGHT_N_FEATURES 12
#define PSK_LIGHT_N_ACTIONS 5 /* DOWN, UP, LEFT, RIGHT, USE */
#define PSK_LIGHT_ROOM 6      /* ROOM_W = ROOM_H = 6, worlds/light.py:11-12 */

/* One scenario (LightScenario, worlds/light.py:163-173), 192 bytes. */
typedef struct psk_light_scenario {
    uint32_t walls[PSK_LIGHT_MAX_BOARD];   /* row x: bit y set = wall (cells beyond the board are walls) */
    uint8_t doors[PSK_LIGHT_MAX_DOORS][2]; /* x, y */
    uint8_t keys[PSK_LIGHT_MAX_KEYS][4];   /* key x, key y, door x, door y (the scenario's initial key set) */
    uint8_t n_doors, n_keys, board_w, board_h;
    uint8_t goal_rx, goal_ry, init_x, init_y;
    uint8_t reserved[8];
} psk_light_scenario;

/* Per-env state u8[n][4]: x, y, bitmask of keys still on the map, reserved.
 * Several keys may lie on one cell (the reference's dict of keys cannot hold that): one USE on the
 * cell picks up every key lying there, in psk_light_step, the fused tick and both teachers.  A key
 * locks its target cell only if a door stands there (worlds/light.py:233); one aimed at any other
 * cell locks nothing. */
#define PSK_LIGHT_STATE_BYTES 4

int psk_light_reset(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                    const uint8_t *mask, int64_t n, void *stream);
int psk_light_step(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                   const uint8_t *action, const uint8_t *active, float *reward,
                   int32_t *err_flags, int64_t n, void *stream);
int psk_light_features(const psk_light_scenario *scen, const int32_t *scen_idx,
                       const uint8_t *state, float *out, int64_t n, void *stream);
int psk_light_satisfies(const psk_light_scenario *scen, const int32_t *scen_idx,
                        const uint8_t *state, uint8_t *out, int64_t n, void *stream);
/* action u8[n] (255 = goal room unreachable, 254 = already in the goal room), dist i16[n].
 * max_keys: the largest n_keys among the scenarios used (sizes the per-warp shared memory).  An env
 * whose scenario has more keys than max_keys, or whose key mask has a bit at or above its scenario's
 * n_keys, is not searched: action 255, dist -2. */
int psk_light_expert(const psk_light_scenario *scen, const int32_t *scen_idx,
                     const uint8_t *state, uint8_t *action, int16_t *dist, int32_t max_keys,
                     int64_t n, void *stream);

/* The teacher as a table.  Its answer depends only on (scenario, x, y, keys on the map) — at most
 * 32 x 32 x 2^n_keys states per scenario, shared by all envs of the scenario — so the backward
 * flood of psk_light_expert runs once per scenario (one CTA each) and every later query is ONE byte
 * load.  Per scenario the table holds u16[1 << max_keys][32][32] — fewest actions to the goal room
 * from cell (x, y) with key subset m on the map, 0xFFFF = unreachable — followed by three u8[32][32]
 * per-cell maps (keys locking the door here, keys lying here, doors here) that replace the door / key
 * loops of step and features in the fused tick, and by u8[1 << max_keys][32][32]: the teacher's action
 * for every state, derived from the distances when the table is built;
 * psk_light_teacher_table_bytes gives the total size.  psk_light_expert_table answers like
 * psk_light_expert (same actions, same dist).  A scenario with more keys than max_keys gets no flood
 * (its table says 254 in the goal room, 255 elsewhere), and a key mask with no layer in the table
 * (mask >= 1 << max_keys: such a scenario's envs after reset, or mask bits the scenario does not
 * have) answers 255 / dist -2 in psk_light_expert_table, psk_light_tick and psk_light_rollout;
 * no lookup reads outside its scenario's block.
 * Tested against oracle/light_oracle.c (tests/test_light.py on the reference's 60 scenarios,
 * tests/test_light_limits_gpu.py on every state of generator draws of all 17 goals up to 7 keys and
 * of synthetic scenarios up to 8 keys / 8 doors / 31 x 31 with shared doors and shared key cells). */
int64_t psk_light_teacher_table_bytes(int64_t n_scen, int32_t max_keys);
int psk_light_teacher_build(const psk_light_scenario *scen, int64_t n_scen, int32_t max_keys,
                            uint16_t *table, void *stream);
int psk_light_expert_table(const psk_light_scenario *scen, const int32_t *scen_idx, const uint8_t *state,
                           const uint16_t *table, int32_t max_keys, uint8_t *action, int16_t *dist,
                           int64_t n, void *stream);

/* One rollout tick for every env, the Craft tick's contract (psk_craft_tick) on this world:
 *     ref = teacher(s); f = s.features(); a = action_in ? action_in[i] : ref
 *     elapsed += 1; done = a not in 0..4 (teacher: 254 already in the goal room, 255 unreachable)
 *                          or elapsed >= max_timesteps
 *     done -> success = s.satisfies(goal); s <- LightScenario.init()       !done -> s = s.step(a)
 * state byte 3 counts the steps of the running episode (0 after psk_light_reset).  features_out
 * f32[n][12] (may be NULL), expert_out u8[n], done_out / success_out u8[n] (may be NULL), stats
 * u64[4] {episodes, successes, env_steps, reserved} (may be NULL). */
int psk_light_tick(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                   const uint16_t *table, int32_t max_keys, const uint8_t *action_in,
                   float *features_out, uint8_t *expert_out, uint8_t *done_out, uint8_t *success_out,
                   unsigned long long *stats, int32_t max_timesteps, int64_t n, void *stream);

/* `ticks` ticks in ONE launch (the contract of psk_craft_rollout on this world): tick t reads
 * action_in[t][n] (NULL = follow the teacher), writes expert_out[t][n], done_out[t][n] / success_out[t][n]
 * (may be NULL) and the feature frame (t % feat_ring) of features_out f32[feat_ring][n][12] (may be
 * NULL).  The final states equal `ticks` calls of psk_light_tick. */
int psk_light_rollout(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                      const uint16_t *table, int32_t max_keys, int32_t ticks, const uint8_t *action_in,
                      float *features_out, int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                      uint8_t *success_out, unsigned long long *stats, int32_t max_timesteps, int64_t n,
                      void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PSK_LIGHT_H */
