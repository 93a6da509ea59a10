// psk_light.cu — batched Light world (worlds/light.py): step, features, satisfies, reset, and a
// warp-cooperative shortest-path teacher over (position, remaining keys).
#include "psk_common.cuh"
#include "../../include/psk_light.h"

// Resident blocks of 256 threads per SM asked of the compiler (same-box A/B at 1 M envs,
// profiles/README.md): the table lookup alone gains from 8 (32 registers: 6.25 -> 5.45 us); the fused
// tick is best at 6 (42 registers: 15.5 us; natural 56 registers 17.95, 5 blocks 16.8, 8 blocks spill:
// 18.4), the rollout at 5 (11.5 us per tick; natural 12.4, 6 blocks 11.6, 8 blocks 12.8).
#ifndef PSK_LIGHT_MINBLOCKS
#define PSK_LIGHT_MINBLOCKS 6
#endif
#ifndef PSK_LIGHT_ROLLOUT_MINBLOCKS
#define PSK_LIGHT_ROLLOUT_MINBLOCKS 5
#endif
#ifndef PSK_LIGHT_LOOKUP_MINBLOCKS
#define PSK_LIGHT_LOOKUP_MINBLOCKS 8
#endif
#ifndef PSK_LIGHT_COALESCED
#define PSK_LIGHT_COALESCED 1
#endif

namespace psk {

__device__ __forceinline__ bool light_wall(const psk_light_scenario &s, int x, int y) {
    if (x < 0 || y < 0 || x >= PSK_LIGHT_MAX_BOARD || y >= PSK_LIGHT_MAX_BOARD) return true;
    return (s.walls[x] >> y) & 1;
}

// is (x, y) a door whose key is still on the map?  (worlds/light.py:233)
__device__ __forceinline__ bool light_locked_door(const psk_light_scenario &s, int x, int y,
                                                  uint32_t alive) {
    bool is_door = false;
    for (int d = 0; d < s.n_doors; d++) is_door |= (s.doors[d][0] == x && s.doors[d][1] == y);
    if (!is_door) return false;
    for (int k = 0; k < s.n_keys; k++)
        if (((alive >> k) & 1) && s.keys[k][2] == x && s.keys[k][3] == y) return true;
    return false;
}

// keys whose target cell is a door: only those lock anything (light_locked_door); a key aimed at
// any other cell is still picked up but opens nothing
__device__ __forceinline__ uint32_t light_door_keys(const psk_light_scenario &s) {
    uint32_t r = 0;
    for (int k = 0; k < s.n_keys; k++)
        for (int d = 0; d < s.n_doors; d++)
            if (s.keys[k][2] == s.doors[d][0] && s.keys[k][3] == s.doors[d][1]) r |= 1u << k;
    return r;
}

__global__ void __launch_bounds__(256)
light_reset_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                   uint8_t *__restrict__ state, const uint8_t *__restrict__ mask, int64_t n) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[e]) continue;
        const psk_light_scenario &s = scen[scen_idx[e]];
        // LightScenario.init: centre of the initial room, every key on the map (light.py:175-180)
        const uint32_t alive = s.n_keys >= 8 ? 0xFFu : ((1u << s.n_keys) - 1u);
        reinterpret_cast<uint32_t *>(state)[e] = uint32_t(s.init_x) | (uint32_t(s.init_y) << 8) | (alive << 16);
    }
}

__global__ void __launch_bounds__(256)
light_step_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                  uint8_t *__restrict__ state, const uint8_t *__restrict__ action,
                  const uint8_t *__restrict__ active, float *__restrict__ reward,
                  int32_t *err_flags, int64_t n) {
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        if (reward) reward[e] = 0.0f;                       // light.py:235
        if (active && !active[e]) continue;
        const psk_light_scenario &s = scen[scen_idx[e]];
        const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
        const int x = st & 0xFF, y = (st >> 8) & 0xFF;
        const uint32_t alive = (st >> 16) & 0xFF;
        uint32_t n_alive = alive;
        const int a = action[e];
        int dx = 0, dy = 0;
        if (a < 4) {                                        // light.py:216-223
            dx = dx_of(a);
            dy = dy_of(a);
        } else if (a == 4) {                                // USE: pick up the key underfoot (:224-228)
            for (int k = 0; k < s.n_keys; k++)
                if (((alive >> k) & 1) && s.keys[k][0] == x && s.keys[k][1] == y) n_alive &= ~(1u << k);
        } else {
            flags |= PSK_FLAG_BAD_ACTION;                   // the reference fails with UnboundLocalError
            continue;
        }
        int nx = x + dx, ny = y + dy;
        if (light_wall(s, nx, ny)) { nx = x; ny = y; }      // light.py:231-232
        // doors are tested against the keys BEFORE this step's pick-up (light.py:233 uses self.keys)
        if (light_locked_door(s, nx, ny, alive)) { nx = x; ny = y; }
        reinterpret_cast<uint32_t *>(state)[e] = uint32_t(nx) | (uint32_t(ny) << 8) | (n_alive << 16) |
                                                 (st & 0xFF000000u);   // byte 3: psk_light_tick's step counter
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// worlds/light.py:191-204 with the precomputed maps of :105-146.  `strength //= 10` leaves 1.0
// only at distance 0, so a door/key contributes (1,1,1,1) exactly when the agent stands on it:
// locked doors -> out[0:4], open doors -> out[4:8], keys still on the map -> out[8:12].
__global__ void __launch_bounds__(256)
light_features_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                      const uint8_t *__restrict__ state, float *__restrict__ out, int64_t n) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        const psk_light_scenario &s = scen[scen_idx[e]];
        const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
        const int x = st & 0xFF, y = (st >> 8) & 0xFF;
        const uint32_t alive = (st >> 16) & 0xFF;
        float locked = 0.f, open = 0.f, key = 0.f;
        for (int d = 0; d < s.n_doors; d++) {
            if (s.doors[d][0] != x || s.doors[d][1] != y) continue;
            bool lk = false;
            for (int k = 0; k < s.n_keys; k++)
                lk |= ((alive >> k) & 1) && s.keys[k][2] == x && s.keys[k][3] == y;
            if (lk) locked += 1.f; else open += 1.f;
        }
        for (int k = 0; k < s.n_keys; k++)
            if (((alive >> k) & 1) && s.keys[k][0] == x && s.keys[k][1] == y &&
                x % PSK_LIGHT_ROOM != 0 && y % PSK_LIGHT_ROOM != 0)
                key += 1.f;
        float4 *o = reinterpret_cast<float4 *>(out + e * PSK_LIGHT_N_FEATURES);
        o[0] = make_float4(locked, locked, locked, locked);
        o[1] = make_float4(open, open, open, open);
        o[2] = make_float4(key, key, key, key);
    }
}

__global__ void __launch_bounds__(256)
light_satisfies_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                       const uint8_t *__restrict__ state, uint8_t *__restrict__ out, int64_t n) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        const psk_light_scenario &s = scen[scen_idx[e]];
        const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
        const int x = st & 0xFF, y = (st >> 8) & 0xFF;
        out[e] = (x / PSK_LIGHT_ROOM == s.goal_rx) && (y / PSK_LIGHT_ROOM == s.goal_ry);   // light.py:208-210
    }
}

// ---------------------------------------------------------------------------------------------
// Teacher (specified here; the reference has none for this world): fewest actions from
// (pos, keys) to any cell of the goal room, where a move costs 1 and picking up a key (USE on the
// key's cell) costs 1 and unlocks its door; the first action of the best plan, ties -> smallest
// action index (DOWN, UP, LEFT, RIGHT, USE).
//
// One WARP per env.  Lane x holds row x of every board as a 32-bit word (boards are <= 31 x 31):
// vertical moves are bit shifts inside the lane, horizontal moves are __shfl_up/down_sync between
// lanes, emptiness tests are __ballot_sync.  The search runs BACKWARD from the goal room over the
// layers "key subset still on the map" (<= 2^n_keys layers, kept in shared memory): R[m] = cells
// from which the goal is reachable within the current number of steps when the keys in m are still
// lying around.  A level adds to R[m]: the passable neighbours of R[m] (a move), and every key
// cell k in m whose lower layer R[m \ {k}] already contains it (USE).  The first level at which
// the agent's cell enters R[alive] is the distance; the action is the smallest a whose successor
// state was in R one level earlier.

__global__ void __launch_bounds__(128)
light_expert_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                    const uint8_t *__restrict__ state, uint8_t *__restrict__ action,
                    int16_t *__restrict__ dist_out, int64_t n, int layer_cap) {
    extern __shared__ uint32_t s_layers[];          // [warps][2][n_layers_cap][32]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    constexpr unsigned FULL = 0xffffffffu;
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const psk_light_scenario &s = scen[scen_idx[e]];
        const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
        const int px = st & 0xFF, py = (st >> 8) & 0xFF;
        const uint32_t alive = (st >> 16) & 0xFF;
        const int nk = s.n_keys;
        const int n_layers = 1 << nk;
        // the scenario has more keys than the caller announced, or the mask names keys it does not have
        if (n_layers > layer_cap || alive >= (uint32_t)n_layers) {
            if (lane == 0) {
                action[e] = 255;
                if (dist_out) dist_out[e] = -2;
            }
            continue;
        }
        uint32_t *R = s_layers + (size_t)warp * 2 * layer_cap * 32;   // reached so far
        uint32_t *P = R + layer_cap * 32;                             // reached one level earlier
        const uint32_t wall_row = s.walls[lane];
        // goal room rows / cells
        uint32_t goal_row = 0;
        if (lane / PSK_LIGHT_ROOM == s.goal_rx)
            goal_row = (0x3Fu << (s.goal_ry * PSK_LIGHT_ROOM)) & ~wall_row;
        // locked-door cells per layer are recomputed on the fly: door d is locked in layer m if a
        // key of m points at it
        const uint32_t door_keys = light_door_keys(s);
        if (((py < 32) && ((__shfl_sync(FULL, goal_row, px & 31) >> py) & 1))) {
            if (lane == 0) {
                action[e] = 254;
                if (dist_out) dist_out[e] = 0;
            }
            continue;
        }
        for (int m = 0; m < n_layers; m++) {
            // a cell of the goal room that is a locked door in layer m cannot be stood on
            uint32_t lockrow = 0;
            for (int k = 0; k < nk; k++)
                if ((((m & door_keys) >> k) & 1) && s.keys[k][2] == lane) lockrow |= 1u << s.keys[k][3];
            R[m * 32 + lane] = goal_row & ~lockrow;
            P[m * 32 + lane] = 0;
        }
        // byte k: the keys lying on key k's cell, for the keys in this lane's row (0 for the others)
        uint64_t same_cell = 0;
        for (int k = 0; k < nk; k++)
            for (int j = 0; j < nk; j++)
                if (s.keys[k][0] == lane && s.keys[j][0] == lane && s.keys[j][1] == s.keys[k][1])
                    same_cell |= 1ull << (8 * k + j);
        __syncwarp();
        int found = -1;
        const int max_levels = 32 * 32 + 64;
        for (int level = 1; level <= max_levels; level++) {
            bool grew = false;
            // only layers that are subsets of `alive` can be reached from the current state
            for (int m = 0; m < n_layers; m++) {
                if ((m & ~alive) != 0) continue;
                uint32_t lockrow = 0;
                for (int k = 0; k < nk; k++)
                    if ((((m & door_keys) >> k) & 1) && s.keys[k][2] == lane) lockrow |= 1u << s.keys[k][3];
                const uint32_t pass = ~wall_row & ~lockrow;      // cells one may stand on in layer m
                const uint32_t cur = R[m * 32 + lane];
                P[m * 32 + lane] = cur;
                // predecessors by a move: p -> p+delta in R, p itself passable (agent stands there)
                const uint32_t up = __shfl_up_sync(FULL, cur, 1), dn = __shfl_down_sync(FULL, cur, 1);
                uint32_t add = (cur << 1) | (cur >> 1) | (lane > 0 ? up : 0u) | (lane < 31 ? dn : 0u);
                // predecessors by USE: standing on key k (in m) with R[m \ gone] containing the cell,
                // where gone = the keys lying on that cell (one USE picks up every key of m there)
                for (int k = 0; k < nk; k++) {
                    const uint32_t gone = (uint32_t)(same_cell >> (8 * k)) & 0xFFu;
                    if (!((m >> k) & 1) || !gone) continue;
                    const uint32_t bit = 1u << s.keys[k][1];
                    // lower layer as of the PREVIOUS level: layers are swept in increasing m and
                    // m \ gone < m was already advanced this level, so read its snapshot P
                    if (P[(m & ~gone) * 32 + lane] & bit) add |= bit;
                }
                const uint32_t nxt = cur | (add & pass);
                R[m * 32 + lane] = nxt;
                grew |= nxt != cur;
            }
            __syncwarp();
            const uint32_t mine = __shfl_sync(FULL, R[alive * 32 + lane], px & 31);
            if ((mine >> py) & 1) { found = level; break; }
            if (!__any_sync(FULL, grew)) break;
        }
        if (found < 0) {
            if (lane == 0) {
                action[e] = 255;
                if (dist_out) dist_out[e] = -1;
            }
            continue;
        }
        // first action: smallest a whose successor was reached one level earlier (snapshot P)
        int best = 255;
        if (lane == 0) {
            for (int a = 0; a < 5 && best == 255; a++) {
                int nx = px, ny = py;
                uint32_t m2 = alive;
                if (a < 4) {
                    nx = px + dx_of(a);
                    ny = py + dy_of(a);
                    if (light_wall(s, nx, ny) || light_locked_door(s, nx, ny, alive)) continue;  // no progress
                } else {
                    for (int k = 0; k < nk; k++)
                        if (((alive >> k) & 1) && s.keys[k][0] == px && s.keys[k][1] == py) m2 &= ~(1u << k);
                    if (m2 == alive) continue;
                }
                const uint32_t *L = (found == 1) ? nullptr : P;
                bool ok;
                if (found == 1) {
                    // successor must be in the goal room itself
                    ok = (nx / PSK_LIGHT_ROOM == s.goal_rx) && (ny / PSK_LIGHT_ROOM == s.goal_ry);
                } else {
                    ok = (L[m2 * 32 + nx] >> ny) & 1;
                }
                if (ok) best = a;
            }
            action[e] = (uint8_t)best;
            if (dist_out) dist_out[e] = (int16_t)found;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// Teacher as a table.  The teacher's answer is a function of (scenario, x, y, keys on the map), a
// state space of at most 32 x 32 x 2^n_keys per scenario, shared by every env of that scenario — so
// instead of one search per env and query (light_expert_kernel above: 8.4 ms per 65,536 envs) the
// backward flood runs ONCE per scenario and records, for every key subset m and cell, the level at
// which the cell entered R[m]: dist u16[n_scen][2^max_keys][32][32] (0xFFFF = goal room unreachable).
// One CTA per scenario; warp w sweeps the layers m = w, w + 8, ...; lane x holds row x; all layers
// advance level by level (Jacobi: a level reads only the previous level's boards, double-buffered in
// shared memory), one __syncthreads_or per level.  A query is then a handful of loads.
// Per-scenario block of the teacher table: dist u16[layer_cap][32][32], then three per-cell byte maps
// that turn the door / key loops of step, features and the teacher query into single loads:
//   cell_lock[x*32+y]   bitmask of the keys that lock the door at this cell (0: no door here)
//   cell_keys[x*32+y]   bitmask of the keys lying on this cell
//   cell_doors[x*32+y]  number of doors at this cell
// and last the teacher's ANSWER per state, so that a query is one byte load instead of six distance
// loads and their wall / lock tests:
//   act u8[layer_cap][32][32]   254 in the goal room, 255 unreachable, else the first action
#define PSK_LIGHT_AUX_BYTES (3 * 1024)
__host__ __device__ constexpr size_t light_block_u16(int layer_cap) {
    return (size_t)layer_cap * 1024 + PSK_LIGHT_AUX_BYTES / 2 + (size_t)layer_cap * 512;
}
struct LightAux {
    const uint8_t *lock, *keys, *doors, *act;
    __device__ __forceinline__ LightAux(const uint16_t *block, int layer_cap) {
        lock = reinterpret_cast<const uint8_t *>(block + (size_t)layer_cap * 1024);
        keys = lock + 1024;
        doors = keys + 1024;
        act = doors + 1024;
    }
    __device__ __forceinline__ bool locked(int x, int y, uint32_t alive) const {     // light.py:233
        return (lock[(x & 31) * 32 + (y & 31)] & alive) != 0;
    }
};

__device__ __forceinline__ void light_teacher_flood(const psk_light_scenario &s, uint16_t *T, uint32_t *s_boards,
                                                    int layer_cap);
__device__ __forceinline__ int light_action_from_dist(const psk_light_scenario &s, const uint16_t *T,
                                                      const LightAux &aux, int x, int y, uint32_t alive,
                                                      int &dist);

__global__ void __launch_bounds__(256)
light_teacher_build_kernel(const psk_light_scenario *__restrict__ scen, uint16_t *__restrict__ table,
                           int layer_cap) {
    extern __shared__ uint32_t s_boards[];           // [2][layer_cap][32]
    const psk_light_scenario &s = scen[blockIdx.x];
    const int n_layers = 1 << s.n_keys;
    uint16_t *T = table + (size_t)blockIdx.x * light_block_u16(layer_cap);
    for (int i = threadIdx.x; i < layer_cap * 1024; i += blockDim.x) T[i] = 0xFFFFu;
    {   // per-cell maps
        uint8_t *aux = reinterpret_cast<uint8_t *>(T + (size_t)layer_cap * 1024);
        for (int c = threadIdx.x; c < 1024; c += blockDim.x) {
            const int x = c >> 5, y = c & 31;
            int nd = 0;
            uint32_t lk = 0, ky = 0;
            for (int d = 0; d < s.n_doors; d++) nd += (s.doors[d][0] == x && s.doors[d][1] == y);
            for (int k = 0; k < s.n_keys; k++) {
                if (nd && s.keys[k][2] == x && s.keys[k][3] == y) lk |= 1u << k;
                if (s.keys[k][0] == x && s.keys[k][1] == y) ky |= 1u << k;
            }
            aux[c] = (uint8_t)lk;
            aux[1024 + c] = (uint8_t)ky;
            aux[2048 + c] = (uint8_t)nd;
        }
    }
    __syncthreads();
    // more keys than announced: no flood, everything outside the goal room stays unreachable
    if (n_layers <= layer_cap) light_teacher_flood(s, T, s_boards, layer_cap);
    __syncthreads();                                 // the distances of this scenario are complete
    {   // the teacher's answer for every (key subset, cell), from the distances
        const LightAux aux(T, layer_cap);
        uint8_t *A = const_cast<uint8_t *>(aux.act);
        for (int i = threadIdx.x; i < layer_cap * 1024; i += blockDim.x) {
            int d;
            A[i] = (uint8_t)light_action_from_dist(s, T, aux, (i >> 5) & 31, i & 31, (uint32_t)(i >> 10), d);
        }
    }
}

__device__ __forceinline__ void light_teacher_flood(const psk_light_scenario &s, uint16_t *T, uint32_t *s_boards,
                                                    int layer_cap) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    constexpr unsigned FULL = 0xffffffffu;
    const int nk = s.n_keys;
    const int n_layers = 1 << nk;
    const uint32_t wall_row = s.walls[lane];
    uint32_t goal_row = 0;
    if (lane / PSK_LIGHT_ROOM == s.goal_rx)
        goal_row = (0x3Fu << (s.goal_ry * PSK_LIGHT_ROOM)) & ~wall_row;
    const uint32_t door_keys = light_door_keys(s);
    auto lock_row = [&](int m) {                     // locked-door cells of this lane's row in layer m
        uint32_t r = 0;
        for (int k = 0; k < nk; k++)
            if ((((m & door_keys) >> k) & 1) && s.keys[k][2] == lane) r |= 1u << s.keys[k][3];
        return r;
    };
    uint32_t *B0 = s_boards, *B1 = s_boards + layer_cap * 32;
    for (int m = warp; m < n_layers; m += nwarps) {
        const uint32_t r = goal_row & ~lock_row(m);
        B0[m * 32 + lane] = r;
        for (uint32_t b = r; b; b &= b - 1) T[(m * 32 + lane) * 32 + (__ffs(b) - 1)] = 0;
    }
    __syncthreads();
    for (int level = 1; level < 0xFFFF; level++) {
        const uint32_t *prev = (level & 1) ? B0 : B1;
        uint32_t *cur = (level & 1) ? B1 : B0;
        int grew = 0;
        for (int m = warp; m < n_layers; m += nwarps) {
            const uint32_t c = prev[m * 32 + lane];
            const uint32_t pass = ~wall_row & ~lock_row(m);
            const uint32_t up = __shfl_up_sync(FULL, c, 1), dn = __shfl_down_sync(FULL, c, 1);
            uint32_t add = (c << 1) | (c >> 1) | (lane > 0 ? up : 0u) | (lane < 31 ? dn : 0u);
            // USE on a key cell: every key of m lying on that cell is picked up (light.py:224-228)
            for (int k = 0; k < nk; k++) {
                if (!((m >> k) & 1) || s.keys[k][0] != lane) continue;
                int gone = 0;
                for (int j = 0; j < nk; j++)
                    if (((m >> j) & 1) && s.keys[j][0] == s.keys[k][0] && s.keys[j][1] == s.keys[k][1])
                        gone |= 1 << j;
                const uint32_t bit = 1u << s.keys[k][1];
                if (prev[(m & ~gone) * 32 + lane] & bit) add |= bit;
            }
            const uint32_t nxt = c | (add & pass);
            cur[m * 32 + lane] = nxt;
            for (uint32_t b = nxt & ~c; b; b &= b - 1)
                T[(m * 32 + lane) * 32 + (__ffs(b) - 1)] = (uint16_t)level;
            grew |= nxt != c;
        }
        if (!__syncthreads_or(grew)) break;
    }
}

// The teacher's answer from the distances (used ONCE per state, when the table is built).  dist 0 = in
// the goal room (action 254), 0xFFFF = unreachable (action 255); else the smallest action whose
// successor is one level closer.
__device__ __forceinline__ int light_action_from_dist(const psk_light_scenario &s, const uint16_t *T,
                                                      const LightAux &aux, int x, int y, uint32_t alive,
                                                      int &dist) {
    if (x / PSK_LIGHT_ROOM == s.goal_rx && y / PSK_LIGHT_ROOM == s.goal_ry && !light_wall(s, x, y)) {
        dist = 0;
        return 254;
    }
    const int d = T[(alive * 32 + (x & 31)) * 32 + (y & 31)];
    if (d == 0xFFFF) {
        dist = -1;
        return 255;
    }
    dist = d;
    // the four neighbours' distances are independent loads: issue them together
    int nd[4];
    bool ok[4];
#pragma unroll
    for (int a = 0; a < 4; a++) {
        const int nx = x + dx_of(a), ny = y + dy_of(a);
        ok[a] = !light_wall(s, nx, ny) && !aux.locked(nx, ny, alive);
        nd[a] = ok[a] ? T[(alive * 32 + (nx & 31)) * 32 + (ny & 31)] : 0xFFFF;
    }
#pragma unroll
    for (int a = 0; a < 4; a++)
        if (ok[a] && nd[a] == d - 1) return a;
    const uint32_t m2 = alive & ~(uint32_t)aux.keys[(x & 31) * 32 + (y & 31)];
    if (m2 != alive && T[(m2 * 32 + x) * 32 + y] == d - 1) return 4;
    return 255;
}

// Teacher query against the table (thread per env): one byte load; the distance only on request.
// A key mask that has no layer in the table (a scenario with more keys than max_keys, or mask bits
// the scenario does not have) answers 255 / dist -2, as the search kernel does, instead of reading
// the next scenario's block or past the end of the table.  The load keeps the mask inside the table
// and the answer is picked after it, off the address path (an early return makes the fused tick spill
// at its 40-register budget).
__device__ __forceinline__ int light_table_action(const LightAux &aux, int layer_cap, int x, int y,
                                                  uint32_t alive) {
    const int a = aux.act[((alive & (uint32_t)(layer_cap - 1)) * 32 + (x & 31)) * 32 + (y & 31)];
    return alive < (uint32_t)layer_cap ? a : 255;
}
__device__ __forceinline__ int light_table_dist(const uint16_t *T, int layer_cap, int action, int x, int y,
                                                uint32_t alive) {
    if (action == 254) return 0;
    if (alive >= (uint32_t)layer_cap) return -2;
    const int d = T[(alive * 32 + (x & 31)) * 32 + (y & 31)];
    return d == 0xFFFF ? -1 : d;
}

__global__ void __launch_bounds__(256, PSK_LIGHT_LOOKUP_MINBLOCKS)
light_expert_table_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                          const uint8_t *__restrict__ state, const uint16_t *__restrict__ table,
                          int layer_cap, uint8_t *__restrict__ action, int16_t *__restrict__ dist_out,
                          int64_t n) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        const int si = scen_idx[e];
        const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
        const uint16_t *T = table + (size_t)si * light_block_u16(layer_cap);
        const LightAux aux(T, layer_cap);
        const int x = st & 0xFF, y = (st >> 8) & 0xFF;
        const uint32_t alive = (st >> 16) & 0xFF;
        const int a = light_table_action(aux, layer_cap, x, y, alive);
        action[e] = (uint8_t)a;
        if (dist_out) dist_out[e] = (int16_t)light_table_dist(T, layer_cap, a, x, y, alive);
    }
}

// Fused Light tick (thread per env) — the Craft tick's contract on this world:
//     ref = teacher(s); f = s.features(); a = action_in ? action_in[e] : ref
//     elapsed += 1; done = a is not one of the 5 actions (the teacher's "already there" 254 /
//                          "unreachable" 255) or elapsed >= max_timesteps
//     done -> success = s.satisfies(goal); s <- LightScenario.init()      !done -> s = s.step(a)
// state byte 3 counts the steps of the running episode.
// One env, one tick: teacher action, the three feature values (each is written four times,
// light.py:191-204), done / success, and the next state word.
struct LightTickOut {
    int ref;
    float locked, open, key;
    bool done, success;
    uint32_t next;
};

__device__ __forceinline__ LightTickOut light_tick_env(const psk_light_scenario &s, const LightAux &aux,
                                                       int layer_cap, uint32_t st, int action_in,
                                                       int max_timesteps) {
    LightTickOut o;
    const int x = st & 0xFF, y = (st >> 8) & 0xFF;
    const uint32_t alive = (st >> 16) & 0xFF;
    o.ref = light_table_action(aux, layer_cap, x, y, alive);
    const int cell = (x & 31) * 32 + (y & 31);
    const float doors_here = (float)aux.doors[cell];
    const bool lk = aux.locked(x, y, alive);
    o.locked = lk ? doors_here : 0.f;
    o.open = lk ? 0.f : doors_here;
    o.key = 0.f;
    if (x % PSK_LIGHT_ROOM != 0 && y % PSK_LIGHT_ROOM != 0)
        o.key = (float)__popc((uint32_t)aux.keys[cell] & alive);
    const int a = action_in >= 0 ? action_in : o.ref;
    const int elapsed = (int)(st >> 24) + 1;
    o.done = a >= PSK_LIGHT_N_ACTIONS || elapsed >= max_timesteps;
    o.success = false;
    if (o.done) {
        o.success = (x / PSK_LIGHT_ROOM == s.goal_rx) && (y / PSK_LIGHT_ROOM == s.goal_ry);
        const uint32_t all = s.n_keys >= 8 ? 0xFFu : ((1u << s.n_keys) - 1u);
        o.next = uint32_t(s.init_x) | (uint32_t(s.init_y) << 8) | (all << 16);
    } else {
        uint32_t n_alive = alive;
        int nx = x, ny = y;
        if (a < 4) {
            nx = x + dx_of(a);
            ny = y + dy_of(a);
            if (light_wall(s, nx, ny) || aux.locked(nx, ny, alive)) { nx = x; ny = y; }
        } else {
            n_alive = alive & ~(uint32_t)aux.keys[cell];
        }
        o.next = uint32_t(nx) | (uint32_t(ny) << 8) | (n_alive << 16) | (uint32_t(elapsed) << 24);
    }
    return o;
}

// The 12 feature floats of the 32 envs of a warp are 1,536 contiguous bytes.  Written per env (three
// float4 at a stride of 48 bytes) every store instruction touches 48 sectors for 512 bytes; instead the
// three values of each env are redistributed with shuffles so that every instruction writes 512
// contiguous bytes.  All 32 lanes must call this (cnt = envs of this warp that exist).
__device__ __forceinline__ void light_store_features_warp(float *warp_rows, const LightTickOut &o, int cnt) {
    const int lane = threadIdx.x & 31;
#if PSK_LIGHT_COALESCED
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int q = j * 32 + lane;                // float4 index among the warp's 96
        const int src = q / 3, part = q - src * 3;
        const float a = __shfl_sync(0xffffffffu, o.locked, src);
        const float b = __shfl_sync(0xffffffffu, o.open, src);
        const float c = __shfl_sync(0xffffffffu, o.key, src);
        const float v = part == 0 ? a : (part == 1 ? b : c);
        if (src < cnt) __stcs(reinterpret_cast<float4 *>(warp_rows) + q, make_float4(v, v, v, v));
    }
#else
    if (lane < cnt) {
        float4 *p = reinterpret_cast<float4 *>(warp_rows + lane * PSK_LIGHT_N_FEATURES);
        __stcs(p, make_float4(o.locked, o.locked, o.locked, o.locked));
        __stcs(p + 1, make_float4(o.open, o.open, o.open, o.open));
        __stcs(p + 2, make_float4(o.key, o.key, o.key, o.key));
    }
#endif
}

// statistics: one atomic per counter per BLOCK (per-warp atomics on three addresses serialise in
// L2 and were a third of the kernel at 1 M envs: 98 k atomics per launch)
__device__ __forceinline__ void light_block_stats(unsigned long long *stats, unsigned n_done, unsigned n_succ,
                                                  unsigned n_live) {
    if (!stats) return;
    __shared__ unsigned red[3][8];
    const unsigned d = __reduce_add_sync(0xffffffffu, n_done);
    const unsigned sc = __reduce_add_sync(0xffffffffu, n_succ);
    const unsigned lv = __reduce_add_sync(0xffffffffu, n_live);
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = d;
        red[1][threadIdx.x >> 5] = sc;
        red[2][threadIdx.x >> 5] = lv;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        unsigned tot = 0;
        for (int w = 0; w < int(blockDim.x >> 5); w++) tot += red[threadIdx.x][w];
        if (tot) atomicAdd(stats + threadIdx.x, (unsigned long long)tot);
    }
}

__global__ void __launch_bounds__(256, PSK_LIGHT_MINBLOCKS)
light_tick_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                  uint8_t *__restrict__ state, const uint16_t *__restrict__ table, int layer_cap,
                  const uint8_t *__restrict__ action_in, float *__restrict__ features_out,
                  uint8_t *__restrict__ expert_out, uint8_t *__restrict__ done_out,
                  uint8_t *__restrict__ success_out, unsigned long long *stats, int max_timesteps,
                  int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned n_done = 0, n_succ = 0, n_live = 0;        // per thread, over its grid-stride iterations
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
        const int64_t e = base + (threadIdx.x & 31);
        LightTickOut o = {};
        if (e < n) {
            const int si = scen_idx[e];
            const uint16_t *T = table + (size_t)si * light_block_u16(layer_cap);
            const LightAux aux(T, layer_cap);
            const uint32_t st = reinterpret_cast<const uint32_t *>(state)[e];
            o = light_tick_env(scen[si], aux, layer_cap, st, action_in ? (int)action_in[e] : -1, max_timesteps);
            expert_out[e] = (uint8_t)o.ref;
            reinterpret_cast<uint32_t *>(state)[e] = o.next;
            if (done_out) done_out[e] = o.done;
            if (success_out) success_out[e] = o.success;
            n_done += o.done;
            n_succ += o.success;
            n_live += 1;
        }
        if (features_out)
            light_store_features_warp(features_out + base * PSK_LIGHT_N_FEATURES, o,
                                      (int)(n - base < 32 ? n - base : 32));
    }
    light_block_stats(stats, n_done, n_succ, n_live);
}

// `ticks` rollout ticks in one launch (the Craft rollout's contract, psk_craft_rollout): the state word,
// the scenario and its table pointers stay in registers; per tick only the outputs are written —
// row t of expert_out / done_out / success_out and frame t % feat_ring of features_out.
__global__ void __launch_bounds__(256, PSK_LIGHT_ROLLOUT_MINBLOCKS)
light_rollout_kernel(const psk_light_scenario *__restrict__ scen, const int32_t *__restrict__ scen_idx,
                     uint8_t *__restrict__ state, const uint16_t *__restrict__ table, int layer_cap,
                     const uint8_t *__restrict__ action_in, float *__restrict__ features_out, int feat_ring,
                     uint8_t *__restrict__ expert_out, uint8_t *__restrict__ done_out,
                     uint8_t *__restrict__ success_out, unsigned long long *stats, int max_timesteps,
                     int ticks, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned n_done = 0, n_succ = 0, n_live = 0;
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
        const int64_t e = base + (threadIdx.x & 31);
        const bool live = e < n;
        const int cnt = (int)(n - base < 32 ? n - base : 32);
        const int si = live ? scen_idx[e] : 0;
        const psk_light_scenario &s = scen[si];
        const uint16_t *T = table + (size_t)si * light_block_u16(layer_cap);
        const LightAux aux(T, layer_cap);
        uint32_t st = live ? reinterpret_cast<const uint32_t *>(state)[e] : 0u;
        for (int t = 0; t < ticks; t++) {
            const int64_t row = (int64_t)t * n + e;
            LightTickOut o = {};
            if (live) {
                o = light_tick_env(s, aux, layer_cap, st, action_in ? (int)action_in[row] : -1, max_timesteps);
                expert_out[row] = (uint8_t)o.ref;
                if (done_out) done_out[row] = o.done;
                if (success_out) success_out[row] = o.success;
                n_done += o.done;
                n_succ += o.success;
                st = o.next;
            }
            if (features_out)
                light_store_features_warp(features_out + ((int64_t)(t % feat_ring) * n + base) * PSK_LIGHT_N_FEATURES,
                                          o, cnt);
        }
        if (live) {
            reinterpret_cast<uint32_t *>(state)[e] = st;
            n_live += ticks;
        }
    }
    light_block_stats(stats, n_done, n_succ, n_live);
}

static inline int lblocks(int64_t n, int per) {
    int64_t b = (n + per - 1) / per;
    return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

}  // namespace psk

using namespace psk;

extern "C" {

static int light_args_ok(const void *scen, const void *idx, const void *state, int64_t n) {
    return n >= 0 && (n == 0 || (scen && idx && state));
}

int psk_light_reset(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                    const uint8_t *mask, int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_reset_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(scen, scen_idx, state, mask, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_step(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                   const uint8_t *action, const uint8_t *active, float *reward,
                   int32_t *err_flags, int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && !action)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_step_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(scen, scen_idx, state, action,
                                                                        active, reward, err_flags, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_features(const psk_light_scenario *scen, const int32_t *scen_idx,
                       const uint8_t *state, float *out, int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && !out)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_features_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(scen, scen_idx, state, out, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_satisfies(const psk_light_scenario *scen, const int32_t *scen_idx,
                        const uint8_t *state, uint8_t *out, int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && !out)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_satisfies_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(scen, scen_idx, state, out, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_expert(const psk_light_scenario *scen, const int32_t *scen_idx,
                     const uint8_t *state, uint8_t *action, int16_t *dist, int32_t max_keys,
                     int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && !action) || max_keys < 0 ||
        max_keys > PSK_LIGHT_MAX_KEYS)
        return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    // two boards (reached / previous level) of 32 rows per key subset and warp
    const int layer_cap = 1 << max_keys;
    const size_t per_warp = (size_t)2 * layer_cap * 32 * sizeof(uint32_t);
    int wpb = (int)((48 * 1024) / per_warp);
    wpb = wpb < 1 ? 1 : (wpb > 4 ? 4 : wpb);
    const size_t smem = (size_t)wpb * per_warp;
    static size_t configured_on[PSK_MAX_DEVICES] = {0};   // the attribute is per device
    size_t &configured = configured_on[current_device()];
    if (smem > configured) {
        if (cudaFuncSetAttribute(light_expert_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem) != cudaSuccess)
            return PSK_ERR_CUDA;
        configured = smem;
    }
    light_expert_kernel<<<lblocks(n, wpb), wpb * 32, smem, (cudaStream_t)stream>>>(
        scen, scen_idx, state, action, dist, n, layer_cap);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int64_t psk_light_teacher_table_bytes(int64_t n_scen, int32_t max_keys) {
    if (n_scen < 0 || max_keys < 0 || max_keys > PSK_LIGHT_MAX_KEYS) return -1;
    return n_scen * (int64_t)light_block_u16(1 << max_keys) * (int64_t)sizeof(uint16_t);
}

int psk_light_teacher_build(const psk_light_scenario *scen, int64_t n_scen, int32_t max_keys,
                            uint16_t *table, void *stream) {
    if (n_scen < 0 || max_keys < 0 || max_keys > PSK_LIGHT_MAX_KEYS || (n_scen && (!scen || !table)))
        return PSK_ERR_BADARG;
    if (n_scen == 0) return PSK_OK;
    const int layer_cap = 1 << max_keys;
    const size_t smem = (size_t)2 * layer_cap * 32 * sizeof(uint32_t);       // 64 KB at 8 keys
    static size_t configured_on[PSK_MAX_DEVICES] = {0};
    size_t &configured = configured_on[current_device()];
    if (smem > configured) {
        if (cudaFuncSetAttribute(light_teacher_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem) != cudaSuccess)
            return PSK_ERR_CUDA;
        configured = smem;
    }
    light_teacher_build_kernel<<<(unsigned)n_scen, 256, smem, (cudaStream_t)stream>>>(scen, table, layer_cap);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_expert_table(const psk_light_scenario *scen, const int32_t *scen_idx, const uint8_t *state,
                           const uint16_t *table, int32_t max_keys, uint8_t *action, int16_t *dist,
                           int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && (!action || !table)) || max_keys < 0 ||
        max_keys > PSK_LIGHT_MAX_KEYS)
        return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_expert_table_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
        scen, scen_idx, state, table, 1 << max_keys, action, dist, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_tick(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                   const uint16_t *table, int32_t max_keys, const uint8_t *action_in,
                   float *features_out, uint8_t *expert_out, uint8_t *done_out, uint8_t *success_out,
                   unsigned long long *stats, int32_t max_timesteps, int64_t n, void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && (!expert_out || !table)) || max_keys < 0 ||
        max_keys > PSK_LIGHT_MAX_KEYS || max_timesteps <= 0 || max_timesteps > 255)
        return PSK_ERR_BADARG;
    if (features_out && (reinterpret_cast<uintptr_t>(features_out) & 15)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    light_tick_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
        scen, scen_idx, state, table, 1 << max_keys, action_in, features_out, expert_out, done_out,
        success_out, stats, max_timesteps, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_light_rollout(const psk_light_scenario *scen, const int32_t *scen_idx, uint8_t *state,
                      const uint16_t *table, int32_t max_keys, int32_t ticks, const uint8_t *action_in,
                      float *features_out, int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                      uint8_t *success_out, unsigned long long *stats, int32_t max_timesteps, int64_t n,
                      void *stream) {
    if (!light_args_ok(scen, scen_idx, state, n) || (n && (!expert_out || !table)) || max_keys < 0 ||
        max_keys > PSK_LIGHT_MAX_KEYS || max_timesteps <= 0 || max_timesteps > 255 || ticks < 0 ||
        (features_out && feat_ring < 1))
        return PSK_ERR_BADARG;
    if (features_out && (reinterpret_cast<uintptr_t>(features_out) & 15)) return PSK_ERR_BADARG;
    if (n == 0 || ticks == 0) return PSK_OK;
    light_rollout_kernel<<<lblocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
        scen, scen_idx, state, table, 1 << max_keys, action_in, features_out, feat_ring, expert_out, done_out,
        success_out, stats, max_timesteps, ticks, n);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

}  // extern "C"
