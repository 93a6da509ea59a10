// psk_craft.cu — sm_100a kernels of the batched Craft environment + BFS teacher and their C ABI.
//
// Kernels (DESIGN.md has the roofline of each):
//   craft_step_kernel      one env per thread; agent record moved as one 256-bit LDG/STG, one
//                          byte gathered from the grid row, recipe table in shared memory.
//   craft_features_kernel  one CTA per tile of E envs; the f32 feature tile is built in shared
//                          memory (zero-fill + scatter of the ~15 non-zeros per env) and leaves
//                          with ONE TMA bulk store (cp.async.bulk, UBLKCP) per tile,
//                          double-buffered so the store of tile i overlaps the build of i+1.
//   craft_expert_kernel    one env per thread; hint-tree walk, then a level-synchronous BFS over
//                          (pos, dir) on 64/128-bit bitboards carrying 4 "first action" colours.
//   craft_advance_kernel   rollout bookkeeping (timer / done / success / auto-reset) + step.
//   craft_tick_kernel      expert + features + advance fused: state read once per tick.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>

#include "psk_common.cuh"

namespace psk {

// =============================================================================================
// step  (worlds/craft.py:332-424)
// =============================================================================================
// Applies `act` to the agent record `a` and the env's grid row.  Cells are read through `rd`
// (global memory, or a shared-memory copy of the row) and cleared through `row` (global).
// flags collects PSK_FLAG_* bits.
template <int W, int H, class TAB>
__device__ __forceinline__ void step_env(const TAB &st, Agent &a, uint8_t *row,
                                         const uint8_t *rd, int act, uint32_t &flags) {
    int x = a.x(), y = a.y(), dir = a.dir();
    if (act < 4) {  // craft.py:341-352 + 418-421: turn always, move iff the target cell is free
        dir = act;
        const int tx = x + dx_of(act), ty = y + dy_of(act);
        if (tx >= 0 && ty >= 0 && tx < W && ty < H && rd[tx * H + ty] == 0) {
            x = tx;
            y = ty;
        }
        a.set_pose(x, y, dir);
    } else if (act == PSK_ACT_USE) {  // craft.py:356-412
        const int fx = x + dx_of(dir), fy = y + dy_of(dir);
        if (fx >= 0 && fy >= 0 && fx < W && fy < H) {  // neighbors(), craft.py:426-437
            const int thing = rd[fx * H + fy];
            const int cls = st.kind_class(thing);
            if (cls == KC_GRAB) {  // craft.py:383-386
                if (thing < PSK_MAX_INV) {
                    if (a.inv(thing) == 255) flags |= PSK_FLAG_INV_OVERFLOW;
                    else a.inv_add(thing, 1);
                }
                row[fx * H + fy] = 0;
            } else if (cls == KC_WORKSHOP) {  // craft.py:388-401: all recipes, in file order
                // only this workshop's recipes are visited (ws_recipes: bit r = recipe r is made here),
                // lowest bit first = file order
                for (uint32_t todo = st.ws_recipes(thing); todo; todo &= todo - 1) {
                    const uint2 rc = st.recipe(__ffs(todo) - 1);
                    const int out = rc.x & 0xFF, n_in = (rc.x >> 16) & 0xFF;
                    const int in0 = rc.x >> 24, c0 = rc.y & 0xFF;
                    const int in1 = (rc.y >> 8) & 0xFF, c1 = (rc.y >> 16) & 0xFF, yld = rc.y >> 24;
                    if (n_in > 0 && a.inv(in0) < c0) continue;
                    if (n_in > 1 && a.inv(in1) < c1) continue;
                    if (a.inv(out) + yld > 255) { flags |= PSK_FLAG_INV_OVERFLOW; continue; }
                    a.inv_add(out, yld);
                    if (n_in > 0) a.inv_add(in0, -c0);
                    if (n_in > 1) a.inv_add(in1, -c1);
                }
            } else if (cls == KC_WATER) {  // craft.py:403-406
                const int bridge = st.bridge_kind();
                if (bridge && a.inv(bridge) > 0) {
                    row[fx * H + fy] = 0;
                    a.inv_add(bridge, -1);
                }
            } else if (cls == KC_STONE) {  // craft.py:408-410 (the axe is kept)
                const int axe = st.axe_kind();
                if (axe && a.inv(axe) > 0) row[fx * H + fy] = 0;
            }
        }
    } else if (act != PSK_ACT_STOP) {
        flags |= PSK_FLAG_BAD_ACTION;  // craft.py:415-416
    }
}

// MODE 0: tables staged in shared memory by the CTA, 256-thread CTAs (the round-1 kernel).
// MODE 1: kind classes / recipes read through the read-only path from the device copy — no table
//         staging, no CTA barrier — 64-thread CTAs so that 65,536 envs spread over all SMs.
// MODE 2: MODE 1 + the warp's 32 grid rows (32 x 64 B, contiguous) copied to shared memory with
//         coalesced 128-bit loads issued TOGETHER with the agent loads, instead of one dependent
//         byte gather after the agent record has arrived: one DRAM round trip instead of two (the
//         kernel is latency-bound at 65,536 envs: 13 MB of traffic), and no extra DRAM traffic —
//         the byte gather already pulled a 32-byte sector of every row.  Rows of 64 bytes only.
// All modes: programmatic dependent launch — the grid may be scheduled while its predecessor in
// the stream drains; nothing is read or written before griddepcontrol.wait.
template <int W, int H, int MODE>
__global__ void __launch_bounds__(MODE == 0 ? 256 : 64)
craft_step_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                  uint8_t *__restrict__ agent, const uint8_t *__restrict__ action,
                  const uint8_t *__restrict__ active, float *__restrict__ reward,
                  int32_t *err_flags, int64_t n, int cell_stride) {
    constexpr int CP = ((W * H + 63) / 64) * 64;
    static_assert(MODE != 2 || CP == 64, "row preload is built for 64-byte rows");
    __shared__ __align__(16) uint8_t s_rows[MODE == 2 ? 64 * CP : 16];
    asm volatile("griddepcontrol.launch_dependents;");
    uint32_t flags = 0;
    auto body = [&](const auto &tab) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        const int lane = threadIdx.x & 31;
        // whole warps iterate so that the cooperative row copy of MODE 2 stays converged
        for (int64_t base = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); base < n;
             base += (int64_t)gridDim.x * blockDim.x) {
            const int64_t e = base + lane;
            const bool valid = e < n;
            const uint8_t *rd = grid + e * cell_stride;
            if (MODE == 2) {
                uint8_t *wrows = s_rows + (threadIdx.x & ~31) * CP;
                const uint4 *g = reinterpret_cast<const uint4 *>(grid + base * CP);
                const int64_t lim = (n - base < 32 ? n - base : 32) * (CP / 16);
                uint4 v[CP / 16];
#pragma unroll
                for (int i = 0; i < CP / 16; i++)
                    if (i * 32 + lane < lim) v[i] = g[i * 32 + lane];
                Agent a0;
                int act0 = PSK_ACT_STOP;
                bool on = valid;
                if (valid) {                                // in flight together with the rows
                    a0 = load_agent(agent, e);
                    act0 = action[e];
                    if (active) on = active[e] != 0;
                }
                __syncwarp();                               // previous iteration's readers are done
#pragma unroll
                for (int i = 0; i < CP / 16; i++)
                    if (i * 32 + lane < lim) reinterpret_cast<uint4 *>(wrows)[i * 32 + lane] = v[i];
                __syncwarp();
                rd = wrows + lane * CP;
                if (!valid) continue;
                if (reward) reward[e] = 0.0f;  // craft.py:338,424
                if (!on) continue;
                Agent a = a0;
                step_env<W, H>(tab, a, grid + e * cell_stride, rd, act0, flags);
                bool changed = false;
#pragma unroll
                for (int i = 0; i < 8; i++) changed |= a.w[i] != a0.w[i];
                if (changed) store_agent(agent, e, a);
            } else {
                if (!valid) continue;
                if (reward) reward[e] = 0.0f;  // craft.py:338,424
                if (active && !active[e]) continue;
                Agent a = load_agent(agent, e);
                const Agent before = a;
                step_env<W, H>(tab, a, grid + e * cell_stride, rd, action[e], flags);
                bool changed = false;
#pragma unroll
                for (int i = 0; i < 8; i++) changed |= a.w[i] != before.w[i];
                if (changed) store_agent(agent, e, a);
            }
        }
    };
    if constexpr (MODE == 0) {
        __shared__ SharedTables sst;
        stage_tables(sst, T);
        body(sst);
    } else {
        body(GlobalTables{T});
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// =============================================================================================
// satisfies  (worlds/craft.py:285-294)  and the hint-tree walk (teachers/base.py:10-25)
// =============================================================================================
template <int W, int H>
__device__ __forceinline__ int facing_kind(const Agent &a, const uint8_t *row) {
    const int fx = a.x() + dx_of(a.dir()), fy = a.y() + dy_of(a.dir());
    if (fx < 0 || fy < 0 || fx >= W || fy >= H) return 0;
    return row[fx * H + fy];
}

__device__ __forceinline__ int node_satisfied(uint32_t nd, const Agent &a, int facing) {
    const int sat = nd & 0xFF, arg = (nd >> 8) & 0xFF;
    if (sat == SAT_INV) return arg < PSK_MAX_INV ? (a.inv(arg) > 0) : 0;
    if (sat == SAT_FACING) return facing == arg;
    return 2;  // None
}

// first incomplete leaf of `task` (node word), or 0 when there is none (-> STOP).
// WARP-CONVERGENT: all 32 lanes call it together; the loop runs in lock-step (vote) so that the
// lanes are converged again when it ends, whatever their individual trip counts were.
__device__ __forceinline__ uint32_t find_incomplete(const SharedTables &st, int task,
                                                    const Agent &a, int facing) {
    const int n = st.task_len(task);
    int i = 0;
    uint32_t leaf = 0;
    while (__any_sync(0xffffffffu, i < n && !leaf)) {
        if (i < n && !leaf) {
            const uint32_t nd = st.node(task, i);
            if (node_satisfied(nd, a, facing) == 1) {
                // bit 0x40 of the leaf byte: last subtask of an (unsatisfied) task — the reference's
                // assert at teachers/base.py:23-24; reported like a bad leaf
                if (nd & 0x00400000u) leaf = (uint32_t(LEAF_BAD) << 16) | 0x80000000u;
                i = nd >> 24;
            } else if ((nd >> 16) & 0x0F) leaf = nd | 0x80000000u;  // bit 31 marks "found"
            else i++;
        }
    }
    return leaf;
}

template <int W, int H>
__global__ void __launch_bounds__(256)
craft_satisfies_kernel(const psk_craft_tables *__restrict__ T,
                       const uint8_t *__restrict__ grid, const uint8_t *__restrict__ agent,
                       const uint8_t *__restrict__ task, uint8_t *__restrict__ out, int64_t n,
                       int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        const Agent a = load_agent_ro(agent, e);
        const int tk = task ? task[e] : a.task();
        const int facing = facing_kind<W, H>(a, grid + e * cell_stride);
        out[e] = st.task_len(tk) ? node_satisfied(st.node(tk, 0), a, facing) : 2;
    }
}

// =============================================================================================
// expert  (teachers/demonstration.py:9-30, teachers/base.py:27-87)
// =============================================================================================
// The reference runs one FIFO BFS per goal cell over states (pos, dir), expanding DOWN, UP,
// LEFT, RIGHT, keeps the strictly shortest path (first goal cell in x-major order wins ties) and
// returns its first action.  Order-independent form used here (proved in DESIGN.md §BFS, checked
// against the literal queue of oracle/craft_oracle.c on every golden state):
//   * the successor of (p, d) under action a is (p', a), p' independent of d, so every state on
//     a shortest path except the last is entered by a successful move: its depth is the plain
//     4-neighbour distance dpos() of its position;
//   * a state facing goal cell g with direction d is entered either by turning in place at
//     q = g - delta(d) (action d is blocked by g) or by moving from q = g - 2*delta(d) into
//     g - delta(d); both cost dpos(q) + 1.  Call such q a "source" of g for direction d;
//   * the FIFO tree path of a node is the lexicographically smallest shortest path to it, so
//     the teacher's action is the smallest first action over all shortest paths to sources of
//     the chosen goal cell.
// So: a colourless forward flood from the agent until the flooded set touches a source gives
// the length D and (lowest bit) the goal cell; a backward flood of D-2 levels from that cell's
// sources tells which neighbours of the agent lie on a shortest path; the action is the
// smallest such direction.  Two floods of ~20 instructions per level on 64/128-bit boards.
// Returns the path length (-1: unreachable); first (0..3) is valid when the length is > 0.
template <int W, int H>
__device__ __forceinline__ typename Board<W, H>::BT spread(typename Board<W, H>::BT v) {
    using B = Board<W, H>;
    return B::template shift<0>(v) | B::template shift<1>(v) | B::template shift<2>(v) |
           B::template shift<3>(v);
}

// WARP-CONVERGENT: all 32 lanes call it together (lanes without a search pass need = false).
// Both floods run in lock-step under a warp vote, so the straight-line code after each loop is
// executed once per warp instead of once per distinct trip count.
template <int W, int H>
__device__ __forceinline__ int bfs_first_action(bool need, typename Board<W, H>::BT occ,
                                                typename Board<W, H>::BT goal, int x, int y,
                                                int d0, int &first, int &goal_idx) {
    using B = Board<W, H>;
    using BT = typename B::BT;
    constexpr unsigned FULL = 0xffffffffu;
    const BT freeb = ~occ & B::all();
    const BT root = B::bit(x * H + y);
    first = -1;
    goal_idx = -1;
    bool face0 = false;
    {  // depth 0: already facing a goal cell (teachers/base.py:57-66 on the first dequeue)
        const int fx = x + dx_of(d0), fy = y + dy_of(d0);
        if (need && fx >= 0 && fy >= 0 && fx < W && fy < H && ((goal >> (fx * H + fy)) & 1)) {
            face0 = true;
            goal_idx = fx * H + fy;
        }
    }
    // T[d]: positions whose d-neighbour is a goal cell
    const BT T0 = B::template unshift<0>(goal), T1 = B::template unshift<1>(goal),
             T2 = B::template unshift<2>(goal), T3 = B::template unshift<3>(goal);
    const BT src_all = T0 | T1 | T2 | T3 |
                       (B::template unshift<0>(freeb & T0)) | (B::template unshift<1>(freeb & T1)) |
                       (B::template unshift<2>(freeb & T2)) | (B::template unshift<3>(freeb & T3));
    // forward flood: VF = positions within k moves of the agent
    const bool run = need && !face0 && goal != 0;
    BT VF = root;
    int k = 0;
    bool h;
    while (true) {
        h = (VF & src_all) != 0;
        const BT nv = VF | (spread<W, H>(VF) & freeb);
        const bool go = run && !h && nv != VF && k < W * H;  // nv == VF: queue drained (base.py:87)
        if (!__any_sync(FULL, go)) break;
        if (go) {
            VF = nv;
            k++;
        }
    }
    const bool reached = run && h;
    // goal cells faced at depth k+1: by a turn at a flooded cell, or one move further
    const BT hit = B::template shift<0>(VF & T0) | B::template shift<1>(VF & T1) |
                   B::template shift<2>(VF & T2) | B::template shift<3>(VF & T3) |
                   B::template shift<0>(B::template shift<0>(VF) & freeb & T0) |
                   B::template shift<1>(B::template shift<1>(VF) & freeb & T1) |
                   B::template shift<2>(B::template shift<2>(VF) & freeb & T2) |
                   B::template shift<3>(B::template shift<3>(VF) & freeb & T3);
    const BT hg = hit & goal;
    const int gi = hg ? B::lowest(hg) : 0;
    const BT g = B::bit(gi);
    // sources of the chosen goal cell, per final action d
    const BT g0 = B::template unshift<0>(g), g1 = B::template unshift<1>(g),
             g2 = B::template unshift<2>(g), g3 = B::template unshift<3>(g);
    const BT s0 = g0 | B::template unshift<0>(freeb & g0), s1 = g1 | B::template unshift<1>(freeb & g1),
             s2 = g2 | B::template unshift<2>(freeb & g2), s3 = g3 | B::template unshift<3>(freeb & g3);
    // backward flood over free cells: VB = cells within k-1 moves of a source (sources lie at
    // forward depth exactly k, otherwise the forward flood had stopped earlier)
    BT VB = (s0 | s1 | s2 | s3) & VF;
    const int kmax = __reduce_max_sync(FULL, reached ? k : 0);
    for (int j = 1; j < kmax; j++) {
        const BT nb = VB | (spread<W, H>(VB) & freeb);
        if (j < k) VB = nb;
    }
    if (face0) return 0;
    if (!reached) return -1;
    goal_idx = gi;
    if (k == 0) {  // the agent's own cell is the source: one action
        first = (root & s0) ? 0 : (root & s1) ? 1 : (root & s2) ? 2 : 3;
        return 1;
    }
    const BT ok = VB & freeb;
    first = (B::template shift<0>(root) & ok) ? 0
          : (B::template shift<1>(root) & ok) ? 1
          : (B::template shift<2>(root) & ok) ? 2 : 3;
    return k + 1;
}

// occupancy / goal bitboards from one env's grid row held in registers.
// Per 4-cell word: bit 7 of every non-zero byte via ((w & 0x7f..) + 0x7f..) | w, the four flag
// bits gathered into a nibble by one multiply (0x00204081 moves bits 7,15,23,31 to 28..31).
__device__ __forceinline__ uint32_t nonzero_flags(uint32_t w) {
    return (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) & 0x80808080u;
}
template <int W, int H>
__device__ __forceinline__ void build_boards(const uint32_t *row_words, int goal_kind,
                                             typename Board<W, H>::BT &occ,
                                             typename Board<W, H>::BT &goal) {
    using BT = typename Board<W, H>::BT;
    constexpr int NW = (W * H + 3) / 4;
    const uint32_t gk = uint32_t(goal_kind) * 0x01010101u;
    uint32_t o[(NW + 7) / 8], q[(NW + 7) / 8];
#pragma unroll
    for (int i = 0; i < (NW + 7) / 8; i++) o[i] = q[i] = 0;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const uint32_t w = row_words[i];
        const uint32_t nz = nonzero_flags(w);
        const uint32_t eq = nonzero_flags(w ^ gk) ^ 0x80808080u;
        const int sh = 4 * (i & 7);
        o[i >> 3] |= ((nz * 0x00204081u) >> 28) << sh;
        q[i >> 3] |= ((eq * 0x00204081u) >> 28) << sh;
    }
    occ = 0;
    goal = 0;
#pragma unroll
    for (int i = 0; i < (NW + 7) / 8; i++) {
        occ |= BT(o[i]) << (32 * i);
        goal |= BT(q[i]) << (32 * i);
    }
    occ &= Board<W, H>::all();
    goal &= Board<W, H>::all();
    if (goal_kind == 0) goal = 0;
}

// Loads one env's grid row into registers with 128-bit loads (row is 16-byte aligned).
template <int NW4>
__device__ __forceinline__ void load_row(const uint8_t *row, uint32_t *words) {
#pragma unroll
    for (int i = 0; i < NW4; i++) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(row) + i);
        words[4 * i + 0] = v.x;
        words[4 * i + 1] = v.y;
        words[4 * i + 2] = v.z;
        words[4 * i + 3] = v.w;
    }
}

// Teacher action for one env.  row_words: the env's grid row in registers.
// WARP-CONVERGENT (see find_incomplete / bfs_first_action): called by all 32 lanes.
template <int W, int H>
__device__ __forceinline__ int expert_env(const SharedTables &st, const Agent &a, int task,
                                          const uint32_t *row_words, int facing, int &dist,
                                          uint32_t &flags) {
    const uint32_t leaf = find_incomplete(st, task, a, facing);
    const int kind = (leaf >> 16) & 0x0F;
    const bool need = leaf && kind == LEAF_GO;
    typename Board<W, H>::BT occ, goal;
    build_boards<W, H>(row_words, need ? (leaf >> 8) & 0xFF : 0, occ, goal);
    int first, gidx;
    const int d = bfs_first_action<W, H>(need, occ, goal, a.x(), a.y(), a.dir(), first, gidx);
    dist = need ? d : -1;
    if (!leaf) return PSK_ACT_STOP;                         // demonstration.py:15-16
    if (kind == LEAF_USE) return PSK_ACT_USE;               // demonstration.py:20-21
    if (kind != LEAF_GO) {                                  // demonstration.py:18 (assert)
        flags |= PSK_FLAG_BAD_LEAF;
        return PSK_ACT_INVALID;
    }
    if (d < 0) return PSK_ACT_STOP;                         // demonstration.py:25-26
    return first >= 0 ? first : PSK_ACT_INVALID;
}

template <int W, int H>
__global__ void __launch_bounds__(128)
craft_expert_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                    const uint8_t *__restrict__ agent, const uint8_t *__restrict__ task,
                    uint8_t *__restrict__ action, int16_t *__restrict__ dist_out,
                    int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    constexpr int NW4 = (W * H + 15) / 16;
    uint32_t flags = 0;
    const int lane = threadIdx.x & 31;
    // whole warps iterate (base is warp-uniform); lanes past the end replay env n-1, unsaved
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); base < n;
         base += (int64_t)gridDim.x * blockDim.x) {
        const bool valid = base + lane < n;
        const int64_t e = valid ? base + lane : n - 1;
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        uint32_t words[NW4 * 4];
        load_row<NW4>(row, words);
        const int tk = task ? task[e] : a.task();
        const int facing = facing_kind<W, H>(a, row);
        int dist;
        uint32_t fl = 0;
        const int act = expert_env<W, H>(st, a, tk, words, facing, dist, fl);
        if (valid) {
            flags |= fl;
            action[e] = (uint8_t)act;
            if (dist_out) dist_out[e] = (int16_t)dist;
        }
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// find_closest_resources (teachers/base.py:27-34) for an explicit kind, with the full
// lexicographically-smallest action sequence reconstructed by re-running the BFS towards the
// chosen goal cell after every move (only the length is used on the training path).
template <int W, int H>
__global__ void __launch_bounds__(128)
craft_find_closest_kernel(const psk_craft_tables *__restrict__ T,
                          const uint8_t *__restrict__ grid, const uint8_t *__restrict__ agent,
                          const uint8_t *__restrict__ kind, uint8_t *__restrict__ goal_out,
                          int16_t *__restrict__ len_out, uint8_t *__restrict__ seq, int seq_cap,
                          int64_t n, int cell_stride) {
    using B = Board<W, H>;
    using BT = typename B::BT;
    constexpr int NW4 = (W * H + 15) / 16;
    const int lane = threadIdx.x & 31;
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); base < n;
         base += (int64_t)gridDim.x * blockDim.x) {
        const bool valid = base + lane < n;
        const int64_t e = valid ? base + lane : n - 1;
        const Agent a = load_agent_ro(agent, e);
        uint32_t words[NW4 * 4];
        load_row<NW4>(grid + e * cell_stride, words);
        BT occ, goal;
        build_boards<W, H>(words, kind[e], occ, goal);
        int first, gidx;
        int x = a.x(), y = a.y(), d = a.dir();
        const int len = bfs_first_action<W, H>(true, occ, goal, x, y, d, first, gidx);
        if (valid) {
            len_out[e] = (int16_t)len;
            if (len < 0) {
                // best_goal keeps the LAST goal cell scanned when none is reachable (base.py:31)
                int last = -1;
                BT g = goal;
                while (g) { last = B::lowest(g); g &= g - 1; }
                goal_out[2 * e] = last < 0 ? 255 : last / H;
                goal_out[2 * e + 1] = last < 0 ? 255 : last % H;
            } else {
                goal_out[2 * e] = gidx / H;
                goal_out[2 * e + 1] = gidx % H;
            }
        }
        if (seq) {
            // replay: apply the action, search again towards the chosen cell (lock-step)
            uint8_t *sq = seq + e * (int64_t)seq_cap;
            const BT g1 = len > 0 ? B::bit(gidx) : BT(0);
            const int lmax = __reduce_max_sync(0xffffffffu, len > 0 ? len : 0);
            int f = first;
            for (int k = 0; k < lmax; k++) {
                const bool on = k < len;
                if (on) {
                    if (valid && k < seq_cap) sq[k] = (uint8_t)f;
                    const int tx = x + dx_of(f), ty = y + dy_of(f);
                    const bool can = tx >= 0 && ty >= 0 && tx < W && ty < H &&
                                     !((occ >> (tx * H + ty)) & 1);
                    if (can) { x = tx; y = ty; }
                    d = f;
                }
                int f2, g2;
                bfs_first_action<W, H>(on && k + 1 < len, occ, g1, x, y, d, f2, g2);
                if (on && k + 1 < len) f = f2;
            }
            if (valid)
                for (int k = len > 0 ? len : 0; k < seq_cap; k++) sq[k] = 255;
        }
    }
}

// =============================================================================================
// enlarged grids (W, H <= 64): one WARP per env, rows of every board spread over the lanes
// =============================================================================================
// Same two floods as bfs_first_action, with the boards laid out row-per-lane: vertical moves
// (y +- 1) are bit shifts inside a lane, horizontal moves (x +- 1) are __shfl_up/down_sync
// between lanes, emptiness tests are __ballot_sync / __any_sync.  Every value is warp-uniform in
// control flow, so there is no divergence at all; the reference's 1000-slot queue
// (teachers/base.py:42) would overflow on these sizes, the floods have no such limit.
// Up to 32 rows: lane x holds row x.  Up to 64 rows: lane l holds rows 2l and 2l+1, so a
// horizontal move is one register move plus one shuffle.  Rows are 32- or 64-bit words.
template <int H> struct RowWord { using type = uint64_t; };
template <> struct RowWord<32> { using type = uint32_t; };

template <int W, int H> struct RowBoard {
    static_assert(W <= 64 && H <= 64, "row-per-lane boards cover up to 64 x 64");
    static constexpr int RPL = W > 32 ? 2 : 1;   // rows per lane
    using RT = typename RowWord<(H > 32 ? 64 : 32)>::type;
    static constexpr unsigned FULL = 0xffffffffu;
    RT r[RPL];

    static __device__ __forceinline__ RT hmask() {
        return H == 8 * (int)sizeof(RT) ? ~RT(0) : ((RT(1) << (H % (8 * (int)sizeof(RT)))) - 1);
    }
    static __device__ __forceinline__ int row_of(int lane, int slot) { return RPL * lane + slot; }
    static __device__ __forceinline__ RowBoard zero() {
        RowBoard b;
#pragma unroll
        for (int s = 0; s < RPL; s++) b.r[s] = 0;
        return b;
    }
    static __device__ __forceinline__ RowBoard bit(int x, int y, int lane) {
        RowBoard b = zero();
#pragma unroll
        for (int s = 0; s < RPL; s++)
            if (row_of(lane, s) == x) b.r[s] = RT(1) << y;
        return b;
    }
    __device__ __forceinline__ RowBoard operator&(const RowBoard &o) const {
        RowBoard b;
#pragma unroll
        for (int s = 0; s < RPL; s++) b.r[s] = r[s] & o.r[s];
        return b;
    }
    __device__ __forceinline__ RowBoard operator|(const RowBoard &o) const {
        RowBoard b;
#pragma unroll
        for (int s = 0; s < RPL; s++) b.r[s] = r[s] | o.r[s];
        return b;
    }
    __device__ __forceinline__ bool lane_any() const {
        RT t = 0;
#pragma unroll
        for (int s = 0; s < RPL; s++) t |= r[s];
        return t != 0;
    }
    __device__ __forceinline__ bool any() const { return __any_sync(FULL, lane_any()); }
    __device__ __forceinline__ bool differs(const RowBoard &o) const {
        bool d = false;
#pragma unroll
        for (int s = 0; s < RPL; s++) d |= r[s] != o.r[s];
        return __any_sync(FULL, d);
    }
    // free cells from an occupancy board: complement within the grid
    __device__ __forceinline__ RowBoard free_of(int lane) const {
        RowBoard b;
#pragma unroll
        for (int s = 0; s < RPL; s++) b.r[s] = row_of(lane, s) < W ? (~r[s] & hmask()) : RT(0);
        return b;
    }
    // positions p + delta(A) for p in this board
    template <int A> __device__ __forceinline__ RowBoard shift(int lane) const {
        RowBoard b;
        if (A == 0) {                                   // DOWN  (0,-1)
#pragma unroll
            for (int s = 0; s < RPL; s++) b.r[s] = r[s] >> 1;
        } else if (A == 1) {                            // UP    (0,+1)
#pragma unroll
            for (int s = 0; s < RPL; s++) b.r[s] = (r[s] << 1) & hmask();
        } else if (A == 2) {                            // LEFT  (-1,0): row x <- row x+1
            const RT nxt = __shfl_down_sync(FULL, r[0], 1);      // first row of the next lane
            if (RPL == 1) b.r[0] = lane < 31 ? nxt : RT(0);
            else {
                b.r[0] = r[RPL - 1];
                b.r[RPL - 1] = lane < 31 ? nxt : RT(0);
            }
        } else {                                        // RIGHT (+1,0): row x <- row x-1
            const RT prv = __shfl_up_sync(FULL, r[RPL - 1], 1);  // last row of the previous lane
            if (RPL == 1) b.r[0] = lane > 0 ? prv : RT(0);
            else {
                b.r[RPL - 1] = r[0];
                b.r[0] = lane > 0 ? prv : RT(0);
            }
        }
#pragma unroll
        for (int s = 0; s < RPL; s++)
            if (row_of(lane, s) >= W) b.r[s] = 0;
        return b;
    }
    template <int A> __device__ __forceinline__ RowBoard unshift(int lane) const {
        return shift<(A ^ 1)>(lane);
    }
    __device__ __forceinline__ RowBoard spread(int lane) const {
        return shift<0>(lane) | shift<1>(lane) | shift<2>(lane) | shift<3>(lane);
    }
    // row `x` of the board, broadcast to every lane
    __device__ __forceinline__ RT row(int x) const {
        RT v = __shfl_sync(FULL, r[0], x / RPL);
        if (RPL == 2) {
            const RT v1 = __shfl_sync(FULL, r[RPL - 1], x / RPL);
            if (x % RPL) v = v1;
        }
        return v;
    }
    static __device__ __forceinline__ int low_bit(RT v) {
        return sizeof(RT) == 8 ? __ffsll((long long)v) - 1 : __ffs((int)v) - 1;
    }
    static __device__ __forceinline__ int high_bit(RT v) {
        return sizeof(RT) == 8 ? 63 - __clzll((long long)v) : 31 - __clz((int)v);
    }
    // lowest / highest cell in x-major order (np.nonzero order); false when empty
    __device__ __forceinline__ bool lowest(int &x, int &y) const {
        const unsigned m = __ballot_sync(FULL, lane_any());
        if (!m) return false;
        const int l = __ffs(m) - 1;
        const RT a = __shfl_sync(FULL, r[0], l), b = __shfl_sync(FULL, r[RPL - 1], l);
        const int slot = (RPL == 2 && a == 0) ? 1 : 0;
        x = RPL * l + slot;
        y = low_bit(slot ? b : a);
        return true;
    }
    __device__ __forceinline__ bool highest(int &x, int &y) const {
        const unsigned m = __ballot_sync(FULL, lane_any());
        if (!m) return false;
        const int l = 31 - __clz(m);
        const RT a = __shfl_sync(FULL, r[0], l), b = __shfl_sync(FULL, r[RPL - 1], l);
        const int slot = (RPL == 2 && b != 0) ? 1 : 0;
        x = RPL * l + slot;
        y = high_bit(slot ? b : a);
        return true;
    }
};

// occupancy / goal boards of this lane's rows from the env's grid row (global memory)
template <int W, int H>
__device__ __forceinline__ void build_rows(const uint8_t *row, int lane, int goal_kind,
                                           RowBoard<W, H> &occ, RowBoard<W, H> &goal) {
    using RB = RowBoard<W, H>;
    using RT = typename RB::RT;
#pragma unroll
    for (int s = 0; s < RB::RPL; s++) {
        RT o = 0, g = 0;
        const int x = RB::row_of(lane, s);
        if (x < W) {
            const uint8_t *p = row + x * H;
            if (H % 4 == 0) {
#pragma unroll
                for (int i = 0; i < H / 4; i++) {
                    const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(p + 4 * i));
                    const uint32_t nz = nonzero_flags(w);
                    const uint32_t eq = nonzero_flags(w ^ (uint32_t(goal_kind) * 0x01010101u)) ^ 0x80808080u;
                    o |= RT((nz * 0x00204081u) >> 28) << (4 * i);
                    g |= RT((eq * 0x00204081u) >> 28) << (4 * i);
                }
            } else {
                for (int y = 0; y < H; y++) {
                    const int k = p[y];
                    o |= RT(k != 0) << y;
                    g |= RT(k == goal_kind) << y;
                }
            }
        } else {
            o = RB::hmask();   // rows beyond the grid are solid
        }
        occ.r[s] = o;
        goal.r[s] = goal_kind ? g : RT(0);
    }
}

// Warp-cooperative twin of bfs_first_action.  All lanes return the same values.
template <int W, int H>
__device__ __forceinline__ int bfs_rows(bool need, const RowBoard<W, H> &occ,
                                        const RowBoard<W, H> &goal, int px, int py, int d0,
                                        int lane, int &first, int &gx, int &gy) {
    using RB = RowBoard<W, H>;
    const RB freeb = occ.free_of(lane);
    const RB root = RB::bit(px, py, lane);
    first = -1;
    gx = gy = -1;
    {   // depth 0: already facing a goal cell
        const int fx = px + dx_of(d0), fy = py + dy_of(d0);
        const bool in = fx >= 0 && fy >= 0 && fx < W && fy < H;
        const typename RB::RT grow = goal.row(in ? fx : 0);
        if (need && in && ((grow >> fy) & 1)) {
            gx = fx;
            gy = fy;
            return 0;
        }
    }
    const RB T0 = goal.template unshift<0>(lane), T1 = goal.template unshift<1>(lane),
             T2 = goal.template unshift<2>(lane), T3 = goal.template unshift<3>(lane);
    const RB src_all = T0 | T1 | T2 | T3 | (freeb & T0).template unshift<0>(lane) |
                       (freeb & T1).template unshift<1>(lane) |
                       (freeb & T2).template unshift<2>(lane) |
                       (freeb & T3).template unshift<3>(lane);
    if (!need || !goal.any()) return -1;
    RB VF = root;
    int k = 0;
    while (!(VF & src_all).any()) {
        const RB nv = VF | (VF.spread(lane) & freeb);
        if (!nv.differs(VF)) return -1;                 // queue drained (base.py:87)
        VF = nv;
        k++;
    }
    const RB hit =
        ((VF & T0).template shift<0>(lane) | (VF & T1).template shift<1>(lane) |
         (VF & T2).template shift<2>(lane) | (VF & T3).template shift<3>(lane) |
         (VF.template shift<0>(lane) & freeb & T0).template shift<0>(lane) |
         (VF.template shift<1>(lane) & freeb & T1).template shift<1>(lane) |
         (VF.template shift<2>(lane) & freeb & T2).template shift<2>(lane) |
         (VF.template shift<3>(lane) & freeb & T3).template shift<3>(lane)) & goal;
    hit.lowest(gx, gy);                                 // lowest cell index (np.nonzero order)
    const RB g = RB::bit(gx, gy, lane);
    const RB g0 = g.template unshift<0>(lane), g1 = g.template unshift<1>(lane),
             g2 = g.template unshift<2>(lane), g3 = g.template unshift<3>(lane);
    const RB s0 = g0 | (freeb & g0).template unshift<0>(lane),
             s1 = g1 | (freeb & g1).template unshift<1>(lane),
             s2 = g2 | (freeb & g2).template unshift<2>(lane),
             s3 = g3 | (freeb & g3).template unshift<3>(lane);
    if (k == 0) {
        first = (root & s0).any() ? 0 : (root & s1).any() ? 1 : (root & s2).any() ? 2 : 3;
        return 1;
    }
    RB VB = (s0 | s1 | s2 | s3) & VF;
    for (int j = 1; j < k; j++) VB = VB | (VB.spread(lane) & freeb);
    const RB ok = VB & freeb;
    first = (root.template shift<0>(lane) & ok).any()   ? 0
            : (root.template shift<1>(lane) & ok).any() ? 1
            : (root.template shift<2>(lane) & ok).any() ? 2
                                                        : 3;
    return k + 1;
}

template <int W, int H>
__global__ void __launch_bounds__(128)
craft_expert_rows_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                         const uint8_t *__restrict__ agent, const uint8_t *__restrict__ task,
                         uint8_t *__restrict__ action, int16_t *__restrict__ dist_out,
                         int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        const int tk = task ? task[e] : a.task();
        const int facing = facing_kind<W, H>(a, row);
        const uint32_t leaf = find_incomplete(st, tk, a, facing);
        const int kind = (leaf >> 16) & 0x0F;
        const bool need = leaf && kind == LEAF_GO;
        RowBoard<W, H> occ, goal;
        build_rows<W, H>(row, lane, need ? (leaf >> 8) & 0xFF : 0, occ, goal);
        int first, gx, gy;
        const int d = bfs_rows<W, H>(need, occ, goal, a.x(), a.y(), a.dir(), lane, first, gx, gy);
        int act;
        if (!leaf) act = PSK_ACT_STOP;
        else if (kind == LEAF_USE) act = PSK_ACT_USE;
        else if (kind != LEAF_GO) { act = PSK_ACT_INVALID; flags |= PSK_FLAG_BAD_LEAF; }
        else if (d < 0) act = PSK_ACT_STOP;
        else act = first >= 0 ? first : PSK_ACT_INVALID;
        if (lane == 0) {
            action[e] = (uint8_t)act;
            if (dist_out) dist_out[e] = (int16_t)(need ? d : -1);
        }
    }
    if (flags && err_flags && lane == 0) atomicOr(err_flags, (int)flags);
}

// Grids up to 16 rows: TWO envs per warp.  Lanes 0-15 hold the rows of one env, lanes 16-31 those of
// another (row x in sub-lane x, one 32-bit word per row); horizontal moves are width-16 shuffles,
// emptiness tests are the half's 16 bits of a ballot.  The two halves usually need different numbers
// of flood levels, so both floods run in lock-step under a warp vote (as in bfs_first_action) and
// every shuffle / ballot is executed by all 32 lanes.  Same answers as bfs_rows (tests/test_stress_gpu.py).
template <int W, int H> struct HalfRows {
    static_assert(W <= 16 && H <= 32, "two envs per warp: up to 16 rows of up to 32 cells");
    static constexpr unsigned FULL = 0xffffffffu;
    static __device__ __forceinline__ uint32_t hmask() { return H == 32 ? ~0u : ((1u << (H % 32)) - 1u); }
    template <int A> static __device__ __forceinline__ uint32_t shift(uint32_t r, int sub) {
        uint32_t b;
        if (A == 0) b = r >> 1;                                   // DOWN  (0,-1)
        else if (A == 1) b = (r << 1) & hmask();                  // UP    (0,+1)
        else if (A == 2) {                                        // LEFT  (-1,0): row x <- row x+1
            const uint32_t nxt = __shfl_down_sync(FULL, r, 1, 16);
            b = sub < 15 ? nxt : 0u;
        } else {                                                  // RIGHT (+1,0): row x <- row x-1
            const uint32_t prv = __shfl_up_sync(FULL, r, 1, 16);
            b = sub > 0 ? prv : 0u;
        }
        return sub < W ? b : 0u;
    }
    template <int A> static __device__ __forceinline__ uint32_t unshift(uint32_t r, int sub) {
        return shift<(A ^ 1)>(r, sub);
    }
    static __device__ __forceinline__ uint32_t spread(uint32_t r, int sub) {
        return shift<0>(r, sub) | shift<1>(r, sub) | shift<2>(r, sub) | shift<3>(r, sub);
    }
    static __device__ __forceinline__ uint32_t half_ballot(bool p, int lane) {
        return (__ballot_sync(FULL, p) >> (lane & 16)) & 0xFFFFu;
    }
    static __device__ __forceinline__ bool any(uint32_t r, int lane) { return half_ballot(r != 0, lane) != 0; }
    static __device__ __forceinline__ uint32_t row(uint32_t r, int x) { return __shfl_sync(FULL, r, x & 15, 16); }
};

// returns the path length (-1 unreachable, 0 already facing); first / (gx, gy) as bfs_rows
template <int W, int H>
__device__ __forceinline__ int bfs_half_rows(bool need, uint32_t occ, uint32_t goal, int px, int py,
                                             int d0, int lane, int &first, int &gx, int &gy) {
    using HR = HalfRows<W, H>;
    constexpr unsigned FULL = 0xffffffffu;
    const int sub = lane & 15;
    const uint32_t freeb = sub < W ? (~occ & HR::hmask()) : 0u;
    const uint32_t root = sub == px ? (1u << py) : 0u;
    first = -1;
    gx = gy = -1;
    bool face0 = false;
    {
        const int fx = px + dx_of(d0), fy = py + dy_of(d0);
        const bool in = fx >= 0 && fy >= 0 && fx < W && fy < H;
        const uint32_t grow = HR::row(goal, in ? fx : 0);
        if (need && in && ((grow >> (fy & 31)) & 1)) {
            face0 = true;
            gx = fx;
            gy = fy;
        }
    }
    const uint32_t T0 = HR::template unshift<0>(goal, sub), T1 = HR::template unshift<1>(goal, sub),
                   T2 = HR::template unshift<2>(goal, sub), T3 = HR::template unshift<3>(goal, sub);
    const uint32_t src_all = T0 | T1 | T2 | T3 | HR::template unshift<0>(freeb & T0, sub) |
                             HR::template unshift<1>(freeb & T1, sub) |
                             HR::template unshift<2>(freeb & T2, sub) |
                             HR::template unshift<3>(freeb & T3, sub);
    const bool has_goal = HR::any(goal, lane);
    const bool run = need && !face0 && has_goal;
    uint32_t VF = root;
    int k = 0;
    bool h;
    while (true) {
        h = HR::any(VF & src_all, lane);
        const uint32_t nv = VF | (HR::spread(VF, sub) & freeb);
        const bool changed = HR::any(nv ^ VF, lane);            // unchanged: queue drained (base.py:87)
        const bool go = run && !h && changed;
        if (!__any_sync(FULL, go)) break;
        if (go) {
            VF = nv;
            k++;
        }
    }
    const bool reached = run && h;
    const uint32_t hit =
        (HR::template shift<0>(VF & T0, sub) | HR::template shift<1>(VF & T1, sub) |
         HR::template shift<2>(VF & T2, sub) | HR::template shift<3>(VF & T3, sub) |
         HR::template shift<0>(HR::template shift<0>(VF, sub) & freeb & T0, sub) |
         HR::template shift<1>(HR::template shift<1>(VF, sub) & freeb & T1, sub) |
         HR::template shift<2>(HR::template shift<2>(VF, sub) & freeb & T2, sub) |
         HR::template shift<3>(HR::template shift<3>(VF, sub) & freeb & T3, sub)) & goal;
    // lowest cell of `hit` in x-major order (np.nonzero order)
    const uint32_t hm = HR::half_ballot(hit != 0, lane);
    const int hx = hm ? __ffs(hm) - 1 : 0;
    const uint32_t hrow = HR::row(hit, hx);
    const int hy = hrow ? __ffs(hrow) - 1 : 0;
    const uint32_t g = (sub == hx) ? (1u << hy) : 0u;
    const uint32_t g0 = HR::template unshift<0>(g, sub), g1 = HR::template unshift<1>(g, sub),
                   g2 = HR::template unshift<2>(g, sub), g3 = HR::template unshift<3>(g, sub);
    const uint32_t s0 = g0 | HR::template unshift<0>(freeb & g0, sub), s1 = g1 | HR::template unshift<1>(freeb & g1, sub),
                   s2 = g2 | HR::template unshift<2>(freeb & g2, sub), s3 = g3 | HR::template unshift<3>(freeb & g3, sub);
    const bool r0 = HR::any(root & s0, lane), r1 = HR::any(root & s1, lane), r2 = HR::any(root & s2, lane);
    uint32_t VB = (s0 | s1 | s2 | s3) & VF;
    const int kmax = __reduce_max_sync(FULL, reached ? k : 0);
    for (int j = 1; j < kmax; j++) {
        const uint32_t nb = VB | (HR::spread(VB, sub) & freeb);
        if (j < k) VB = nb;
    }
    const uint32_t ok = VB & freeb;
    const bool n0 = HR::any(HR::template shift<0>(root, sub) & ok, lane),
               n1 = HR::any(HR::template shift<1>(root, sub) & ok, lane),
               n2 = HR::any(HR::template shift<2>(root, sub) & ok, lane);
    if (face0) return 0;
    if (!reached) return -1;
    gx = hx;
    gy = hy;
    if (k == 0) {
        first = r0 ? 0 : r1 ? 1 : r2 ? 2 : 3;
        return 1;
    }
    first = n0 ? 0 : n1 ? 1 : n2 ? 2 : 3;
    return k + 1;
}

template <int W, int H>
__global__ void __launch_bounds__(128)
craft_expert_half_rows_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                              const uint8_t *__restrict__ agent, const uint8_t *__restrict__ task,
                              uint8_t *__restrict__ action, int16_t *__restrict__ dist_out,
                              int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int sub = lane & 15, half = lane >> 4;
    uint32_t flags = 0;
    const int64_t pairs = (n + 1) / 2;
    for (int64_t pr = blockIdx.x * (int64_t)wpb + warp; pr < pairs; pr += (int64_t)gridDim.x * wpb) {
        const bool valid = 2 * pr + half < n;
        const int64_t e = valid ? 2 * pr + half : n - 1;          // a dead half replays the last env, unsaved
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        const int tk = task ? task[e] : a.task();
        const int facing = facing_kind<W, H>(a, row);
        const uint32_t leaf = find_incomplete(st, tk, a, facing);
        const int kind = (leaf >> 16) & 0x0F;
        const bool need = leaf && kind == LEAF_GO;
        const int goal_kind = need ? (leaf >> 8) & 0xFF : 0;
        uint32_t occ = HalfRows<W, H>::hmask(), goal = 0;         // rows beyond the grid are solid
        if (sub < W) {
            occ = goal = 0;
            const uint8_t *p = row + sub * H;
            if (H % 4 == 0) {
#pragma unroll
                for (int i = 0; i < H / 4; i++) {
                    const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(p + 4 * i));
                    const uint32_t nz = nonzero_flags(w);
                    const uint32_t eq = nonzero_flags(w ^ (uint32_t(goal_kind) * 0x01010101u)) ^ 0x80808080u;
                    occ |= ((nz * 0x00204081u) >> 28) << (4 * i);
                    goal |= ((eq * 0x00204081u) >> 28) << (4 * i);
                }
            } else {
                for (int y = 0; y < H; y++) {
                    const int c = p[y];
                    occ |= uint32_t(c != 0) << y;
                    goal |= uint32_t(c == goal_kind) << y;
                }
            }
            if (!goal_kind) goal = 0;
        }
        int first, gx, gy;
        const int d = bfs_half_rows<W, H>(need, occ, goal, a.x(), a.y(), a.dir(), lane, first, gx, gy);
        int act;
        if (!leaf) act = PSK_ACT_STOP;
        else if (kind == LEAF_USE) act = PSK_ACT_USE;
        else if (kind != LEAF_GO) { act = PSK_ACT_INVALID; if (valid) flags |= PSK_FLAG_BAD_LEAF; }
        else if (d < 0) act = PSK_ACT_STOP;
        else act = first >= 0 ? first : PSK_ACT_INVALID;
        if (sub == 0 && valid) {
            action[e] = (uint8_t)act;
            if (dist_out) dist_out[e] = (int16_t)(need ? d : -1);
        }
    }
    if (flags && err_flags && sub == 0) atomicOr(err_flags, (int)flags);
}

template <int W, int H>
__global__ void __launch_bounds__(128)
craft_find_closest_rows_kernel(const uint8_t *__restrict__ grid, const uint8_t *__restrict__ agent,
                               const uint8_t *__restrict__ kind, uint8_t *__restrict__ goal_out,
                               int16_t *__restrict__ len_out, uint8_t *__restrict__ seq,
                               int seq_cap, int64_t n, int cell_stride) {
    using RB = RowBoard<W, H>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        RB occ, goal;
        build_rows<W, H>(row, lane, kind[e], occ, goal);
        int x = a.x(), y = a.y(), d = a.dir(), first, gx, gy;
        const int len = bfs_rows<W, H>(true, occ, goal, x, y, d, lane, first, gx, gy);
        if (len < 0) {
            // last goal cell in scan order (teachers/base.py:31 keeps replacing while None)
            if (!goal.highest(gx, gy)) gx = gy = 255;
        }
        if (lane == 0) {
            len_out[e] = (int16_t)len;
            goal_out[2 * e] = (uint8_t)gx;
            goal_out[2 * e + 1] = (uint8_t)gy;
        }
        if (seq) {
            uint8_t *sq = seq + e * (int64_t)seq_cap;
            const RB g1 = len > 0 ? RB::bit(gx, gy, lane) : RB::zero();
            int f = first;
            for (int k = 0; k < len; k++) {
                if (lane == 0 && k < seq_cap) sq[k] = (uint8_t)f;
                const int tx = x + dx_of(f), ty = y + dy_of(f);
                const bool in = tx >= 0 && ty >= 0 && tx < W && ty < H;
                const typename RB::RT orow = occ.row(in ? tx : 0);
                if (in && !((orow >> ty) & 1)) { x = tx; y = ty; }
                d = f;
                if (k + 1 < len) {
                    int g2x, g2y;
                    bfs_rows<W, H>(true, occ, g1, x, y, d, lane, f, g2x, g2y);
                }
            }
            for (int k = (len > 0 ? len : 0) + lane; k < seq_cap; k += 32) sq[k] = 255;
        }
    }
}

// =============================================================================================
// features  (worlds/craft.py:296-330)
// =============================================================================================
// Streaming store of the vector path: st.global.cs (evict-first).  Plain st.global and
// st.global.wt were tried through a run-time knob and were never faster (profiles/README.md);
// the knob cost a branch per store and is gone.
__device__ __forceinline__ void store_out16(float4 *p, const float4 &t) { __stcs(p, t); }

// Shared-space stores by 32-bit address (no generic-address conversion in the hot loop).
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts_u8(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// The feature tile in shared memory holds one element of ESZ bytes per feature: f32 (ESZ 4, the
// TMA path copies the tile to HBM as it is) or u8 (ESZ 1, the vector path widens u8 -> f32 on the
// way out: every feature is a small exact integer, and a byte tile costs a quarter of the
// shared-memory wavefronts for zero-fill and read-out — the L1/LSU data pipe, not HBM, was the
// busiest unit of the rollout kernel with an f32 tile, profiles/README.md).
template <int ESZ> __device__ __forceinline__ void sts_feat(uint32_t addr, uint32_t count) {
    if (ESZ == 4) sts_f32(addr, (float)count);
    else sts_u8(addr, count);
}
// element := 1 iff k != 0, as a predicated store (never a branch)
template <int ESZ> __device__ __forceinline__ void sts_one_if(uint32_t addr, uint32_t k) {
    if (ESZ == 4)
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p st.shared.f32 [%0], %2;\n\t}" ::"r"(addr),
            "r"(k), "f"(1.0f)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p st.shared.u8 [%0], %2;\n\t}" ::"r"(addr),
            "r"(k), "r"(1)
            : "memory");
}
__device__ __forceinline__ void sts_zero16(uint32_t addr) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "r"(0) : "memory");
}

// The grid-row bytes one feature thread owns: NCH chunks of 8 consecutive cells.  Grids above
// 128 cells are not copied at all (WINDOWED): the features only depend on the WIN^2 x WIN^2
// window around the agent, so the scatter gathers those cells straight from the row.
template <int W, int H, int TPE> struct RowChunks {
    static constexpr bool WINDOWED = W * H > 128;
    static constexpr int CP = ((W * H + 63) / 64) * 64;
    static constexpr int NCH = WINDOWED ? 1 : CP / (8 * TPE);
    uint2 v[NCH];
    const uint8_t *row;
    // thread j of the env reads cells [j*NCH*8, (j+1)*NCH*8) (global or shared, 8-byte aligned)
    __device__ __forceinline__ void load(const uint8_t *r, int j) {
        row = r;
        if constexpr (!WINDOWED) {
#pragma unroll
            for (int c = 0; c < NCH; c++)
                v[c] = *reinterpret_cast<const uint2 *>(r + (j * NCH + c) * 8);
        }
    }
    // same from global memory, as volatile asm: the load is issued where it is written (the
    // prefetch of the next chunk), not sunk by the compiler to its first use an iteration later
    __device__ __forceinline__ void prefetch(const uint8_t *r, int j) {
        row = r;
        if constexpr (!WINDOWED) {
#pragma unroll
            for (int c = 0; c < NCH; c++)
                asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];"
                             : "=r"(v[c].x), "=r"(v[c].y)
                             : "l"(r + (j * NCH + c) * 8));
        }
    }
};

// Scatter of one env's non-zero features into its f32 row at shared address `frow_s`, done by
// the TPE threads of the env; thread j owns the cells in `cells`.  K is the number of kinds.
// The centre block of the pooled WIN^2 x WIN^2 window is exactly the local WIN x WIN window
// (bhw = hw*WIN + hw), so one pass over the cells writes both feature groups.
template <int W, int H, int WIN, int TPE, int ESZ>
__device__ __forceinline__ void scatter_features(uint32_t frow_s, uint32_t trash_s,
                                                 const RowChunks<W, H, TPE> &cells,
                                                 const Agent &a, int K, int j) {
    constexpr int HW = WIN / 2, BHW = (WIN * WIN) / 2;  // craft.py:299-302
    constexpr int WW = WIN * WIN;
    constexpr int NCH = RowChunks<W, H, TPE>::NCH;
    const int px = a.x(), py = a.y();
    const int K4 = K * ESZ;   // bytes per cell of the tile
    const uint32_t big_s = frow_s + WW * K4;
    if (RowChunks<W, H, TPE>::WINDOWED) {
        // gather the WW x WW window cells (thread j takes every TPE-th)
        for (int idx = j; idx < WW * WW; idx += TPE) {
            const int bx = idx / WW, by = idx % WW;
            const int x = px - BHW + bx, y = py - BHW + by;
            if (x < 0 || y < 0 || x >= W || y >= H) continue;
            const int k = __ldg(cells.row + x * H + y);
            if (k == 0) continue;
            sts_feat<ESZ>(big_s + (((bx / WIN) * WIN + (by / WIN)) * K + k) * ESZ, 1);
            if (bx / WIN == HW && by / WIN == HW)
                sts_feat<ESZ>(frow_s + (((bx - HW * WIN) * WIN + (by - HW * WIN)) * K + k) * ESZ, 1);
        }
    } else
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
        const int cc = (j * NCH + ch) * 8;
        const uint2 v = cells.v[ch];
        if (cc >= W * H || (v.x | v.y) == 0) continue;
        if (H == 8 && WIN == 3) {
            // 8x8 grid, 3x3 window (craft_medium): the thread's 8 cells are column x.  The column
            // is shifted so that byte `by` of (z2:z1:z0) is the kind at window row by
            // (y = py - BHW + by; rows outside the grid and columns outside the window read 0);
            // the 9 window rows then sit at compile-time byte positions and every store is one
            // byte extract, one address add and one predicated st.shared (no branches, no
            // per-cell range checks).
            const int x = cc / 8;
            const int bx = x - px + BHW;
            const bool bx_ok = (unsigned)bx < (unsigned)WW;
            const int bi = bx / WIN;
            const uint32_t vx = bx_ok ? v.x : 0u, vy = bx_ok ? v.y : 0u;
            const int sh = 8 * py;                       // = 8 * (py - BHW + 4): 0..56
            const bool hi_word = sh >= 32;
            const uint32_t a0 = hi_word ? vx : 0u, a1 = hi_word ? vy : vx, a2 = hi_word ? 0u : vy;
            const uint32_t z0 = __funnelshift_r(a0, a1, sh & 31);
            const uint32_t z1 = __funnelshift_r(a1, a2, sh & 31);
            const uint32_t z2 = a2 >> (sh & 31);
            const uint32_t big_col = big_s + bi * (WIN * K4);
#pragma unroll
            for (int by = 0; by < 9; by++) {             // pooled window, block (bi, by / 3)
                const uint32_t z = by < 4 ? z0 : (by < 8 ? z1 : z2);
                const uint32_t k = (z >> ((by & 3) * 8)) & 0xFF;
                sts_one_if<ESZ>(big_col + (by / WIN) * K4 + k * ESZ, k);
            }
            // local window = centre block; ravel order (dx, dy, kind)  (craft.py:304-305)
            const bool centre_col = bx_ok && bi == HW;
            const uint32_t c0 = centre_col ? z0 : 0u, c1 = centre_col ? z1 : 0u;
            const uint32_t loc_col = frow_s + (bx - HW * WIN) * (WIN * K4);
#pragma unroll
            for (int dy = 0; dy < 3; dy++) {
                const int by = HW * WIN + dy;
                const uint32_t k = ((by < 4 ? c0 : c1) >> ((by & 3) * 8)) & 0xFF;
                sts_one_if<ESZ>(loc_col + dy * K4 + k * ESZ, k);
            }
        } else if (H % 8 == 0) {
            // the 8 cells share one column x; y = y0 + b.  Stores are unconditional: a cell that
            // contributes nothing writes into the warp's trash slot instead (no branches).
            const int x = cc / H, y0 = cc % H;
            const int bx = x - px + BHW;
            const bool bx_ok = (unsigned)bx < (unsigned)WW;
            const int bi = bx / WIN;
            const uint32_t big_col = big_s + bi * (WIN * K4);
            const bool centre_col = bx_ok && bi == HW;
            const uint32_t loc_col = frow_s + (bx - HW * WIN) * (WIN * K4) - HW * WIN * K4;
            const int by0 = y0 - py + BHW;
#pragma unroll
            for (int b = 0; b < 8; b++) {
                const int k = ((b < 4 ? v.x : v.y) >> ((b & 3) * 8)) & 0xFF;
                const int by = by0 + b;
                const bool ok = bx_ok && (unsigned)by < (unsigned)WW && k != 0;
                const int bj = by / WIN;
                const uint32_t off = by * K4 + k * ESZ;
                // pooled window, block (bi, bj)  (craft.py:306-310)
                sts_feat<ESZ>(ok ? big_col + bj * K4 + k * ESZ : trash_s, 1);
                // local window, ravel order (dx, dy, kind)  (craft.py:304-305)
                sts_feat<ESZ>((ok && centre_col && bj == HW) ? loc_col + off : trash_s, 1);
            }
        } else {
#pragma unroll
            for (int b = 0; b < 8; b++) {
                const int k = ((b < 4 ? v.x : v.y) >> ((b & 3) * 8)) & 0xFF;
                const int c = cc + b;
                if (k == 0 || c >= W * H) continue;
                const int dx = c / H - px, dy = c % H - py;
                if ((unsigned)(dx + HW) < (unsigned)WIN && (unsigned)(dy + HW) < (unsigned)WIN)
                    sts_feat<ESZ>(frow_s + (((dx + HW) * WIN + (dy + HW)) * K + k) * ESZ, 1);
                const int bx = dx + BHW, by = dy + BHW;
                if ((unsigned)bx < (unsigned)WW && (unsigned)by < (unsigned)WW)
                    sts_feat<ESZ>(big_s + (((bx / WIN) * WIN + (by / WIN)) * K + k) * ESZ, 1);
            }
        }
    }
    // inventory counts (craft.py:325): thread j converts inventory word j (4 kinds)
    const uint32_t tail_s = frow_s + 2 * WW * K4;
    for (int wi = j; wi < 6; wi += TPE) {
        const uint32_t w = a.inv_word(wi);
        if (w == 0) continue;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int cnt = (w >> (8 * b)) & 0xFF;
            if (cnt && wi * 4 + b < K) sts_feat<ESZ>(tail_s + (wi * 4 + b) * ESZ, cnt);
        }
    }
    if (j == TPE - 1) sts_feat<ESZ>(tail_s + (K + a.dir()) * ESZ, 1);  // craft.py:321-322; last stays 0
}

// TMA helpers (cp.async.bulk, shared::cta -> global)
__device__ __forceinline__ void bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
                 "r"(ssrc), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// One warp builds the feature rows of up to EPW = 32/TPE consecutive envs in its own shared-
// memory tile(s) and sends each finished chunk to HBM; no CTA-level barrier is involved: warps
// are autonomous pipelines.  Two ways out of shared memory:
//   USE_TMA  f32 tile; one cp.async.bulk (UBLKCP) per chunk, issued by lane 0, two tiles per warp
//            so the store of chunk i overlaps the build of chunk i+1; the tile is zero-filled per
//            chunk;
//   else     u8 tile (see sts_feat); all lanes read one 32-bit word (4 features), widen it to a
//            float4 and write coalesced 128-bit st.global.cs; every word read out is zeroed in
//            the same pass, so one tile per warp stays clean (feature_buffer_init zeroes it once).
//   wbuf_s  shared address of this warp's tile(s); it = this warp's chunk counter (parity)
//   gdst    where the chunk's rows go; ne = live envs in the chunk (<= EPW)
//   cells/a the lane's share of its env's grid row and the env's agent record
// KC > 0 fixes the number of kinds at compile time (KC == K) so that the loops unroll.
// Each tile is EPW*nf elements (rounded up to 16 bytes) + one 16-byte trash slot for the
// scatter's no-op stores.
// Element size of the tile on the vector-store path (profiles/README.md).  Round 1: the stand-alone
// features kernel was 4 % faster with the u8 tile, the fused kernels 3 % slower (their feature warps
// share the issue slots with the teacher, widening costs 8 more instructions per 16 bytes).  Round 2,
// with tile chaining and the shorter USE path the balance flipped: u8 tile 15.36 vs 15.40 us per tick
// in the rollout kernel, 17.65 vs 18.35 us in the single-tick kernel (same box, interleaved) — u8
// everywhere now; -DPSK_ESZ_FUSED_KERNELS=4 rebuilds the f32 tile for A/B runs.
#define PSK_ESZ_FEATURES_KERNEL 1
#ifndef PSK_ESZ_FUSED_KERNELS          // experiment builds: -DPSK_ESZ_FUSED_KERNELS=4 + PSK_LIB
#define PSK_ESZ_FUSED_KERNELS 1
#endif
__host__ __device__ constexpr int feature_tile_bytes(bool tma, int epw, int nf, int vec_esz) {
    return ((epw * nf * (tma ? 4 : vec_esz) + 15) / 16) * 16 + 16;
}
// all tiles of one warp
__host__ __device__ constexpr int feature_buffer_bytes(bool tma, int epw, int nf, int vec_esz) {
    return (tma ? 2 : 1) * feature_tile_bytes(tma, epw, nf, vec_esz);
}

template <int TPE, int KC, bool USE_TMA, int VEC_ESZ>
__device__ __forceinline__ void feature_buffer_init(uint32_t wbuf_s, int nf) {
    constexpr int EPW = 32 / TPE;
    const int lane = threadIdx.x & 31;
    const int bytes = feature_buffer_bytes(USE_TMA, EPW, nf, VEC_ESZ);      // a multiple of 16
    for (int i = lane; i < bytes / 16; i += 32) sts_zero16(wbuf_s + i * 16);
    __syncwarp();
}

// u8 x4 -> float4, exact: byte b of the word is merged under the exponent of 2^23 (one PRMT) and
// 2^23 is subtracted (one FADD)
__device__ __forceinline__ float4 widen_u8x4(uint32_t w) {
    float4 t;
    t.x = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7440)) - 8388608.0f;
    t.y = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7441)) - 8388608.0f;
    t.z = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7442)) - 8388608.0f;
    t.w = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7443)) - 8388608.0f;
    return t;
}

template <int W, int H, int WIN, int TPE, int KC, bool USE_TMA, int VEC_ESZ>
__device__ __forceinline__ void warp_feature_chunk(uint32_t wbuf_s, int it, float *gdst, int ne,
                                                   const RowChunks<W, H, TPE> &cells,
                                                   const Agent &a, int K, int nf) {
    constexpr int EPW = 32 / TPE;
    constexpr int ESZ = USE_TMA ? 4 : VEC_ESZ;
    if (KC > 0) {
        K = KC;
        nf = 2 * WIN * WIN * KC + KC + 5;
    }
    const int lane = threadIdx.x & 31;
    const int le = lane / TPE, j = lane % TPE;
    const uint32_t buf_s = wbuf_s + (USE_TMA ? (uint32_t)(it & 1) * feature_tile_bytes(true, EPW, nf, 4) : 0u);
    const uint32_t trash_s = buf_s + feature_tile_bytes(USE_TMA, EPW, nf, VEC_ESZ) - 16;
    const int n16 = EPW * nf / 4;        // float4s of a full chunk (EPW is a multiple of 4)
    if (USE_TMA) {
        // the tile was handed to the TMA two chunks ago: wait until it has been read, re-zero
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
        if (KC > 0) {
#pragma unroll
            for (int i = 0; i < (n16 + 31) / 32; i++)
                if (i * 32 + lane < n16) sts_zero16(buf_s + (i * 32 + lane) * 16);
        } else {
            for (int i = lane; i < n16; i += 32) sts_zero16(buf_s + i * 16);
        }
        __syncwarp();
    }
    if (le < ne)
        scatter_features<W, H, WIN, TPE, ESZ>(buf_s + le * nf * ESZ, trash_s, cells, a, K, j);
    const uint32_t bytes = (uint32_t)ne * (uint32_t)nf * 4u;
    // 16-byte paths need the chunk size AND its destination aligned (a frame of a feature ring
    // starts at slot*n*nf floats, which is not a multiple of 16 bytes for every n and nf)
    const bool vec_ok = (bytes & 15u) == 0 && (reinterpret_cast<uintptr_t>(gdst) & 15) == 0;
    if (USE_TMA) {
        if (vec_ok) {
            fence_async_smem();  // generic-proxy writes -> visible to the async proxy
            __syncwarp();
            if (lane == 0) bulk_store(gdst, buf_s, bytes);
        } else {
            __syncwarp();
            for (int i = lane; i < ne * nf; i += 32) {
                float t;
                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(t) : "r"(buf_s + i * 4));
                gdst[i] = t;
            }
            __syncwarp();
        }
    } else if (ESZ == 4) {
        // f32 tile, 128-bit read-out
        __syncwarp();
        if (vec_ok) {
            float4 *g4 = reinterpret_cast<float4 *>(gdst);
            const int m16 = (int)(bytes / 16);
            auto move16 = [&](int i) {
                float4 t;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(t.x), "=f"(t.y), "=f"(t.z), "=f"(t.w)
                             : "r"(buf_s + i * 16));
                sts_zero16(buf_s + i * 16);
                store_out16(g4 + i, t);
            };
            if (KC > 0 && m16 == n16) {
                // the shared-memory instructions are volatile asm and keep their source order, so
                // the order is written out: four loads in flight, then their re-zeroing, then the
                // four global stores (one load latency per four 16-byte pieces instead of one each)
                constexpr int NIT = (EPW * (2 * WIN * WIN * KC + KC + 5) / 4 + 31) / 32;
#pragma unroll
                for (int i0 = 0; i0 < NIT; i0 += 4) {
                    float4 t[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16)
                            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                                         : "=f"(t[u].x), "=f"(t[u].y), "=f"(t[u].z), "=f"(t[u].w)
                                         : "r"(buf_s + i * 16));
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16) sts_zero16(buf_s + i * 16);
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16) store_out16(g4 + i, t[u]);
                    }
                }
            } else {
                for (int i = lane; i < m16; i += 32) move16(i);
                for (int i = m16 + lane; i < n16; i += 32) sts_zero16(buf_s + i * 16);
            }
        } else {
            for (int i = lane; i < ne * nf; i += 32) {
                float t;
                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(t) : "r"(buf_s + i * 4));
                gdst[i] = t;
            }
            __syncwarp();
            for (int i = lane; i < n16; i += 32) sts_zero16(buf_s + i * 16);
        }
        __syncwarp();
    } else {
        __syncwarp();
        if (vec_ok) {
            float4 *g4 = reinterpret_cast<float4 *>(gdst);
            const int m16 = (int)(bytes / 16);
            auto move16 = [&](int i) {            // features 4i .. 4i+3 of the chunk
                uint32_t w;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(buf_s + i * 4));
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(buf_s + i * 4), "r"(0) : "memory");
                store_out16(g4 + i, widen_u8x4(w));
            };
            if (KC > 0 && m16 == n16) {
                constexpr int NIT = (EPW * (2 * WIN * WIN * KC + KC + 5) / 4 + 31) / 32;
#pragma unroll
                for (int i0 = 0; i0 < NIT; i0 += 4) {      // same ordering as the f32 read-out
                    uint32_t w[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16)
                            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[u]) : "r"(buf_s + i * 4));
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16)
                            asm volatile("st.shared.u32 [%0], %1;" ::"r"(buf_s + i * 4), "r"(0) : "memory");
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = (i0 + u) * 32 + lane;
                        if (i0 + u < NIT && i < n16) store_out16(g4 + i, widen_u8x4(w[u]));
                    }
                }
            } else {
                for (int i = lane; i < m16; i += 32) move16(i);
                // rows of dead lanes were touched by nobody, but stay safe
                for (int i = m16 + lane; i < n16; i += 32)
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(buf_s + i * 4), "r"(0) : "memory");
            }
        } else {
            for (int i = lane; i < ne * nf; i += 32) {
                uint32_t b;
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(buf_s + i));
                gdst[i] = (float)b;
            }
            __syncwarp();
            for (int i = lane; i < n16; i += 32)
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(buf_s + i * 4), "r"(0) : "memory");
        }
        __syncwarp();
    }
}

// Compact observation frame: the same feature rows as bytes (u8[n][nf]; every feature is an exact
// integer <= 255: 0/1 indicators and inventory counts, which are u8 in the state already).  A
// quarter of the f32 frame — for consumers on the far side of PCIe (psk_craft_host_tick_resident).
// The u8 tile is what the vector path builds anyway; here it leaves as it is, 4 features per store.
template <int W, int H, int WIN, int TPE, int KC>
__device__ __forceinline__ void warp_feature_chunk_u8(uint32_t wbuf_s, uint8_t *gdst, int ne,
                                                      const RowChunks<W, H, TPE> &cells,
                                                      const Agent &a, int K, int nf) {
    constexpr int EPW = 32 / TPE;
    if (KC > 0) {
        K = KC;
        nf = 2 * WIN * WIN * KC + KC + 5;
    }
    const int lane = threadIdx.x & 31;
    const int le = lane / TPE, j = lane % TPE;
    const uint32_t trash_s = wbuf_s + feature_tile_bytes(false, EPW, nf, 1) - 16;
    if (le < ne) scatter_features<W, H, WIN, TPE, 1>(wbuf_s + le * nf, trash_s, cells, a, K, j);
    __syncwarp();
    const int n4 = EPW * nf / 4;                 // words of a full chunk (EPW is a multiple of 4)
    const int bytes = ne * nf;
    if ((bytes & 3) == 0 && (reinterpret_cast<uintptr_t>(gdst) & 3) == 0) {
        uint32_t *g4 = reinterpret_cast<uint32_t *>(gdst);
        for (int i = lane; i < n4; i += 32) {
            uint32_t w;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(wbuf_s + i * 4));
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(wbuf_s + i * 4), "r"(0) : "memory");
            if (i < bytes / 4) __stcs(g4 + i, w);
        }
    } else {
        for (int i = lane; i < bytes; i += 32) {
            uint32_t b;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(wbuf_s + i));
            gdst[i] = (uint8_t)b;
        }
        __syncwarp();
        for (int i = lane; i < n4; i += 32)
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(wbuf_s + i * 4), "r"(0) : "memory");
    }
    __syncwarp();
}

// WPB autonomous warps per CTA; warp w of CTA b takes chunks (b*WPB + w) + k*gridDim.x*WPB.
// The inputs of the next chunk are fetched before the current one is built (software prefetch).
template <int W, int H, int WIN, int WPB, int TPE, int KC, bool USE_TMA, typename OUT = float>
__global__ void __launch_bounds__(WPB * 32)
craft_features_kernel(const uint8_t *__restrict__ grid, const uint8_t *__restrict__ agent,
                      OUT *__restrict__ out, int64_t n, int cell_stride, int K, int nf) {
    constexpr bool OUT_U8 = sizeof(OUT) == 1;
    static_assert(!(OUT_U8 && USE_TMA), "the u8 frame uses the vector path");
    constexpr int EPW = 32 / TPE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int le = lane / TPE, j = lane % TPE;
    const uint32_t wbuf_s = smem_u32(smem_raw) + (uint32_t)warp * feature_buffer_bytes(USE_TMA, EPW, nf, PSK_ESZ_FEATURES_KERNEL);
    if (!USE_TMA) feature_buffer_init<TPE, KC, USE_TMA, PSK_ESZ_FEATURES_KERNEL>(wbuf_s, nf);
    const int64_t n_chunks = (n + EPW - 1) / EPW;
    const int64_t stride = (int64_t)gridDim.x * WPB;
    int64_t ch = (int64_t)blockIdx.x * WPB + warp;
    Agent a, a_next;
    RowChunks<W, H, TPE> cells, cells_next;
    auto fetch = [&](int64_t c, Agent &ag, RowChunks<W, H, TPE> &rc) {
        int64_t e = c * EPW + le;
        if (e >= n) e = n - 1;
        ag = load_agent_ro(agent, e);
        rc.prefetch(grid + e * cell_stride, j);
    };
    if (ch < n_chunks) fetch(ch, a, cells);
    for (int it = 0; ch < n_chunks; ch += stride, it++) {
        const bool more = ch + stride < n_chunks;
        if (more) fetch(ch + stride, a_next, cells_next);
        const int64_t e0 = ch * EPW;
        const int ne = (int)((n - e0) < EPW ? (n - e0) : EPW);
        if constexpr (OUT_U8)
            warp_feature_chunk_u8<W, H, WIN, TPE, KC>(wbuf_s, out + e0 * nf, ne, cells, a, K, nf);
        else
            warp_feature_chunk<W, H, WIN, TPE, KC, USE_TMA, PSK_ESZ_FEATURES_KERNEL>(wbuf_s, it, out + e0 * nf, ne, cells, a,
                                                                                     K, nf);
        if (more) {
            a = a_next;
            cells = cells_next;
        }
    }
    if (USE_TMA && lane == 0) bulk_wait_read<0>();  // smem must outlive the last store's read
}

// =============================================================================================
// reset / advance  (worlds/craft.py:258-273; trainers/imitation.py:63-73)
// =============================================================================================
__global__ void __launch_bounds__(256)
craft_reset_kernel(uint8_t *__restrict__ grid, uint8_t *__restrict__ agent,
                   const uint8_t *__restrict__ scen_grid, const int32_t *__restrict__ scen_idx,
                   const uint8_t *__restrict__ init_agent, const uint8_t *__restrict__ mask,
                   int64_t n, int cell_stride) {
    // one 16-byte chunk per thread: chunks [0, cs/16) are the grid row, the last two the agent
    const int chunks = cell_stride / 16 + 2;
    const int64_t total = n * chunks;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / chunks;
        const int c = (int)(i % chunks);
        if (mask && !mask[e]) continue;
        if (c < cell_stride / 16) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(
                                      scen_grid + (int64_t)scen_idx[e] * cell_stride) + c);
            reinterpret_cast<uint4 *>(grid + e * cell_stride)[c] = v;
        } else {
            const int h = c - cell_stride / 16;
            reinterpret_cast<uint4 *>(agent + e * PSK_AGENT_BYTES)[h] =
                __ldg(reinterpret_cast<const uint4 *>(init_agent + e * PSK_AGENT_BYTES) + h);
        }
    }
}

// Per-env end of a rollout tick.  Cells are read through `rd` (global row or its shared copy) and
// written through `row` (global).  Returns true when the episode ended (state was reset).
template <int W, int H>
__device__ __forceinline__ bool advance_env(const SharedTables &st, Agent &a, uint8_t *row,
                                            const uint8_t *rd, int act, const uint8_t *scen_row,
                                            const uint8_t *init_agent_row, int cell_stride,
                                            bool &success, uint32_t &flags) {
    const int timer = a.timer() - 1;                          // imitation.py:63
    const bool done = (act == PSK_ACT_STOP) || timer <= 0;    // imitation.py:64-65
    if (done) {
        const int facing = facing_kind<W, H>(a, rd);
        success = st.task_len(a.task())
                      ? node_satisfied(st.node(a.task(), 0), a, facing) == 1
                      : false;                                // imitation.py:69
        // auto-reset: CraftScenario.init (craft.py:270-273)
        for (int c = 0; c < cell_stride / 16; c++)
            reinterpret_cast<uint4 *>(row)[c] = __ldg(reinterpret_cast<const uint4 *>(scen_row) + c);
        const uint4 lo = __ldg(reinterpret_cast<const uint4 *>(init_agent_row));
        const uint4 hi = __ldg(reinterpret_cast<const uint4 *>(init_agent_row) + 1);
        a.w[0] = lo.x; a.w[1] = lo.y; a.w[2] = lo.z; a.w[3] = lo.w;
        a.w[4] = hi.x; a.w[5] = hi.y; a.w[6] = hi.z; a.w[7] = hi.w;
    } else {
        success = false;
        step_env<W, H>(st, a, row, rd, act, flags);           // imitation.py:72
        a.set_timer(timer);
    }
    return done;
}

__device__ __forceinline__ void add_stats(unsigned long long *stats, bool done, bool success,
                                          bool counted) {
    const unsigned full = __activemask();
    const int n_done = __popc(__ballot_sync(full, done));
    const int n_succ = __popc(__ballot_sync(full, success));
    const int n_step = __popc(__ballot_sync(full, counted));
    const int leader = __ffs(full) - 1;
    if (stats && (int)(threadIdx.x & 31) == leader) {
        if (n_done) atomicAdd(stats + 0, (unsigned long long)n_done);
        if (n_succ) atomicAdd(stats + 1, (unsigned long long)n_succ);
        if (n_step) atomicAdd(stats + 2, (unsigned long long)n_step);
    }
}

template <int W, int H>
__global__ void __launch_bounds__(256)
craft_advance_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                     uint8_t *__restrict__ agent, const uint8_t *__restrict__ action,
                     const uint8_t *__restrict__ scen_grid, const int32_t *__restrict__ scen_idx,
                     const uint8_t *__restrict__ init_agent, uint8_t *__restrict__ done_out,
                     uint8_t *__restrict__ success_out, unsigned long long *stats,
                     int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        Agent a = load_agent(agent, e);
        bool success;
        const bool done = advance_env<W, H>(st, a, grid + e * cell_stride,
                                            grid + e * cell_stride, action[e],
                                            scen_grid + (int64_t)scen_idx[e] * cell_stride,
                                            init_agent + e * PSK_AGENT_BYTES, cell_stride,
                                            success, flags);
        store_agent(agent, e, a);
        if (done_out) done_out[e] = done;
        if (success_out) success_out[e] = success;
        add_stats(stats, done, success, true);
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// =============================================================================================
// fused tick: expert + features + advance, state read once
// =============================================================================================
// Warp-specialised: CTA = NE env threads + NFW feature warps = one super-tile of NE envs at a time.
//   all warps      : coalesced 128-bit copy of the super-tile's grid rows and agent records into
//                    shared memory (the only read of the state).
//   env warps      (one env per thread): teacher action (hint walk + bitboard floods), then
//                    advance (step / done / success / auto-reset) with write-back to HBM.
//   feature warps  : each an autonomous pipeline over its share of the super-tile's envs
//                    (warp_feature_chunk: zero-fill + scatter into its smem buffers, TMA store).
// The integer-ALU-bound teacher and the store-bound feature stream therefore overlap inside
// every CTA instead of alternating.
// OUT = float: the reference's f32 feature rows; OUT = uint8_t: the compact byte frame
// (psk_craft_tick_u8 / psk_craft_rollout_u8; vector-store path only: the tile IS the frame).
// STEP_FIRST: PSK_TICK_STEP_FIRST, a separate instantiation so that the other orders' code is
// exactly what it was without it.  On 10 x 10 grids it is held to 80 registers, the budget of the
// other orders' instantiations there (left alone, ptxas takes up to 126 and fits 4 CTAs per SM
// instead of 6).
template <int W, int H, int WIN, int NE, int NFW, int KC, bool USE_TMA, typename OUT = float,
          bool STEP_FIRST = false>
__global__ void __launch_bounds__(NE + NFW * 32,
                                  STEP_FIRST && W * H > 64 ? 65536 / ((NE + NFW * 32) * 80) : 0)
craft_tick_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                  uint8_t *__restrict__ agent, const uint8_t *__restrict__ action_in,
                  const uint8_t *__restrict__ scen_grid, const int32_t *__restrict__ scen_idx,
                  const uint8_t *__restrict__ init_agent, OUT *__restrict__ features_out,
                  uint8_t *__restrict__ expert_out, uint8_t *__restrict__ done_out,
                  uint8_t *__restrict__ success_out, unsigned long long *stats,
                  int32_t *err_flags, int64_t n, int cell_stride, int K, int nf, int adv_first,
                  uint32_t *chain, int64_t chain_g0) {
    if constexpr (STEP_FIRST) adv_first = 1;
    constexpr int NT = NE + NFW * 32;
    constexpr int TPE = 8, EPW = 32 / TPE;
    constexpr int SPW = NE / NFW;              // env slots per feature warp
    static_assert(SPW % EPW == 0, "feature warps take whole chunks");
    constexpr int CP = ((W * H + 63) / 64) * 64;
    constexpr int NW4 = (W * H + 15) / 16;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ SharedTables st;
    __shared__ __align__(16) uint8_t s_rows[NE * CP];
    __shared__ __align__(16) uint32_t s_agent[NE * 8];
    __shared__ uint32_t s_ticket[NE / PSK_CHAIN_GROUP];
    const int tid = threadIdx.x;
    const bool env_warp = tid < NE;
    // tile chaining (psk_common.cuh): one ticket per group of envs this CTA owns, taken before the
    // next grid may launch; chain == NULL (persistent grids, huge batches) falls back to waiting
    // for the whole previous grid
    const int64_t grp0 = (int64_t)blockIdx.x * (NE / PSK_CHAIN_GROUP);
    // groups are identified by the ADDRESS of their agent records (chain_g0 = group of env 0), so
    // that launches on different slices of one batch agree on which counters guard which envs
    auto grp = [&](int j) { return (chain_g0 + grp0 + j) & (PSK_CHAIN_GROUPS - 1); };
    const bool chain_thread = chain && tid < NE / PSK_CHAIN_GROUP &&
                              (grp0 + tid) * PSK_CHAIN_GROUP < n;
    // The table loads are ISSUED first and committed to shared memory after the ticket round trip:
    // the two global latencies of a CTA's start-up overlap instead of adding up (a single-tick CTA
    // lives ~10 us, ~3 us of which used to be start-up latency: ticket, tables, state).
    constexpr int TW = (int)(sizeof(psk_craft_tables) / 16);
    uint4 tv[(TW + NT - 1) / NT];
#pragma unroll
    for (int k = 0; k < (TW + NT - 1) / NT; k++)
        if (tid + k * NT < TW) tv[k] = __ldg(reinterpret_cast<const uint4 *>(T) + tid + k * NT);
    uint32_t flags = 0;             // PSK_FLAG_* seen by this thread, OR-ed into *err_flags at the end
    if (chain) {
        if (chain_thread) s_ticket[tid] = chain_enter(chain, grp(tid));
        __syncthreads();
    }
    // Programmatic dependent launch: let the next kernel in the stream (normally the next tick)
    // be scheduled while this one drains, and do everything that does not depend on the previous
    // kernel (tables, buffer init) before waiting for it.  Both are no-ops for a plain launch.
    asm volatile("griddepcontrol.launch_dependents;");
    if (!USE_TMA && !env_warp && features_out)
        feature_buffer_init<8, KC, USE_TMA, PSK_ESZ_FUSED_KERNELS>(
            smem_u32(smem_raw) + (uint32_t)((tid - NE) >> 5) * feature_buffer_bytes(false, 4, nf, PSK_ESZ_FUSED_KERNELS),
            nf);
#pragma unroll
    for (int k = 0; k < (TW + NT - 1) / NT; k++)
        if (tid + k * NT < TW) reinterpret_cast<uint4 *>(st.words)[tid + k * NT] = tv[k];
    if (chain) {
        if (chain_thread && !chain_wait(chain, grp(tid), s_ticket[tid])) flags = PSK_FLAG_CHAIN_TIMEOUT;
        __syncthreads();            // nobody touches the state before the chain threads' acquire
    } else {
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    // (without chaining the tables become visible with the barrier that follows the state load)
    int it = 0;  // this feature warp's chunk counter
    const int64_t n_super = (n + NE - 1) / NE;
    for (int64_t sp = blockIdx.x; sp < n_super; sp += gridDim.x) {
        const int64_t e_base = sp * NE;
        const int ne_sp = (int)((n - e_base) < NE ? (n - e_base) : NE);
        {   // ---- state super-tile -> shared memory
            const uint4 *grow = reinterpret_cast<const uint4 *>(grid + e_base * CP);
            uint4 *srow = reinterpret_cast<uint4 *>(s_rows);
            for (int i = tid; i < ne_sp * (CP / 16); i += NT) srow[i] = grow[i];
            const uint4 *gag = reinterpret_cast<const uint4 *>(agent + e_base * PSK_AGENT_BYTES);
            uint4 *sag = reinterpret_cast<uint4 *>(s_agent);
            for (int i = tid; i < ne_sp * 2; i += NT) sag[i] = gag[i];
        }
        __syncthreads();
        if (adv_first) {
            // "step, then observe" (PSK_TICK_ADVANCE_FIRST, or PSK_TICK_STEP_FIRST without the episode
            // rules): the env threads apply action_in to the tile in shared memory first — the teacher
            // and the feature warps then see the NEW state
            if (env_warp && tid < ne_sp) {
                const int64_t e = e_base + tid;
                bool done = false, success = false;
                if (action_in) {
                    Agent a;
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const uint4 v = reinterpret_cast<const uint4 *>(s_agent)[tid * 2 + i];
                        a.w[4 * i] = v.x; a.w[4 * i + 1] = v.y; a.w[4 * i + 2] = v.z; a.w[4 * i + 3] = v.w;
                    }
                    const Agent before = a;
                    uint8_t *srow_w = s_rows + tid * CP;
                    const int act = action_in[e];
                    if constexpr (STEP_FIRST)   // CraftState.step only: no timer, no done, no auto-reset
                        step_env<W, H>(st, a, srow_w, srow_w, act, flags);
                    else
                        done = advance_env<W, H>(st, a, srow_w, srow_w, act,
                                                 scen_grid + (int64_t)scen_idx[e] * CP,
                                                 init_agent + e * PSK_AGENT_BYTES, CP, success, flags);
                    bool changed = false;
#pragma unroll
                    for (int i = 0; i < 8; i++) changed |= a.w[i] != before.w[i];
                    if (changed) {
                        store_agent(agent, e, a);
                        uint4 *sag = reinterpret_cast<uint4 *>(s_agent) + tid * 2;
                        sag[0] = make_uint4(a.w[0], a.w[1], a.w[2], a.w[3]);
                        sag[1] = make_uint4(a.w[4], a.w[5], a.w[6], a.w[7]);
                    }
                    if (done || act == PSK_ACT_USE) {      // the only transitions that touch cells
#pragma unroll
                        for (int i = 0; i < CP / 16; i++)
                            reinterpret_cast<uint4 *>(grid + e * CP)[i] = reinterpret_cast<const uint4 *>(srow_w)[i];
                    }
                }
                if (done_out) done_out[e] = done;
                if (success_out) success_out[e] = success;
                if constexpr (!STEP_FIRST) add_stats(stats, done, success, action_in != nullptr);
            }
            __syncthreads();
        }
        if (env_warp) {
            const bool live = tid < ne_sp;
            const int slot = live ? tid : 0;             // dead lanes replay slot 0, unsaved
            const int64_t e = e_base + slot;
            bool done = false, success = false;
            Agent a;
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const uint4 v = reinterpret_cast<const uint4 *>(s_agent)[slot * 2 + i];
                a.w[4 * i] = v.x; a.w[4 * i + 1] = v.y; a.w[4 * i + 2] = v.z; a.w[4 * i + 3] = v.w;
            }
            const uint8_t *srow = s_rows + slot * CP;
            uint32_t words[NW4 * 4];
#pragma unroll
            for (int i = 0; i < NW4; i++) {
                const uint4 v = reinterpret_cast<const uint4 *>(srow)[i];
                words[4 * i] = v.x; words[4 * i + 1] = v.y; words[4 * i + 2] = v.z; words[4 * i + 3] = v.w;
            }
            const int facing = facing_kind<W, H>(a, srow);
            int dist;
            uint32_t fl = 0;
            int act = expert_env<W, H>(st, a, a.task(), words, facing, dist, fl);
            if (live) flags |= fl;
            if (live && adv_first) expert_out[e] = (uint8_t)act;
            if (live && !adv_first) {
                const Agent before = a;
                expert_out[e] = (uint8_t)act;
                if (action_in) act = action_in[e];
                done = advance_env<W, H>(st, a, grid + e * CP, srow, act,
                                         scen_grid + (int64_t)scen_idx[e] * CP,
                                         init_agent + e * PSK_AGENT_BYTES, CP, success, flags);
                bool changed = false;
#pragma unroll
                for (int i = 0; i < 8; i++) changed |= a.w[i] != before.w[i];
                if (changed) store_agent(agent, e, a);
                if (done_out) done_out[e] = done;
                if (success_out) success_out[e] = success;
            }
            if (!adv_first) add_stats(stats, done, success, live);
        } else if (features_out) {
            const int fw = (tid - NE) >> 5, lane = tid & 31;
            const uint32_t wbuf_s = smem_u32(smem_raw) + (uint32_t)fw * feature_buffer_bytes(USE_TMA, EPW, nf, PSK_ESZ_FUSED_KERNELS);
            for (int c = 0; c < SPW / EPW; c++) {
                const int s0 = fw * SPW + c * EPW;      // first env slot of the chunk
                if (s0 >= ne_sp) break;
                const int ne = (ne_sp - s0) < EPW ? (ne_sp - s0) : EPW;
                int se = s0 + lane / TPE;
                if (se >= ne_sp) se = s0;
                Agent b;
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const uint4 v = reinterpret_cast<const uint4 *>(s_agent)[se * 2 + i];
                    b.w[4 * i] = v.x; b.w[4 * i + 1] = v.y; b.w[4 * i + 2] = v.z; b.w[4 * i + 3] = v.w;
                }
                RowChunks<W, H, TPE> cells;
                cells.load(s_rows + se * CP, lane % TPE);
                if constexpr (sizeof(OUT) == 1) {
                    static_assert(sizeof(OUT) != 1 || (!USE_TMA && PSK_ESZ_FUSED_KERNELS == 1), "u8 frame: vector path, u8 tile");
                    warp_feature_chunk_u8<W, H, WIN, TPE, KC>(wbuf_s, features_out + (e_base + s0) * nf, ne,
                                                              cells, b, K, nf);
                } else {
                    warp_feature_chunk<W, H, WIN, TPE, KC, USE_TMA, PSK_ESZ_FUSED_KERNELS>(
                        wbuf_s, it, features_out + (e_base + s0) * nf, ne, cells, b, K, nf);
                }
                it++;
            }
        }
        __syncthreads();  // s_rows / s_agent are recycled by the next super-tile
    }
    if (chain_thread) chain_leave(chain, grp(tid), s_ticket[tid]);   // after the barrier above
    if (USE_TMA && !env_warp && (tid & 31) == 0) bulk_wait_read<0>();
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// =============================================================================================
// multi-tick rollout: the fused tick with the tick loop inside the kernel
// =============================================================================================
// Environments never interact, so a CTA can keep its NE envs for `ticks` consecutive ticks: the
// state lives in shared memory (double-buffered: the feature warps read the state of tick t while
// the env warps write the state of tick t+1) and in the env threads' registers; HBM sees one
// state read, one state write and `ticks` feature/action frames per launch.  This removes the
// per-tick launch, table staging and state reload, which is what bounds the single-tick kernel
// at 65,536 envs.  Valid whenever the actions do not depend on anything outside the kernel:
// teacher-driven rollouts (action_in == NULL) or replay of given action sequences.
//   action_in   u8[ticks][n] or NULL;  expert_out u8[ticks][n];  done_out/success_out u8[ticks][n] or NULL
//   features_out f32[feat_ring][n][nf] or NULL: tick t writes slot t % feat_ring
// Register cap: 896 threads per SM at 72 registers, i.e. 7 CTAs of 64 + 2 warps (128 threads) or
// 9 CTAs of 32 + 2 warps (96 threads); one register more and a CTA less fits per SM (17.5 -> 21 us
// per tick at 65,536 envs when a change pushed the kernel to 80 registers).
__host__ __device__ constexpr int rollout_threads(int ne, int nfw) { return (ne + 31) / 32 * 32 + nfw * 32; }
template <int W, int H, int WIN, int NE, int NFW, int KC, bool USE_TMA, typename OUT = float>
__global__ void __launch_bounds__(rollout_threads(NE, NFW),
                                  (W * H <= 64 && rollout_threads(NE, NFW) <= 128) ? 896 / rollout_threads(NE, NFW) : 1)
craft_rollout_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                     uint8_t *__restrict__ agent, const uint8_t *__restrict__ action_in,
                     const uint8_t *__restrict__ scen_grid, const int32_t *__restrict__ scen_idx,
                     const uint8_t *__restrict__ init_agent, OUT *__restrict__ features_out,
                     int feat_ring, uint8_t *__restrict__ expert_out, uint8_t *__restrict__ done_out,
                     uint8_t *__restrict__ success_out, unsigned long long *stats,
                     int32_t *err_flags, int64_t n, int cell_stride, int K, int nf, int ticks,
                     uint32_t *chain, int64_t chain_g0) {
    constexpr int NEW = (NE + 31) / 32 * 32;   // env-warp threads (lanes >= NE idle when NE < 32)
    constexpr int NT = NEW + NFW * 32;
    constexpr int TPE = 8, EPW = 32 / TPE;
    constexpr int SPW = NE / NFW;
    static_assert(SPW % EPW == 0, "feature warps take whole chunks");
    constexpr int CP = ((W * H + 63) / 64) * 64;
    constexpr int NW4 = (W * H + 15) / 16;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ SharedTables st;
    __shared__ __align__(16) uint8_t s_rows[2][NE * CP];
    __shared__ __align__(16) uint32_t s_agent[2][NE * 8];
    __shared__ uint32_t s_ticket[NE / PSK_CHAIN_GROUP];
    const int tid = threadIdx.x;
    const bool env_warp = tid < NEW;
    const int64_t grp0 = (int64_t)blockIdx.x * (NE / PSK_CHAIN_GROUP);     // tile chaining, see the tick kernel
    auto grp = [&](int j) { return (chain_g0 + grp0 + j) & (PSK_CHAIN_GROUPS - 1); };
    const bool chain_thread = chain && tid < NE / PSK_CHAIN_GROUP &&
                              (grp0 + tid) * PSK_CHAIN_GROUP < n;
    uint32_t flags = 0;
    if (chain) {
        if (chain_thread) s_ticket[tid] = chain_enter(chain, grp(tid));
        __syncthreads();
    }
    asm volatile("griddepcontrol.launch_dependents;");
    stage_tables(st, T);
    if (!USE_TMA && !env_warp && features_out)
        feature_buffer_init<8, KC, USE_TMA, PSK_ESZ_FUSED_KERNELS>(
            smem_u32(smem_raw) + (uint32_t)((tid - NEW) >> 5) * feature_buffer_bytes(false, 4, nf, PSK_ESZ_FUSED_KERNELS),
            nf);
    if (chain) {
        if (chain_thread && !chain_wait(chain, grp(tid), s_ticket[tid])) flags = PSK_FLAG_CHAIN_TIMEOUT;
        __syncthreads();
    } else {
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    int it = 0;
    const int64_t n_super = (n + NE - 1) / NE;
    for (int64_t sp = blockIdx.x; sp < n_super; sp += gridDim.x) {
        const int64_t e_base = sp * NE;
        const int ne_sp = (int)((n - e_base) < NE ? (n - e_base) : NE);
        {   // ---- state super-tile -> shared memory (buffer 0)
            const uint4 *grow = reinterpret_cast<const uint4 *>(grid + e_base * CP);
            uint4 *srow = reinterpret_cast<uint4 *>(s_rows[0]);
            for (int i = tid; i < ne_sp * (CP / 16); i += NT) srow[i] = grow[i];
            const uint4 *gag = reinterpret_cast<const uint4 *>(agent + e_base * PSK_AGENT_BYTES);
            uint4 *sag = reinterpret_cast<uint4 *>(s_agent[0]);
            for (int i = tid; i < ne_sp * 2; i += NT) sag[i] = gag[i];
        }
        __syncthreads();
        const bool live = env_warp && tid < ne_sp;   // ne_sp <= NE
        const int slot = live ? tid : 0;
        const int64_t e = e_base + slot;
        Agent a;
        const uint8_t *scen_row = nullptr;
        int n_done = 0, n_succ = 0;
        if (env_warp) {
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const uint4 v = reinterpret_cast<const uint4 *>(s_agent[0])[slot * 2 + i];
                a.w[4 * i] = v.x; a.w[4 * i + 1] = v.y; a.w[4 * i + 2] = v.z; a.w[4 * i + 3] = v.w;
            }
            scen_row = scen_grid + (int64_t)scen_idx[e] * CP;
        }
        for (int t = 0; t < ticks; t++) {
            const int cur = t & 1, nxt = cur ^ 1;
            if (env_warp) {
                const uint8_t *srow = s_rows[cur] + slot * CP;
                uint8_t *nrow = s_rows[nxt] + slot * CP;
                uint32_t words[NW4 * 4];
#pragma unroll
                for (int i = 0; i < NW4; i++) {
                    const uint4 v = reinterpret_cast<const uint4 *>(srow)[i];
                    words[4 * i] = v.x; words[4 * i + 1] = v.y; words[4 * i + 2] = v.z; words[4 * i + 3] = v.w;
                    if (live) reinterpret_cast<uint4 *>(nrow)[i] = v;     // next state starts as a copy
                }
                const int facing = facing_kind<W, H>(a, srow);
                int dist;
                uint32_t fl = 0;
                int act = expert_env<W, H>(st, a, a.task(), words, facing, dist, fl);
                if (live) {
                    flags |= fl;
                    const int64_t o = (int64_t)t * n + e;
                    expert_out[o] = (uint8_t)act;
                    if (action_in) act = action_in[o];
                    bool success;
                    const bool done = advance_env<W, H>(st, a, nrow, srow, act, scen_row,
                                                        init_agent + e * PSK_AGENT_BYTES, CP,
                                                        success, flags);
                    if (done_out) done_out[o] = done;
                    if (success_out) success_out[o] = success;
                    n_done += done;
                    n_succ += success;
                    uint4 *sag = reinterpret_cast<uint4 *>(s_agent[nxt]) + slot * 2;
                    sag[0] = make_uint4(a.w[0], a.w[1], a.w[2], a.w[3]);
                    sag[1] = make_uint4(a.w[4], a.w[5], a.w[6], a.w[7]);
                }
            } else if (features_out) {
                const int fw = (tid - NEW) >> 5, lane = tid & 31;
                const uint32_t wbuf_s = smem_u32(smem_raw) +
                                        (uint32_t)fw * feature_buffer_bytes(USE_TMA, EPW, nf, PSK_ESZ_FUSED_KERNELS);
                OUT *fout = features_out + (int64_t)(t % feat_ring) * n * nf;
                for (int c = 0; c < SPW / EPW; c++) {
                    const int s0 = fw * SPW + c * EPW;
                    if (s0 >= ne_sp) break;
                    const int ne = (ne_sp - s0) < EPW ? (ne_sp - s0) : EPW;
                    int se = s0 + lane / TPE;
                    if (se >= ne_sp) se = s0;
                    Agent b;
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const uint4 v = reinterpret_cast<const uint4 *>(s_agent[cur])[se * 2 + i];
                        b.w[4 * i] = v.x; b.w[4 * i + 1] = v.y; b.w[4 * i + 2] = v.z; b.w[4 * i + 3] = v.w;
                    }
                    RowChunks<W, H, TPE> cells;
                    cells.load(s_rows[cur] + se * CP, lane % TPE);
                    if constexpr (sizeof(OUT) == 1) {
                        static_assert(sizeof(OUT) != 1 || (!USE_TMA && PSK_ESZ_FUSED_KERNELS == 1), "u8 frame: vector path, u8 tile");
                        warp_feature_chunk_u8<W, H, WIN, TPE, KC>(wbuf_s, fout + (e_base + s0) * nf, ne, cells,
                                                                  b, K, nf);
                    } else {
                        warp_feature_chunk<W, H, WIN, TPE, KC, USE_TMA, PSK_ESZ_FUSED_KERNELS>(
                            wbuf_s, it, fout + (e_base + s0) * nf, ne, cells, b, K, nf);
                    }
                    it++;
                }
            }
            __syncthreads();   // state of tick t+1 complete, state of tick t no longer read
        }
        // ---- final state -> HBM, statistics
        if (env_warp) {
            if (live) {
                store_agent(agent, e, a);
                const uint8_t *frow = s_rows[ticks & 1] + slot * CP;
#pragma unroll
                for (int i = 0; i < NW4; i++)
                    reinterpret_cast<uint4 *>(grid + e * CP)[i] = reinterpret_cast<const uint4 *>(frow)[i];
            }
            const int d = __reduce_add_sync(0xffffffffu, n_done);
            const int sc = __reduce_add_sync(0xffffffffu, n_succ);
            const int lv = __reduce_add_sync(0xffffffffu, live ? ticks : 0);
            if (stats && (tid & 31) == 0) {
                if (d) atomicAdd(stats + 0, (unsigned long long)d);
                if (sc) atomicAdd(stats + 1, (unsigned long long)sc);
                if (lv) atomicAdd(stats + 2, (unsigned long long)lv);
            }
        }
        __syncthreads();
    }
    if (chain_thread) chain_leave(chain, grp(tid), s_ticket[tid]);   // after the barrier above
    if (USE_TMA && !env_warp && (tid & 31) == 0) bulk_wait_read<0>();
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// =============================================================================================
// host side: dispatch on (width, height, window)
// =============================================================================================
static int num_sms() {
    static int sms[PSK_MAX_DEVICES] = {0};
    const int dev = current_device();
    if (!sms[dev]) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sms[dev] = n > 0 ? n : 148;
    }
    return sms[dev];
}

// Run-time tuning knobs (psk_set_tuning in include/psk_craft.h): -1 = automatic.  Each knob starts
// from the environment variable PSK_<NAME> (upper case) the first time any knob is read, and can be
// changed at any time afterwards, so tests and A/B runs can force every kernel variant.
enum TuneKey { TUNE_ROLLOUT_VARIANT, TUNE_ROLLOUT_TMA, TUNE_TICK_VARIANT, TUNE_TICK_TMA,
               TUNE_TICK_PERSIST, TUNE_FEAT_PERSIST, TUNE_TICK_PDL, TUNE_STEP_VARIANT,
               TUNE_TILE_CHAIN, TUNE_COUNT };
static const char *const tune_names[TUNE_COUNT] = {
    "rollout_variant", "rollout_tma", "tick_variant", "tick_tma", "tick_persist", "feat_persist",
    "tick_pdl", "step_variant", "tile_chain"};
static std::atomic<int> tune_val[TUNE_COUNT];
static std::once_flag tune_once;
static void tune_init() {
    for (int i = 0; i < TUNE_COUNT; i++) {
        char name[64] = "PSK_";
        size_t j = 4;
        for (const char *c = tune_names[i]; *c && j + 1 < sizeof(name); c++)
            name[j++] = (char)(*c >= 'a' && *c <= 'z' ? *c - 32 : *c);
        name[j] = 0;
        const char *v = getenv(name);
        tune_val[i].store(v ? atoi(v) : -1);
    }
}
static inline int tune(TuneKey k) {
    std::call_once(tune_once, tune_init);
    return tune_val[k].load(std::memory_order_relaxed);
}

static inline int grid_for(int64_t n, int block, int ctas_per_sm) {
    int64_t need = (n + block - 1) / block;
    int64_t cap = (int64_t)num_sms() * ctas_per_sm;
    return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

static inline int check(cudaError_t e) { return e == cudaSuccess ? PSK_OK : PSK_ERR_CUDA; }

// Device copies of the callers' tables: a small per-device cache keyed by content, so that batches
// with different tables (or on different streams) never share a slot that is being rewritten.
// Filling a slot is a pageable H2D copy: it must not happen inside a CUDA-graph capture, so call any
// entry point once with new tables before capturing (every caller's warm-up does).  When more than
// SLOTS distinct tables are alive on a device the oldest slot is recycled after a device-wide sync.
static const psk_craft_tables *device_tables(const psk_craft_tables *caller_tables, cudaStream_t st) {
    constexpr int MAX_DEV = PSK_MAX_DEVICES, SLOTS = 8;
    struct Slot {
        psk_craft_tables host;
        psk_craft_tables *dev = nullptr;
    };
    struct PerDevice {
        Slot slot[SLOTS];
        int used = 0, last = 0, next_victim = 0;
    };
    static PerDevice cache[MAX_DEV];
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
    // ws_recipes is derived data: always rebuilt from recipes[] here, whatever the caller put there
    psk_craft_tables canon = *caller_tables;
    memset(canon.ws_recipes, 0, sizeof(canon.ws_recipes));
    for (int r = 0; r < canon.n_recipes && r < PSK_MAX_RECIPES; r++)
        canon.ws_recipes[canon.recipes[r][1] & (PSK_MAX_KINDS - 1)] |= (uint16_t)(1u << r);
    const psk_craft_tables *t = &canon;
    std::lock_guard<std::mutex> lock(mu);
    PerDevice &c = cache[dev];
    if (c.used && memcmp(&c.slot[c.last].host, t, sizeof(psk_craft_tables)) == 0) return c.slot[c.last].dev;
    for (int i = 0; i < c.used; ++i)
        if (memcmp(&c.slot[i].host, t, sizeof(psk_craft_tables)) == 0) {
            c.last = i;
            return c.slot[i].dev;
        }
    int i;
    if (c.used < SLOTS) {
        i = c.used;
        if (cudaMalloc(&c.slot[i].dev, sizeof(psk_craft_tables)) != cudaSuccess) return nullptr;
        ++c.used;
    } else {
        i = c.next_victim;
        c.next_victim = (c.next_victim + 1) % SLOTS;
        if (cudaDeviceSynchronize() != cudaSuccess) return nullptr;   // nobody may still read the slot
    }
    memset(&c.slot[i].host, 0xFF, sizeof(psk_craft_tables));           // invalid until the copy is queued
    if (cudaMemcpyAsync(c.slot[i].dev, t, sizeof(psk_craft_tables), cudaMemcpyHostToDevice, st) != cudaSuccess)
        return nullptr;
    // kernels on other streams may use this slot later: make the copy visible to them as well
    if (cudaStreamSynchronize(st) != cudaSuccess) return nullptr;
    c.slot[i].host = *t;
    c.last = i;
    return c.slot[i].dev;
}
// Tile-chaining counters (psk_common.cuh), one zero-initialised array per device, allocated on the
// first call (like the table copies: outside a CUDA-graph capture).  NULL = do not chain.
static uint32_t *chain_counters(const psk_craft_state &s, int64_t *g0) {
    static uint32_t *ctr[PSK_MAX_DEVICES] = {nullptr};
    static std::mutex mu;
    const int64_t n = s.n;
    if (tune(TUNE_TILE_CHAIN) == 0 || tune(TUNE_TICK_PDL) == 0) return nullptr;
    if ((n + PSK_CHAIN_GROUP - 1) / PSK_CHAIN_GROUP > PSK_CHAIN_GROUPS) return nullptr;
    // groups are keyed by the address of their agent records: only batches (or slices) that start
    // on a group boundary chain; anything else waits for the whole previous grid
    constexpr uintptr_t GROUP_BYTES = (uintptr_t)PSK_CHAIN_GROUP * PSK_AGENT_BYTES;
    if (reinterpret_cast<uintptr_t>(s.agent) % GROUP_BYTES) return nullptr;
    *g0 = (int64_t)(reinterpret_cast<uintptr_t>(s.agent) / GROUP_BYTES);
    const int dev = current_device();
    std::lock_guard<std::mutex> lock(mu);
    if (!ctr[dev]) {
        const size_t bytes = (size_t)2 * PSK_CHAIN_GROUPS * sizeof(uint32_t);
        if (cudaMalloc(&ctr[dev], bytes) != cudaSuccess) return nullptr;
        if (cudaMemset(ctr[dev], 0, bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
            cudaFree(ctr[dev]);
            ctr[dev] = nullptr;
        }
    }
    return ctr[dev];
}

#define PSK_DT(var)                                   \
    const psk_craft_tables *var = device_tables(t, st); \
    if (!var) return PSK_ERR_CUDA

template <int W, int H, int WIN> struct Config {
    static constexpr int CP = ((W * H + 63) / 64) * 64;
    static constexpr int TPE = 8;   // threads per env in the feature scatter
    // <= 128 cells: one env per thread on 64/128-bit bitboards; larger: one env per warp, row per lane
    static constexpr bool BITBOARD = W * H <= 128;

    static bool matches(const psk_craft_tables *t) {
        return t->width == W && t->height == H && t->window_w == WIN && t->window_h == WIN &&
               t->n_kinds <= PSK_MAX_INV;
    }
    static int nf(const psk_craft_tables *t) { return 2 * WIN * WIN * t->n_kinds + t->n_kinds + 5; }

    static int step(const psk_craft_tables *t, psk_craft_state s, const uint8_t *action,
                    const uint8_t *active, float *reward, int32_t *err, cudaStream_t st) {
        PSK_DT(dt);
        // step_variant: 0 (default) tables staged in shared memory, 256-thread CTAs; 1 tables through
        // the read-only path, 64-thread CTAs; 2 = 1 + row preload.  Same box, 65,536 envs, after the
        // per-workshop recipe mask: 3.07 / ~3.3 / 3.6 us (profiles/README.md) — with the USE path
        // short, staging once per CTA beats per-thread table loads again.
        int mode = tune(TUNE_STEP_VARIANT);
        if (mode < 0 || mode > 2) mode = 0;
        if (mode == 2 && CP != 64) mode = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.blockDim = dim3(mode == 0 ? 256 : 64);
        cfg.gridDim = dim3((unsigned)(mode == 0 ? grid_for(s.n, 256, 8) : grid_for(s.n, 64, 32)));
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = tune(TUNE_TICK_PDL) != 0 ? 1 : 0;
        const int cell_stride = s.cell_stride;
        const int64_t n = s.n;
        if (mode == 0)
            return check(cudaLaunchKernelEx(&cfg, craft_step_kernel<W, H, 0>, dt, s.grid, s.agent, action,
                                            active, reward, err, n, cell_stride));
        if constexpr (CP == 64) {
            if (mode == 2)
                return check(cudaLaunchKernelEx(&cfg, craft_step_kernel<W, H, 2>, dt, s.grid, s.agent,
                                                action, active, reward, err, n, cell_stride));
        }
        return check(cudaLaunchKernelEx(&cfg, craft_step_kernel<W, H, 1>, dt, s.grid, s.agent, action,
                                        active, reward, err, n, cell_stride));
    }
    static int satisfies(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                         uint8_t *out, cudaStream_t st) {
        PSK_DT(dt);
        craft_satisfies_kernel<W, H><<<grid_for(s.n, 256, 8), 256, 0, st>>>(
            dt, s.grid, s.agent, task, out, s.n, s.cell_stride);
        return check(cudaGetLastError());
    }
    static int expert(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                      uint8_t *action, int16_t *dist, int32_t *err, cudaStream_t st) {
        PSK_DT(dt);
        if constexpr (BITBOARD)
            craft_expert_kernel<W, H><<<grid_for(s.n, 128, 8), 128, 0, st>>>(
                dt, s.grid, s.agent, task, action, dist, err, s.n, s.cell_stride);
        else if constexpr (W <= 16 && H <= 32)      // two envs per warp (half a warp of rows each)
            craft_expert_half_rows_kernel<W, H><<<grid_for((s.n + 1) / 2, 4, 16), 128, 0, st>>>(
                dt, s.grid, s.agent, task, action, dist, err, s.n, s.cell_stride);
        else
            craft_expert_rows_kernel<W, H><<<grid_for(s.n, 4, 16), 128, 0, st>>>(
                dt, s.grid, s.agent, task, action, dist, err, s.n, s.cell_stride);
        return check(cudaGetLastError());
    }
    static int find_closest(const psk_craft_tables *t, psk_craft_state s, const uint8_t *kind,
                            uint8_t *goal, int16_t *len, uint8_t *seq, int seq_cap,
                            cudaStream_t st) {
        PSK_DT(dt);
        if constexpr (BITBOARD)
            craft_find_closest_kernel<W, H><<<grid_for(s.n, 128, 8), 128, 0, st>>>(
                dt, s.grid, s.agent, kind, goal, len, seq, seq_cap, s.n, s.cell_stride);
        else
            craft_find_closest_rows_kernel<W, H><<<grid_for(s.n, 4, 16), 128, 0, st>>>(
                s.grid, s.agent, kind, goal, len, seq, seq_cap, s.n, s.cell_stride);
        return check(cudaGetLastError());
    }
    template <bool TMA, typename OUT = float>
    static int features_impl(const psk_craft_tables *t, psk_craft_state s, OUT *out,
                             cudaStream_t st) {
        constexpr int WPB = 4, EPW = 32 / TPE;
        const int f = nf(t);
        const size_t smem = (size_t)WPB * feature_buffer_bytes(TMA, EPW, f, PSK_ESZ_FEATURES_KERNEL);
        // the default cookbook has 21 kinds: that case is compiled with K fixed
        auto kern = t->n_kinds == 21 ? craft_features_kernel<W, H, WIN, WPB, TPE, 21, TMA, OUT>
                                     : craft_features_kernel<W, H, WIN, WPB, TPE, 0, TMA, OUT>;
        // opt in to > 48 KB dynamic smem (both instantiations, once per size)
        static size_t configured_on[PSK_MAX_DEVICES] = {0};   // the attribute is per device
        size_t &configured = configured_on[current_device()];
        if (configured != smem) {
            if (cudaFuncSetAttribute(craft_features_kernel<W, H, WIN, WPB, TPE, 21, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(craft_features_kernel<W, H, WIN, WPB, TPE, 0, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
                return PSK_ERR_CUDA;
            configured = smem;
        }
        int per_sm = (int)((224 * 1024) / (smem + 1024));
        if (per_sm > 16) per_sm = 16;
        const int64_t ctas = (s.n + (int64_t)WPB * EPW - 1) / ((int64_t)WPB * EPW);
        int64_t g = (int64_t)num_sms() * (per_sm > 0 ? per_sm : 1);
        // One CTA per tile, dispatched in index order, keeps the DRAM write front compact:
        // 270 us vs 330 us at 1 M envs for a persistent grid-stride grid (profiles/README.md).
        const int persist = tune(TUNE_FEAT_PERSIST) > 0;
        if (g > ctas || !persist) g = ctas > 0 ? ctas : 1;
        kern<<<(int)g, WPB * 32, smem, st>>>(s.grid, s.agent, out, s.n, s.cell_stride, t->n_kinds, f);
        return check(cudaGetLastError());
    }
    static int features(const psk_craft_tables *t, psk_craft_state s, float *out, int impl,
                        cudaStream_t st) {
        if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) impl = 1;
        return impl == 2 ? features_impl<true>(t, s, out, st) : features_impl<false>(t, s, out, st);
    }
    static int features_u8(const psk_craft_tables *t, psk_craft_state s, uint8_t *out, cudaStream_t st) {
        return features_impl<false, uint8_t>(t, s, out, st);
    }
    static int advance(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                       const uint8_t *action, uint8_t *done, uint8_t *success,
                       unsigned long long *stats, int32_t *err, cudaStream_t st) {
        PSK_DT(dt);
        craft_advance_kernel<W, H><<<grid_for(s.n, 256, 8), 256, 0, st>>>(
            dt, s.grid, s.agent, action, ep.scen_grid, ep.scen_idx, ep.init_agent, done, success,
            stats, err, s.n, s.cell_stride);
        return check(cudaGetLastError());
    }
    template <int NE, int NFW, bool TMA, typename OUT = float>
    static int tick_variant(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                            const uint8_t *action_in, OUT *features_out, uint8_t *expert_out,
                            uint8_t *done, uint8_t *success, unsigned long long *stats,
                            int32_t *err, cudaStream_t st, int adv_first) {
        constexpr int EPW = 32 / TPE;
        const int f = nf(t);
        const size_t smem = (size_t)NFW * feature_buffer_bytes(TMA, EPW, f, PSK_ESZ_FUSED_KERNELS);
        auto kern = adv_first == 2
                        ? (t->n_kinds == 21 ? craft_tick_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT, true>
                                            : craft_tick_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT, true>)
                        : (t->n_kinds == 21 ? craft_tick_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT>
                                            : craft_tick_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT>);
        static size_t configured_on[PSK_MAX_DEVICES] = {0};   // the attribute is per device
        size_t &configured = configured_on[current_device()];
        if (configured != smem) {
            if (cudaFuncSetAttribute(craft_tick_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(craft_tick_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(craft_tick_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT, true>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(craft_tick_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT, true>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
                return PSK_ERR_CUDA;
            configured = smem;
        }
        const size_t static_smem = sizeof(SharedTables) + (size_t)NE * (CP + 32);
        int per_sm = (int)((224 * 1024) / (smem + static_smem + 1024));
        const int by_threads = 2048 / (NE + NFW * 32);
        if (per_sm > by_threads) per_sm = by_threads;
        const int64_t tiles = (s.n + NE - 1) / NE;
        int64_t g = (int64_t)num_sms() * (per_sm > 0 ? per_sm : 1);
        const int persist = tune(TUNE_TICK_PERSIST) > 0;   // see features_impl: in-order tiles win
        if (g > tiles || !persist) g = tiles > 0 ? tiles : 1;
        PSK_DT(dt);
        const int pdl = tune(TUNE_TICK_PDL) != 0;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)g);
        cfg.blockDim = dim3(NE + NFW * 32);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = pdl ? 1 : 0;
        const int cell_stride = s.cell_stride, K = t->n_kinds;
        int64_t chain_g0 = 0;
        // one tile per CTA only; not with TMA stores: a single-tick CTA would pay the release fence of
        // chain_leave while its bulk stores are in flight (1 M envs, same box: 342 us chained vs 304 not;
        // vector stores at 262,144 envs: 72.4 chained vs 78.5 not — profiles/README.md)
        uint32_t *chain = (g == tiles && pdl && !TMA) ? chain_counters(s, &chain_g0) : nullptr;
        return check(cudaLaunchKernelEx(&cfg, kern, dt, s.grid, s.agent, action_in, ep.scen_grid,
                                        ep.scen_idx, ep.init_agent, features_out, expert_out, done,
                                        success, stats, err, s.n, cell_stride, K, f, adv_first, chain,
                                        chain_g0));
    }
    template <int NE, int NFW, bool TMA, typename OUT = float>
    static int rollout_variant(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                               int ticks, const uint8_t *action_in, OUT *features_out,
                               int feat_ring, uint8_t *expert_out, uint8_t *done,
                               uint8_t *success, unsigned long long *stats, int32_t *err,
                               cudaStream_t st) {
        constexpr int EPW = 32 / TPE;
        const int f = nf(t);
        const size_t smem = (size_t)NFW * feature_buffer_bytes(TMA, EPW, f, PSK_ESZ_FUSED_KERNELS);
        auto kern = t->n_kinds == 21 ? craft_rollout_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT>
                                     : craft_rollout_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT>;
        static size_t configured_on[PSK_MAX_DEVICES] = {0};   // the attribute is per device
        size_t &configured = configured_on[current_device()];
        if (configured != smem) {
            if (cudaFuncSetAttribute(craft_rollout_kernel<W, H, WIN, NE, NFW, 21, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
                cudaFuncSetAttribute(craft_rollout_kernel<W, H, WIN, NE, NFW, 0, TMA, OUT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
                return PSK_ERR_CUDA;
            configured = smem;
        }
        const int64_t tiles = (s.n + NE - 1) / NE;
        PSK_DT(dt);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(tiles > 0 ? tiles : 1));
        cfg.blockDim = dim3(rollout_threads(NE, NFW));
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const int cell_stride = s.cell_stride, K = t->n_kinds;
        int64_t chain_g0 = 0;
        uint32_t *chain = chain_counters(s, &chain_g0);
        return check(cudaLaunchKernelEx(&cfg, kern, dt, s.grid, s.agent, action_in, ep.scen_grid,
                                        ep.scen_idx, ep.init_agent, features_out, feat_ring,
                                        expert_out, done, success, stats, err, s.n, cell_stride, K,
                                        f, ticks, chain, chain_g0));
    }
    static int rollout(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep, int ticks,
                       const uint8_t *action_in, float *features_out, int feat_ring,
                       uint8_t *expert_out, uint8_t *done, uint8_t *success,
                       unsigned long long *stats, int32_t *err, cudaStream_t st) {
        if constexpr (!BITBOARD) {
            return PSK_ERR_UNSUPPORTED;
        } else if constexpr (WIN != 3) {
            // craft_large (10 x 10, window 5, 128-bit boards, 1,076 features): the multi-tick kernel was
            // built and measured — 185 registers, 3 CTAs per SM, 73.6 us per tick at 65,536 envs against
            // 56.0 us for chained single ticks (profiles/README.md) — so psk_craft_rollout loops over
            // craft_tick_kernel launches for this geometry
            return PSK_ERR_UNSUPPORTED;
        } else {
            // CTA shape and store path (sweeps in profiles/README.md): 32 env threads + 2 feature warps
            // (96 threads, 9 CTAs per SM) at every batch size — in round 1 a single wave of 64 + 2 CTAs
            // won below 65,536 envs, with tile chaining the smaller CTAs win there too (32,768 envs:
            // 8.10 vs 8.65 us per tick; 4,096: 3.89 vs 4.87); vector stores up to 196,608 envs, TMA above.
            // rollout_variant (0 = 64 + 2, 2 = 32 + 2, 3 = 16 + 2, 4 = 16 + 1) and rollout_tma override.
            const int env_tma = tune(TUNE_ROLLOUT_TMA), env_variant = tune(TUNE_ROLLOUT_VARIANT);
            const int tma = env_tma >= 0 ? env_tma : (s.n > 196608 ? 1 : 0);
            const int variant = env_variant >= 0 ? env_variant : 2;
#define PSK_ROLLOUT_ARGS t, s, ep, ticks, action_in, features_out, feat_ring, expert_out, done, success, stats, err, st
            if (variant == 2)
                return tma ? rollout_variant<32, 2, true>(PSK_ROLLOUT_ARGS)
                           : rollout_variant<32, 2, false>(PSK_ROLLOUT_ARGS);
            if (variant == 3)   // 16 envs per CTA (half an env warp) + 2 feature warps: 3 waves at 65,536 envs
                return tma ? rollout_variant<16, 2, true>(PSK_ROLLOUT_ARGS)
                           : rollout_variant<16, 2, false>(PSK_ROLLOUT_ARGS);
            if (variant == 4)   // 16 envs + 1 feature warp (64 threads, 14 CTAs per SM)
                return tma ? rollout_variant<16, 1, true>(PSK_ROLLOUT_ARGS)
                           : rollout_variant<16, 1, false>(PSK_ROLLOUT_ARGS);
            return tma ? rollout_variant<64, 2, true>(PSK_ROLLOUT_ARGS)
                       : rollout_variant<64, 2, false>(PSK_ROLLOUT_ARGS);
#undef PSK_ROLLOUT_ARGS
        }
    }
    // the byte frame through the fused kernels: one CTA shape (32 + 2), vector stores
    static int tick_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                       const uint8_t *action_in, uint8_t *features_out, uint8_t *expert_out, uint8_t *done,
                       uint8_t *success, unsigned long long *stats, int32_t *err, cudaStream_t st,
                       int adv_first) {
        if constexpr (!BITBOARD) {
            return PSK_ERR_UNSUPPORTED;
        } else if constexpr (WIN != 3) {
            return tick_variant<64, 2, false, uint8_t>(t, s, ep, action_in, features_out, expert_out, done,
                                                       success, stats, err, st, adv_first);
        } else {
            return tick_variant<32, 2, false, uint8_t>(t, s, ep, action_in, features_out, expert_out, done,
                                                       success, stats, err, st, adv_first);
        }
    }
    static int rollout_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep, int ticks,
                          const uint8_t *action_in, uint8_t *features_out, int feat_ring,
                          uint8_t *expert_out, uint8_t *done, uint8_t *success,
                          unsigned long long *stats, int32_t *err, cudaStream_t st) {
        if constexpr (!BITBOARD || WIN != 3) {
            return PSK_ERR_UNSUPPORTED;
        } else {
            return rollout_variant<32, 2, false, uint8_t>(t, s, ep, ticks, action_in, features_out, feat_ring,
                                                          expert_out, done, success, stats, err, st);
        }
    }
    static int tick_fused(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                          const uint8_t *action_in, float *features_out, uint8_t *expert_out,
                          uint8_t *done, uint8_t *success, unsigned long long *stats,
                          int32_t *err, cudaStream_t st, int adv_first) {
        if constexpr (!BITBOARD) {
            return PSK_ERR_UNSUPPORTED;   // psk_craft_tick falls back to the three-kernel pipeline
        } else {
        // Defaults from the sweeps in profiles/README.md: 32 env threads + 2 feature warps at
        // every batch size measured (65,536: 20.4 vs 20.9 us for 64 + 2; 262,144: 71.2 vs 72.9),
        // vector stores up to 262,144 envs, TMA stores above (1 M: 294 vs 318 us).
        // PSK_TICK_VARIANT / PSK_TICK_TMA override.
        const int env_variant = tune(TUNE_TICK_VARIANT), env_tma = tune(TUNE_TICK_TMA);
        const bool big = s.n > 262144;
        const int variant = env_variant >= 0 ? env_variant : 4;
        const int tma = env_tma >= 0 ? env_tma : (big ? 1 : 0);
#define PSK_TV(NE, NFW)                                                                          \
    return tma ? tick_variant<NE, NFW, true>(t, s, ep, action_in, features_out, expert_out, done, \
                                             success, stats, err, st, adv_first)                 \
               : tick_variant<NE, NFW, false>(t, s, ep, action_in, features_out, expert_out, done, \
                                              success, stats, err, st, adv_first)
        if constexpr (WIN != 3) {
            (void)variant;
            PSK_TV(64, 2);
        } else {
            switch (variant) {
                case 1: PSK_TV(128, 4);
                case 2: PSK_TV(32, 1);
                case 3: PSK_TV(64, 4);
                case 4: PSK_TV(32, 2);
                default: PSK_TV(64, 2);
            }
        }
#undef PSK_TV
        }
    }
};

using Medium = Config<8, 8, 3>;    // configs/worlds/craft_medium.yaml
using Large = Config<10, 10, 5>;   // configs/worlds/craft_large.yaml
using Stress16 = Config<16, 16, 3>;  // enlarged-grid stress tests (BASELINE configs[4])
using Stress32 = Config<32, 32, 3>;
using Stress64 = Config<64, 64, 3>;

#define PSK_DISPATCH(t, CALL)                             \
    do {                                                  \
        if (Medium::matches(t)) return Medium::CALL;      \
        if (Large::matches(t)) return Large::CALL;        \
        if (Stress16::matches(t)) return Stress16::CALL;  \
        if (Stress32::matches(t)) return Stress32::CALL;  \
        if (Stress64::matches(t)) return Stress64::CALL;  \
        return PSK_ERR_UNSUPPORTED;                       \
    } while (0)

static bool state_ok(const psk_craft_tables *t, const psk_craft_state &s) {
    if (!t || s.n < 0) return false;
    if (s.n == 0) return true;
    if (!s.grid || !s.agent) return false;
    const int need = ((t->width * t->height + 63) / 64) * 64;
    if (s.cell_stride != need) return false;
    if ((reinterpret_cast<uintptr_t>(s.grid) & 15) || (reinterpret_cast<uintptr_t>(s.agent) & 31))
        return false;
    return true;
}

}  // namespace psk

using namespace psk;

extern "C" {

const char *psk_version(void) { return "psketch_b200 0.2 sm_100a"; }

int psk_set_tuning(const char *key, int32_t value) {
    if (!key) return PSK_ERR_BADARG;
    tune(TUNE_ROLLOUT_VARIANT);   // environment defaults are read before the first override
    for (int i = 0; i < TUNE_COUNT; i++)
        if (strcmp(key, tune_names[i]) == 0) {
            tune_val[i].store(value);
            return PSK_OK;
        }
    return PSK_ERR_BADARG;
}

int psk_get_tuning(const char *key, int32_t *value) {
    if (!key || !value) return PSK_ERR_BADARG;
    for (int i = 0; i < TUNE_COUNT; i++)
        if (strcmp(key, tune_names[i]) == 0) {
            *value = tune((TuneKey)i);
            return PSK_OK;
        }
    return PSK_ERR_BADARG;
}

int psk_craft_supported(const psk_craft_tables *t) {
    if (!t) return 0;
    return Medium::matches(t) || Large::matches(t) || Stress16::matches(t) || Stress32::matches(t) ||
           Stress64::matches(t);
}

int psk_craft_n_features(const psk_craft_tables *t) {
    if (!psk_craft_supported(t)) return -1;
    return 2 * t->window_w * t->window_h * t->n_kinds + t->n_kinds + 5;
}

int psk_craft_step(const psk_craft_tables *t, psk_craft_state s, const uint8_t *action,
                   const uint8_t *active, float *reward, int32_t *err_flags, void *stream) {
    if (!state_ok(t, s) || (!action && s.n)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, step(t, s, action, active, reward, err_flags, (cudaStream_t)stream));
}

int psk_craft_features(const psk_craft_tables *t, psk_craft_state s, float *out, int impl,
                       void *stream) {
    if (!state_ok(t, s) || (!out && s.n)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, features(t, s, out, impl, (cudaStream_t)stream));
}

int psk_craft_features_u8(const psk_craft_tables *t, psk_craft_state s, uint8_t *out, void *stream) {
    if (!state_ok(t, s) || (!out && s.n)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, features_u8(t, s, out, (cudaStream_t)stream));
}

int psk_craft_satisfies(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                        uint8_t *out, void *stream) {
    if (!state_ok(t, s) || (!out && s.n)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, satisfies(t, s, task, out, (cudaStream_t)stream));
}

int psk_craft_expert(const psk_craft_tables *t, psk_craft_state s, const uint8_t *task,
                     uint8_t *action, int16_t *dist, int32_t *err_flags, void *stream) {
    if (!state_ok(t, s) || (!action && s.n)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, expert(t, s, task, action, dist, err_flags, (cudaStream_t)stream));
}

int psk_craft_find_closest(const psk_craft_tables *t, psk_craft_state s, const uint8_t *kind,
                           uint8_t *goal, int16_t *length, uint8_t *seq, int32_t seq_cap,
                           void *stream) {
    if (!state_ok(t, s) || ((!kind || !goal || !length) && s.n) || seq_cap < 0)
        return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    PSK_DISPATCH(t, find_closest(t, s, kind, goal, length, seq, seq_cap, (cudaStream_t)stream));
}

int psk_craft_reset(psk_craft_state s, psk_craft_episodes ep, const uint8_t *mask, void *stream) {
    if (s.n < 0 || s.cell_stride <= 0 || s.cell_stride % 64) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    if (!s.grid || !s.agent || !ep.scen_grid || !ep.scen_idx || !ep.init_agent)
        return PSK_ERR_BADARG;
    const int64_t total = s.n * (s.cell_stride / 16 + 2);
    craft_reset_kernel<<<grid_for(total, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        s.grid, s.agent, ep.scen_grid, ep.scen_idx, ep.init_agent, mask, s.n, s.cell_stride);
    return check(cudaGetLastError());
}

// craft_tick_kernel's adv_first argument for a tick order: 0 = observe, then advance (PSK_TICK_FUSED);
// 1 = advance, then observe (PSK_TICK_ADVANCE_FIRST); 2 = step, then observe (PSK_TICK_STEP_FIRST)
static int tick_order_arg(int order) {
    return order == PSK_TICK_ADVANCE_FIRST ? 1 : order == PSK_TICK_STEP_FIRST ? 2 : 0;
}

int psk_craft_tick(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                   const uint8_t *action_in, float *features_out, uint8_t *expert_out,
                   uint8_t *done_out, uint8_t *success_out, unsigned long long *stats,
                   int32_t *err_flags, int fused, void *stream) {
    if (!state_ok(t, s)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    if (!expert_out || !ep.scen_grid || !ep.scen_idx || !ep.init_agent) return PSK_ERR_BADARG;
    if (features_out && (reinterpret_cast<uintptr_t>(features_out) & 15)) return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int adv_first = tick_order_arg(fused);
    if (fused && t->width * t->height <= 128) {
        PSK_DISPATCH(t, tick_fused(t, s, ep, action_in, features_out, expert_out, done_out,
                                   success_out, stats, err_flags, st, adv_first));
    }
    if (adv_first) {        // step, then observe — as separate launches (grids above 128 cells)
        if (action_in && adv_first == 2) {      // CraftState.step only; done / success stay 0
            const int rc = psk_craft_step(t, s, action_in, nullptr, nullptr, err_flags, stream);
            if (rc) return rc;
        }
        if (action_in && adv_first == 1) {
            int rc = PSK_ERR_UNSUPPORTED;
            do {
                if (Medium::matches(t)) { rc = Medium::advance(t, s, ep, action_in, done_out, success_out, stats, err_flags, st); break; }
                if (Large::matches(t)) { rc = Large::advance(t, s, ep, action_in, done_out, success_out, stats, err_flags, st); break; }
                if (Stress16::matches(t)) { rc = Stress16::advance(t, s, ep, action_in, done_out, success_out, stats, err_flags, st); break; }
                if (Stress32::matches(t)) { rc = Stress32::advance(t, s, ep, action_in, done_out, success_out, stats, err_flags, st); break; }
                if (Stress64::matches(t)) { rc = Stress64::advance(t, s, ep, action_in, done_out, success_out, stats, err_flags, st); break; }
            } while (0);
            if (rc) return rc;
        } else {
            if (done_out && cudaMemsetAsync(done_out, 0, (size_t)s.n, st) != cudaSuccess) return PSK_ERR_CUDA;
            if (success_out && cudaMemsetAsync(success_out, 0, (size_t)s.n, st) != cudaSuccess) return PSK_ERR_CUDA;
        }
        int rc = psk_craft_expert(t, s, nullptr, expert_out, nullptr, err_flags, stream);
        if (rc) return rc;
        return features_out ? psk_craft_features(t, s, features_out, 0, stream) : PSK_OK;
    }
    int rc = psk_craft_expert(t, s, nullptr, expert_out, nullptr, err_flags, stream);
    if (rc) return rc;
    if (features_out) {
        rc = psk_craft_features(t, s, features_out, 0, stream);
        if (rc) return rc;
    }
    const uint8_t *act = action_in ? action_in : expert_out;
    PSK_DISPATCH(t, advance(t, s, ep, act, done_out, success_out, stats, err_flags, st));
}

// Fault injection for the tile-chaining safety net (tests only): hands out one ticket of the group that
// owns env `env` of this batch without ever finishing it — what an aborted launch leaves behind.  The
// next fused launch on these envs must time out on that group (PSK_FLAG_CHAIN_TIMEOUT), not hang, and
// leave the counters in step again.
__global__ void chain_skip_ticket_kernel(uint32_t *chain, int64_t g) { atomicAdd(chain + 2 * g, 1u); }

int psk_debug_chain_skip_ticket(psk_craft_state s, int64_t env, void *stream) {
    if (env < 0 || env >= s.n || !s.agent) return PSK_ERR_BADARG;
    int64_t g0 = 0;
    uint32_t *chain = chain_counters(s, &g0);
    if (!chain) return PSK_ERR_UNSUPPORTED;          // this batch does not chain
    const int64_t g = (g0 + env / PSK_CHAIN_GROUP) & (PSK_CHAIN_GROUPS - 1);
    chain_skip_ticket_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(chain, g);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_craft_tick_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                      const uint8_t *action_in, uint8_t *features_out, uint8_t *expert_out,
                      uint8_t *done_out, uint8_t *success_out, unsigned long long *stats,
                      int32_t *err_flags, int order, void *stream) {
    if (!state_ok(t, s)) return PSK_ERR_BADARG;
    if (s.n == 0) return PSK_OK;
    if (!expert_out || !features_out || !ep.scen_grid || !ep.scen_idx || !ep.init_agent) return PSK_ERR_BADARG;
    if (reinterpret_cast<uintptr_t>(features_out) & 3) return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int adv_first = tick_order_arg(order);
    if (t->width * t->height <= 128)
        PSK_DISPATCH(t, tick_u8(t, s, ep, action_in, features_out, expert_out, done_out, success_out, stats,
                                err_flags, st, adv_first));
    // grids above 128 cells: the feature kernel writes the bytes, the tick does the rest
    if (!adv_first) {
        const int rc = psk_craft_features_u8(t, s, features_out, stream);
        if (rc) return rc;
    }
    int rc = psk_craft_tick(t, s, ep, action_in, nullptr, expert_out, done_out, success_out, stats, err_flags,
                            order, stream);
    if (!rc && adv_first) rc = psk_craft_features_u8(t, s, features_out, stream);
    return rc;
}

int psk_craft_rollout_u8(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                         int32_t ticks, const uint8_t *action_in, uint8_t *features_out,
                         int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                         uint8_t *success_out, unsigned long long *stats, int32_t *err_flags,
                         void *stream) {
    if (!state_ok(t, s) || ticks < 0 || !features_out || feat_ring <= 0) return PSK_ERR_BADARG;
    if (s.n == 0 || ticks == 0) return PSK_OK;
    if (!expert_out || !ep.scen_grid || !ep.scen_idx || !ep.init_agent) return PSK_ERR_BADARG;
    if (reinterpret_cast<uintptr_t>(features_out) & 3) return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = PSK_ERR_UNSUPPORTED;
    if (Medium::matches(t))
        rc = Medium::rollout_u8(t, s, ep, ticks, action_in, features_out, feat_ring, expert_out, done_out,
                                success_out, stats, err_flags, st);
    if (rc != PSK_ERR_UNSUPPORTED) return rc;
    const int nfeat = psk_craft_n_features(t);
    for (int k = 0; k < ticks; k++) {
        const int64_t o = (int64_t)k * s.n;
        rc = psk_craft_tick_u8(t, s, ep, action_in ? action_in + o : nullptr,
                               features_out + (int64_t)(k % feat_ring) * s.n * nfeat, expert_out + o,
                               done_out ? done_out + o : nullptr, success_out ? success_out + o : nullptr,
                               stats, err_flags, PSK_TICK_FUSED, stream);
        if (rc) return rc;
    }
    return PSK_OK;
}

int psk_craft_rollout(const psk_craft_tables *t, psk_craft_state s, psk_craft_episodes ep,
                      int32_t ticks, const uint8_t *action_in, float *features_out,
                      int32_t feat_ring, uint8_t *expert_out, uint8_t *done_out,
                      uint8_t *success_out, unsigned long long *stats, int32_t *err_flags,
                      void *stream) {
    if (!state_ok(t, s) || ticks < 0 || (features_out && feat_ring <= 0)) return PSK_ERR_BADARG;
    if (s.n == 0 || ticks == 0) return PSK_OK;
    if (!expert_out || !ep.scen_grid || !ep.scen_idx || !ep.init_agent) return PSK_ERR_BADARG;
    if (features_out && (reinterpret_cast<uintptr_t>(features_out) & 15)) return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = PSK_ERR_UNSUPPORTED;
    if (Medium::matches(t))
        rc = Medium::rollout(t, s, ep, ticks, action_in, features_out, feat_ring, expert_out, done_out,
                             success_out, stats, err_flags, st);

    if (rc != PSK_ERR_UNSUPPORTED) return rc;
    // other geometries: one fused / pipelined tick per iteration, same outputs
    const int nfeat = psk_craft_n_features(t);
    for (int k = 0; k < ticks; k++) {
        const int64_t o = (int64_t)k * s.n;
        rc = psk_craft_tick(t, s, ep, action_in ? action_in + o : nullptr,
                            features_out ? features_out + (int64_t)(k % feat_ring) * s.n * nfeat : nullptr,
                            expert_out + o, done_out ? done_out + o : nullptr,
                            success_out ? success_out + o : nullptr, stats, err_flags, 1, stream);
        if (rc) return rc;
    }
    return PSK_OK;
}

}  // extern "C"
