// psk_craft_generic.cu — the Craft primitives for every geometry of the generic domain
// (include/psk_craft.h: 1 <= W, H <= 64, odd windows of 1..9 cells on each axis, n_kinds <= 24).
//
// The specialised kernels of psk_craft.cu are templates on (W, H, WIN) and are built for five
// geometries.  The kernels here read W, H, the window and K from the device tables at run time, so
// one build serves any world yaml the reference accepts; psk_craft.cu dispatches to them when no
// specialised configuration matches (or when the tuning key `generic` forces them).  Algorithms are
// those of the specialised kernels:
//   craft_generic_step_kernel / _satisfies / _advance   one env per thread (step_env, advance_env)
//   craft_generic_expert_kernel / _find_closest         one env per warp: hint walk, then the two
//                                                       floods of bfs_rows on boards of u64 rows,
//                                                       rows 2l and 2l+1 in lane l
//   craft_generic_features_kernel                       one env per warp: zero-filled byte row in
//                                                       shared memory, scatter of the non-zeros,
//                                                       coalesced read-out as f32 or u8
#include "psk_common.cuh"

namespace psk {

__device__ __forceinline__ bool on_grid(int x, int y, int W, int H) {
    return x >= 0 && y >= 0 && x < W && y < H;
}

// step_env (psk_craft.cu) with W, H as values; worlds/craft.py:332-424
__device__ __forceinline__ void gen_step_env(const SharedTables &st, int W, int H, Agent &a,
                                             uint8_t *row, int act, uint32_t &flags) {
    int x = a.x(), y = a.y(), dir = a.dir();
    if (act < 4) {  // craft.py:341-352 + 418-421: turn always, move iff the target cell is free
        dir = act;
        const int tx = x + dx_of(act), ty = y + dy_of(act);
        if (on_grid(tx, ty, W, H) && row[tx * H + ty] == 0) {
            x = tx;
            y = ty;
        }
        a.set_pose(x, y, dir);
    } else if (act == PSK_ACT_USE) {  // craft.py:356-412
        const int fx = x + dx_of(dir), fy = y + dy_of(dir);
        if (on_grid(fx, fy, W, H)) {  // neighbors(), craft.py:426-437
            const int thing = row[fx * H + fy];
            const int cls = st.kind_class(thing);
            if (cls == KC_GRAB) {  // craft.py:383-386
                if (thing < PSK_MAX_INV) {
                    if (a.inv(thing) == 255) flags |= PSK_FLAG_INV_OVERFLOW;
                    else a.inv_add(thing, 1);
                }
                row[fx * H + fy] = 0;
            } else if (cls == KC_WORKSHOP) {  // craft.py:388-401: this workshop's recipes, file order
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

__device__ __forceinline__ int gen_facing_kind(const Agent &a, const uint8_t *row, int W, int H) {
    const int fx = a.x() + dx_of(a.dir()), fy = a.y() + dy_of(a.dir());
    return on_grid(fx, fy, W, H) ? row[fx * H + fy] : 0;
}

__global__ void __launch_bounds__(GENERIC_THREAD_CTA)
craft_generic_step_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                          uint8_t *__restrict__ agent, const uint8_t *__restrict__ action,
                          const uint8_t *__restrict__ active, float *__restrict__ reward,
                          int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int W = st.t().width, H = st.t().height;
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        if (reward) reward[e] = 0.0f;  // craft.py:338,424
        if (active && !active[e]) continue;
        Agent a = load_agent(agent, e);
        const Agent before = a;
        gen_step_env(st, W, H, a, grid + e * cell_stride, action[e], flags);
        bool changed = false;
#pragma unroll
        for (int i = 0; i < 8; i++) changed |= a.w[i] != before.w[i];
        if (changed) store_agent(agent, e, a);
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

__global__ void __launch_bounds__(GENERIC_THREAD_CTA)
craft_generic_satisfies_kernel(const psk_craft_tables *__restrict__ T,
                               const uint8_t *__restrict__ grid, const uint8_t *__restrict__ agent,
                               const uint8_t *__restrict__ task, uint8_t *__restrict__ out, int64_t n,
                               int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int W = st.t().width, H = st.t().height;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        const Agent a = load_agent_ro(agent, e);
        const int tk = task ? task[e] : a.task();
        const int facing = gen_facing_kind(a, grid + e * cell_stride, W, H);
        out[e] = st.task_len(tk) ? node_satisfied(st.node(tk, 0), a, facing) : 2;
    }
}

// advance_env (psk_craft.cu): timer / done / success / auto-reset, else step; imitation.py:63-73
__global__ void __launch_bounds__(GENERIC_THREAD_CTA)
craft_generic_advance_kernel(const psk_craft_tables *__restrict__ T, uint8_t *__restrict__ grid,
                             uint8_t *__restrict__ agent, const uint8_t *__restrict__ action,
                             const uint8_t *__restrict__ scen_grid, const int32_t *__restrict__ scen_idx,
                             const uint8_t *__restrict__ init_agent, uint8_t *__restrict__ done_out,
                             uint8_t *__restrict__ success_out, unsigned long long *stats,
                             int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int W = st.t().width, H = st.t().height;
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n;
         e += (int64_t)gridDim.x * blockDim.x) {
        Agent a = load_agent(agent, e);
        uint8_t *row = grid + e * cell_stride;
        const int act = action[e];
        const int timer = a.timer() - 1;                          // imitation.py:63
        const bool done = (act == PSK_ACT_STOP) || timer <= 0;    // imitation.py:64-65
        bool success = false;
        if (done) {
            const int facing = gen_facing_kind(a, row, W, H);
            success = st.task_len(a.task()) ? node_satisfied(st.node(a.task(), 0), a, facing) == 1
                                            : false;              // imitation.py:69
            // auto-reset: CraftScenario.init (craft.py:270-273)
            const uint4 *scen = reinterpret_cast<const uint4 *>(scen_grid + (int64_t)scen_idx[e] * cell_stride);
            for (int c = 0; c < cell_stride / 16; c++) reinterpret_cast<uint4 *>(row)[c] = __ldg(scen + c);
            const uint4 *ia = reinterpret_cast<const uint4 *>(init_agent + e * PSK_AGENT_BYTES);
            const uint4 lo = __ldg(ia), hi = __ldg(ia + 1);
            a.w[0] = lo.x; a.w[1] = lo.y; a.w[2] = lo.z; a.w[3] = lo.w;
            a.w[4] = hi.x; a.w[5] = hi.y; a.w[6] = hi.z; a.w[7] = hi.w;
        } else {
            gen_step_env(st, W, H, a, row, act, flags);           // imitation.py:72
            a.set_timer(timer);
        }
        store_agent(agent, e, a);
        if (done_out) done_out[e] = done;
        if (success_out) success_out[e] = success;
        add_stats(stats, done, success, true);
    }
    if (flags && err_flags) atomicOr(err_flags, (int)flags);
}

// =============================================================================================
// teacher: RowBoard of psk_craft.cu with W and H as values.  Two u64 rows per lane (rows 2l and
// 2l+1), so up to 64 rows of 64 cells; rows at or beyond W and bits at or beyond H stay zero.
// =============================================================================================
struct GenGeo {
    int W, H, lane;
    uint64_t hm;      // the H valid bits of a row
    bool v0, v1;      // this lane's rows lie on the grid
    __device__ __forceinline__ GenGeo(int W_, int H_, int lane_)
        : W(W_), H(H_), lane(lane_), hm(H_ == 64 ? ~0ull : ((1ull << H_) - 1)),
          v0(2 * lane_ < W_), v1(2 * lane_ + 1 < W_) {}
};

struct GenRows {
    static constexpr unsigned FULL = 0xffffffffu;
    uint64_t r0, r1;

    static __device__ __forceinline__ GenRows zero() { return GenRows{0, 0}; }
    static __device__ __forceinline__ GenRows bit(int x, int y, const GenGeo &g) {
        GenRows b{0, 0};
        if (x == 2 * g.lane) b.r0 = 1ull << y;
        if (x == 2 * g.lane + 1) b.r1 = 1ull << y;
        return b;
    }
    __device__ __forceinline__ GenRows operator&(const GenRows &o) const { return GenRows{r0 & o.r0, r1 & o.r1}; }
    __device__ __forceinline__ GenRows operator|(const GenRows &o) const { return GenRows{r0 | o.r0, r1 | o.r1}; }
    __device__ __forceinline__ bool lane_any() const { return (r0 | r1) != 0; }
    __device__ __forceinline__ bool any() const { return __any_sync(FULL, lane_any()); }
    __device__ __forceinline__ bool differs(const GenRows &o) const {
        return __any_sync(FULL, r0 != o.r0 || r1 != o.r1);
    }
    // free cells from an occupancy board: complement within the grid
    __device__ __forceinline__ GenRows free_of(const GenGeo &g) const {
        return GenRows{g.v0 ? (~r0 & g.hm) : 0ull, g.v1 ? (~r1 & g.hm) : 0ull};
    }
    // positions p + delta(A) for p in this board
    template <int A> __device__ __forceinline__ GenRows shift(const GenGeo &g) const {
        GenRows b;
        if (A == 0) {                                   // DOWN  (0,-1)
            b.r0 = r0 >> 1;
            b.r1 = r1 >> 1;
        } else if (A == 1) {                            // UP    (0,+1)
            b.r0 = (r0 << 1) & g.hm;
            b.r1 = (r1 << 1) & g.hm;
        } else if (A == 2) {                            // LEFT  (-1,0): row x <- row x+1
            const uint64_t nxt = __shfl_down_sync(FULL, r0, 1);
            b.r0 = r1;
            b.r1 = g.lane < 31 ? nxt : 0ull;
        } else {                                        // RIGHT (+1,0): row x <- row x-1
            const uint64_t prv = __shfl_up_sync(FULL, r1, 1);
            b.r1 = r0;
            b.r0 = g.lane > 0 ? prv : 0ull;
        }
        if (!g.v0) b.r0 = 0;
        if (!g.v1) b.r1 = 0;
        return b;
    }
    template <int A> __device__ __forceinline__ GenRows unshift(const GenGeo &g) const {
        return shift<(A ^ 1)>(g);
    }
    __device__ __forceinline__ GenRows spread(const GenGeo &g) const {
        return shift<0>(g) | shift<1>(g) | shift<2>(g) | shift<3>(g);
    }
    // row `x` of the board, broadcast to every lane
    __device__ __forceinline__ uint64_t row(int x) const {
        const uint64_t a = __shfl_sync(FULL, r0, x >> 1), b = __shfl_sync(FULL, r1, x >> 1);
        return (x & 1) ? b : a;
    }
    // lowest / highest cell in x-major order (np.nonzero order); false when empty
    __device__ __forceinline__ bool lowest(int &x, int &y) const {
        const unsigned m = __ballot_sync(FULL, lane_any());
        if (!m) return false;
        const int l = __ffs(m) - 1;
        const uint64_t a = __shfl_sync(FULL, r0, l), b = __shfl_sync(FULL, r1, l);
        const int slot = a == 0 ? 1 : 0;
        x = 2 * l + slot;
        y = __ffsll((long long)(slot ? b : a)) - 1;
        return true;
    }
    __device__ __forceinline__ bool highest(int &x, int &y) const {
        const unsigned m = __ballot_sync(FULL, lane_any());
        if (!m) return false;
        const int l = 31 - __clz(m);
        const uint64_t a = __shfl_sync(FULL, r0, l), b = __shfl_sync(FULL, r1, l);
        const int slot = b != 0 ? 1 : 0;
        x = 2 * l + slot;
        y = 63 - __clzll((long long)(slot ? b : a));
        return true;
    }
};

// occupancy / goal rows of this lane from the env's grid row (global memory); rows beyond the grid
// are solid
__device__ __forceinline__ void gen_build_rows(const uint8_t *row, const GenGeo &g, int goal_kind,
                                               GenRows &occ, GenRows &goal) {
    uint64_t o[2], q[2];
#pragma unroll
    for (int s = 0; s < 2; s++) {
        const int x = 2 * g.lane + s;
        uint64_t ov = g.hm, gv = 0;
        if (x < g.W) {
            ov = 0;
            const uint8_t *p = row + x * g.H;
            for (int y = 0; y < g.H; y++) {
                const int k = __ldg(p + y);
                ov |= uint64_t(k != 0) << y;
                gv |= uint64_t(k == goal_kind) << y;
            }
        }
        o[s] = ov;
        q[s] = goal_kind ? gv : 0ull;
    }
    occ = GenRows{o[0], o[1]};
    goal = GenRows{q[0], q[1]};
}

// bfs_rows (psk_craft.cu) on GenRows: returns the path length (-1 unreachable, 0 already facing);
// first = the teacher's first action, (gx, gy) = the chosen goal cell.  All lanes return the same.
__device__ __forceinline__ int gen_bfs_rows(bool need, const GenRows &occ, const GenRows &goal, int px,
                                            int py, int d0, const GenGeo &g, int &first, int &gx, int &gy) {
    const GenRows freeb = occ.free_of(g);
    const GenRows root = GenRows::bit(px, py, g);
    first = -1;
    gx = gy = -1;
    {   // depth 0: already facing a goal cell
        const int fx = px + dx_of(d0), fy = py + dy_of(d0);
        const bool in = on_grid(fx, fy, g.W, g.H);
        const uint64_t grow = goal.row(in ? fx : 0);
        if (need && in && ((grow >> fy) & 1)) {
            gx = fx;
            gy = fy;
            return 0;
        }
    }
    const GenRows T0 = goal.unshift<0>(g), T1 = goal.unshift<1>(g), T2 = goal.unshift<2>(g),
                  T3 = goal.unshift<3>(g);
    const GenRows src_all = T0 | T1 | T2 | T3 | (freeb & T0).unshift<0>(g) | (freeb & T1).unshift<1>(g) |
                            (freeb & T2).unshift<2>(g) | (freeb & T3).unshift<3>(g);
    if (!need || !goal.any()) return -1;
    GenRows VF = root;
    int k = 0;
    while (!(VF & src_all).any()) {
        const GenRows nv = VF | (VF.spread(g) & freeb);
        if (!nv.differs(VF)) return -1;                 // queue drained (base.py:87)
        VF = nv;
        k++;
    }
    const GenRows hit =
        ((VF & T0).shift<0>(g) | (VF & T1).shift<1>(g) | (VF & T2).shift<2>(g) | (VF & T3).shift<3>(g) |
         (VF.shift<0>(g) & freeb & T0).shift<0>(g) | (VF.shift<1>(g) & freeb & T1).shift<1>(g) |
         (VF.shift<2>(g) & freeb & T2).shift<2>(g) | (VF.shift<3>(g) & freeb & T3).shift<3>(g)) & goal;
    hit.lowest(gx, gy);                                 // lowest cell index (np.nonzero order)
    const GenRows gb = GenRows::bit(gx, gy, g);
    const GenRows g0 = gb.unshift<0>(g), g1 = gb.unshift<1>(g), g2 = gb.unshift<2>(g), g3 = gb.unshift<3>(g);
    const GenRows s0 = g0 | (freeb & g0).unshift<0>(g), s1 = g1 | (freeb & g1).unshift<1>(g),
                  s2 = g2 | (freeb & g2).unshift<2>(g), s3 = g3 | (freeb & g3).unshift<3>(g);
    if (k == 0) {
        first = (root & s0).any() ? 0 : (root & s1).any() ? 1 : (root & s2).any() ? 2 : 3;
        return 1;
    }
    GenRows VB = (s0 | s1 | s2 | s3) & VF;
    for (int j = 1; j < k; j++) VB = VB | (VB.spread(g) & freeb);
    const GenRows ok = VB & freeb;
    first = (root.shift<0>(g) & ok).any()   ? 0
            : (root.shift<1>(g) & ok).any() ? 1
            : (root.shift<2>(g) & ok).any() ? 2
                                            : 3;
    return k + 1;
}

__global__ void __launch_bounds__(GENERIC_WARP_CTA)
craft_generic_expert_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                            const uint8_t *__restrict__ agent, const uint8_t *__restrict__ task,
                            uint8_t *__restrict__ action, int16_t *__restrict__ dist_out,
                            int32_t *err_flags, int64_t n, int cell_stride) {
    __shared__ SharedTables st;
    stage_tables(st, T);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const GenGeo g(st.t().width, st.t().height, lane);
    uint32_t flags = 0;
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        const int tk = task ? task[e] : a.task();
        const int facing = gen_facing_kind(a, row, g.W, g.H);
        const uint32_t leaf = find_incomplete(st, tk, a, facing);
        const int kind = (leaf >> 16) & 0x0F;
        const bool need = leaf && kind == LEAF_GO;
        GenRows occ, goal;
        gen_build_rows(row, g, need ? (leaf >> 8) & 0xFF : 0, occ, goal);
        int first, gx, gy;
        const int d = gen_bfs_rows(need, occ, goal, a.x(), a.y(), a.dir(), g, first, gx, gy);
        int act;
        if (!leaf) act = PSK_ACT_STOP;                              // demonstration.py:15-16
        else if (kind == LEAF_USE) act = PSK_ACT_USE;               // demonstration.py:20-21
        else if (kind != LEAF_GO) { act = PSK_ACT_INVALID; flags |= PSK_FLAG_BAD_LEAF; }
        else if (d < 0) act = PSK_ACT_STOP;                         // demonstration.py:25-26
        else act = first >= 0 ? first : PSK_ACT_INVALID;
        if (lane == 0) {
            action[e] = (uint8_t)act;
            if (dist_out) dist_out[e] = (int16_t)(need ? d : -1);
        }
    }
    if (flags && err_flags && lane == 0) atomicOr(err_flags, (int)flags);
}

// find_closest_resources (teachers/base.py:27-34): length, goal cell and the lexicographically
// smallest action sequence (re-running the search towards the chosen cell after every move)
__global__ void __launch_bounds__(GENERIC_WARP_CTA)
craft_generic_find_closest_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                                  const uint8_t *__restrict__ agent, const uint8_t *__restrict__ kind,
                                  uint8_t *__restrict__ goal_out, int16_t *__restrict__ len_out,
                                  uint8_t *__restrict__ seq, int seq_cap, int64_t n, int cell_stride) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const GenGeo g(__ldg(&T->width), __ldg(&T->height), lane);
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        GenRows occ, goal;
        gen_build_rows(row, g, kind[e], occ, goal);
        int x = a.x(), y = a.y(), d = a.dir(), first, gx, gy;
        const int len = gen_bfs_rows(true, occ, goal, x, y, d, g, first, gx, gy);
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
            const GenRows g1 = len > 0 ? GenRows::bit(gx, gy, g) : GenRows::zero();
            int f = first;
            for (int k = 0; k < len; k++) {
                if (lane == 0 && k < seq_cap) sq[k] = (uint8_t)f;
                const int tx = x + dx_of(f), ty = y + dy_of(f);
                const bool in = on_grid(tx, ty, g.W, g.H);
                const uint64_t orow = occ.row(in ? tx : 0);
                if (in && !((orow >> ty) & 1)) { x = tx; y = ty; }
                d = f;
                if (k + 1 < len) {
                    int g2x, g2y;
                    gen_bfs_rows(true, occ, g1, x, y, d, g, f, g2x, g2y);
                }
            }
            for (int k = (len > 0 ? len : 0) + lane; k < seq_cap; k += 32) sq[k] = 255;
        }
    }
}

// =============================================================================================
// features (worlds/craft.py:296-330): local window (ww x wh x K, ravel order (dx, dy, kind)), the
// (ww^2 x wh^2) window max-pooled in ww x wh blocks (same size), inventory, direction one-hot, 0.
// The pooled window's centre block IS the local window, so one pass over its cells writes both.
// =============================================================================================
constexpr int GEN_MAX_WIN = 9;
constexpr int GEN_ROW_BYTES =
    ((2 * GEN_MAX_WIN * GEN_MAX_WIN * PSK_MAX_INV + PSK_MAX_INV + 5) + 15) / 16 * 16;   // 3,920

__global__ void __launch_bounds__(GENERIC_WARP_CTA)
craft_generic_features_kernel(const psk_craft_tables *__restrict__ T, const uint8_t *__restrict__ grid,
                              const uint8_t *__restrict__ agent, float *__restrict__ out_f32,
                              uint8_t *__restrict__ out_u8, int64_t n, int cell_stride) {
    __shared__ __align__(16) uint8_t s_rows[GENERIC_WARP_CTA / 32][GEN_ROW_BYTES];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int W = __ldg(&T->width), H = __ldg(&T->height), K = __ldg(&T->n_kinds);
    const int ww = __ldg(&T->window_w), wh = __ldg(&T->window_h);
    const int hw = ww / 2, hh = wh / 2;                       // craft.py:299-300
    const int bhw = (ww * ww) / 2, bhh = (wh * wh) / 2;       // craft.py:301-302
    const int nf = 2 * ww * wh * K + K + 5;
    const int big = ww * wh * K, tail = 2 * ww * wh * K;
    uint8_t *r = s_rows[warp];
    uint32_t *r4 = reinterpret_cast<uint32_t *>(r);
    const int nw = (nf + 3) / 4;
    for (int i = lane; i < nw; i += 32) r4[i] = 0;
    for (int64_t e = blockIdx.x * (int64_t)wpb + warp; e < n; e += (int64_t)gridDim.x * wpb) {
        const Agent a = load_agent_ro(agent, e);
        const uint8_t *row = grid + e * cell_stride;
        const int px = a.x(), py = a.y();
        __syncwarp();                                         // the zero fill has landed
        // the on-grid part of the pooled window
        const int x0 = max(px - bhw, 0), x1 = min(px + bhw, W - 1);
        const int y0 = max(py - bhh, 0), y1 = min(py + bhh, H - 1);
        const int ny = y1 - y0 + 1, cells = (x1 - x0 + 1) * ny;
        for (int i = lane; i < cells; i += 32) {
            const int x = x0 + i / ny, y = y0 + i % ny;
            const int k = __ldg(row + x * H + y);
            if (k == 0 || k >= K) continue;
            const int bx = x - px + bhw, by = y - py + bhh;
            const int bi = bx / ww, bj = by / wh;
            r[big + (bi * wh + bj) * K + k] = 1;
            if (bi == hw && bj == hh) r[((bx - hw * ww) * wh + (by - hh * wh)) * K + k] = 1;
        }
        if (lane < K) r[tail + lane] = (uint8_t)a.inv(lane);   // craft.py:325
        if (lane == 0) r[tail + K + a.dir()] = 1;              // craft.py:321-322; last feature 0
        __syncwarp();
        // read-out, then the row's words back to zero for the next env
        if (out_f32) {
            float *o = out_f32 + e * nf;
            for (int j = lane; j < nf; j += 32) o[j] = (float)r[j];
        } else {
            uint8_t *o = out_u8 + e * nf;
            for (int j = lane; j < nf; j += 32) o[j] = r[j];
        }
        __syncwarp();
        for (int i = lane; i < nw; i += 32) r4[i] = 0;
    }
}

// =============================================================================================
// host launchers (dispatch: psk_craft.cu)
// =============================================================================================
static inline int launched() { return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA; }

int generic_step(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *action,
                 const uint8_t *active, float *reward, int32_t *err, cudaStream_t st) {
    craft_generic_step_kernel<<<grid, GENERIC_THREAD_CTA, 0, st>>>(dt, s.grid, s.agent, action, active, reward,
                                                                   err, s.n, s.cell_stride);
    return launched();
}

int generic_satisfies(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *task,
                      uint8_t *out, cudaStream_t st) {
    craft_generic_satisfies_kernel<<<grid, GENERIC_THREAD_CTA, 0, st>>>(dt, s.grid, s.agent, task, out, s.n,
                                                                        s.cell_stride);
    return launched();
}

int generic_advance(int grid, const psk_craft_tables *dt, psk_craft_state s, psk_craft_episodes ep,
                    const uint8_t *action, uint8_t *done, uint8_t *success, unsigned long long *stats,
                    int32_t *err, cudaStream_t st) {
    craft_generic_advance_kernel<<<grid, GENERIC_THREAD_CTA, 0, st>>>(
        dt, s.grid, s.agent, action, ep.scen_grid, ep.scen_idx, ep.init_agent, done, success, stats, err, s.n,
        s.cell_stride);
    return launched();
}

int generic_expert(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *task,
                   uint8_t *action, int16_t *dist, int32_t *err, cudaStream_t st) {
    craft_generic_expert_kernel<<<grid, GENERIC_WARP_CTA, 0, st>>>(dt, s.grid, s.agent, task, action, dist, err,
                                                                   s.n, s.cell_stride);
    return launched();
}

int generic_find_closest(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *kind,
                         uint8_t *goal, int16_t *len, uint8_t *seq, int seq_cap, cudaStream_t st) {
    craft_generic_find_closest_kernel<<<grid, GENERIC_WARP_CTA, 0, st>>>(dt, s.grid, s.agent, kind, goal, len,
                                                                         seq, seq_cap, s.n, s.cell_stride);
    return launched();
}

int generic_features(int grid, const psk_craft_tables *dt, psk_craft_state s, float *out_f32,
                     uint8_t *out_u8, cudaStream_t st) {
    craft_generic_features_kernel<<<grid, GENERIC_WARP_CTA, 0, st>>>(dt, s.grid, s.agent, out_f32, out_u8, s.n,
                                                                     s.cell_stride);
    return launched();
}

}  // namespace psk
