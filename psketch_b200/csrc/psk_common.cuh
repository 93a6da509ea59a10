// Shared device helpers: tables staged in shared memory, the packed agent record, bitboards.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/psk_craft.h"

namespace psk {

enum : int { KC_FREE = 0, KC_INERT = 1, KC_WORKSHOP = 2, KC_WATER = 3, KC_STONE = 4, KC_GRAB = 5 };
enum : int { SAT_NEVER = 0, SAT_INV = 1, SAT_FACING = 2 };
enum : int { LEAF_NONE = 0, LEAF_USE = 1, LEAF_GO = 2, LEAF_BAD = 3 };

// coord_change of DOWN, UP, LEFT, RIGHT (worlds/craft.py:77-91)
__device__ __forceinline__ int dx_of(int a) { return a == 2 ? -1 : (a == 3 ? 1 : 0); }
__device__ __forceinline__ int dy_of(int a) { return a == 0 ? -1 : (a == 1 ? 1 : 0); }

// ---------------------------------------------------------------------------------------------
// Domain tables in shared memory.  Threads index them divergently (per-env task ids, per-cell
// kind classes), which constant memory would serialise, so every CTA stages the 2.3 KB struct
// from its device copy into shared memory first.
struct __align__(16) SharedTables {
    uint32_t words[sizeof(psk_craft_tables) / 4];

    __device__ __forceinline__ const psk_craft_tables &t() const {
        return *reinterpret_cast<const psk_craft_tables *>(words);
    }
    __device__ __forceinline__ int kind_class(int k) const { return t().kind_class[k & 31]; }
    __device__ __forceinline__ uint2 recipe(int r) const {
        return reinterpret_cast<const uint2 *>(t().recipes)[r];
    }
    __device__ __forceinline__ uint32_t node(int task, int i) const {
        return reinterpret_cast<const uint32_t *>(t().task_nodes)[(task & 31) * PSK_MAX_TASK_NODES + i];
    }
    __device__ __forceinline__ int task_len(int task) const { return t().task_len[task & 31]; }
    __device__ __forceinline__ uint32_t ws_recipes(int k) const { return t().ws_recipes[k & 31]; }
    __device__ __forceinline__ int n_recipes() const { return t().n_recipes; }
    __device__ __forceinline__ int bridge_kind() const { return t().bridge_kind; }
    __device__ __forceinline__ int axe_kind() const { return t().axe_kind; }
};

static_assert(sizeof(psk_craft_tables) % 16 == 0, "tables are staged with 128-bit loads");

// The same accessors straight from the device copy (read-only path, L1-resident after the first
// touch).  For kernels that use a few dozen bytes of the tables per thread and are too short to pay
// for staging 2.3 KB + a CTA barrier (craft_step_kernel: 160 bytes of kind classes and recipes).
struct GlobalTables {
    const psk_craft_tables *p;
    __device__ __forceinline__ int kind_class(int k) const { return __ldg(p->kind_class + (k & 31)); }
    __device__ __forceinline__ uint2 recipe(int r) const {
        return __ldg(reinterpret_cast<const uint2 *>(p->recipes) + r);
    }
    __device__ __forceinline__ uint32_t ws_recipes(int k) const { return __ldg(p->ws_recipes + (k & 31)); }
    __device__ __forceinline__ int n_recipes() const { return __ldg(&p->n_recipes); }
    __device__ __forceinline__ int bridge_kind() const { return __ldg(&p->bridge_kind); }
    __device__ __forceinline__ int axe_kind() const { return __ldg(&p->axe_kind); }
};

// T points at the device copy of the tables (see device_tables() in psk_craft.cu): one coalesced
// 128-bit load per thread.  (Indexing the struct as a kernel parameter instead costs one
// serialised constant-bank access per lane: 9 % of the stall samples of the first fused kernel.)
__device__ __forceinline__ void stage_tables(SharedTables &st, const psk_craft_tables *T) {
    const uint4 *src = reinterpret_cast<const uint4 *>(T);
    uint4 *dst = reinterpret_cast<uint4 *>(st.words);
    for (int i = threadIdx.x; i < int(sizeof(psk_craft_tables) / 16); i += blockDim.x)
        dst[i] = __ldg(src + i);
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Agent record: 32 bytes, moved with one 256-bit load/store (LDG.E.256 / STG.E.256 on sm_100a).
struct Agent {
    uint32_t w[8];  // w[0..5] inventory bytes, w[6] = x | y<<8 | dir<<16 | task<<24, w[7] = timer | ...

    __device__ __forceinline__ int x() const { return w[6] & 0xFF; }
    __device__ __forceinline__ int y() const { return (w[6] >> 8) & 0xFF; }
    __device__ __forceinline__ int dir() const { return (w[6] >> 16) & 0x3; }
    __device__ __forceinline__ int task() const { return w[6] >> 24; }
    __device__ __forceinline__ int timer() const { return w[7] & 0xFF; }
    __device__ __forceinline__ void set_pose(int x, int y, int dir) {
        w[6] = (w[6] & 0xFF000000u) | uint32_t(x) | (uint32_t(y) << 8) | (uint32_t(dir) << 16);
    }
    __device__ __forceinline__ void set_timer(int t) { w[7] = (w[7] & 0xFFFFFF00u) | uint32_t(t & 0xFF); }

    __device__ __forceinline__ uint32_t inv_word(int wi) const {
        uint32_t r = w[0];
#pragma unroll
        for (int i = 1; i < 6; i++) r = (wi == i) ? w[i] : r;
        return r;
    }
    __device__ __forceinline__ int inv(int k) const { return (inv_word(k >> 2) >> ((k & 3) * 8)) & 0xFF; }
    // count += delta (delta may be negative); the caller guarantees 0 <= result <= 255
    __device__ __forceinline__ void inv_add(int k, int delta) {
        const uint32_t d = uint32_t(delta) << ((k & 3) * 8);
        const int wi = k >> 2;
#pragma unroll
        for (int i = 0; i < 6; i++) w[i] += (wi == i) ? d : 0u;
    }
};

__device__ __forceinline__ Agent load_agent(const uint8_t *agent, int64_t e) {
    Agent a;
    const uint8_t *p = agent + e * PSK_AGENT_BYTES;
    asm volatile("ld.global.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.w[0]), "=r"(a.w[1]), "=r"(a.w[2]), "=r"(a.w[3]), "=r"(a.w[4]),
                   "=r"(a.w[5]), "=r"(a.w[6]), "=r"(a.w[7])
                 : "l"(p));
    return a;
}
__device__ __forceinline__ Agent load_agent_ro(const uint8_t *agent, int64_t e) {
    Agent a;
    const uint8_t *p = agent + e * PSK_AGENT_BYTES;
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.w[0]), "=r"(a.w[1]), "=r"(a.w[2]), "=r"(a.w[3]), "=r"(a.w[4]),
                   "=r"(a.w[5]), "=r"(a.w[6]), "=r"(a.w[7])
                 : "l"(p));
    return a;
}
__device__ __forceinline__ void store_agent(uint8_t *agent, int64_t e, const Agent &a) {
    uint8_t *p = agent + e * PSK_AGENT_BYTES;
    asm volatile("st.global.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.w[0]),
                 "r"(a.w[1]), "r"(a.w[2]), "r"(a.w[3]), "r"(a.w[4]), "r"(a.w[5]), "r"(a.w[6]),
                 "r"(a.w[7])
                 : "memory");
}

// ---------------------------------------------------------------------------------------------
// satisfies (worlds/craft.py:285-294) and the hint-tree walk (teachers/base.py:10-25), shared by the
// specialised kernels (psk_craft.cu) and the run-time-geometry ones (psk_craft_generic.cu).
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

// episode / success / env-step counters of a rollout tick, one atomic per warp and counter
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

// ---------------------------------------------------------------------------------------------
// Bitboards over the grid: bit (x*H + y).  uint64_t for W*H <= 64, unsigned __int128 up to 128.
template <int CELLS> struct BoardOf { using type = unsigned __int128; };
template <> struct BoardOf<64> { using type = uint64_t; };

template <int W, int H> struct Board {
    static constexpr int CELLS = W * H;
    static_assert(CELLS <= 128, "bitboard path covers up to 128 cells");
    using BT = typename BoardOf<(CELLS <= 64 ? 64 : 128)>::type;
    static constexpr int BITS = (CELLS <= 64 ? 64 : 128);

    static constexpr BT one() { return BT(1); }
    static constexpr BT all() { return CELLS == BITS ? ~BT(0) : ((BT(1) << (CELLS % BITS)) - 1); }
    static constexpr BT y0() {
        BT m = 0;
        for (int x = 0; x < W; x++) m |= BT(1) << (x * H);
        return m;
    }
    static constexpr BT yh() {
        BT m = 0;
        for (int x = 0; x < W; x++) m |= BT(1) << (x * H + H - 1);
        return m;
    }
    // positions p + delta(A) for p in b (off-grid results dropped)
    template <int A> static __device__ __forceinline__ BT shift(BT b) {
        constexpr BT NOT_Y0 = ~y0(), NOT_YH = ~yh(), ALL = all();
        if (A == 0) return (b & NOT_Y0) >> 1;            // DOWN  (0,-1)
        if (A == 1) return ((b & NOT_YH) << 1);          // UP    (0,+1)
        if (A == 2) return b >> H;                       // LEFT  (-1,0)
        return (b << H) & ALL;                           // RIGHT (+1,0)
    }
    template <int A> static __device__ __forceinline__ BT unshift(BT b) {
        return shift<(A ^ 1)>(b);                        // opposite action: 0<->1, 2<->3
    }
    static __device__ __forceinline__ int lowest(BT b) {
        if (BITS == 64) return __ffsll((long long)(uint64_t)b) - 1;
        const uint64_t lo = (uint64_t)b;
        if (lo) return __ffsll((long long)lo) - 1;
        return 64 + __ffsll((long long)(uint64_t)(b >> (BITS / 2))) - 1;
    }
    static __device__ __forceinline__ BT bit(int idx) { return BT(1) << idx; }
};

// nibble of "byte != 0" flags of a 32-bit word holding 4 cells, from a per-byte 0xFF/0x00 mask
__device__ __forceinline__ uint32_t mask_nibble(uint32_t bytemask) {
    return ((bytemask & 0x01010101u) * 0x10204080u) >> 28;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// ---------------------------------------------------------------------------------------------
// Tile chaining: fine-grained ordering between consecutive launches of the fused kernels.
// Envs never interact, so tile b of launch k+1 depends only on the launch-k CTA that owned the same
// envs — not on the whole grid.  With programmatic dependent launch the next grid becomes resident
// while the current one drains; instead of griddepcontrol.wait (= the WHOLE previous grid complete
// and flushed) its CTAs wait for their own predecessors through a pair of counters per group of
// PSK_CHAIN_GROUP envs:  chain[2g] tickets handed out, chain[2g+1] ticket holders finished.
// A CTA takes one ticket per group it owns (its position in that group's launch order), waits until
// every earlier holder has finished (ld.acquire: also drops stale L1 lines), and on exit publishes
// its state writes with st.release (after the CTA barrier).  The ticket is taken BEFORE launch_dependents, so a
// dependent CTA can never overtake its predecessor's ticket; the earliest holder of a group never
// waits on an unfinished CTA, so the chain always drains.  Counters only ever increase (u32 wrap
// is harmless under ==), which is what makes the scheme work under CUDA-graph replay.
#define PSK_CHAIN_GROUP 16
#define PSK_CHAIN_GROUPS (1 << 20)
__device__ __forceinline__ uint32_t chain_enter(uint32_t *chain, int64_t g) {
    return atomicAdd(chain + 2 * g, 1u);
}
// Returns false if the predecessor did not finish within PSK_CHAIN_SPIN_LIMIT polls (seconds; a healthy
// wait is microseconds): something outside this scheme went wrong — a previous launch on these envs was
// aborted, or the counters were overwritten.  The caller raises PSK_FLAG_CHAIN_TIMEOUT and goes on
// instead of hanging the GPU; its chain_leave puts the counter back in step for its successors.
#define PSK_CHAIN_SPIN_LIMIT (1u << 22)
#ifndef PSK_CHAIN_BOUNDED
#define PSK_CHAIN_BOUNDED 1
#endif
__device__ __forceinline__ bool chain_wait(const uint32_t *chain, int64_t g, uint32_t ticket) {
    uint32_t v;
#if PSK_CHAIN_BOUNDED
#pragma unroll 1        // unrolled (nvcc does, 16 x) the single tick loses 0.8 us: keep the poll loop tight
    for (uint32_t spins = 0; spins < PSK_CHAIN_SPIN_LIMIT; spins++) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(chain + 2 * g + 1) : "memory");
        if (v == ticket) return true;
        __nanosleep(64);
    }
    return false;
#else
    while (true) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(chain + 2 * g + 1) : "memory");
        if (v == ticket) return true;
        __nanosleep(64);
    }
#endif
}
__device__ __forceinline__ void chain_leave(uint32_t *chain, int64_t g, uint32_t ticket) {
    // st.release.gpu IS fence + store (SASS: MEMBAR.ALL.GPU; ST): with the CTA barrier before it, it
    // publishes every thread's state writes.  (A __threadfence() in front adds a second, sequentially
    // consistent MEMBAR.SC.GPU for nothing.)
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(chain + 2 * g + 1), "r"(ticket + 1) : "memory");
}

// Host-side per-device caches (SM count, shared-memory attributes, table copies) are indexed by this.
#define PSK_MAX_DEVICES 32
static inline int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= PSK_MAX_DEVICES) dev = 0;
    return dev;
}

// ---------------------------------------------------------------------------------------------
// Generic tier (psk_craft_generic.cu): the primitives for any geometry of the generic domain
// (include/psk_craft.h), geometry and K read from the device tables `dt` at run time.  `grid` is
// the launch's CTA count: step, satisfies and advance run 256-thread CTAs of one env per thread,
// expert, find_closest and features 128-thread CTAs of one env per warp.  Launches are
// asynchronous on `st`; the return value is a PSK_* code.
constexpr int GENERIC_THREAD_CTA = 256, GENERIC_WARP_CTA = 128;
int generic_step(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *action,
                 const uint8_t *active, float *reward, int32_t *err, cudaStream_t st);
int generic_satisfies(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *task,
                      uint8_t *out, cudaStream_t st);
int generic_expert(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *task,
                   uint8_t *action, int16_t *dist, int32_t *err, cudaStream_t st);
int generic_find_closest(int grid, const psk_craft_tables *dt, psk_craft_state s, const uint8_t *kind,
                         uint8_t *goal, int16_t *len, uint8_t *seq, int seq_cap, cudaStream_t st);
int generic_features(int grid, const psk_craft_tables *dt, psk_craft_state s, float *out_f32,
                     uint8_t *out_u8, cudaStream_t st);
int generic_advance(int grid, const psk_craft_tables *dt, psk_craft_state s, psk_craft_episodes ep,
                    const uint8_t *action, uint8_t *done, uint8_t *success, unsigned long long *stats,
                    int32_t *err, cudaStream_t st);
// true when psk_craft_tick / _tick_u8 run the fused kernel for these tables (one of the five built
// geometries, generic tier not forced); the host contexts' zero-copy route needs it
bool craft_fused_built(const psk_craft_tables *t);

}  // namespace psk
