// psk_scenario.cu — scenario sampling on the device (reset path, SURVEY §8 row R1).
//
// Restates make_data.py:74-144 (`random_free`, `sample_scenario`) with a counter-based Philox
// generator instead of numpy's RandomState: boundary ring, then every item of `place_kinds` in
// order (the reference: 2 x iron, grass, wood, then the 3 workshops) and finally the agent, each
// at a uniformly random cell drawn by rejection until the cell is free AND, with the cell
// occupied, (i) all free cells are still mutually reachable and (ii) every occupied interior
// cell still touches a free cell (make_data.py:84-97 — a flood started from an occupied cell can
// only leave through a free neighbour).  One scenario per thread; grids are 64/128-bit
// bitboards, the connectivity test is a flood fill of shifts and ORs.
//
// Bit-equality with numpy's stream is not a goal (BASELINE.json); the procedure, and therefore
// the distribution, is the reference's.  tests/test_scenario_gpu.py checks the invariants, the
// kind histogram, solvability of all tasks and the cell-occupancy statistics against scenarios
// sampled by the reference itself (tests/golden/sampler_stats.npz); tests/test_sampler_gpu.py
// compares every output byte of the three kernels with a plain C restatement
// (oracle/sampler_oracle.c), which tests/test_sampler_cpu.py pins to the Philox known answers.
#include "psk_common.cuh"

namespace psk {

// Philox4x32-10 (Salmon et al., SC'11): counter (c0..c3), key (k0,k1).
struct Philox {
    uint32_t k0, k1;
    uint32_t c0, c1, c2, c3;
    uint32_t out[4];
    int have;

    __device__ __forceinline__ Philox(uint64_t seed, uint64_t stream, uint64_t offset)
        : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), c0((uint32_t)offset),
          c1((uint32_t)(offset >> 32)), c2((uint32_t)stream), c3((uint32_t)(stream >> 32)), have(0) {}

    __device__ __forceinline__ void round(uint32_t &a, uint32_t &b, uint32_t &c, uint32_t &d,
                                          uint32_t ka, uint32_t kb) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, a), lo0 = 0xD2511F53u * a;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c), lo1 = 0xCD9E8D57u * c;
        a = hi1 ^ b ^ ka;
        b = lo1;
        c = hi0 ^ d ^ kb;
        d = lo0;
    }
    __device__ __forceinline__ void refill() {
        uint32_t a = c0, b = c1, c = c2, d = c3, ka = k0, kb = k1;
#pragma unroll
        for (int i = 0; i < 10; i++) {
            round(a, b, c, d, ka, kb);
            ka += 0x9E3779B9u;
            kb += 0xBB67AE85u;
        }
        out[0] = a; out[1] = b; out[2] = c; out[3] = d;
        have = 4;
        if (++c0 == 0) ++c1;
    }
    __device__ __forceinline__ uint32_t next() {
        if (have == 0) refill();
        return out[--have];
    }
    // uniform integer in [0, n)  (numpy randint(n)); multiply-shift, bias < 2^-32 * n
    __device__ __forceinline__ int below(int n) { return (int)(((uint64_t)next() * (uint64_t)n) >> 32); }
};

template <int W, int H>
__device__ __forceinline__ bool keeps_connected(typename Board<W, H>::BT occ) {
    using B = Board<W, H>;
    using BT = typename B::BT;
    const BT freeb = ~occ & B::all();
    if (!freeb) return true;
    // (i) all free cells mutually reachable (make_data.py:27-72 from the first free cell)
    BT v = B::bit(B::lowest(freeb));
    while (true) {
        BT nv = v;
#pragma unroll
        for (int r = 0; r < 2; r++)
            nv |= (B::template shift<0>(nv) | B::template shift<1>(nv) | B::template shift<2>(nv) |
                   B::template shift<3>(nv)) & freeb;
        if (nv == v) break;
        v = nv;
    }
    if (v != freeb) return false;
    // (ii) every occupied interior cell touches a free cell (make_data.py:89-97)
    BT interior = 0;
    {
        BT ring = 0;
        for (int x = 0; x < W; x++) ring |= B::bit(x * H) | B::bit(x * H + H - 1);
        for (int y = 0; y < H; y++) ring |= B::bit(y) | B::bit((W - 1) * H + y);
        interior = B::all() & ~ring;
    }
    const BT near_free = B::template shift<0>(freeb) | B::template shift<1>(freeb) |
                         B::template shift<2>(freeb) | B::template shift<3>(freeb);
    return (occ & interior & ~near_free) == 0;
}

// random_free (make_data.py:74-103): returns the cell index, or -1 after max_tries draws
template <int W, int H>
__device__ __forceinline__ int random_free(Philox &rng, typename Board<W, H>::BT occ,
                                           bool keep_connected, int max_tries) {
    using B = Board<W, H>;
    for (int t = 0; t < max_tries; t++) {
        const int x = rng.below(W), y = rng.below(H);
        const int c = x * H + y;
        if ((occ >> c) & 1) continue;
        if (!keep_connected || keeps_connected<W, H>(occ | B::bit(c))) return c;
    }
    return -1;
}

template <int W, int H>
__global__ void __launch_bounds__(128)
craft_sample_scenarios_kernel(uint8_t *__restrict__ scen_grid, uint8_t *__restrict__ init_pos,
                              const uint8_t *__restrict__ place_kinds, int n_place,
                              int boundary_kind, uint64_t seed, uint64_t offset, int64_t n,
                              int cell_stride, int32_t *fail_count) {
    using B = Board<W, H>;
    using BT = typename B::BT;
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < n;
         s += (int64_t)gridDim.x * blockDim.x) {
        Philox rng(seed, (uint64_t)s + offset, 0);
        uint8_t *row = scen_grid + s * cell_stride;
        BT occ = 0;
        for (int c = 0; c < cell_stride; c++) {
            const int x = c / H, y = c % H;
            const bool ring = c < W * H && (x == 0 || y == 0 || x == W - 1 || y == H - 1);
            row[c] = ring ? (uint8_t)boundary_kind : 0;   // make_data.py:107-112
            if (ring) occ |= B::bit(c);
        }
        bool ok = true;
        for (int i = 0; i < n_place && ok; i++) {         // make_data.py:128-139
            const int c = random_free<W, H>(rng, occ, true, 4096);
            if (c < 0) { ok = false; break; }
            row[c] = place_kinds[i];
            occ |= B::bit(c);
        }
        int p = ok ? random_free<W, H>(rng, occ, true, 4096) : -1;   // make_data.py:142
        if (p < 0) {
            ok = false;
            p = 0;
        }
        init_pos[2 * s] = (uint8_t)(p / H);
        init_pos[2 * s + 1] = (uint8_t)(p % H);
        if (!ok && fail_count) atomicAdd(fail_count, 1);
    }
}

// Dataset instance positions (make_data.py:203-208): `per_group` DISTINCT uniformly random free
// cells of a scenario per group, random_free(keep_connected=False) with re-draw on repeats.
template <int W, int H>
__global__ void __launch_bounds__(128)
craft_sample_positions_kernel(const uint8_t *__restrict__ scen_grid,
                              const int32_t *__restrict__ group_scen, int per_group,
                              uint8_t *__restrict__ out_pos, uint64_t seed, uint64_t offset,
                              int64_t n_groups, int cell_stride, int32_t *fail_count) {
    using B = Board<W, H>;
    using BT = typename B::BT;
    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n_groups;
         g += (int64_t)gridDim.x * blockDim.x) {
        Philox rng(seed, (uint64_t)g + offset, 1);
        const uint8_t *row = scen_grid + (int64_t)group_scen[g] * cell_stride;
        BT occ = ~B::all();
        for (int c = 0; c < W * H; c++)
            if (row[c]) occ |= B::bit(c);
        BT taken = occ;
        for (int i = 0; i < per_group; i++) {
            const int c = random_free<W, H>(rng, taken, false, 1 << 16);
            uint8_t *o = out_pos + (g * per_group + i) * 2;
            if (c < 0) {
                if (fail_count) atomicAdd(fail_count, 1);
                o[0] = o[1] = 255;
                continue;
            }
            taken |= B::bit(c);
            o[0] = (uint8_t)(c / H);
            o[1] = (uint8_t)(c % H);
        }
    }
}

// Off-policy action source (SURVEY §8(d) config 2): action[e] ~ U{0..n_actions-1} from the first
// word of Philox stream (seed, env) at counter start t (include/psk_craft.h): reproducible whatever
// the launch geometry.
// out u8[ticks][n]: row k holds the actions of clock t + k (ticks = 1: the plain per-tick form; a
// block of rows feeds psk_craft_rollout's action_in, so the off-policy variant also runs `ticks`
// ticks per launch).
__global__ void __launch_bounds__(256)
random_actions_kernel(uint8_t *__restrict__ out, int64_t n, int ticks, int n_actions, uint64_t seed,
                      uint64_t t, const unsigned long long *__restrict__ t_dev) {
    if (t_dev) t += *t_dev;   // device-side clock (e.g. the env-step counter): advances under graph replay
    const int64_t total = n * ticks;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = i / n, e = i - k * n;
        Philox rng(seed, (uint64_t)e, t + (uint64_t)k);
        out[i] = (uint8_t)rng.below(n_actions);
    }
}

static inline int blocks_for(int64_t n) {
    int64_t b = (n + 127) / 128;
    return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

}  // namespace psk

using namespace psk;

extern "C" {

int psk_craft_sample_scenarios(const psk_craft_tables *t, uint8_t *scen_grid, uint8_t *init_pos,
                               const uint8_t *place_kinds, int32_t n_place, int32_t boundary_kind,
                               uint64_t seed, uint64_t offset, int64_t n, int32_t cell_stride,
                               int32_t *fail_count, void *stream) {
    if (!t || n < 0 || !place_kinds || n_place < 0) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    if (!scen_grid || !init_pos || cell_stride != ((t->width * t->height + 63) / 64) * 64)
        return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (t->width == 8 && t->height == 8)
        craft_sample_scenarios_kernel<8, 8><<<blocks_for(n), 128, 0, st>>>(
            scen_grid, init_pos, place_kinds, n_place, boundary_kind, seed, offset, n, cell_stride, fail_count);
    else if (t->width == 10 && t->height == 10)
        craft_sample_scenarios_kernel<10, 10><<<blocks_for(n), 128, 0, st>>>(
            scen_grid, init_pos, place_kinds, n_place, boundary_kind, seed, offset, n, cell_stride, fail_count);
    else
        return PSK_ERR_UNSUPPORTED;
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_random_actions(uint8_t *out, int64_t n, int32_t n_actions, uint64_t seed, uint64_t t,
                       const unsigned long long *t_dev, void *stream) {
    if (n < 0 || n_actions <= 0 || n_actions > 255 || (n && !out)) return PSK_ERR_BADARG;
    if (n == 0) return PSK_OK;
    int64_t b = (n + 255) / 256;
    if (b > 148 * 8) b = 148 * 8;
    random_actions_kernel<<<(int)b, 256, 0, (cudaStream_t)stream>>>(out, n, 1, n_actions, seed, t, t_dev);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_random_actions_block(uint8_t *out, int64_t n, int32_t ticks, int32_t n_actions, uint64_t seed,
                             uint64_t t, const unsigned long long *t_dev, void *stream) {
    if (n < 0 || ticks < 0 || n_actions <= 0 || n_actions > 255 || (n && ticks && !out)) return PSK_ERR_BADARG;
    if (n == 0 || ticks == 0) return PSK_OK;
    int64_t b = (n * ticks + 255) / 256;
    if (b > 148 * 8) b = 148 * 8;
    random_actions_kernel<<<(int)b, 256, 0, (cudaStream_t)stream>>>(out, n, ticks, n_actions, seed, t, t_dev);
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

int psk_craft_sample_positions(const psk_craft_tables *t, const uint8_t *scen_grid,
                               const int32_t *group_scen, int32_t per_group, uint8_t *out_pos,
                               uint64_t seed, uint64_t offset, int64_t n_groups,
                               int32_t cell_stride, int32_t *fail_count, void *stream) {
    if (!t || n_groups < 0 || per_group <= 0) return PSK_ERR_BADARG;
    if (n_groups == 0) return PSK_OK;
    if (!scen_grid || !group_scen || !out_pos || cell_stride < t->width * t->height) return PSK_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (t->width == 8 && t->height == 8)
        craft_sample_positions_kernel<8, 8><<<blocks_for(n_groups), 128, 0, st>>>(
            scen_grid, group_scen, per_group, out_pos, seed, offset, n_groups, cell_stride, fail_count);
    else if (t->width == 10 && t->height == 10)
        craft_sample_positions_kernel<10, 10><<<blocks_for(n_groups), 128, 0, st>>>(
            scen_grid, group_scen, per_group, out_pos, seed, offset, n_groups, cell_stride, fail_count);
    else
        return PSK_ERR_UNSUPPORTED;
    return cudaGetLastError() == cudaSuccess ? PSK_OK : PSK_ERR_CUDA;
}

}  // extern "C"
