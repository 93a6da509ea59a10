/*
 * TEST INFRASTRUCTURE ONLY — CPU restatement (plain C) of the Philox sampler kernels
 * (psketch_b200/csrc/psk_scenario.cu): the scenario sampler, the dataset's start cells and the
 * off-policy random actions.  Restated from the documented procedure (include/psk_craft.h), not
 * from the kernel's bitboards: cells are a byte array indexed x * H + y, and the acceptance rule is
 * a literal breadth-first search over a cell list.
 *
 * Generator: Philox4x32-10 (Salmon et al., SC'11) on 32-bit words with 64-bit multiplies,
 * checked against the Random123 known-answer vectors (tests/test_sampler_cpu.py).  A stream
 * (seed, stream, start) has key = (seed lo, seed hi) and counter = (start lo, start hi, stream lo,
 * stream hi); counter word 0 is incremented after each block, carrying into word 1; the words of a
 * block are consumed out[3], out[2], out[1], out[0]; below(n) = (u64(word) * n) >> 32.
 */
#include <stdint.h>
#include <string.h>

#define MAXC 256 /* cells per grid: the sampler serves 8 x 8 and 10 x 10 */

void orc_philox_block(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t x0 = ctr[0], x1 = ctr[1], x2 = ctr[2], x3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        if (r) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        const uint64_t p0 = (uint64_t)0xD2511F53u * x0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * x2;
        const uint32_t y0 = (uint32_t)(p1 >> 32) ^ x1 ^ k0;
        const uint32_t y1 = (uint32_t)p1;
        const uint32_t y2 = (uint32_t)(p0 >> 32) ^ x3 ^ k1;
        const uint32_t y3 = (uint32_t)p0;
        x0 = y0; x1 = y1; x2 = y2; x3 = y3;
    }
    out[0] = x0; out[1] = x1; out[2] = x2; out[3] = x3;
}

int orc_below(uint32_t word, int n) { return (int)(((uint64_t)word * (uint64_t)n) >> 32); }

typedef struct {
    uint32_t key[2], ctr[4], out[4];
    int have;
} rng_t;

static void rng_init(rng_t *r, uint64_t seed, uint64_t stream, uint64_t start) {
    r->key[0] = (uint32_t)seed;
    r->key[1] = (uint32_t)(seed >> 32);
    r->ctr[0] = (uint32_t)start;
    r->ctr[1] = (uint32_t)(start >> 32);
    r->ctr[2] = (uint32_t)stream;
    r->ctr[3] = (uint32_t)(stream >> 32);
    r->have = 0;
}

static uint32_t rng_word(rng_t *r) {
    if (r->have == 0) {
        orc_philox_block(r->ctr, r->key, r->out);
        r->have = 4;
        if (++r->ctr[0] == 0) ++r->ctr[1];
    }
    return r->out[--r->have];
}

static int rng_below(rng_t *r, int n) { return orc_below(rng_word(r), n); }

/* The acceptance rule of random_free(keep_connected=True) on a grid whose occupied cells are
 * occ[x * H + y] != 0.  Returns 0 when it holds; bit 0: (i) some free cell is not reachable from
 * the first free cell (lowest index); bit 1: (ii) some occupied interior cell has no free
 * 4-neighbour. */
int orc_rule_violations(const uint8_t *occ, int W, int H) {
    static const int DX[4] = {1, -1, 0, 0}, DY[4] = {0, 0, 1, -1};
    int queue[MAXC];
    uint8_t seen[MAXC];
    int n_free = 0, first = -1, res = 0;
    memset(seen, 0, sizeof(seen));
    for (int c = 0; c < W * H; c++)
        if (!occ[c]) {
            if (first < 0) first = c;
            n_free++;
        }
    if (n_free) {
        int head = 0, tail = 0;
        queue[tail++] = first;
        seen[first] = 1;
        while (head < tail) {
            const int c = queue[head++], x = c / H, y = c % H;
            for (int d = 0; d < 4; d++) {
                const int nx = x + DX[d], ny = y + DY[d];
                if (nx < 0 || ny < 0 || nx >= W || ny >= H) continue;
                const int q = nx * H + ny;
                if (!occ[q] && !seen[q]) {
                    seen[q] = 1;
                    queue[tail++] = q;
                }
            }
        }
        if (tail != n_free) res |= 1;
    }
    for (int x = 1; x < W - 1; x++)
        for (int y = 1; y < H - 1; y++) {
            if (!occ[x * H + y]) continue;
            int near_free = 0;
            for (int d = 0; d < 4; d++) near_free |= !occ[(x + DX[d]) * H + y + DY[d]];
            if (!near_free) res |= 2;
        }
    return res;
}

/* random_free: draw x, then y; reject an occupied cell; with keep_connected, occupy the cell and
 * accept it only if the rule above holds.  The cell index, or -1 after max_tries draws. */
static int random_free(rng_t *r, uint8_t *occ, int W, int H, int keep_connected, int max_tries) {
    for (int t = 0; t < max_tries; t++) {
        const int x = rng_below(r, W);
        const int y = rng_below(r, H);
        const int c = x * H + y;
        if (occ[c]) continue;
        if (!keep_connected) return c;
        occ[c] = 1;
        const int ok = orc_rule_violations(occ, W, H) == 0;
        occ[c] = 0;
        if (ok) return c;
    }
    return -1;
}

/* Scenario s from stream (seed, s + offset), counter start 0: the ring of boundary_kind, then
 * place[0..n_place) in order, then the agent, each by random_free(keep_connected, 4096 tries).  A
 * scenario that runs out of draws keeps the items placed so far, gets init_pos (0, 0) and counts
 * as failed.  Rows are written at cell_stride with the tail zeroed.  Returns the failure count. */
int64_t orc_sample_scenarios(int W, int H, const uint8_t *place, int n_place, int boundary_kind,
                             uint64_t seed, uint64_t offset, int64_t n, int cell_stride,
                             uint8_t *grid, uint8_t *init_pos) {
    int64_t fails = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : fails)
    for (int64_t s = 0; s < n; s++) {
        rng_t r;
        rng_init(&r, seed, (uint64_t)s + offset, 0);
        uint8_t *row = grid + s * cell_stride;
        uint8_t occ[MAXC];
        memset(row, 0, (size_t)cell_stride);
        memset(occ, 0, sizeof(occ));
        for (int x = 0; x < W; x++)
            for (int y = 0; y < H; y++)
                if (x == 0 || y == 0 || x == W - 1 || y == H - 1) {
                    row[x * H + y] = (uint8_t)boundary_kind;
                    occ[x * H + y] = 1;
                }
        int ok = 1;
        for (int i = 0; i < n_place; i++) {
            const int c = random_free(&r, occ, W, H, 1, 4096);
            if (c < 0) {
                ok = 0;
                break;
            }
            row[c] = place[i];
            occ[c] = 1;
        }
        int p = ok ? random_free(&r, occ, W, H, 1, 4096) : -1;
        if (p < 0) {
            ok = 0;
            p = 0;
        }
        init_pos[2 * s] = (uint8_t)(p / H);
        init_pos[2 * s + 1] = (uint8_t)(p % H);
        fails += !ok;
    }
    return fails;
}

/* Start cells: group g from stream (seed, g + offset), counter start 1; per_group draws of
 * random_free(keep_connected=False, 65536 tries) over the cells of row group_scen[g] that are 0,
 * each drawn cell taken for the rest of the group.  A slot that runs out of draws is 255/255 and
 * counts as failed; the next slot continues from the same generator state.  (Draws never leave the
 * W x H grid, so the bitboard bits beyond it need no counterpart here.) */
int64_t orc_sample_positions(int W, int H, const uint8_t *grid, const int32_t *group_scen,
                             int per_group, uint64_t seed, uint64_t offset, int64_t n_groups,
                             int cell_stride, uint8_t *out) {
    int64_t fails = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : fails)
    for (int64_t g = 0; g < n_groups; g++) {
        rng_t r;
        rng_init(&r, seed, (uint64_t)g + offset, 1);
        const uint8_t *row = grid + (int64_t)group_scen[g] * cell_stride;
        uint8_t taken[MAXC];
        for (int c = 0; c < W * H; c++) taken[c] = row[c] != 0;
        for (int i = 0; i < per_group; i++) {
            uint8_t *o = out + (g * per_group + i) * 2;
            const int c = random_free(&r, taken, W, H, 0, 1 << 16);
            if (c < 0) {
                fails++;
                o[0] = o[1] = 255;
                continue;
            }
            taken[c] = 1;
            o[0] = (uint8_t)(c / H);
            o[1] = (uint8_t)(c % H);
        }
    }
    return fails;
}

/* Off-policy actions: out[k * n + e] = below(n_actions) of the first word of stream (seed, e)
 * at counter start t + k (mod 2^64); t already includes the device clock. */
void orc_random_actions(uint8_t *out, int64_t n, int ticks, int n_actions, uint64_t seed, uint64_t t) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n * ticks; i++) {
        const int64_t k = i / n, e = i - k * n;
        rng_t r;
        rng_init(&r, seed, (uint64_t)e, t + (uint64_t)k);
        out[i] = (uint8_t)rng_below(&r, n_actions);
    }
}
