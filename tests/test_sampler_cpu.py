"""The C restatement of the Philox sampler kernels (oracle/sampler_oracle.c), no GPU: the generator
against the Random123 known answers and against a Python reading of the stream layout, the
acceptance rule on the reference's own grids and on boards where each half of it rejects alone, and
the cell statistics of oracle scenarios against the reference's sampler.  tests/test_sampler_gpu.py
shows that the kernels equal this oracle byte for byte, so the statistics hold for them too.  Also
the input checks in front of the sampler entry points."""
import ctypes
import os

import numpy as np
import pytest

from oracle import sampler_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
M32 = 0xFFFFFFFF


def _words(v):
    return [v & M32, (v >> 32) & M32]


def test_philox_known_answers():
    """Philox4x32-10 known-answer vectors of Random123 (kat_vectors): any change to a multiplier,
    a Weyl constant, the round structure or the key schedule fails here."""
    cases = [
        ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
        ([M32] * 4, [M32] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
        ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
         [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
    ]
    for ctr, key, want in cases:
        assert so.philox_block(ctr, key).tolist() == want, (ctr, key)


def test_below_edges():
    for n in (1, 6, 8, 10, 255):
        assert so.below(0, n) == 0
        assert so.below(M32, n) == n - 1
        assert so.below(0x80000000, n) == n // 2
    assert so.below(0x2AAAAAAB, 6) == 1 and so.below(0x2AAAAAAA, 6) == 0     # 2^32 / 6 = 0x2AAAAAAA.AB


def test_random_actions_read_the_documented_block():
    """Row k, env e is below(n_actions) of word 3 of the block with key (seed lo, seed hi) and
    counter (t + k lo, t + k hi, e lo, e hi), for clocks and seeds on both sides of 2^32 and a
    clock that wraps past 2^64."""
    n, ticks = 37, 5
    for seed in (0, 123, (1 << 32) + 123, (1 << 64) - 1):
        for t in (0, (1 << 32) - 3, (1 << 64) - 2):
            for n_actions in (1, 6, 255):
                got = so.random_actions(n, ticks, n_actions, seed, t)
                for k in range(ticks):
                    tk = (t + k) % (1 << 64)
                    for e in (0, 1, n - 1):
                        w = so.philox_block(_words(tk) + _words(e), _words(seed))[3]
                        assert got[k, e] == so.below(w, n_actions), (seed, t, n_actions, k, e)
    # the seed's high word and the clock's high word reach the output
    a = so.random_actions(4096, 1, 255, 123, 7)
    assert not np.array_equal(a, so.random_actions(4096, 1, 255, (1 << 32) + 123, 7))
    assert not np.array_equal(a, so.random_actions(4096, 1, 255, 123, (1 << 32) + 7))


def _stream_words(seed, stream):
    """Words of stream (seed, stream) from counter start 0, in the documented order: block c is
    Philox(counter = (c lo, c hi, stream lo, stream hi), key = (seed lo, seed hi)), read out[3] first."""
    c = 0
    while True:
        for w in so.philox_block(_words(c) + _words(stream), _words(seed))[::-1]:
            yield int(w)
        c += 1


def _first_interior_draw(W, H, seed, stream):
    words = _stream_words(seed, stream)
    while True:
        x = so.below(next(words), W)
        y = so.below(next(words), H)
        if 0 < x < W - 1 and 0 < y < H - 1:
            return x, y


@pytest.mark.parametrize("W", [8, 10])
def test_scenario_stream_layout(W):
    """With nothing to place, the agent lands on the first draw inside the ring (one occupied cell
    cannot break either rule on an empty interior): checks the stream = scenario + offset, the
    counter start 0, the x-then-y order and the word order across block boundaries."""
    for seed, offset in ((123, 0), ((1 << 32) + 123, 0), (5, (1 << 32) - 3), ((1 << 64) - 1, (1 << 64) - 2)):
        n = 40
        _, pos, fails = so.sample_scenarios(W, W, [], 1, seed, offset, n)
        assert fails == 0
        for s in range(n):
            want = _first_interior_draw(W, W, seed, (s + offset) % (1 << 64))
            assert tuple(pos[s]) == want, (seed, offset, s)


def _free_nbr_ok(g):
    """Python check of both rules on one final grid (ids[W, H], 0 = free)."""
    W, H = g.shape
    free = g == 0
    cells = list(zip(*np.nonzero(free)))
    seen, stack = {cells[0]}, [cells[0]]
    while stack:
        x, y = stack.pop()
        for q in ((x + 1, y), (x - 1, y), (x, y + 1), (x, y - 1)):
            if 0 <= q[0] < W and 0 <= q[1] < H and free[q] and q not in seen:
                seen.add(q)
                stack.append(q)
    if len(seen) != len(cells):
        return False
    return all(free[x + 1, y] or free[x - 1, y] or free[x, y + 1] or free[x, y - 1]
               for x in range(1, W - 1) for y in range(1, H - 1) if not free[x, y])


def test_rule_holds_on_the_reference_grids():
    ref = np.load(os.path.join(GOLDEN, "sampler_stats.npz"))
    grids = ref["example_grids"].reshape(-1, 8, 8)
    assert len(grids) == 64
    for g in grids:
        assert so.rule_violations(g != 0) == 0
        assert _free_nbr_ok(g)


def _ring(W):
    occ = np.zeros((W, W), bool)
    occ[0, :] = occ[-1, :] = occ[:, 0] = occ[:, -1] = True
    return occ


@pytest.mark.parametrize("W", [8, 10])
def test_each_rule_rejects_on_its_own(W):
    assert so.rule_violations(_ring(W)) == 0
    # a wall across the interior: the last item cuts the corridor, every item still sees a free cell
    wall = _ring(W)
    wall[3, 1:W - 2] = True
    assert so.rule_violations(wall) == 0
    wall[3, W - 2] = True
    assert so.rule_violations(wall) == 1
    # an item sealed in by four others; the free cells stay connected
    seal = _ring(W)
    seal[3, 4] = seal[5, 4] = seal[4, 3] = True
    assert so.rule_violations(seal) == 0
    seal[4, 5] = True
    assert so.rule_violations(seal) == 1          # (4, 4) is a free cell cut off from the rest
    seal[4, 4] = True
    assert so.rule_violations(seal) == 2
    # (ii) looks at interior cells only: an occupied edge cell may be shut in
    edge = np.zeros((W, W), bool)
    edge[0, 0] = edge[0, 1] = edge[1, 0] = True
    assert so.rule_violations(edge) == 0
    # both at once: a sealed item and a cut corridor
    both = seal | wall
    assert so.rule_violations(both) == 3


def _kind_counts(g, K):
    return np.stack([(g == k).sum(axis=(1, 2)) for k in range(K)], axis=1)


@pytest.mark.parametrize("world", ["craft_medium", "craft_large"])
def test_oracle_scenarios_invariants(world):
    """Every oracle scenario holds the default placement, the ring, a free start cell, and the
    rule with the start cell occupied (the state random_free accepted last)."""
    from psketch_b200.data import default_placement
    from psketch_b200.tables import CraftTables
    t = CraftTables(world_config=world)
    W, H, n = t.W, t.H, 3000
    grid, pos, fails = so.sample_for(t, n, seed=123)
    assert fails == 0
    assert (grid[:, W * H:] == 0).all()
    g = grid[:, :W * H].reshape(n, W, H)
    want = np.bincount(default_placement(t), minlength=t.K)
    want[1] = 2 * (W + H) - 4
    want[0] = W * H - want.sum()
    assert (_kind_counts(g, t.K) == want).all()
    ring = _ring(W)
    assert (g[:, ring] == 1).all() and (g[:, ~ring] != 1).all()
    assert (g[np.arange(n), pos[:, 0], pos[:, 1]] == 0).all()
    for i in range(0, n, 7):
        occ = g[i] != 0
        occ[pos[i, 0], pos[i, 1]] = True
        assert so.rule_violations(occ) == 0


def test_oracle_statistics_match_the_reference_sampler():
    """tests/test_scenario_gpu.py's comparison with 3,000 scenarios of the reference's own sampler,
    on 20,000 oracle scenarios: kind-cell and start-cell occupancy at 5 sigma, free-neighbour
    profile of the items within 1 %."""
    from psketch_b200.tables import CraftTables
    t = CraftTables(world_config="craft_medium")
    n = 20000
    grid, pos, fails = so.sample_for(t, n, seed=123)
    assert fails == 0
    g = grid[:, :64].reshape(n, 8, 8)
    ref = np.load(os.path.join(GOLDEN, "sampler_stats.npz"))
    m = int(ref["n_scen"])
    for k in (2, 3, 4, 7, 8, 9):
        p_ref = ref["kind_cell"][k][1:7, 1:7] / m
        p_orc = (g == k).mean(axis=0)[1:7, 1:7]
        sigma = np.sqrt(np.maximum(p_orc * (1 - p_orc), 1e-4) * (1.0 / m + 1.0 / n))
        assert np.abs(p_ref - p_orc).max() < 5 * sigma.max(), k
    p_ref = ref["pos_cell"][1:7, 1:7] / m
    p_orc = np.zeros((8, 8))
    np.add.at(p_orc, (pos[:, 0], pos[:, 1]), 1.0 / n)
    assert np.abs(p_ref - p_orc[1:7, 1:7]).max() < 5 * np.sqrt(0.03 * (1.0 / m + 1.0 / n))
    free = g == 0
    fn = np.zeros_like(g, dtype=np.int64)
    fn[:, 1:7, 1:7] = (free[:, 2:8, 1:7].astype(int) + free[:, 0:6, 1:7] + free[:, 1:7, 2:8] + free[:, 1:7, 0:6])
    items = g > 1
    nb = np.asarray([(fn[items] == v).sum() for v in range(5)], np.float64)
    assert np.abs(nb / nb.sum() - ref["n_free_nbr"] / ref["n_free_nbr"].sum()).max() < 0.01


def test_oracle_failure_path_and_positions_edges():
    """The oracle's own failure answers: too many items keep the partial row, start (0, 0) and
    count; a group asking for more cells than are free gets every free cell once, then 255/255."""
    W = 8
    grid, pos, fails = so.sample_scenarios(W, W, [7] * 30, 1, 123, 0, 16)
    assert fails == 16 and (pos == 0).all()
    placed = (grid[:, :64] == 7).sum(axis=1)
    assert placed.min() > 0 and placed.max() < 30
    good, _, f = so.sample_scenarios(W, W, [7, 8, 9], 1, 5, 0, 4)
    assert f == 0
    n_free = (good[:, :64] == 0).sum(axis=1)
    out, f = so.sample_positions(W, W, good, [0, 3, 3], int(n_free[3]) + 2, 9)
    assert f == 2 * 2 + max(0, 2 + int(n_free[3]) - int(n_free[0]))
    for gi, s in enumerate((0, 3, 3)):
        cells = [tuple(c) for c in out[gi] if c[0] != 255]
        assert len(cells) == len(set(cells)) == min(len(out[gi]), n_free[s])
        assert all(good[s, x * W + y] == 0 for x, y in cells)
        assert (out[gi, len(cells):] == 255).all()


# ------------------------------------------------------------------------------- input checks
def test_sample_scenarios_rejects_kind_ids_before_device_work(medium_tables):
    from psketch_b200 import data
    for bad in ([7, 0, 8], [medium_tables.K], [7, 255], [-1]):
        with pytest.raises(ValueError, match="place_kinds"):
            data.sample_scenarios(medium_tables, 4, seed=1, place_kinds=bad, device="cpu")


def test_sample_positions_rejects_rows_out_of_range(medium_tables):
    torch = pytest.importorskip("torch")
    from psketch_b200 import data
    sg = torch.zeros((3, 64), dtype=torch.uint8)
    for bad in ([0, 3], [-1], [2, 0, 7]):
        with pytest.raises(ValueError, match="group_scen"):
            data.sample_positions(medium_tables, sg, bad, 1, seed=1)


def test_sampler_entry_points_reject_bad_arguments(medium_tables, large_tables):
    """The C checks that answer before any CUDA call (the pointers are never dereferenced)."""
    from psketch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(64)
    for t in (medium_tables, large_tables):
        ct = _lib.make_tables(t)
        C = t.W * t.H
        for cs in (C - 1, 0, -64):
            assert lib.psk_craft_sample_positions(ctypes.byref(ct), fake, fake, 1, fake, 1, 0, 4, cs,
                                                  None, None) == _lib.PSK_ERR_BADARG
        for cs in (C - 1, so.cell_stride(t.W, t.H) + 1):
            assert lib.psk_craft_sample_scenarios(ctypes.byref(ct), fake, fake, fake, 1, 1, 1, 0, 4, cs,
                                                  None, None) == _lib.PSK_ERR_BADARG
    for n_actions in (0, 256, -1):
        assert lib.psk_random_actions(fake, 4, n_actions, 1, 0, None, None) == _lib.PSK_ERR_BADARG
        assert lib.psk_random_actions_block(fake, 4, 2, n_actions, 1, 0, None, None) == _lib.PSK_ERR_BADARG
