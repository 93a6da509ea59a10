"""Pins the CPU oracle (oracle/craft_oracle.c) against the reference's golden vectors and
against outputs exported from the unmodified reference (tests/golden/, made by
oracle/gen_golden.py).  CPU only."""
import numpy as np
import pytest

ERR_ASSERT, ERR_TYPE = 255, 254


def _replay(oracle, grids, ienv, itask, ipos, ref, ref_len):
    """Teacher/step replay of make_data.py:146-152 for all instances at once."""
    n = len(ienv)
    C = grids.shape[1]
    grid = grids[ienv.astype(np.int64)].copy()
    inv = np.zeros((n, oracle.K), np.int32)
    pos = ipos.astype(np.int32).copy()
    dirs = np.zeros(n, np.int32)
    task = itask.astype(np.int32)
    alive = np.ones(n, bool)
    mism = 0
    for t in range(ref.shape[1]):
        idx = np.nonzero(alive)[0]
        if len(idx) == 0:
            break
        a, _, _ = oracle.expert(grid[idx], inv[idx], pos[idx], dirs[idx], task[idx])
        mism += int((a != ref[idx, t]).sum())
        stop = a == 5
        # every trajectory ends satisfied (make_data.py:151)
        if stop.any():
            sat = oracle.satisfies(grid[idx][stop], inv[idx][stop], pos[idx][stop],
                                   dirs[idx][stop], task[idx][stop])
            assert (sat == 1).all()
            assert (ref_len[idx][stop] == t + 1).all()
        g2, i2, p2, d2, st = oracle.step(grid[idx], inv[idx], pos[idx], dirs[idx], a)
        assert (st == 0).all()
        grid[idx], inv[idx], pos[idx], dirs[idx] = g2, i2, p2, d2
        alive[idx[stop]] = False
    assert not alive.any()
    return mism


@pytest.mark.parametrize("split", ["dev", "test", "train"])
def test_oracle_reproduces_golden_trajectories(split, splits, medium_oracle):
    mism = _replay(medium_oracle, splits[split + "_grids"], splits[split + "_inst_env"],
                   splits[split + "_inst_task"], splits[split + "_inst_pos"],
                   splits[split + "_ref_actions"], splits[split + "_ref_len"])
    assert mism == 0


def test_split_sizes(splits):
    # experiments/dagger_no_mix/run.log:41-43
    assert len(splits["train_inst_env"]) == 17600
    assert len(splits["dev_inst_env"]) == 2200 and len(splits["test_inst_env"]) == 2200
    assert int(splits["dev_ref_len"].sum()) == 21981
    assert int(splits["test_ref_len"].sum()) == 23207
    for s in ("train", "dev", "test"):
        g = splits[s + "_grids"]
        assert ((g != 0).sum(axis=1) == 37).all()          # SURVEY §8: 37 occupied cells


def _check_states(oracle, S):
    grid, inv = S["grid"], S["inv"].astype(np.int32)
    pos, dirs = S["pos"].astype(np.int32), S["dir"].astype(np.int32)
    n = len(grid)
    # features (worlds/craft.py:296-330)
    f = oracle.features(grid, inv, pos, dirs)
    assert f.dtype == np.float32
    assert np.array_equal(f, S["features"].astype(np.float32))
    # step for all six actions (worlds/craft.py:332-424)
    for a in range(6):
        g2, i2, p2, d2, st = oracle.step(grid, inv, pos, dirs, np.full(n, a))
        assert (st == 0).all()
        assert np.array_equal(g2, S["step_grid"][:, a])
        assert np.array_equal(i2, S["step_inv"][:, a])
        assert np.array_equal(p2, S["step_pos"][:, a])
        assert np.array_equal(d2, S["step_dir"][:, a])
    assert (S["step_reward"] == 0).all()
    for bad in (-1, 6, 7, 200):
        assert (oracle.step(grid[:4], inv[:4], pos[:4], dirs[:4], np.full(4, bad))[4] == -1).all()
    # satisfies + expert for every task id
    n_tasks = S["satisfies"].shape[1]
    for tid in range(1, n_tasks):
        sat = oracle.satisfies(grid, inv, pos, dirs, np.full(n, tid))
        assert np.array_equal(sat, S["satisfies"][:, tid]), tid
        a, dist, st = oracle.expert(grid, inv, pos, dirs, np.full(n, tid))
        ref = S["expert"][:, tid].astype(np.int32)
        raised = ref == ERR_TYPE
        # where the reference raises TypeError the oracle flags status 2
        assert np.array_equal(st == 2, raised), tid
        ok = ~raised
        assert np.array_equal(a[ok], ref[ok]), tid
    # find_closest_resources
    for j, kind in enumerate(S["go_kinds"]):
        goal, length, st, seq = oracle.find_closest(grid, pos, dirs, np.full(n, kind), seq_cap=48)
        rst = S["closest_status"][:, j]
        assert np.array_equal(st, rst)
        ok = rst == 0
        assert np.array_equal(length[ok], S["closest_len"][ok, j])
        assert np.array_equal(goal[ok], S["closest_goal"][ok, j])
        assert np.array_equal(seq[ok], S["closest_seq"][ok, j])
        none = rst == 1
        assert (length[none] == -1).all()
        has_goal = none & (S["closest_goal"][:, j, 0] != 255)
        assert np.array_equal(goal[has_goal], S["closest_goal"][has_goal, j])


def test_oracle_matches_reference_states_medium(medium_oracle, medium_states):
    _check_states(medium_oracle, medium_states)


def test_oracle_matches_reference_states_large(large_oracle, large_states):
    assert large_oracle.n_features == 1076
    _check_states(large_oracle, large_states)


def test_oracle_matches_reference_states_custom_cookbook(custom_oracle, custom_tables, custom_states):
    """Another cookbook and hint file (tests/golden/custom/): kind ids in a different order
    (boundary is 2, water 1), forward references, _yield 2 and 3, input counts of 2 — the table
    builder and the oracle against 2,000 states exported from the reference running those files."""
    cb = custom_tables.cookbook
    assert cb.index["water"] == 1 and cb.index["boundary"] == 2 and cb.index["plank"] == 13
    assert custom_tables.K == 20 and custom_tables.n_features == 385
    assert int(custom_states["K"]) == 20 and custom_states["features"].shape[1] == 385
    _check_states(custom_oracle, custom_states)


def test_feature_check_vector(medium_oracle, medium_tables):
    """SURVEY Appendix A.3 check vector (probed on the reference)."""
    cb = medium_tables.cookbook
    g = np.zeros((8, 8), np.uint8)
    g[0, :] = g[7, :] = g[:, 0] = g[:, 7] = cb.index["boundary"]
    g[4, 3] = cb.index["wood"]
    g[2, 2] = cb.index["iron"]
    inv = np.zeros((1, 21), np.int32)
    inv[0, cb.index["plank"]] = 2
    f = medium_oracle.features(g.reshape(1, 64), inv, [[3, 3]], [3])[0]
    nz = np.nonzero(f)[0].tolist()
    assert nz == [7, 156, 190, 211, 232, 253, 280, 282, 295, 316, 337, 358, 390, 402]
    assert f[390] == 2 and f.sum() == 15


def test_chain_crafting(medium_oracle, medium_tables):
    """One USE fires every enabled recipe of the workshop in YAML order, inventory updated in
    between (SURVEY §8 row S1, probed on the reference)."""
    cb = medium_tables.cookbook
    ix = cb.index

    def use_at(ws, have):
        g = np.zeros((8, 8), np.uint8)
        g[0, :] = g[7, :] = g[:, 0] = g[:, 7] = ix["boundary"]
        g[3, 4] = ix[ws]
        inv = np.zeros((1, 21), np.int32)
        for k, v in have.items():
            inv[0, ix[k]] = v
        _, i2, _, _, _ = medium_oracle.step(g.reshape(1, 64), inv, [[3, 3]], [1], [4])
        return {cb.index.get(k): int(v) for k, v in enumerate(i2[0]) if v}

    assert use_at("workshop1", {"wood": 1, "iron": 1}) == {"shears": 1}
    assert use_at("workshop0", {"wood": 2, "grass": 1}) == {"wood": 1, "plank": 1, "rope": 1}
    assert use_at("workshop2", {"grass": 1, "wood": 1, "iron": 1, "plank": 1, "stick": 1}) == \
        {"cloth": 1, "bridge": 1, "ladder": 1}


def test_unsatisfied_task_whose_last_subtask_is_satisfied_asserts(tmp_path):
    """teachers/base.py:23-24: `assert incomplete_subtask is not None` fires when every subtask of an
    unsatisfied task is satisfied.  Cannot happen with the stock hint file (last subtasks are use[...]
    / makeat[...]); a custom file whose last subtask is a get/make/go node can trigger it.  The table
    builder marks such nodes, the oracle (and the kernels, tests/test_craft_gpu.py) report the
    reference's AssertionError (action 255 + PSK_FLAG_BAD_LEAF) instead of walking on."""
    import yaml
    from oracle.craft_oracle import CraftOracle
    from psketch_b200.tables import Cookbook, CraftTables, TaskManager
    hints = {"use[none]": [], "go[wood]": [], "get[wood]": ["go[wood]", "use[none]"],
             "make[plank]": ["get[wood]"]}
    hp = str(tmp_path / "hints.yaml")
    yaml.safe_dump(hints, open(hp, "w"), sort_keys=False)
    tables = CraftTables(Cookbook(), TaskManager(hp), "craft_medium")
    assert tables.may_assert and "plank" in tables.may_assert[0][0]
    o = CraftOracle(tables)
    cb = tables.cookbook
    grid = np.zeros((2, 8, 8), np.uint8)
    grid[:, 0, :] = grid[:, 7, :] = grid[:, :, 0] = grid[:, :, 7] = 1
    grid[:, 3, 5] = cb.index["wood"]
    grid = grid.reshape(2, 64)
    inv = np.zeros((2, tables.K), np.int32)
    inv[1, cb.index["wood"]] = 1                      # env 1 already holds wood, has no plank
    pos = np.asarray([[3, 3], [3, 3]], np.int32)
    dirs = np.zeros(2, np.int32)
    task = np.full(2, tables.task_manager["make[plank]"].task_id, np.int32)
    act, _, _ = o.expert(grid, inv, pos, dirs, task)
    # the reference's answers on these two states: env 0 walks UP towards the wood; env 1 asserts
    assert act[0] == 1 and act[1] == 255
