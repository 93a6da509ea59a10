"""PSK_TICK_STEP_FIRST (VecCraft.step_observe): CraftState.step alone — no timer, no done, no
auto-reset, STOP the idle action — then the teacher's action and the features of the NEW state, in one
launch.  The language trainers' decoding step (trainers/primitive_language.py:47-70, 93-113).

Every tick is checked against oracle/craft_oracle.c: the step (with the u8 inventory rule of
psk_craft_step, tests/test_edge_states_cpu.step_u8), then the teacher and the features of the new
state, in f32 and u8 frames.  Outputs are poisoned before every call."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_edge_states_cpu import edge_states, step_u8           # noqa: E402
from test_fused_states_gpu import tuning                         # noqa: E402

pytestmark = pytest.mark.gpu

AG_X, AG_DIR, AG_TASK, AG_TIMER = 24, 26, 27, 28
POISON = 0xA5


class Model(object):
    """The oracle's copy of a batch: grid u8[n, C], inv i32[n, K], pos, dir, task, timer."""

    def __init__(self, tables, oracle, grid, inv, pos, dirs, task, timer):
        self.tables, self.oracle = tables, oracle
        self.grid, self.inv = np.asarray(grid, np.uint8).copy(), np.asarray(inv, np.int32).copy()
        self.pos, self.dir = np.asarray(pos, np.int32).copy(), np.asarray(dirs, np.int32).copy()
        self.task, self.timer = np.asarray(task, np.int32), np.asarray(timer, np.uint8)

    def env(self):
        from psketch_b200.vec import VecCraft
        env = VecCraft.from_states(self.tables, self.grid, self.inv, self.pos, self.dir, task=self.task)
        env.agent[:, AG_TIMER] = torch.from_numpy(self.timer).to(env.device)
        return env

    def step(self, actions):
        """Returns the PSK_FLAG_* bits the step raises."""
        a = np.asarray(actions, np.int32)
        bad = a > 5
        g, inv, pos, dirs, over, _ = step_u8(self.tables, self.grid, self.inv, self.pos, self.dir,
                                              np.where(bad, 5, a))
        self.grid, self.inv, self.pos, self.dir = g, inv.astype(np.int32), pos, dirs
        return (1 if bad.any() else 0) | (2 if over.any() else 0)

    def observe(self):
        o = self.oracle
        act, _, _ = o.expert(self.grid, self.inv, self.pos, self.dir, self.task)
        return act.astype(np.uint8), o.features(self.grid, self.inv, self.pos, self.dir)

    def assert_state(self, env):
        agent = env.agent.cpu().numpy()
        assert np.array_equal(env.cells.cpu().numpy(), self.grid)
        assert np.array_equal(agent[:, :self.tables.K], self.inv)
        assert np.array_equal(agent[:, AG_X:AG_X + 2], self.pos)
        assert np.array_equal(agent[:, AG_DIR], self.dir)
        assert np.array_equal(agent[:, AG_TASK], self.task)
        assert np.array_equal(agent[:, AG_TIMER], self.timer)     # the timer is not touched


def raw_tick(env, actions, order, u8=False):
    """psk_craft_tick(_u8) with every output poisoned, done / success and stats included."""
    from psketch_b200 import _lib
    n, dev = env.n, env.device
    feats = torch.full((n, env.n_features), POISON, dtype=torch.uint8 if u8 else torch.float32, device=dev)
    expert, done, success = (torch.full((n,), POISON, dtype=torch.uint8, device=dev) for _ in range(3))
    acts = None if actions is None else torch.as_tensor(np.asarray(actions, np.uint8)).to(dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    entry = env.lib.psk_craft_tick_u8 if u8 else env.lib.psk_craft_tick
    with torch.cuda.device(dev):
        rc = entry(ctypes.byref(env.ct), env._state(), env._episodes(), p(acts), p(feats), p(expert), p(done),
                   p(success), p(env.stats), p(env.err_flags), order, env._stream())
    _lib.check(rc, "psk_craft_tick")
    return dict(features=feats, expert=expert, done=done, success=success)


def check_tick(env, model, actions, u8=False, raw=False):
    """One step_observe tick on the device and on the oracle; every output and the state compared."""
    from psketch_b200 import _lib
    env.err_flags.zero_()
    stats = env.stats.clone()
    if raw:
        out = raw_tick(env, actions, _lib.TICK_STEP_FIRST, u8)
        assert (out["done"] == 0).all() and (out["success"] == 0).all()
    else:
        feats = torch.full((env.n, env.n_features), POISON, dtype=torch.uint8 if u8 else torch.float32,
                           device=env.device)
        out = env.step_observe(actions, features_out=feats,
                               out={"expert": torch.full((env.n,), POISON, dtype=torch.uint8, device=env.device)})
    want_flags = model.step(actions) if actions is not None else 0
    act, feats = model.observe()
    torch.cuda.synchronize()
    model.assert_state(env)
    assert np.array_equal(out["expert"].cpu().numpy(), act)
    got = out["features"].cpu().numpy()
    assert np.array_equal(got.astype(np.float32) if u8 else got, feats)
    assert torch.equal(env.stats, stats)                          # stats are not touched
    flags = int(env.err_flags.item())
    assert flags & (_lib.FLAG_BAD_ACTION | _lib.FLAG_INV_OVERFLOW) == want_flags, (flags, want_flags)
    assert not flags & _lib.FLAG_CHAIN_TIMEOUT
    env.err_flags.zero_()


def _random_actions(rng, n, bad=False):
    a = rng.randint(0, 6, size=n)
    a = np.where(rng.rand(n) < 0.3, 4, a)                          # plenty of USE
    if bad:
        a = np.where(rng.rand(n) < 0.1, rng.randint(6, 256, size=n), a)
    return a.astype(np.uint8)


def _edge_model(tables, oracle, S, n, seed):
    st = edge_states(tables, S, n, seed)
    rng = np.random.RandomState(seed)
    task = rng.randint(1, tables.n_tasks, size=n)
    return Model(tables, oracle, st["grid"], st["inv"], st["pos"], st["dir"], task,
                 rng.randint(0, 256, size=n))


@pytest.fixture(params=["medium", "large", "custom"])
def world(request, medium_tables, medium_oracle, medium_states, large_tables, large_oracle, large_states,
          custom_tables, custom_oracle, custom_states):
    return dict(medium=(medium_tables, medium_oracle, medium_states),
                large=(large_tables, large_oracle, large_states),
                custom=(custom_tables, custom_oracle, custom_states))[request.param]


@pytest.mark.parametrize("u8", [False, True])
def test_step_observe_on_edge_states_with_random_actions(world, u8):
    """Exported states facing what USE acts on, inventories up to 255, random timers; random action
    streams with USE, STOP and bytes 6..255 (BAD_ACTION, the env untouched)."""
    tables, oracle, S = world
    model = _edge_model(tables, oracle, S, 2000, seed=3)
    env = model.env()
    rng = np.random.RandomState(4)
    check_tick(env, model, None, u8)                              # observe only: nothing moves
    for k in range(12):
        check_tick(env, model, _random_actions(rng, env.n, bad=k % 3 == 1), u8, raw=k % 2 == 0)


def test_step_observe_along_golden_dev_trajectories(splits, medium_tables, medium_oracle):
    """The dev instances follow their reference action sequences (STOP last, then idle on STOP)."""
    g = splits["dev_grids"][splits["dev_inst_env"]]
    n = len(g)
    model = Model(medium_tables, medium_oracle, g, np.zeros((n, medium_tables.K)), splits["dev_inst_pos"],
                  np.zeros(n), splits["dev_inst_task"], np.full(n, 40))
    env = model.env()
    ref = splits["dev_ref_actions"]
    check_tick(env, model, None)
    for t in range(ref.shape[1]):
        a = np.where(ref[:, t] == 255, 5, ref[:, t])
        check_tick(env, model, a, u8=t % 2 == 1)


@pytest.mark.parametrize("n", [1, 31, 33, 4097, 65573])
def test_step_observe_batch_sizes(n, splits, medium_tables, medium_oracle):
    rng = np.random.RandomState(n)
    pick = rng.randint(0, len(splits["train_inst_env"]), size=n)
    model = Model(medium_tables, medium_oracle, splits["train_grids"][splits["train_inst_env"][pick]],
                  np.zeros((n, medium_tables.K)), splits["train_inst_pos"][pick], rng.randint(0, 4, size=n),
                  splits["train_inst_task"][pick], rng.randint(0, 256, size=n))
    env = model.env()
    for k in range(4):
        check_tick(env, model, _random_actions(rng, n), u8=k == 3, raw=k == 2)


def test_step_observe_16x16_takes_separate_launches():
    """Grids above 128 cells: psk_craft_step, then teacher and features (the same results)."""
    from oracle.craft_oracle import CraftOracle
    from test_stress_gpu import _random_states, _tables
    tables = _tables(16)
    grid, inv, pos, dirs, task = _random_states(tables, 700, seed=5, wall_frac=0.2)
    rng = np.random.RandomState(6)
    model = Model(tables, CraftOracle(tables), grid, inv, pos, dirs, task, rng.randint(0, 256, size=len(grid)))
    n = len(grid)
    env = model.env()
    check_tick(env, model, None)
    for k in range(8):
        check_tick(env, model, _random_actions(rng, n, bad=k == 3), u8=k % 2 == 1, raw=k % 3 == 0)


def test_step_observe_chained_with_the_other_orders(splits, medium_tables, medium_oracle):
    """50 back-to-back launches, then launches interleaved with ADVANCE_FIRST, FUSED and psk_craft_rollout
    on the same batch (tile chaining at its default and off, and under CUDA-graph replay); the oracle
    follows every step and the final state / observations must agree."""
    from psketch_b200 import _lib
    n = 20000
    rng = np.random.RandomState(7)
    pick = rng.randint(0, len(splits["train_inst_env"]), size=n)
    for chain in (None, 0):
        with tuning(tile_chain=chain):
            model = Model(medium_tables, medium_oracle, splits["train_grids"][splits["train_inst_env"][pick]],
                          np.zeros((n, medium_tables.K)), splits["train_inst_pos"][pick], np.zeros(n),
                          splits["train_inst_task"][pick], np.full(n, 255))
            env = model.env()
            acts = [_random_actions(rng, n) for _ in range(50)]
            feats = torch.empty((n, env.n_features), device=env.device)
            for a in acts:
                out = env.step_observe(a, features_out=feats)
                model.step(a)
            torch.cuda.synchronize()
            check_tick(env, model, None)
            # interleaved: the other orders move the state (and the timer) through the oracle's rollout
            # rules, so each is checked on its own outcome: pure-step envs are those it leaves alone
            for k in range(6):
                a = _random_actions(rng, n)
                env.step_observe(a, features_out=feats)
                model.step(a)
                snap = env.snapshot()
                other = k % 3
                if other == 0:
                    env.tick(actions=np.full(n, 5, np.uint8), advance_first=True)    # STOP: every env resets
                elif other == 1:
                    env.tick(fused=True)
                else:
                    env.rollout(3)
                env.restore(snap)          # back to the step-first state: the chain must have kept order
                check_tick(env, model, _random_actions(rng, n))
            # CUDA-graph replay of 5 step-first ticks with fixed actions
            a_dev = torch.from_numpy(np.stack([_random_actions(rng, n) for _ in range(5)])).to(env.device)
            env.step_observe(None, features_out=feats)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            snap = env.snapshot()
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    for t in range(5):
                        env.step_observe(a_dev[t], features_out=feats)
            torch.cuda.current_stream().wait_stream(side)
            env.restore(snap)
            for _ in range(2):
                g.replay()
                for t in range(5):
                    model.step(a_dev[t].cpu().numpy())
            torch.cuda.synchronize()
            check_tick(env, model, None)
            assert int(env.err_flags.item()) & _lib.FLAG_CHAIN_TIMEOUT == 0


def test_step_observe_every_variant_gives_the_same_bytes(medium_tables, medium_oracle, medium_states):
    """tick_variant / tick_tma / tick_persist / tick_pdl forced through psk_set_tuning."""
    knobs = [dict(tick_variant=v) for v in range(5)] + [dict(tick_tma=1), dict(tick_tma=0),
                                                         dict(tick_persist=1), dict(tick_pdl=0)]
    for kn in knobs:
        with tuning(**kn):
            model = _edge_model(medium_tables, medium_oracle, medium_states, 3000, seed=11)
            env = model.env()
            rng = np.random.RandomState(12)
            for k in range(3):
                check_tick(env, model, _random_actions(rng, env.n, bad=k == 1), u8=k == 2)


def test_step_observe_stays_inside_its_buffers(splits, medium_tables):
    from test_bounds_gpu import Arena, _carved_env, _instances
    from psketch_b200.vec import VecCraft
    for n, skew in ((33, 0), (4097, 16)):
        ref = VecCraft.from_instances(medium_tables, *_instances(splits, n, seed=n), max_timesteps=40)
        arena = Arena(n * (64 + 32) * 3 + n * (404 * 4 + 8) * 2 + (1 << 20), ref.device)
        env = _carved_env(medium_tables, arena, ref)
        feats = arena.carve((n, env.n_features), torch.float32, skew=skew)
        feats8 = arena.carve((n, env.n_features), torch.uint8, skew=skew)
        expert = arena.carve((n,), torch.uint8, skew=skew)
        acts = arena.carve((n,), torch.uint8, skew=skew)
        rng = np.random.RandomState(n)
        for k in range(6):
            acts.copy_(torch.from_numpy(_random_actions(rng, n)))
            env.step_observe(acts, features_out=feats8 if k % 2 else feats, out={"expert": expert})
            ref.step_observe(acts)
        torch.cuda.synchronize()
        assert arena.guards_intact()
        assert torch.equal(env.grid, ref.grid) and torch.equal(env.agent, ref.agent)
