"""psketch_b200.students.GraphedDecode — one decoding pass of the language trainers as one CUDA graph
of step-then-observe ticks — against the eager psketch_b200.rollout.language_decode (bit for bit), the
record of the reference's own PrimitiveLanguageTrainer run, and the C oracle."""
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
T = 40
POISON = 0xA5


def _script(rng, n, never_stop_frac=0.2):
    """Random actions u8[T, n] with a STOP at a random time, except for envs that never stop."""
    a = rng.randint(0, 5, size=(T, n))
    stop_at = rng.randint(0, T + 10, size=n)
    stop_at[rng.rand(n) < never_stop_frac] = T + 10
    a[stop_at[None, :] == np.arange(T)[:, None]] = 5
    return a.astype(np.uint8)


def _point(env, splits, rows):
    """Re-points the env at other train instances, as examples/train_dagger.Batches.next does."""
    dev = env.device
    env.scen_idx.copy_(torch.from_numpy(splits["train_inst_env"][rows].astype(np.int32)).to(dev))
    env.init_agent[:, 24:26] = torch.from_numpy(splits["train_inst_pos"][rows].astype(np.uint8)).to(dev)
    env.init_agent[:, 27] = torch.from_numpy(splits["train_inst_task"][rows].astype(np.uint8)).to(dev)


def _poison(dec):
    for t in (dec.feats, dec.acts, dec.lengths, dec.steps) + ((dec.agents,) if dec.record else ()):
        t.fill_(POISON if t.dtype != torch.bool else True)


def _eager(env, script, record=True):
    feats = torch.full((T, env.n, env.n_features), float("nan"), device=env.device)

    def pol(f, t):
        feats[t].copy_(f)
        return script[t]
    from psketch_b200.rollout import language_decode
    out = language_decode(env, pol, T, record=record)
    return out, feats


def _compare(got, want, want_feats):
    assert torch.equal(got["actions"], want["actions"])
    assert torch.equal(got["lengths"], want["lengths"])
    assert got["steps"] == want["steps"]
    L = int(want["lengths"].max())
    assert got["timesteps"] == L
    if want["agents"] is not None:
        assert torch.equal(got["agents"], want["agents"][:L + 1])
    live = torch.arange(T, device=want["lengths"].device)[:, None] < want["lengths"][None, :]   # [T, n]
    assert torch.equal(got["features"][live], want_feats[live])


@pytest.mark.parametrize("n", [33, 1024, 65573])
def test_graphed_decode_equals_eager_decode(n, splits, medium_tables):
    from psketch_b200.students import GraphedDecode
    from psketch_b200.vec import VecCraft
    rng = np.random.RandomState(n)
    rows = rng.randint(0, len(splits["train_inst_env"]), size=n)
    env = VecCraft.from_instances(medium_tables, splits["train_grids"], splits["train_inst_env"][rows],
                                  splits["train_inst_pos"][rows], splits["train_inst_task"][rows], max_timesteps=40)
    script = torch.from_numpy(_script(rng, n)).to(env.device)
    for record in (True, False):
        dec = GraphedDecode(env, lambda f, t: script[t], T, record=record)
        for rep in range(2):
            if rep:      # a pure replay on other instances and another script
                rows = rng.randint(0, len(splits["train_inst_env"]), size=n)
                _point(env, splits, rows)
                script.copy_(torch.from_numpy(_script(rng, n)))
            _poison(dec)
            got = dec.run()
            assert len(dec.graphs) == 1
            want, feats = _eager(env, script, record)
            _compare(got, want, feats)


def test_graphed_decode_on_craft_large(large_tables, large_states):
    from psketch_b200.students import GraphedDecode
    from psketch_b200.vec import VecCraft
    S = large_states
    n = 97
    rng = np.random.RandomState(5)
    ii = rng.randint(0, len(S["grid"]), size=n)
    env = VecCraft.from_states(large_tables, S["grid"][ii], S["inv"][ii], S["pos"][ii], S["dir"][ii],
                               task=rng.randint(1, large_tables.n_tasks, size=n))
    script = torch.from_numpy(_script(rng, n)).to(env.device)
    dec = GraphedDecode(env, lambda f, t: script[t], T, record=True)
    for rep in range(2):
        script.copy_(torch.from_numpy(_script(rng, n)))
        _poison(dec)
        got = dec.run()
        want, feats = _eager(env, script)
        _compare(got, want, feats)


def test_graphed_passes_reproduce_the_reference_trainer(splits, medium_tables):
    """The first 12 iterations of tests/golden/config4_primitive_language.npz (the reference's own
    PrimitiveLanguageTrainer run): both decoding passes through GraphedDecode with the recorded
    actions, describe_batch on the graph's agent records — descriptions (with the random words drawn
    while the teacher learns the action ids), final action sequences, success and num_steps."""
    from psketch_b200.students import GraphedDecode
    from psketch_b200.teachers import PrimitiveLanguageTeacher
    from psketch_b200.vec import VecCraft
    fx = np.load(os.path.join(GOLDEN, "config4_primitive_language.npz"))
    rng = np.random.RandomState(123)
    teacher = PrimitiveLanguageTeacher(type("Cfg", (), {"random": rng})())
    order = list(range(len(splits["train_inst_env"])))
    rng.shuffle(order)                                             # data/dataset.py:70-72
    env = p1 = p2 = d1 = d2 = None
    for r in range(12):
        B = int(fx["n_env"][r])
        rows = order[32 * r:32 * r + 32]
        assert rows == fx["batch"][r, :B].tolist()
        if env is None:
            env = VecCraft.from_instances(medium_tables, splits["train_grids"], splits["train_inst_env"][rows],
                                          splits["train_inst_pos"][rows], splits["train_inst_task"][rows],
                                          max_timesteps=40)
            p1 = torch.empty((T, B), dtype=torch.uint8, device=env.device)
            p2 = torch.empty_like(p1)
            d1 = GraphedDecode(env, lambda f, t: p1[t], T, record=True)
            d2 = GraphedDecode(env, lambda f, t: p2[t], T, record=False)
        else:
            _point(env, splits, np.asarray(rows))
        p1.copy_(torch.from_numpy(fx["acts"][r][:, :B]))           # 255 = terminated (never executed)
        p2.copy_(torch.from_numpy(fx["phase2_acts"][r][:, :B]))
        _poison(d1)
        _poison(d2)
        first = d1.run()
        L = first["timesteps"]
        desc = teacher.describe_batch(first["actions"][:, :L].long(), first["agents"], first["lengths"], n_kinds=env.K)
        second = d2.run()
        success = (env.satisfies() == 1).cpu().numpy()
        acts = second["actions"].cpu().numpy()
        for i in range(B):
            wd = [int(w) for w in fx["descriptions"][r, i] if w != 255]
            gd = desc[i].cpu().numpy()
            assert gd[gd >= 0].tolist() == wd, (r, i)
            Ls = int(fx["seq_len"][r, i])
            assert acts[i, :Ls].tolist() == fx["phase2_acts"][r, :Ls, i].tolist(), (r, i)
            assert (acts[i, Ls:] == 255).all()
        assert success.tolist() == fx["success"][r, :B].astype(bool).tolist(), r
        assert first["steps"] == int(fx["num_steps"][r]), r
    assert len(teacher.student_action_map) >= 5


@pytest.mark.parametrize("greedy", [True, False])
def test_seq2seq_decode_replays_on_the_oracle(greedy, splits, medium_tables, medium_oracle):
    """examples/train_language.DecodeStep (Seq2SeqPolicy, time index t, Gumbel-max or argmax) in the
    graph: replaying the executed actions on the CPU oracle reproduces the features the policy saw,
    the agent records and the lengths; greedy passes are identical to each other."""
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    from train_language import DecodeStep, decode
    from psketch_b200.students import GraphedDecode, Seq2SeqPolicy, task_tokens
    from psketch_b200.vec import VecCraft
    n = 300
    rng = np.random.RandomState(8)
    rows = rng.randint(0, len(splits["train_inst_env"]), size=n)
    env = VecCraft.from_instances(medium_tables, splits["train_grids"], splits["train_inst_env"][rows],
                                  splits["train_inst_pos"][rows], splits["train_inst_task"][rows], max_timesteps=40)
    torch.manual_seed(0)
    vocab = medium_tables.task_manager.vocab
    model = Seq2SeqPolicy(env.n_features, 6, len(vocab) + 1, vocab["<PAD>"]).to(env.device)
    dec = GraphedDecode(env, DecodeStep(model, n, env.device, greedy=greedy), T, record=True)
    with torch.no_grad():
        mem = model.encode(task_tokens(medium_tables, env.task, reverse=False))
    runs = []
    for rep in range(2):
        _poison(dec)
        got = decode(dec, mem)
        runs.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in got.items()})
    if greedy:
        for k in ("actions", "lengths", "agents", "features"):
            assert torch.equal(runs[0][k], runs[1][k]), k
    got = runs[1]
    acts, lengths = got["actions"].cpu().numpy(), got["lengths"].cpu().numpy()
    feats, agents = got["features"].cpu().numpy(), got["agents"].cpu().numpy()
    o, K = medium_oracle, medium_tables.K
    grid = splits["train_grids"][splits["train_inst_env"][rows]].copy()
    inv, pos = np.zeros((n, K), np.int32), splits["train_inst_pos"][rows].astype(np.int32)
    dirs = np.zeros(n, np.int32)
    for t in range(T):
        live = t < lengths
        assert np.array_equal(feats[t][live], o.features(grid, inv, pos, dirs)[live]), t
        assert ((acts[:, t] != 255) == live).all()
        a = np.where(live, acts[:, t], 5).astype(np.int32)
        stop = live & (a == 5)
        assert (lengths[stop] == t + 1).all()
        grid, inv, pos, dirs, _ = o.step(grid, inv, pos, dirs, a)
        if t + 1 < len(agents):
            assert np.array_equal(agents[t + 1][:, :K], inv) and np.array_equal(agents[t + 1][:, 24:26], pos)
            assert np.array_equal(agents[t + 1][:, 26], dirs)
    never = lengths == T
    assert (acts[never] != 5)[:, :-1].all()
