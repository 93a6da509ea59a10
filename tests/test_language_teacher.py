"""Language teachers (host word logic): fixed expectations, and the batched forms against the
per-rollout ones.  Same words, learned action map and random-stream use as the reference's
teachers/primitive_language.py are pinned by the record of the reference's own training run
(tests/test_config4.py).  CPU only (fake states: ``describe`` reads just .pos and .inventory)."""
import types

import numpy as np
import pytest


class _S(object):
    def __init__(self, pos, inv):
        self.pos, self.inventory = pos, np.asarray(inv, float)


def _world():
    names = ("DOWN", "UP", "LEFT", "RIGHT", "USE", "STOP")
    acts = types.SimpleNamespace(**{n: types.SimpleNamespace(index=i) for i, n in enumerate(names)})
    return types.SimpleNamespace(actions=acts, action_space=[getattr(acts, n) for n in names])


def _episodes(rng, n=40):
    eps = []
    perm = rng.permutation(6)            # the student's private action ids
    delta = {0: (0, -1), 1: (0, 1), 2: (-1, 0), 3: (1, 0)}
    for _ in range(n):
        L = rng.randint(1, 9)
        pos, inv = (3, 3), [0, 0, 0]
        states, actions = [_S(pos, inv)], []
        for t in range(L):
            real = rng.randint(0, 6)
            actions.append(int(perm[real]))
            if real < 4 and rng.rand() < 0.7:
                pos = (pos[0] + delta[real][0], pos[1] + delta[real][1])
            elif real == 4 and rng.rand() < 0.5:
                inv = [inv[0] + 1, inv[1], inv[2]]
            states.append(_S(pos, list(inv)))
        eps.append((actions, states))
    return eps


def test_instruct_and_describe():
    from psketch_b200.teachers import PrimitiveLanguageTeacher
    from psketch_b200.teachers.primitive_language import instruct_batch
    world = _world()
    cfg = types.SimpleNamespace(random=np.random.RandomState(5))
    t = PrimitiveLanguageTeacher(cfg)
    assert t.instruct(world, [1, 0, 2, 3, 4, 5]) == ["up", "down", "left", "right", "use", "stop"]
    with pytest.raises(AssertionError):
        t.instruct(world, [6])
    ids = instruct_batch(np.asarray([[1, 4, 5, 255]], np.uint8))
    assert ids.tolist() == [[2, 5, 6, 0]]
    eps = _episodes(np.random.RandomState(1))
    mine = [t.describe(world, a, s) for a, s in eps]
    assert all(len(m) == len(a) for m, (a, _) in zip(mine, eps))
    assert len(t.student_action_map) >= 4


def _pack(eps, L):
    """Episodes of _episodes() -> (actions [N, L], agent records [L + 1, N, 32], lengths [N])."""
    n = len(eps)
    acts = np.zeros((n, L), np.int64)
    agent = np.zeros((L + 1, n, 32), np.uint8)
    lengths = np.zeros(n, np.int64)
    for i, (a, states) in enumerate(eps):
        lengths[i] = len(a)
        acts[i, :len(a)] = a
        for t in range(L + 1):
            s = states[min(t, len(states) - 1)]
            agent[t, i, 24], agent[t, i, 25] = s.pos[0] + 100, s.pos[1] + 100   # only differences matter
            agent[t, i, :3] = s.inventory
    return acts, agent, lengths


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_describe_batch_equals_describe(seed):
    """describe_batch (tensor operations over [N, L], host loop only per new action-map entry)
    against describe called rollout by rollout: same words, same learned map after every call,
    same position of the shared random stream — over several consecutive batches, starting from an
    empty map (so the first calls exercise the learning / guessing / last-id-inference paths)."""
    import torch
    from psketch_b200.teachers import PrimitiveLanguageTeacher
    from psketch_b200.teachers.primitive_language import ACTION_WORDS
    world = _world()
    a = PrimitiveLanguageTeacher(types.SimpleNamespace(random=np.random.RandomState(seed)))
    b = PrimitiveLanguageTeacher(types.SimpleNamespace(random=np.random.RandomState(seed)))
    rng = np.random.RandomState(100 + seed)
    perm_rng = np.random.RandomState(seed)               # one student = one private id permutation
    for call in range(6):
        eps = _episodes(np.random.RandomState(rng.randint(1 << 30)), n=3 if call < 3 else 40)
        perm = perm_rng.permutation(6) if call == 0 else perm
        # re-label with a permutation that stays fixed across calls
        eps = [([int(perm[x % 6]) for x in acts], states) for acts, states in eps]
        want = [a.describe(world, acts, states) for acts, states in eps]
        acts, agent, lengths = _pack(eps, 9)
        got = b.describe_batch(torch.from_numpy(acts), torch.from_numpy(agent), torch.from_numpy(lengths), n_kinds=3)
        got = [[ACTION_WORDS[w] for w in row[:n]] for row, n in zip(got.tolist(), lengths)]
        assert got == want, call
        assert a.student_action_map == b.student_action_map, call
    assert a.random.randint(1 << 30) == b.random.randint(1 << 30)
    assert len(b.student_action_map) == 6
