"""Zero-copy student ingestion (SURVEY §8(f) N3, BASELINE configs[3]).

The reference's student (students/imitation.py:71-84) turns a Python list of per-env float64
ndarrays into a tensor, copies it to the GPU, decodes one step, and copies the sampled actions back
to the host — every timestep.  Here the env's ``f32[N, 404]`` feature tensor is already on the
device, the policy reads it in place, samples on the device, and the sampled ``u8[N]`` actions go
straight into the env kernel; one whole rollout (40 timesteps of: fused tick in "step, then
observe" order -> decode -> sample) is ONE CUDA graph replay with no host round trip
(``GraphedRollout``).

``GraphedDecode`` does the same for the language trainers' decoding passes (step, then observe,
without the imitation trainer's episode rules).

``Seq2SeqPolicy`` has the architecture of the reference's ``models/lstm_seq2seq.py:LSTMSeq2SeqModel``
(task-token encoder LSTM with source-position embeddings, decoder LSTM over [features, time
embedding], dot-product attention over the encoder outputs, two-layer predictor), organised for
batched device-resident decoding: checkpoints interchange with the reference through
``load_reference_state_dict`` / ``to_reference_state_dict``, and tests/test_students.py pins its
logits to the reference model's on the same weights.  The student is dense PyTorch (cuDNN LSTM,
cuBLAS) exactly as in the reference: it is the consumer of the hot path, not part of it.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .tables import STOP

TIME_EMBED = 64            # models/lstm_seq2seq.py:80
MAX_POSITIONS = 100        # models/lstm_seq2seq.py:112-113

# reference parameter name -> name here
_REFERENCE_KEYS = {
    "encoder.lstm.lstm.weight_ih_l0": "enc.weight_ih_l0", "encoder.lstm.lstm.weight_hh_l0": "enc.weight_hh_l0",
    "encoder.lstm.lstm.bias_ih_l0": "enc.bias_ih_l0", "encoder.lstm.lstm.bias_hh_l0": "enc.bias_hh_l0",
    "decoder.lstm.lstm.weight_ih_l0": "dec.weight_ih_l0", "decoder.lstm.lstm.weight_hh_l0": "dec.weight_hh_l0",
    "decoder.lstm.lstm.bias_ih_l0": "dec.bias_ih_l0", "decoder.lstm.lstm.bias_hh_l0": "dec.bias_hh_l0",
    "attention.linear_in_h.weight": "att_q.weight", "attention.linear_in_h.bias": "att_q.bias",
    "attention.linear_in_v.weight": "att_v.weight", "attention.linear_in_v.bias": "att_v.bias",
    "predictor.0.weight": "head1.weight", "predictor.0.bias": "head1.bias",
    "predictor.2.weight": "head2.weight", "predictor.2.bias": "head2.bias",
    "enc2dec.0.weight": "enc2dec.weight", "enc2dec.0.bias": "enc2dec.bias",
    "embedding.weight": "word.weight",
    "src_time_embedding.weight": "src_time.weight", "tgt_time_embedding.weight": "tgt_time.weight",
}
# the reference's encoder owns an nn.Embedding it never uses (models/lstm_seq2seq.py:24,37-38)
_REFERENCE_UNUSED = "encoder.embedding.weight"


class Seq2SeqPolicy(nn.Module):
    def __init__(self, n_features, n_actions, vocab_size, pad_idx, hidden=256, word_embed=128):
        super().__init__()
        self.hidden, self.n_features, self.n_actions = hidden, n_features, n_actions
        self.word = nn.Embedding(vocab_size, word_embed, padding_idx=pad_idx)
        self.src_time = nn.Embedding(MAX_POSITIONS, TIME_EMBED)
        self.tgt_time = nn.Embedding(MAX_POSITIONS, TIME_EMBED)
        self.enc = nn.LSTM(word_embed + TIME_EMBED, hidden, 1, batch_first=True)
        self.dec = nn.LSTM(n_features + TIME_EMBED, hidden, 1)
        self.enc2dec = nn.Linear(hidden, hidden)
        self.att_q = nn.Linear(hidden, hidden // 2)
        self.att_v = nn.Linear(hidden, hidden // 2)
        self.head1 = nn.Linear(2 * hidden, hidden)
        self.head2 = nn.Linear(hidden, n_actions)

    # ---- checkpoints of the reference (students/imitation.py:100-111)
    def load_reference_state_dict(self, sd):
        mine = {ours: sd[theirs] for theirs, ours in _REFERENCE_KEYS.items()}
        self.load_state_dict(mine, strict=True)

    def to_reference_state_dict(self):
        sd = self.state_dict()
        out = {theirs: sd[ours].clone() for theirs, ours in _REFERENCE_KEYS.items()}
        out[_REFERENCE_UNUSED] = torch.zeros(
            (self.word.num_embeddings, self.word.embedding_dim + TIME_EMBED), dtype=sd["word.weight"].dtype,
            device=sd["word.weight"].device)
        return out

    # ---- model.init (models/lstm_seq2seq.py:118-134)
    def encode(self, tokens, mask=None):
        """tokens i64[N, L] -> memory dict: the encoder outputs, their attention keys, the decoder's
        initial state.  ``mask`` bool[N, L] marks padding positions (set to -inf before the softmax)."""
        n, L = tokens.shape
        pos = torch.arange(L, device=tokens.device).unsqueeze(0).expand(n, L)
        x = torch.cat([self.word(tokens), self.src_time(pos)], dim=2)
        ctx, (h, c) = self.enc(x)
        h0 = torch.tanh(self.enc2dec(h))                    # [1, N, H]
        return {"ctx": ctx, "keys": self.att_v(ctx), "h0": h0, "c0": c, "mask": mask}

    def _head(self, o, mem):
        """o [M, H] decoder outputs, mem rows aligned with o -> action logits [M, n_actions]."""
        q = self.att_q(o).unsqueeze(2)                      # [M, H/2, 1]
        score = torch.bmm(mem["keys"], q).squeeze(2)        # [M, L]
        if mem["mask"] is not None:
            score = score.masked_fill(mem["mask"], float("-inf"))
        attn = F.softmax(score, dim=1).unsqueeze(1)
        wc = torch.bmm(attn, mem["ctx"]).squeeze(1)         # [M, H]
        return self.head2(torch.tanh(self.head1(torch.cat([o, wc], dim=1))))

    # ---- model.decode (models/lstm_seq2seq.py:136-150), one timestep
    def decode_step(self, features, time_idx, state, mem):
        """features f32[N, n_features] (the env's device tensor, read in place), time_idx i64[N],
        state (h, c) each [1, N, H] -> (logits [N, n_actions], new state)."""
        x = torch.cat([features, self.tgt_time(time_idx)], dim=1).unsqueeze(0)
        o, state = self.dec(x, state)
        return self._head(o[0], mem), state

    # ---- the same decode over a recorded window, for learning: one cuDNN call over T steps
    def decode_sequence(self, features, time_idx, mem):
        """features f32[T, N, n_features], time_idx i64[T, N] -> logits [T, N, n_actions], the same
        function of the same inputs as T calls of decode_step from (h0, c0)."""
        T, n, _ = features.shape
        x = torch.cat([features, self.tgt_time(time_idx)], dim=2)
        o, _ = self.dec(x, (mem["h0"], mem["c0"]))
        rep = {"ctx": mem["ctx"].repeat(T, 1, 1), "keys": mem["keys"].repeat(T, 1, 1),
               "mask": None if mem["mask"] is None else mem["mask"].repeat(T, 1)}
        return self._head(o.reshape(T * n, -1), rep).view(T, n, -1)


def task_tokens(tables, task_ids, reverse=True):
    """task ids (tensor [N]) -> i64[N, 2] vocabulary encodings (data/task.py:65-66); reversed like
    students/imitation.py:60-63 by default (PrimitiveLanguageStudent does not reverse, :78-80)."""
    tm = tables.task_manager
    table = torch.zeros((len(tm.tasks), 2), dtype=torch.long)
    for t in tm.tasks:
        table[t.task_id] = torch.tensor(list(reversed(t.encoding)) if reverse else t.encoding)
    return table.to(task_ids.device)[task_ids.long()]


def imitation_loss(logits, refs):
    """students/imitation.py:86-98: per timestep the mean cross-entropy over the envs whose label is
    not -1 (done envs), summed over the timesteps; returns (loss to backpropagate, loss / T)."""
    T = logits.shape[0]
    ce = F.cross_entropy(logits.reshape(-1, logits.shape[-1]), refs.reshape(-1), ignore_index=-1,
                         reduction="none").view(T, -1)
    live = (refs >= 0).float()
    per_t = (ce * live).sum(dim=1) / live.sum(dim=1).clamp(min=1.0)
    used = (live.sum(dim=1) > 0).float()
    total = (per_t * used).sum()
    return total, total / used.sum().clamp(min=1.0)


class GraphedRollout(object):
    """trainers/imitation.py:18-77 for a whole VecCraft batch with the student in the loop, captured
    as ONE CUDA graph: per timestep one psk_craft_tick launch in "step, then observe" order (applies
    the previous actions with the trainer's timer / done / success rules, returns the features and the
    teacher's DAgger label of the new states) -> decode_step -> on-device sampling (Gumbel-max over
    pre-drawn noise; argmax when greedy).  Nothing crosses PCIe during a rollout; what the learner
    needs stays on the device:

        feats f32[T, N, F]   the states the student saw        refs i64[T, N]  teacher labels, -1 = done
        acts  u8[T, N]       what was executed, 255 = done     success bool[N], steps i64[] env-steps taken
    """

    def __init__(self, env, policy, max_timesteps=40, greedy=False, with_teacher=True, use_graph=True):
        from . import _lib
        self.env, self.policy, self.T = env, policy, _lib.check_max_timesteps(max_timesteps)
        self.greedy, self.with_teacher = greedy, with_teacher
        n, dev = env.n, env.device
        self.feats = torch.zeros((self.T, n, env.n_features), dtype=torch.float32, device=dev)
        self.refs = torch.full((self.T, n), -1, dtype=torch.long, device=dev)
        self.acts = torch.full((self.T, n), 255, dtype=torch.uint8, device=dev)
        self.noise = torch.zeros((self.T, n, policy.n_actions), dtype=torch.float32, device=dev)
        self.success = torch.zeros(n, dtype=torch.bool, device=dev)
        self.done = torch.zeros(n, dtype=torch.bool, device=dev)
        self.steps = torch.zeros((), dtype=torch.long, device=dev)
        self.interactions = torch.zeros((), dtype=torch.long, device=dev)
        self.zero_time = torch.zeros(n, dtype=torch.long, device=dev)    # students/imitation.py:58,75:
        self.out = {}                                                    # self.time is never advanced
        self.mem = None
        self.graph = None
        self.use_graph = use_graph

    def _body(self):
        env, pol, mem = self.env, self.policy, self.mem
        state = (mem["h0"], mem["c0"])
        self.done.zero_()
        self.success.zero_()
        self.steps.zero_()
        self.interactions.zero_()
        env.timer.fill_(self.T)                 # the kernel's timer is the trainer's (imitation.py:30,63)
        prev = None
        for t in range(self.T + 1):
            # ONE env launch per timestep: apply the previous actions (timer / done / success /
            # step inside the kernel), then the features and the teacher's label of the new states
            last = t == self.T
            out = env.tick(actions=prev, features_out=None if last else self.feats[t],
                           want_features=not last, out=self.out, advance_first=True)
            if prev is not None:
                ended = ~self.done & out["done"].bool()
                self.success |= ended & out["success"].bool()
                self.done |= ended
                self.steps += (~self.done).sum()
            if last:
                break
            logits, state = pol.decode_step(self.feats[t], self.zero_time, state, mem)
            if self.greedy:
                a = logits.argmax(dim=1)
            else:
                a = (logits - torch.log(-torch.log(self.noise[t]))).argmax(dim=1)   # Gumbel-max sample
            a8 = a.to(torch.uint8)
            live = ~self.done
            if self.with_teacher:
                self.refs[t] = torch.where(live, out["expert"].long(), torch.full_like(a, -1))
                self.interactions += live.sum()
            self.acts[t] = torch.where(live, a8, torch.full_like(a8, 255))
            prev = torch.where(live, a8, torch.full_like(a8, STOP))     # finished envs idle

    @torch.no_grad()
    def run(self, mem):
        """One rollout from the env's episode starts.  ``mem`` = policy.encode(...) of the envs' tasks."""
        env = self.env
        env.reset()
        if not self.greedy:
            self.noise.uniform_(1e-20, 1.0)
        if self.mem is None:
            self.mem = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in mem.items()}
        else:
            for k, v in mem.items():
                if torch.is_tensor(v):
                    self.mem[k].copy_(v)
        if not self.use_graph:
            self._body()
            return self
        if self.graph is None:
            self.graph = capture_graph(env, self._body)
        self.graph.replay()
        return self


def capture_graph(env, body):
    """``body`` captured as one CUDA graph.  A warm-up run first (allocations, cuDNN plans, and the
    first call with the env's tables outside the capture), then the capture on a side stream; leaves
    the envs at their episode starts."""
    body()
    env.reset()
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=env.device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            body()
    torch.cuda.current_stream().wait_stream(side)
    env.reset()
    return graph


class GraphedDecode(object):
    """psketch_b200.rollout.language_decode — one decoding pass of the language trainers
    (trainers/primitive_language.py:47-70, 93-113) from the envs' episode starts — as ONE CUDA graph:
    T + 1 step-then-observe ticks (``VecCraft.step_observe``: CraftState.step alone, every action of a
    running env executed, STOP a no-op, finished envs keep their state), the first without actions,
    and per timestep ``policy(features, t) -> actions [N]``, any capturable callable that reads only
    tensors whose addresses do not change between replays.  The bookkeeping of language_decode runs
    as device ops; nothing crosses PCIe inside a replay.

    ``run(key)`` returns what language_decode returns — actions u8[N, T] padded with 255, lengths
    i64[N], agents u8[L + 1, N, 32] (None unless ``record``), steps — plus ``features``, the frames
    the policy saw (f32[T, N, F]).  The pass always runs T timesteps and ``timesteps`` is
    lengths.max() (language_decode rounds up to its polling interval; timesteps where no env runs
    add nothing to the trainers' losses).  One graph is kept per ``key``: a policy whose static
    tensors change shape (instructions of another length) gives each shape its own key."""

    def __init__(self, env, policy, max_timesteps=40, record=True, use_graph=True):
        from . import _lib
        self.env, self.policy, self.T = env, policy, _lib.check_max_timesteps(max_timesteps)
        self.record, self.use_graph = record, use_graph
        n, dev = env.n, env.device
        self.feats = torch.zeros((self.T + 1, n, env.n_features), dtype=torch.float32, device=dev)
        self.acts = torch.full((n, self.T), 255, dtype=torch.uint8, device=dev)
        self.lengths = torch.zeros(n, dtype=torch.long, device=dev)
        self.agents = torch.zeros((self.T + 1, n, env.agent.shape[1]), dtype=torch.uint8, device=dev) if record else None
        self.done = torch.zeros(n, dtype=torch.bool, device=dev)
        self.steps = torch.zeros((), dtype=torch.long, device=dev)
        self.out = {}
        self.graphs = {}

    def _body(self):
        env, T = self.env, self.T
        self.done.zero_()
        self.lengths.zero_()
        self.steps.zero_()
        self.acts.fill_(255)
        if self.record:
            self.agents[0].copy_(env.agent)
        prev = None
        for t in range(T + 1):
            # ONE env launch per timestep: the previous actions (none at t = 0), then the features of
            # the new states (frame T, of the final states, is seen by nobody)
            env.step_observe(actions=prev, features_out=self.feats[t], out=self.out)
            if self.record and t > 0:
                self.agents[t].copy_(env.agent)
            if t == T:
                break
            a = self.policy(self.feats[t], t).to(torch.uint8)
            live = ~self.done
            self.acts[:, t] = torch.where(live, a, self.acts[:, t])
            prev = torch.where(live, a, torch.full_like(a, STOP))      # finished envs idle
            self.steps += live.sum()
            self.lengths += live
            self.done |= (a == STOP) | (t == T - 1)

    @torch.no_grad()
    def run(self, key=None):
        from . import _lib
        env = self.env
        env.reset()
        if not self.use_graph:
            self._body()
        else:
            if key not in self.graphs:
                self.graphs[key] = capture_graph(env, self._body)
            self.graphs[key].replay()
        # the pass does not use the teacher's labels that come with every tick: the teacher's assertion
        # (FLAG_BAD_LEAF, a state where the reference's teacher would raise) is not an error of the pass
        env.err_flags.bitwise_and_(~_lib.FLAG_BAD_LEAF)
        env.check_errors()
        L = int(self.lengths.max().item())
        return dict(actions=self.acts, lengths=self.lengths, agents=self.agents[:L + 1] if self.record else None,
                    steps=int(self.steps.item()), timesteps=L, features=self.feats[:self.T])
