#!/usr/bin/env python
"""BASELINE configs[3], second loop: configs/experiments/primitive_language.yaml at GPU batch sizes —
the reference's PrimitiveLanguageTrainer / PrimitiveLanguageStudent / PrimitiveLanguageTeacher
(trainers/primitive_language.py:16-143, students/primitive_language.py:97-196,
teachers/primitive_language.py:17-90) with the Craft env, the teacher's words and both student
models on the device.

    python examples/train_language.py --batch 1024 --iters 600 --eval-every 100

Per iteration, the reference's algorithm on a batch of training instances:
  instruct   the teacher's words for the instance's reference actions (``instruct_batch``)
  pass 1     the INSTRUCTED model (conditioned on those words) explores: sampled actions from the
             episode starts, every action executed, the agent records kept (``GraphedDecode``: the
             whole pass is one CUDA graph, one step-then-observe env launch per timestep)
  describe   the teacher names what the executed actions did (``describe_batch``: position /
             inventory deltas -> words, with its stateful student-action map and random fallback)
  receive    the instructed model, conditioned on the DESCRIPTIONS, re-scores the visited states;
             targets = the actions it took (hindsight relabelling, students/...:115-126)
  pass 2     the instructed model, greedy, follows the original instructions from the same starts
  imitate    the MAIN model (conditioned on the task only) re-scores pass 2's states; targets =
             pass 2's actions (:128-137);  loss = instructed + main, one AdamW step (:180-193)
Evaluation = the main model, greedy, on the whole dev split (2,200 instances, one batch).
The three decoding passes (pass 1, pass 2, evaluation) run as CUDA graphs (GraphedDecode);
tests/test_language_graph_gpu.py pins them to the eager psketch_b200.rollout.language_decode.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))

from train_dagger import Batches, load_split  # noqa: E402
from psketch_b200.students import GraphedDecode, Seq2SeqPolicy, task_tokens  # noqa: E402
from psketch_b200.tables import CraftTables  # noqa: E402
from psketch_b200.teachers.primitive_language import ACTION_WORDS, PrimitiveLanguageTeacher, instruct_batch  # noqa: E402
from psketch_b200.vec import VecCraft  # noqa: E402

T_MAX = 40


class DecodeStep(object):
    """``policy(features, t)`` for GraphedDecode: one decoder step of ``model`` at time index t (the
    language student advances time, students/primitive_language.py), reading only static tensors.
    ``load(mem)`` copies the encoder memory into the static tensors of its shape before a replay and
    draws the sampling noise; actions are Gumbel-max samples over that noise (exploring) or the
    argmax (greedy)."""

    def __init__(self, model, n, device, greedy):
        self.model, self.greedy = model, greedy
        self.time = torch.arange(T_MAX, device=device).unsqueeze(1).expand(T_MAX, n).contiguous()
        self.noise = torch.zeros((T_MAX, n, model.n_actions), dtype=torch.float32, device=device)
        self.static = {}            # encoder memories by shape (instruction length): one graph each
        self.mem = self.state = None

    def load(self, mem):
        """Returns the key of the graph that reads the static copy of ``mem``."""
        key = tuple(None if v is None else tuple(v.shape) for v in mem.values())
        if key not in self.static:
            self.static[key] = {k: None if v is None else v.clone() for k, v in mem.items()}
        else:
            for k, v in mem.items():
                if v is not None:
                    self.static[key][k].copy_(v)
        self.mem = self.static[key]
        if not self.greedy:
            self.noise.uniform_(1e-20, 1.0)
        return key

    def __call__(self, features, t):
        if t == 0:
            self.state = (self.mem["h0"], self.mem["c0"])
        logits, self.state = self.model.decode_step(features, self.time[t], self.state, self.mem)
        if self.greedy:
            return logits.argmax(dim=1)
        return (logits - torch.log(-torch.log(self.noise[t]))).argmax(dim=1)     # Gumbel-max sample


def decode(dec, mem):
    """One decoding pass of ``dec`` (a GraphedDecode over a DecodeStep) conditioned on ``mem``."""
    return dec.run(dec.policy.load(mem))


def sequence_loss(logits, actions):
    """students/primitive_language.py:171-178: per timestep the mean cross-entropy over the envs that
    were still running (target -1 = terminated), summed over the timesteps."""
    T = logits.shape[0]
    tgt = actions[:, :T].t().long()
    tgt = torch.where(tgt == 255, torch.full_like(tgt, -1), tgt)
    ce = F.cross_entropy(logits.reshape(-1, logits.shape[-1]), tgt.reshape(-1), ignore_index=-1,
                         reduction="none").view(T, -1)
    live = (tgt >= 0).float()
    return ((ce * live).sum(dim=1) / live.sum(dim=1).clamp(min=1.0)).sum()


def words_to_tokens(word_idx, vocab, device):
    """i64[N, L] indices into ACTION_WORDS (-1 = beyond the rollout) -> (tokens, padding mask)."""
    lut = torch.tensor([vocab[w] for w in ACTION_WORDS] + [vocab["<PAD>"]], device=device)
    return lut[word_idx.clamp(min=-1)], word_idx < 0         # index -1 = the <PAD> entry


def evaluate(main, tables, split, device, cache={}):
    key = id(split)
    if key not in cache:
        env = VecCraft.from_instances(tables, split["grids"], split["inst_env"], split["inst_pos"],
                                      split["inst_task"], max_timesteps=255, device=device)
        cache[key] = (env, GraphedDecode(env, DecodeStep(main, env.n, device, greedy=True), T_MAX, record=False))
    env, dec = cache[key]
    main.eval()
    with torch.no_grad():
        decode(dec, main.encode(task_tokens(tables, env.task, reverse=False)))
    main.train()
    return float((env.satisfies() == 1).float().mean())


def train(args):
    device = torch.device("cuda:0")
    torch.manual_seed(args.seed)
    tables = CraftTables()
    vocab = tables.task_manager.vocab
    train_split, dev_split = load_split("train"), load_split("dev")
    data = Batches(tables, train_split, args.batch, device, args.seed)
    d_ref = torch.from_numpy(train_split["ref_actions"]).to(device)
    n_vocab, pad = len(vocab) + 1, vocab["<PAD>"]
    instructed = Seq2SeqPolicy(404, 6, n_vocab, pad, hidden=args.hidden).to(device)
    main = Seq2SeqPolicy(404, 6, n_vocab, pad, hidden=args.hidden).to(device)
    opt = torch.optim.AdamW(list(instructed.parameters()) + list(main.parameters()), lr=args.lr)
    teacher = PrimitiveLanguageTeacher()
    teacher.random = np.random.RandomState(args.seed)
    explore = GraphedDecode(data.env, DecodeStep(instructed, args.batch, device, greedy=False), T_MAX, record=True)
    follow = GraphedDecode(data.env, DecodeStep(instructed, args.batch, device, greedy=True), T_MAX, record=False)
    log, t0 = [], time.time()
    env_steps = episodes = 0
    for it in range(args.iters):
        env, tasks = data.next()
        rows = data.rows
        ref = d_ref[rows]
        L_ref = int((ref != 255).sum(dim=1).max())
        ref = ref[:, :max(L_ref, 1)]
        instr_tok = instruct_batch(ref, vocab=vocab)
        instr_tok = torch.where(ref == 255, torch.full_like(instr_tok, pad), instr_tok)
        instr_mask = ref == 255
        # pass 1: exploring, instructed
        instructed.train()
        with torch.no_grad():
            first = decode(explore, instructed.encode(instr_tok, instr_mask))
        T1 = first["timesteps"]
        L1 = int(first["lengths"].max())
        desc = teacher.describe_batch(first["actions"][:, :L1].long(), first["agents"][:L1 + 1], first["lengths"],
                                      n_kinds=env.K)
        # receive: the descriptions condition the instructed model on what it actually did
        desc_tok, desc_mask = words_to_tokens(desc, vocab, device)
        mem = instructed.encode(desc_tok, desc_mask)
        logits = instructed.decode_sequence(first["features"][:T1], explore.policy.time[:T1], mem)
        instructed_loss = sequence_loss(logits, first["actions"])
        # pass 2: greedy, original instructions, same starts
        instructed.eval()
        with torch.no_grad():
            second = decode(follow, instructed.encode(instr_tok, instr_mask))
        instructed.train()
        T2 = second["timesteps"]
        success = env.satisfies() == 1
        # imitate: the task-conditioned model learns pass 2's behaviour
        mem = main.encode(task_tokens(tables, tasks, reverse=False))
        logits = main.decode_sequence(second["features"][:T2], follow.policy.time[:T2], mem)
        main_loss = sequence_loss(logits, second["actions"])
        loss = instructed_loss + main_loss
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        env_steps += first["steps"] + second["steps"]
        episodes += 2 * args.batch
        rec = dict(iter=it + 1)
        if (it + 1) % args.log_every == 0 or (it + 1) % args.eval_every == 0 or it == args.iters - 1:
            follows = float(((second["actions"][:, :ref.shape[1]] == ref) | (ref == 255)).all(dim=1).float().mean())
            rec.update(instructed_loss=float(instructed_loss.detach()) / T1, main_loss=float(main_loss.detach()) / T2,
                       instructed_success=float(success.float().mean()), follows_reference=follows,
                       words_known=len(teacher.student_action_map))
        if (it + 1) % args.eval_every == 0 or it == args.iters - 1:
            rec["dev_success"] = evaluate(main, tables, dev_split, device)
        if len(rec) > 1:
            log.append(rec)
            print("iter %5d  instructed loss %.4f  main loss %.4f  instructed success %.3f (follows the reference "
                  "actions %.3f)%s  | %.2e env-steps/s overall"
                  % (it + 1, rec["instructed_loss"], rec["main_loss"], rec["instructed_success"],
                     rec["follows_reference"],
                     "  dev success (main model) %.3f" % rec["dev_success"] if "dev_success" in rec else "",
                     env_steps / (time.time() - t0)), flush=True)
    env.check_errors()
    summary = dict(batch=args.batch, iters=args.iters, episodes=episodes, env_steps=env_steps,
                   wall_s=time.time() - t0, env_steps_per_s=env_steps / (time.time() - t0),
                   final=log[-1], best_dev=max((r.get("dev_success", 0.0) for r in log), default=0.0),
                   teacher_action_map={int(k): v for k, v in teacher.student_action_map.items()})
    return log, (instructed, main), summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=600)
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--seed", type=int, default=123)
    ap.add_argument("--log-every", type=int, default=25)
    ap.add_argument("--eval-every", type=int, default=100)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    log, _, summary = train(args)
    print(json.dumps(summary))
    if args.json:
        json.dump(dict(summary=summary, log=log), open(args.json, "w"))


if __name__ == "__main__":
    main()
