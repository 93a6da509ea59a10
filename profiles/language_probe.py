#!/usr/bin/env python
"""Where the time of the primitive-language loop (examples/train_language.py) goes, with the decoding
passes eager (psketch_b200.rollout.language_decode: a feature launch, the decoder step, sampling, a step
launch and the mask ops per timestep, a host poll every 8) and graphed (psketch_b200.students.
GraphedDecode: one CUDA graph per pass, one step-then-observe launch per timestep).

On the train split at batch 128, 1,024 and 8,192 with Seq2SeqPolicy at hidden 256:
  decode     one greedy 40-step pass (STOP masked, so that no env ends early), eager against graphed
  iteration  one whole training iteration, split into decoding passes / describe_batch / learning
Both forms run in the same process, interleaved, after a warm-up; every number is a mean over CUDA-event
windows of at least --window seconds.  One JSON line with the GPU's name and power limit.

    python profiles/language_probe.py --out profiles/bench_runs/r3_language_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))

from train_dagger import Batches, load_split  # noqa: E402
from train_language import T_MAX, DecodeStep, decode, sequence_loss, words_to_tokens  # noqa: E402
from psketch_b200.rollout import language_decode  # noqa: E402
from psketch_b200.students import GraphedDecode, Seq2SeqPolicy, task_tokens  # noqa: E402
from psketch_b200.tables import STOP, CraftTables  # noqa: E402
from psketch_b200.teachers.primitive_language import PrimitiveLanguageTeacher, instruct_batch  # noqa: E402


class EagerStep(object):
    """The eager form of train_language's decoding policy (the example's loop before GraphedDecode):
    decoder step, softmax + multinomial or argmax, the frames kept for learning."""

    def __init__(self, model, n, device, greedy):
        self.model, self.greedy = model, greedy
        self.feats = torch.empty((T_MAX, n, 404), dtype=torch.float32, device=device)
        self.time = torch.arange(T_MAX, device=device).unsqueeze(1).expand(T_MAX, n).contiguous()

    def start(self, mem):
        self.mem, self.state = mem, (mem["h0"], mem["c0"])

    def __call__(self, features, t):
        self.feats[t].copy_(features)
        with torch.no_grad():
            logits, self.state = self.model.decode_step(features, self.time[t], self.state, self.mem)
        if self.greedy:
            return logits.argmax(dim=1)
        return torch.multinomial(torch.softmax(logits, dim=1), 1).squeeze(1)


class NoStop(object):
    """``model`` with its STOP logit masked, for the decode timing: every env runs all 40 steps in both
    forms (language_decode stops polling once every env is done, an untrained model stops early)."""

    def __init__(self, model):
        self.model, self.n_actions = model, model.n_actions

    def decode_step(self, *args):
        logits, state = self.model.decode_step(*args)
        logits[:, STOP] = float("-inf")
        return logits, state


class Loop(object):
    """train_language's models, optimiser, teacher and data at one batch size, with both decoders."""

    def __init__(self, batch, device, seed=123):
        torch.manual_seed(seed)
        self.tables = CraftTables()
        self.vocab = self.tables.task_manager.vocab
        split = load_split("train")
        self.data = Batches(self.tables, split, batch, device, seed)
        self.d_ref = torch.from_numpy(split["ref_actions"]).to(device)
        nv, self.pad = len(self.vocab) + 1, self.vocab["<PAD>"]
        self.instructed = Seq2SeqPolicy(404, 6, nv, self.pad, hidden=256).to(device)
        self.main = Seq2SeqPolicy(404, 6, nv, self.pad, hidden=256).to(device)
        self.opt = torch.optim.AdamW(list(self.instructed.parameters()) + list(self.main.parameters()), lr=1e-3)
        self.teacher = PrimitiveLanguageTeacher()
        self.teacher.random = np.random.RandomState(seed)
        env = self.data.env
        self.g_explore = GraphedDecode(env, DecodeStep(self.instructed, batch, device, greedy=False), T_MAX)
        self.g_follow = GraphedDecode(env, DecodeStep(self.instructed, batch, device, greedy=True), T_MAX,
                                      record=False)
        self.e_explore = EagerStep(self.instructed, batch, device, greedy=False)
        self.e_follow = EagerStep(self.instructed, batch, device, greedy=True)
        self.device = device

    def capture_all(self):
        """Captures both passes' graphs for every instruction length of the split (one graph each) —
        what a training run does once per length — so that no capture falls into a timed window."""
        n = self.data.batch
        for L in range(1, int((self.d_ref != 255).sum(dim=1).max()) + 1):
            tok = torch.full((n, L), self.pad, dtype=torch.long, device=self.device)
            with torch.no_grad():
                mem = self.instructed.encode(tok, torch.zeros((n, L), dtype=torch.bool, device=self.device))
            decode(self.g_explore, mem)
            decode(self.g_follow, mem)

    def _pass(self, graphed, explore, mem):
        """(result, feature frames, time indices) of one decoding pass."""
        if graphed:
            dec = self.g_explore if explore else self.g_follow
            out = decode(dec, mem)
            return out, out["features"], dec.policy.time
        rec = self.e_explore if explore else self.e_follow
        rec.start(mem)
        out = language_decode(self.data.env, rec, T_MAX, record=explore)
        return out, rec.feats, rec.time

    def iteration(self, graphed, ev):
        """One train_language iteration; ev = 5 CUDA events: start, pass 1 done, describe done, pass 2
        done, learning done (pass 2 and the learning on pass 1 are timed apart)."""
        env, tasks = self.data.next()
        ref = self.d_ref[self.data.rows]
        ref = ref[:, :max(int((ref != 255).sum(dim=1).max()), 1)]
        instr_tok = instruct_batch(ref, vocab=self.vocab)
        instr_tok = torch.where(ref == 255, torch.full_like(instr_tok, self.pad), instr_tok)
        instr_mask = ref == 255
        ev[0].record()
        with torch.no_grad():
            first, f1, time1 = self._pass(graphed, True, self.instructed.encode(instr_tok, instr_mask))
        T1 = first["timesteps"]
        L1 = int(first["lengths"].max())
        ev[1].record()
        desc = self.teacher.describe_batch(first["actions"][:, :L1].long(), first["agents"][:L1 + 1],
                                           first["lengths"], n_kinds=env.K)
        desc_tok, desc_mask = words_to_tokens(desc, self.vocab, self.device)
        ev[2].record()
        with torch.no_grad():
            second, f2, time2 = self._pass(graphed, False, self.instructed.encode(instr_tok, instr_mask))
        T2 = second["timesteps"]
        ev[3].record()
        mem = self.instructed.encode(desc_tok, desc_mask)
        loss = sequence_loss(self.instructed.decode_sequence(f1[:T1], time1[:T1], mem), first["actions"])
        mem = self.main.encode(task_tokens(self.tables, tasks, reverse=False))
        loss = loss + sequence_loss(self.main.decode_sequence(f2[:T2], time2[:T2], mem), second["actions"])
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.opt.step()
        ev[4].record()


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "nvidia-smi failed: %s" % e
    return info


def windowed(fn, window_s):
    """Mean ms per call of fn over CUDA-event windows, calls repeated until window_s has passed."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, t0 = 0, time.time()
    s.record()
    while True:
        fn()
        calls += 1
        if time.time() - t0 >= window_s:
            break
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / calls, calls


def probe(batch, window_s, rounds):
    dev = torch.device("cuda:0")
    lp = Loop(batch, dev)
    env = lp.data.env
    lp.data.next()
    with torch.no_grad():
        mem = lp.main.encode(task_tokens(lp.tables, env.task, reverse=False))
    g_dec = GraphedDecode(env, DecodeStep(NoStop(lp.main), batch, dev, greedy=True), T_MAX, record=False)
    e_rec = EagerStep(NoStop(lp.main), batch, dev, greedy=True)
    lp.capture_all()

    def eager_pass():
        with torch.no_grad():
            e_rec.start(mem)
            language_decode(env, e_rec, T_MAX, record=False)

    def graph_pass():
        with torch.no_grad():
            decode(g_dec, mem)
    for _ in range(3):                                  # warm-up: captures, cuDNN plans, allocations
        eager_pass()
        graph_pass()
    for graphed in (False, True, False, True):
        for _ in range(3):
            lp.iteration(graphed, [torch.cuda.Event(enable_timing=True) for _ in range(5)])
    torch.cuda.synchronize()
    out = dict(batch=batch, decode_ms=dict(eager=[], graphed=[]), iteration_ms=dict(eager=[], graphed=[]))
    for _ in range(rounds):
        for name, fn in (("eager", eager_pass), ("graphed", graph_pass)):
            ms, calls = windowed(fn, window_s)
            out["decode_ms"][name].append(ms)
        for graphed in (False, True):
            evs, t0 = [], time.time()
            while time.time() - t0 < window_s:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
                lp.iteration(graphed, ev)
                evs.append(ev)
            torch.cuda.synchronize()
            parts = np.array([[ev[0].elapsed_time(ev[1]) + ev[2].elapsed_time(ev[3]), ev[1].elapsed_time(ev[2]),
                               ev[3].elapsed_time(ev[4]), ev[0].elapsed_time(ev[4])] for ev in evs])
            m = parts.mean(axis=0)
            out["iteration_ms"]["graphed" if graphed else "eager"].append(
                dict(decode_passes=m[0], describe_batch=m[1], learning=m[2], total=m[3], iterations=len(evs)))
    summ = lambda xs: float(np.median(xs))
    out["decode_ms_median"] = {k: summ(v) for k, v in out["decode_ms"].items()}
    out["decode_speedup"] = out["decode_ms_median"]["eager"] / out["decode_ms_median"]["graphed"]
    out["iteration_ms_median"] = {k: {p: summ([r[p] for r in v]) for p in ("decode_passes", "describe_batch",
                                                                        "learning", "total")}
                                  for k, v in out["iteration_ms"].items()}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="128,1024,8192")
    ap.add_argument("--window", type=float, default=0.5, help="seconds per timing window (at least 0.5)")
    ap.add_argument("--rounds", type=int, default=3, help="interleaved eager / graphed rounds")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("language_probe.py measures the GPU: no CUDA device")
    assert args.window >= 0.5
    rec = dict(probe="language_probe", **gpu_info(), window_s=args.window, rounds=args.rounds,
               rows=[probe(int(b), args.window, args.rounds) for b in args.batches.split(",")])
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
