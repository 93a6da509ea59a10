#!/usr/bin/env python
"""bench.py — env-steps/s of the Craft hot path (teacher action + features + step) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one rollout tick of the whole batch: for every env the BFS teacher's action, the
f32[404] feature vector and the state transition (with done / success / auto-reset), i.e. the body
of trainers/imitation.py:42-73.  Workload at N=1: BASELINE.json configs[1] — craft_medium train
tasks (17,600 instances, regenerated with the reference's make_data.py, committed as
tests/golden/craft_medium_splits.npz) tiled to 65,536 envs; weak scaling for N>1 (same envs per
GPU, no data-path collective; one NCCL all-reduce of the episode statistics after the timed
region).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/s (step+features+expert)"
UNIT = "env-steps/s"
# algorithmic bytes per env-step at craft_medium (SURVEY.md §8(d), DESIGN.md §"Rooflines")
BYTES_FUSED = 1815
BYTES_STEP, BYTES_FEATURES, BYTES_EXPERT = 198, 1712, 97
DUMP_BYTES = 60 * 10**6          # --dump-outputs: all arrays together, with room for the .npy headers


def load_workload(n_envs, split="train"):
    sp = np.load(os.path.join(ROOT, "tests", "golden", "craft_medium_splits.npz"))
    n_inst = len(sp[split + "_inst_env"])
    idx = np.arange(n_envs) % n_inst
    return dict(grids=sp[split + "_grids"], env=sp[split + "_inst_env"][idx],
                pos=sp[split + "_inst_pos"][idx], task=sp[split + "_inst_task"][idx],
                n_instances=n_inst, raw=sp)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = [r for r in self.rows if t0 - 0.05 <= r[0] <= t1 + 0.15] or self.rows
        for _, line in rows:
            p = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU baselines
def cpu_python_port(budget_s=20.0, procs=None, rounds=1, warm=0):
    """The reference's Python loop, restated (oracle/craft_ref_port.py), one process per core on a
    bounded sample of dev-split instances (BASELINE config 1).  Returns one dict per round."""
    from oracle import craft_ref_port as port
    procs = procs or os.cpu_count() or 1
    sp = load_workload(1, "dev")["raw"]
    # ~4.8k env-steps/s/core and ~10 env-steps per instance
    n_inst = int(min(2200 * 32, max(procs * 20, budget_s * 450 * procs)))     # ~5 k env-steps/s/core, ~10 per instance
    idx = np.arange(n_inst) % 2200
    runner = port.ParallelRunner("craft_medium", sp["dev_grids"], procs)
    out = []
    try:
        for r in range(warm + rounds):
            steps, secs = runner.run(sp["dev_inst_env"][idx], sp["dev_inst_pos"][idx],
                                     sp["dev_inst_task"][idx], n_inst)
            if r >= warm:
                out.append({"value": steps / secs, "unit": UNIT, "cores": procs, "kind": "port",
                            "sample": "%d dev-split instances (%d env-steps) through "
                                      "oracle/craft_ref_port.py (pure-Python port of the reference "
                                      "loop), %d processes, %.2f s" % (n_inst, steps, procs, secs),
                            "seconds": secs})
    finally:
        runner.close()
    return out


def cpu_native_oracle(n_envs=65536, ticks=20):
    """The C restatement (oracle/craft_oracle.c) with OpenMP on all cores — a much stronger CPU
    baseline than the reference's Python, reported for context."""
    from psketch_b200.tables import CraftTables
    from oracle.craft_oracle import CraftOracle
    tables = CraftTables()
    o = CraftOracle(tables)
    o.set_threads(os.cpu_count() or 1)
    w = load_workload(n_envs)
    init_grid = w["grids"][w["env"].astype(np.int64)]
    state, _, _, _ = o.rollout(1, 40, init_grid, w["pos"].astype(np.int32), w["task"].astype(np.int32))
    t0 = time.perf_counter()
    state, stats, _, _ = o.rollout(ticks, 40, init_grid, w["pos"].astype(np.int32),
                                   w["task"].astype(np.int32), state=state)
    dt = time.perf_counter() - t0
    return {"value": int(stats[2]) / dt, "unit": UNIT, "cores": os.cpu_count(), "kind": "port-c",
            "sample": "%d envs x %d ticks through oracle/craft_oracle.c (OpenMP), %.2f s" % (n_envs, ticks, dt)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = cpu_python_port(budget_s=max(0.25, 60.0 / max(1, args.steps + args.warmup)),
                               rounds=args.steps, warm=args.warmup)
    base = per_step[-1]
    value = float(np.mean([b["value"] for b in per_step]))
    ms = float(np.mean([b["seconds"] for b in per_step])) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "craft_medium dev-split instances, teacher+features+step per env "
                               "in a Python loop (pure-Python port of the reference, one process per core)"},
        "cpu_baseline": dict(base, value=value),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def time_kernel(fn, torch, inner=10, reps=20):
    """Average device time of one launch: `inner` launches captured in a CUDA graph (so that the
    Python/ctypes launch cost is not what is measured), replayed `reps` times between events."""
    fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(inner):
                fn()
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        g.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e-3 / (reps * inner)


# Port-vs-reference calibration of the CPU arm, measured in the build container (the unmodified
# reference cannot travel to the GPU box): same 660 dev instances, one core, unmodified reference
# 5,117 env-steps/s vs oracle/craft_ref_port.py 6,993 — the port is 1.37x FASTER, so every ratio
# against the port understates the ratio against the reference by that factor.
PORT_VS_REFERENCE = {"factor": 1.37, "reference_env_steps_per_s_per_core": 5117,
                     "port_env_steps_per_s_per_core": 6993,
                     "how": "build container, one core, 660 dev instances, unmodified /root/reference "
                            "(oracle/ref_shim.py) vs oracle/craft_ref_port.py; VERDICT r1 item 10"}


def oracle_parity_sample(env, tables, wl_arrays, snap, out, feat_ring, ticks, first_slot, sample):
    """Bit-exact check of one launch against the CPU oracle on a strided sample of envs: the oracle
    starts from the sampled envs' state before the launch (``snap``) and is advanced tick by tick;
    teacher action of every tick, every feature frame still in the ring, and the final state."""
    import torch
    from oracle.craft_oracle import CraftOracle
    o = CraftOracle(tables)
    grids, ienv, ipos, itask = wl_arrays
    ds = torch.from_numpy(sample).to(env.device)
    g0, a0 = snap[0][ds].cpu().numpy(), snap[1][ds].cpu().numpy()
    C, K = env.C, env.K
    state = dict(grid=np.ascontiguousarray(g0[:, :C]), inv=a0[:, :K].astype(np.int32),
                 pos=a0[:, 24:26].astype(np.int32), dir=a0[:, 26].astype(np.int32),
                 timer=a0[:, 28].astype(np.int32))
    init_grid = np.ascontiguousarray(grids[ienv[sample].astype(np.int64)])
    init_pos, task = ipos[sample].astype(np.int32), itask[sample].astype(np.int32)
    ring = feat_ring.shape[0]
    frames = 0
    for t in range(ticks):
        state, _, f, a = o.rollout(1, env.max_timesteps, init_grid, init_pos, task, state=state,
                                   want_features=True)
        got = out["expert"][t][ds].cpu().numpy().astype(np.int32)
        if not np.array_equal(got, a):
            raise AssertionError("parity: teacher action differs from the oracle at tick %d" % t)
        if t >= ticks - ring:                       # frame not overwritten later in the launch
            if not np.array_equal(feat_ring[(first_slot + t) % ring][ds].cpu().numpy(), f):
                raise AssertionError("parity: features differ from the oracle at tick %d" % t)
            frames += 1
    fin = env.agent[ds].cpu().numpy()
    ok = (np.array_equal(env.cells[ds].cpu().numpy(), state["grid"]) and
          np.array_equal(fin[:, :K].astype(np.int32), state["inv"]) and
          np.array_equal(fin[:, 24:26].astype(np.int32), state["pos"]) and
          np.array_equal(fin[:, 26].astype(np.int32), state["dir"]) and
          np.array_equal(fin[:, 28].astype(np.int32), state["timer"]))
    if not ok:
        raise AssertionError("parity: final state differs from the oracle")
    return {"sample_envs": int(len(sample)), "ticks": int(ticks), "feature_frames": frames,
            "against": "oracle/craft_oracle.c, advanced tick by tick from the pre-launch state"}


def last_step_outputs(torch, features, out, row, n):
    """What one step hands its caller — the f32 feature frame, the teacher's actions and the done /
    success flags — as float arrays on the device.  Larger batches are cut to a fixed, seeded sample of
    envs (``env_index``) so that all arrays together stay under DUMP_BYTES."""
    per_env = 4 * features.shape[-1] + 4 * 3 + 8
    m = min(n, DUMP_BYTES // per_env)
    envs = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    idx = torch.from_numpy(envs).to(features.device)
    res = {"env_index": torch.from_numpy(envs.astype(np.float64)), "features": features[idx]}
    for k in ("expert", "done", "success"):
        res[k] = (out[k] if row is None else out[k][row])[idx].float()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from psketch_b200 import dist as pdist
    from psketch_b200.tables import CraftTables
    from psketch_b200.vec import VecCraft

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    rank, world, local = pdist.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    distributed = world > 1

    n = args.envs_per_gpu
    K, W = args.steps, args.warmup
    tables = CraftTables()
    wl = load_workload(n)
    # each rank owns its own slice of the batch: rotate the instance tiling by rank
    shift = (rank * n) % wl["n_instances"]
    wl_arrays = (wl["grids"], np.roll(wl["env"], -shift), np.roll(wl["pos"], -shift, axis=0),
                 np.roll(wl["task"], -shift))
    env = VecCraft.from_instances(tables, *wl_arrays, max_timesteps=40, device=dev)
    nf = env.n_features
    feat_bytes = n * nf * 4
    fused = not args.unfused
    rand_act = torch.empty(n, dtype=torch.uint8, device=dev) if args.policy == "random" else None
    # Teacher-driven rollouts need nothing from outside the kernel, so T ticks run per launch
    # (psk_craft_rollout: state stays in shared memory between ticks).  T = 1, the random policy
    # and --unfused use one psk_craft_tick launch per step.
    T = max(1, args.ticks_per_launch) if fused else 1
    rand_block = (torch.empty((T, n), dtype=torch.uint8, device=dev)
                  if (rand_act is not None and T > 1) else None)
    # Ring of output frames: larger than L2 (126 MB), and at least T + 1 frames so that no frame is
    # written twice within one launch — a CTA that came back to the same lines a few ticks later
    # would find them still dirty in L2, the writes would merge there and never reach HBM, and the
    # "bandwidth" would exceed what HBM can do (seen: 8.3 TB/s with a ring of 2 at 1 M envs).
    ring = max(2, int(np.ceil(1.5 * 126e6 / feat_bytes)) + 1, T + 1 if T > 1 else 0)
    ring = min(ring, 64)
    feat_ring = torch.empty((ring, n, nf), dtype=torch.float32, device=dev)
    feats = [feat_ring[i] for i in range(ring)]
    outs = [dict() for _ in range(ring)]

    def tick(i):
        if rand_act is not None:        # off-policy variant: U{0..5} actions from Philox(123, (env, t))
            env.random_actions(0, seed=123, out=rand_act, device_clock=True)
        env.tick(actions=rand_act, features_out=feats[i % ring], fused=fused, out=outs[i % ring])

    routs = {}

    def launch_rollout(ticks=None):
        # tick t of a launch writes ring slot t % ring: nothing is written twice within a launch,
        # and between two launches' writes to the same line >= 850 MB pass through the 126 MB L2
        ticks = ticks or T
        acts = None
        if rand_block is not None:      # off-policy: one Philox launch fills the action block of the rollout
            acts = rand_block[:ticks]
            env.random_actions(0, seed=123, out=acts, device_clock=True, ticks=ticks)
        env.rollout(ticks, actions=acts, features_out=feat_ring, out=routs.setdefault(ticks, {}), want_flags=True)

    for i in range(ring):           # allocate output tensors outside the graph
        tick(i)
    if T > 1:
        launch_rollout()
    torch.cuda.synchronize()
    per_tick_launches = (1 if fused else 3) + (1 if rand_act is not None else 0)
    launches = [0]
    graphs = {}

    def plan_for(r):
        return ([T] * (r // T) + ([r % T] if r % T else [])) if T > 1 else list(range(r))

    def capture(plan):
        """CUDA graph of a list of launches; plan entries are tick counts (T > 1) or tick indices."""
        for tc in set(plan) if T > 1 else ():
            launch_rollout(tc)                      # output tensors exist before the capture
        torch.cuda.synchronize()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for j, tc in enumerate(plan):
                    if T > 1:
                        launch_rollout(tc)
                    else:
                        tick(j)
        torch.cuda.current_stream().wait_stream(side)
        return g

    # A request of k ticks = (k // chunk) replays of the main graph (4 full launches, or one ring
    # of single ticks) + one tail graph with the exact remainder.
    chunk = (ring if T == 1 else 4) * T

    def prepare(k):
        if args.no_graph:
            return
        if k >= chunk and "main" not in graphs:
            graphs["main"] = capture(plan_for(chunk))
        r = k % chunk
        if r and r not in graphs:
            graphs[r] = capture(plan_for(r))

    def n_launches(plan):
        return len(plan) * ((2 if rand_block is not None else 1) if T > 1 else per_tick_launches)

    ticks_done = [0]

    def run_steps(k):
        """Exactly k ticks."""
        ticks_done[0] += k
        if args.no_graph:
            done = 0
            while T > 1 and k - done >= T:
                launch_rollout()
                done += T
                launches[0] += 2 if rand_block is not None else 1
            while done < k:
                if T > 1:
                    launch_rollout(k - done)
                    launches[0] += 2 if rand_block is not None else 1
                    done = k
                else:
                    tick(done)
                    done += 1
                    launches[0] += per_tick_launches
            return
        prepare(k)
        for _ in range(k // chunk):
            graphs["main"].replay()
            launches[0] += n_launches(plan_for(chunk))
        if k % chunk:
            graphs[k % chunk].replay()
            launches[0] += n_launches(plan_for(k % chunk))

    graph = None if args.no_graph else True
    prepare(max(W, 3))
    prepare(K)
    prepare(ring * 8)

    sampler = ClockSampler(local) if rank == 0 else None
    run_steps(K)                                    # one untimed pass of the K-step plan: graph upload
    # where the last of K steps leaves its outputs: the plan's last launch runs K % T (or T) ticks and
    # writes the frame of tick t to ring slot t; one tick per launch: step j writes slot j % ring
    tl = K % T or T
    last_step = ((feat_ring[tl - 1], routs[tl], tl - 1) if T > 1 else
                 (feats[(K - 1) % ring], outs[(K - 1) % ring], None))
    env.stats.zero_()
    ticks_before = ticks_done[0]
    phase0 = (40 - env.timer.to(torch.int64)).cpu().numpy()      # ticks into the running episode, per env
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    # the warm-up is still running when the first event is queued, so the timed region starts with
    # the K-step plan already submitted instead of measuring its submission
    run_steps(max(W, 3))
    launches[0] = 0
    m0.record()
    run_steps(K)                                    # the timed region: exactly K steps
    m1.record()
    timed_launches = launches[0]
    torch.cuda.synchronize()
    t1 = time.time()
    if distributed:
        dist.barrier()
    # what the last timed step returned, sampled before anything else runs on the envs
    dumped = last_step_outputs(torch, *last_step, n) if args.dump_outputs and rank == 0 else None
    total = torch.tensor([m0.elapsed_time(m1) * 1e-3], dtype=torch.float64, device=dev)
    stats = env.stats.clone()
    # Size-independent invariant over the WHOLE timed region (every launch, chained or not): teacher-
    # driven episodes of instance i last exactly ref_len[i] ticks and always succeed, so the number of
    # episodes that end inside the region is known in closed form; one env whose state was corrupted
    # anywhere would break the count.
    episodes_ok = None
    if rand_act is None:
        ref_len = np.roll(wl["raw"]["train_ref_len"][np.arange(n) % wl["n_instances"]], -shift).astype(np.int64)
        expected = int(((phase0 + (ticks_done[0] - ticks_before)) // ref_len).sum())
        local = stats.cpu().numpy()
        episodes_ok = bool(int(local[0]) == expected and int(local[1]) == expected)
        assert episodes_ok, "episodes %d / successes %d, expected %d" % (local[0], local[1], expected)
    counted_steps = n * world * (ticks_done[0] - ticks_before)
    if distributed:
        dist.all_reduce(total, op=dist.ReduceOp.MAX)
    ar0, ar1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar0.record()
    pdist.allreduce_stats(stats)                            # the path's only collective (NCCL)
    ar1.record()
    torch.cuda.synchronize()
    stats_allreduce_us = ar0.elapsed_time(ar1) * 1e3
    elapsed = float(total.item())                           # seconds for the K timed steps, MAX over ranks
    clocks = None
    if sampler:
        t1c, window = t1, "timed region"
        if t1 - t0 < 0.6:
            # nvidia-smi cannot sample faster than ~20 ms: keep the same step running (untimed)
            # so that the clocks are read under the same load
            tc = time.time()
            while time.time() - tc < 0.8:
                run_steps(ring * 8)
                torch.cuda.synchronize()
            t1c, window = time.time(), "timed region + 0.8 s untimed continuation of the same step"
        clocks = sampler.stop(t0, t1c)
        clocks["window"] = window
    env.check_errors()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a.cpu().numpy())
    total_steps = n * K * world
    value = total_steps / elapsed
    st = stats.cpu().numpy()
    assert int(st[2]) == counted_steps, "kernel step counter disagrees with the host's"

    # ---- parity of the timed kernel: one more replay of the SAME K-step plan, the last launch of
    # it checked against the CPU oracle on a strided sample (untimed)
    parity = None
    if not args.no_parity and T > 1 and rand_act is None:
        torch.cuda.synchronize()
        plan = plan_for(K)
        if len(plan) > 1:
            run_steps(K - plan[-1])                 # everything but the last launch
        snap = env.snapshot()
        torch.cuda.synchronize()
        launch_rollout(plan[-1])                    # same entry point, arguments and dispatch as the graph node
        torch.cuda.synchronize()
        sample = np.unique(np.concatenate([np.arange(0, n, max(1, n // 2048)), np.arange(max(0, n - 64), n)]))
        parity = oracle_parity_sample(env, tables, wl_arrays, snap, routs[plan[-1]], feat_ring,
                                      plan[-1], 0, sample)
        parity["launch"] = "psk_craft_rollout(ticks=%d) on %d envs, same dispatch as the timed launches" % (plan[-1], n)
        env.check_errors()

    # ---- yardstick for a kernel that only writes: the same ring filled by a plain store kernel (the
    # roofline denominator is a COPY bandwidth, half reads; a store-only stream runs faster than that)
    write_ceiling = None
    if rank == 0:
        try:
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            feat_ring.fill_(0.0)
            torch.cuda.synchronize()
            w0.record()
            for _ in range(5):
                feat_ring.fill_(0.0)
            w1.record()
            torch.cuda.synchronize()
            gbs = 5 * feat_ring.numel() * feat_ring.element_size() / (w0.elapsed_time(w1) * 1e-3) / 1e9
            write_ceiling = {"GBps": gbs, "how": "torch fill_ of the %.0f MB feature ring, 5 passes between CUDA "
                                                 "events, after the timed region" % (feat_ring.numel() * feat_ring.element_size() / 1e6)}
        except Exception as ex:  # noqa: BLE001
            write_ceiling = {"error": repr(ex)}

    # ---- end to end through the public API with host buffers (rank-local, then aggregated)
    e2e = measure_e2e(torch, dist if distributed else None, tables, wl, n, dev, args, world)

    # ---- BASELINE config 3 (8 M envs over the ranks): world > 1 only
    config3 = None
    if distributed and not args.no_config3:
        config3 = measure_config3(torch, dist, pdist, tables, rank, world, dev, args)

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    per_tick_s = elapsed / K             # seconds per tick (= per step)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "timed_region_ms": elapsed * 1e3,
        "ms_per_step": per_tick_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {
            "workload": "craft_medium train tasks (17,600 instances tiled), %d parallel envs per GPU, "
                        "teacher BFS + f32[404] features + step/auto-reset per tick" % n,
            "envs_per_gpu": n, "max_timesteps": 40, "policy": args.policy, "ticks_per_launch": T,
            "kernel": ("craft_rollout_kernel (fused tick, %d ticks per launch)" % T if T > 1 else
                       "craft_tick_kernel (fused, warp-specialised)") if fused else "expert+features+advance",
            "cuda_graph": graph is not None,
            "timing": "one untimed replay of the K-step plan, then the warm-up and the K timed steps "
                      "queued back to back, CUDA events around the K steps; value = envs x K / their time, "
                      "MAX over ranks",
            "l2": "feature outputs rotate through a ring of %d frames (%.0f MB > 126 MB L2); tick t of a "
                  "launch writes slot t %% ring, so a line is rewritten only after >= 850 MB of other "
                  "writes" % (ring, ring * feat_bytes / 1e6),
        },
        "clocks": clocks,
        "gpu_launches": timed_launches,
        "parity_checked": parity is not None, "parity": parity,
        "episodes_match_closed_form": episodes_ok,
        "stats_allreduce_us": stats_allreduce_us if distributed else None,
        "e2e": e2e["headline"], "e2e_variants": e2e["variants"],
        "episodes": int(st[0]), "successes": int(st[1]),
    }
    if config3 is not None:
        line["config3"] = config3
    # ---- roofline of the dominant kernel
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        tr = tr["craft_rollout_kernel" if T > 1 else "craft_tick_kernel"]
        if tr["n_envs"] == n and tr.get("ticks_per_launch", 1) == T:
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass
    if fused:
        # per env: T x (404 f32 features + action + done + success) + one state read and write
        bytes_per_tick = BYTES_FUSED if T == 1 else (1616 + 3) + (2 * 96 + 4) / T
        launch_s = elapsed / max(1, timed_launches)
        ticks_per_launch_eff = K / max(1, timed_launches)
        achieved = bytes_per_tick * ticks_per_launch_eff * n / launch_s / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": "craft_rollout_kernel" if T > 1 else "craft_tick_kernel",
                            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": traffic, "peak_source": peak_src,
                            "algorithmic_bytes_per_env_step": bytes_per_tick,
                            "launch_us": launch_s * 1e6, "ticks_per_launch": ticks_per_launch_eff}
        if write_ceiling and "GBps" in write_ceiling:
            # why frac can exceed 1: this kernel only writes; against a store-only stream it is below 1
            line["roofline"]["write_only_ceiling"] = dict(write_ceiling, frac=achieved / write_ceiling["GBps"])
    # per-kernel numbers (north star: step and features as a fraction of the HBM roofline)
    line["kernels"] = per_kernel_table(torch, env, n, nf, dev, peak, min(ring, 8))
    if not fused:
        k = line["kernels"]["features_tma"]
        line["roofline"] = {"bound": "hbm", "kernel": "craft_features_kernel", "achieved": k["GBps"],
                            "peak": peak, "unit": "GB/s", "frac": k["frac"], "traffic": None,
                            "peak_source": peak_src, "algorithmic_bytes_per_env_step": BYTES_FEATURES}
    line["single_tick"] = dict(line["kernels"].pop("tick_fused"), kernel="craft_tick_kernel (one tick per "
                               "launch: the student-in-the-loop path)", algorithmic_bytes_per_env_step=BYTES_FUSED)
    if fused and world == 1:
        try:
            line["u8_frame"] = u8_frame_record(torch, env, n, nf, dev, peak)
        except Exception as ex:  # noqa: BLE001
            line["u8_frame"] = {"error": repr(ex)}
    if fused and world == 1 and T > 1 and rand_act is None:
        # SURVEY 8(d) config 2, off-policy variant: actions ~ U{0..5} from Philox(123, (env, t)); one Philox
        # launch fills the action block of each T-tick rollout launch (the full run: --policy random)
        try:
            ablock, oout = torch.empty((T, n), dtype=torch.uint8, device=dev), {}

            def off_policy_launch():
                env.random_actions(0, seed=123, out=ablock, device_clock=True, ticks=T)
                env.rollout(T, actions=ablock, features_out=feat_ring, out=oout, want_flags=True)

            for _ in range(3):
                off_policy_launch()
            o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            o0.record()
            for _ in range(60):
                off_policy_launch()
            o1.record()
            torch.cuda.synchronize()
            env.check_errors()
            sec = o0.elapsed_time(o1) * 1e-3 / (60 * T)
            bpt = (1616 + 3) + (2 * 96 + 4) / T + 1         # + the action byte read per env-tick
            line["off_policy"] = {"value": n / sec, "unit": UNIT, "us_per_tick": sec * 1e6,
                                  "frac": bpt * n / sec / 1e9 / peak, "launches": "60 x (Philox block + rollout of "
                                  "%d ticks), eager, CUDA events" % T}
        except Exception as ex:  # noqa: BLE001
            line["off_policy"] = {"error": repr(ex)}
    del env, feat_ring, feats
    torch.cuda.empty_cache()
    if world == 1 and not args.no_1m:
        n1 = 1 << 20
        w1 = load_workload(n1)
        env1 = VecCraft.from_instances(tables, w1["grids"], w1["env"], w1["pos"], w1["task"],
                                       max_timesteps=40, device=dev)
        for _ in range(13):             # states spread over their episodes, as in the 65,536-env table
            env1.tick(want_features=False)
        k1 = per_kernel_table(torch, env1, n1, nf, dev, peak, 3)
        k1["tick"] = k1.pop("tick_fused")
        k1["n_envs"] = n1
        line["kernels_1m"] = k1
        del env1
        torch.cuda.empty_cache()
    if world == 1 and not args.no_light:
        try:
            line["student_in_loop"] = student_in_loop_record(torch, tables, dev)
        except Exception as ex:  # noqa: BLE001
            line["student_in_loop"] = {"error": repr(ex)}
        try:
            line["stress_grids"] = stress_record(torch, dev)
        except Exception as ex:  # noqa: BLE001
            line["stress_grids"] = {"error": repr(ex)}
        try:
            line["light_world"] = light_record(torch, dev, peak)
        except Exception as ex:  # noqa: BLE001
            line["light_world"] = {"error": repr(ex)}
    # ---- CPU baselines on this box's host cores (bounded samples; single-GPU runs only)
    if not args.no_cpu and world == 1:
        line["cpu_baseline"] = dict(cpu_python_port(budget_s=12.0)[0], port_vs_reference=PORT_VS_REFERENCE)
        try:
            line["cpu_baseline_native"] = cpu_native_oracle()
        except Exception as ex:  # noqa: BLE001
            line["cpu_baseline_native"] = {"error": str(ex)}
    print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


def per_kernel_table(torch, env, n, nf, dev, peak, n_bufs):
    """Stand-alone kernels of the path at this batch size (CUDA-graph-timed, outputs rotating over
    n_bufs frames): µs per launch, GB/s on the algorithmic bytes, fraction of the measured peak."""
    kern = {}
    act = env.expert()
    big = [torch.empty((n, nf), dtype=torch.float32, device=dev) for _ in range(n_bufs)]
    cnt = [0]
    tout = {}

    def f_feat(impl):
        def g():
            env.features(out=big[cnt[0] % len(big)], impl=impl)
            cnt[0] += 1
        return g

    def f_tick():
        env.tick(features_out=big[cnt[0] % len(big)], fused=True, out=tout)
        cnt[0] += 1

    snap = env.snapshot()
    for name, fn, b in (("features_tma", f_feat(2), BYTES_FEATURES), ("features_plain", f_feat(1), BYTES_FEATURES),
                        ("expert", lambda: env.expert(out=act), BYTES_EXPERT),
                        ("step", lambda: env.step(act), BYTES_STEP),
                        ("tick_fused", f_tick, BYTES_FUSED)):
        env.restore(snap)               # every kernel is timed from the same states
        dt = time_kernel(fn, torch, inner=len(big) if name != "expert" and name != "step" else 10)
        kern[name] = {"us": dt * 1e6, "GBps": b * n / dt / 1e9, "frac": b * n / dt / 1e9 / peak,
                      "env_per_s": n / dt}
    env.restore(snap)
    del big
    return kern


def u8_frame_record(torch, env, n, nf, dev, peak, ticks=8, ring=16):
    """Secondary record: the same rollout with the opt-in byte frame (psk_craft_rollout_u8 /
    psk_craft_tick_u8) — every feature is an exact integer <= 255, so the frame is the f32 one cast.
    407 B per env-step instead of 1,619: the kernel is no longer write-bound, and the fraction of the
    copy bandwidth says how far the BFS + window arithmetic is from being hidden behind it."""
    snap = env.snapshot()
    frames = torch.empty((ring, n, nf), dtype=torch.uint8, device=dev)    # 16 x 26 MB > L2
    out, cnt = {}, [0]

    def roll():
        s = (cnt[0] * ticks) % ring
        env.rollout(ticks, features_out=frames[s:s + ticks], out=out)
        cnt[0] += 1

    def tick():
        env.tick(features_out=frames[cnt[0] % ring], out=out)
        cnt[0] += 1

    rec = {}
    for name, fn, per_launch in (("rollout", roll, ticks), ("single_tick", tick, 1)):
        env.restore(snap)
        dt = time_kernel(fn, torch, inner=ring // per_launch if per_launch > 1 else ring)
        b = (nf + 3) + (2 * 96 + 4) / per_launch
        rec[name] = {"us_per_tick": dt * 1e6 / per_launch, "env_steps_per_s": n * per_launch / dt,
                     "algorithmic_bytes_per_env_step": b, "GBps": b * n * per_launch / dt / 1e9,
                     "frac": b * n * per_launch / dt / 1e9 / peak, "ticks_per_launch": per_launch}
    env.restore(snap)
    del frames
    return rec


def light_record(torch, dev, peak):
    """Secondary record: the Light world (worlds/light.py) ported the same way — fused tick (table
    teacher + 12 features + step / auto-reset, one launch) on the reference's 60 scenarios."""
    from psketch_b200.worlds.light import LightWorld, VecLight
    goals = ("LL", "LD", "RD", "UL", "UR", "URU", "DRU", "LLD", "RDD", "LUR")
    w = LightWorld()
    scens = [w.sample_scenario_with_goal(g) for rep in range(6) for g in goals]
    rec = {"scenarios": len(scens), "algorithmic_bytes_per_env_step": 63}
    for n in (65536, 1 << 20):
        v = VecLight(scens, np.arange(n) % len(scens), device=dev)
        t0 = time.perf_counter()
        v._table = None
        v.teacher_table()
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        out = {}
        feats = [torch.empty((n, 12), dtype=torch.float32, device=dev) for _ in range(4)]
        cnt = [0]

        def f():
            v.tick(features_out=feats[cnt[0] % 4], out=out, max_timesteps=100)
            cnt[0] += 1
        for _ in range(30):
            f()                                    # envs spread over their episodes
        dt = time_kernel(f, torch, inner=8, reps=30)
        dt_lookup = time_kernel(lambda: v.expert(), torch, inner=8, reps=20)
        r = {"tick_us": dt * 1e6, "env_steps_per_s": n / dt, "GBps": 63 * n / dt / 1e9,
             "frac": 63 * n / dt / 1e9 / peak, "teacher_lookup_us": dt_lookup * 1e6,
             "teacher_table_build_ms_wall": build_ms}
        # T ticks per launch (psk_light_rollout): state, scenario and table pointers stay in registers
        T = 8
        slices = max(2, int(np.ceil(1.5 * 126e6 / (n * 48 * T))))          # ring of slices > L2
        ring = torch.empty((slices * T, n, 12), dtype=torch.float32, device=dev)
        rout = {}

        def g():
            k = cnt[0] % slices
            v.rollout(T, features_out=ring[k * T:(k + 1) * T], out=rout, max_timesteps=100)
            cnt[0] += 1
        dt_r = time_kernel(g, torch, inner=slices if slices <= 8 else 8, reps=20) / T
        b_r = 51 + 12 / T
        r.update({"rollout_ticks_per_launch": T, "rollout_us_per_tick": dt_r * 1e6,
                  "rollout_env_steps_per_s": n / dt_r, "rollout_GBps": b_r * n / dt_r / 1e9,
                  "rollout_frac": b_r * n / dt_r / 1e9 / peak})
        del ring
        if n == 65536:
            dt_search = time_kernel(lambda: v.expert(search=True), torch, inner=2, reps=3)
            r["teacher_search_kernel_us"] = dt_search * 1e6       # round 1: one flood per env
        rec["n_%d" % n] = r
        del v, feats
    return rec


def student_in_loop_record(torch, tables, dev, n=16384):
    """BASELINE configs[3]'s rollout with a policy in the loop: psketch_b200.students.GraphedRollout
    (40 timesteps of fused step-then-observe tick -> LSTM decode -> on-device sampling, one CUDA graph)
    with a randomly initialised student of the reference's architecture (models/lstm_seq2seq.py)."""
    from psketch_b200.students import GraphedRollout, Seq2SeqPolicy, task_tokens
    from psketch_b200.vec import VecCraft
    wl = load_workload(n)
    env = VecCraft.from_instances(tables, wl["grids"], wl["env"], wl["pos"], wl["task"], max_timesteps=255, device=dev)
    torch.manual_seed(0)
    pol = Seq2SeqPolicy(env.n_features, 6, len(tables.task_manager.vocab) + 1, tables.task_manager.vocab["<PAD>"]).to(dev)
    roll = GraphedRollout(env, pol, max_timesteps=40, greedy=False)
    with torch.no_grad():
        mem = pol.encode(task_tokens(tables, env.task))
    for _ in range(2):
        roll.run(mem)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, steps = 5, 0
    s.record()
    for _ in range(reps):
        roll.run(mem)
        steps += int(roll.interactions)
    e.record()
    torch.cuda.synchronize()
    dt = s.elapsed_time(e) * 1e-3
    return {"envs": n, "env_steps_per_s": steps / dt, "env_timesteps_per_s": reps * n * 40 / dt,
            "rollouts_per_s": reps * n / dt,
            "ms_per_rollout_of_40_timesteps": dt / reps * 1e3,
            "how": "GraphedRollout: per timestep one psk_craft_tick (step, then observe) + Seq2SeqPolicy.decode_step "
                   "(cuDNN LSTM 468->256, attention, predictor) + Gumbel-max sampling on the device; env_steps = "
                   "teacher-labelled states of running episodes (an untrained student samples STOP after ~6 steps "
                   "and idles for the rest of the 40), env_timesteps = every env x 40; training runs: "
                   "profiles/bench_runs/r2_dagger_*.json",
            "reference": "experiments/dagger_no_mix/run.log: ~1.5e3 interactions/s including learning"}


def stress_record(torch, dev, n=65536):
    """Secondary record (BASELINE configs[4]): the enlarged-grid BFS stress test — the row-per-lane
    warp-cooperative teacher (one warp per env), features and step on 16x16 / 32x32 / 64x64 grids
    with 20 % obstacles (tests/test_stress_gpu.py checks these kernels against the oracle)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_stress_gpu import _random_states, _tables
    from psketch_b200.vec import VecCraft
    rec = {"envs": n}
    for size in (16, 32, 64):
        tables = _tables(size)
        m = min(n, 4096 if size < 64 else 512)
        grid, inv, pos, dirs, task = _random_states(tables, m, seed=size, wall_frac=0.2)
        rep = (n + m - 1) // m
        tile = lambda a: np.concatenate([a] * rep)[:n]
        env = VecCraft.from_states(tables, tile(grid), tile(inv), tile(pos), tile(dirs), task=tile(task), device=dev)
        act = env.expert()
        feats = env.features()
        snap = env.snapshot()
        dt_e = time_kernel(lambda: env.expert(out=act), torch, inner=5, reps=6)
        dt_f = time_kernel(lambda: env.features(out=feats), torch, inner=5, reps=6)
        dt_s = time_kernel(lambda: env.step(act), torch, inner=5, reps=6)
        env.restore(snap)
        rec["%dx%d" % (size, size)] = {"expert_us": dt_e * 1e6, "expert_env_per_s": n / dt_e,
                                        "features_us": dt_f * 1e6, "step_us": dt_s * 1e6}
        del env, feats
    return rec


def measure_config3(torch, dist, pdist, tables, rank, world, dev, args):
    """BASELINE configs[2]: 8,388,608 envs sharded over the ranks (contiguous slices), T ticks per
    launch, one NCCL all-reduce of the episode statistics per 40-tick rollout."""
    from psketch_b200.vec import VecCraft
    total = 1 << 23
    n = total // world
    wl = load_workload(n)
    shift = (rank * n) % wl["n_instances"]
    env = VecCraft.from_instances(tables, wl["grids"], np.roll(wl["env"], -shift),
                                  np.roll(wl["pos"], -shift, axis=0), np.roll(wl["task"], -shift),
                                  max_timesteps=40, device=dev)
    nf = env.n_features
    T = max(1, args.ticks_per_launch)
    ring = T + 1
    feat_ring = torch.empty((ring, n, nf), dtype=torch.float32, device=dev)
    out = {}

    def launch():
        env.rollout(T, features_out=feat_ring, out=out, want_flags=True)

    per_rollout = 40 // T                           # launches per 40-tick rollout
    for _ in range(2):
        launch()
    env.stats.zero_()
    torch.cuda.synchronize()
    dist.barrier()
    rounds = 3
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar_ms = []
    s.record()
    for _ in range(rounds):
        for _ in range(per_rollout):
            launch()
        st = env.stats.clone()
        a0.record()
        pdist.allreduce_stats(st)                   # NCCL SUM of {episodes, successes, env_steps}
        a1.record()
        a1.synchronize()
        ar_ms.append(a0.elapsed_time(a1))
    e.record()
    torch.cuda.synchronize()
    el = torch.tensor([s.elapsed_time(e) * 1e-3], dtype=torch.float64, device=dev)
    dist.all_reduce(el, op=dist.ReduceOp.MAX)
    env.check_errors()
    steps = rounds * per_rollout * T
    peak, _ = measured_peaks()
    bytes_per_tick = (1616 + 3) + (2 * 96 + 4) / T
    value = total * steps / float(el.item())
    res = {"workload": "BASELINE configs[2]: craft_medium, 8,388,608 envs sharded over %d GPUs (%d per GPU), "
                       "%d ticks per launch, NCCL all-reduce of the statistics every 40 ticks" % (world, n, T),
           "value": value, "unit": UNIT, "envs_total": total, "envs_per_gpu": n, "steps": steps,
           "ms_per_step": float(el.item()) / steps * 1e3,
           "roofline_frac_per_gpu": bytes_per_tick * n * steps / float(el.item()) / 1e9 / peak,
           "stats_allreduce_ms": ar_ms, "env_steps_counted": int(st[2])}
    del env, feat_ring
    torch.cuda.empty_cache()
    return res


def measure_e2e(torch, dist, tables, wl, n, dev, args, world):
    """The same tick through the reference-facing C ABI with HOST buffers, copies inside the timed
    region, MAX over ranks.  Four forms, all checked against the step counter:
      host_in_loop_f32         psk_craft_host_tick_resident, step-then-observe: the host's actions
                               go up every step, the f32[n,404] frame + teacher actions + flags come down
      host_in_loop_f32_wire_u8 the same f32 host frame, but bytes cross PCIe and host threads widen them
                               (headline = the faster of these two)
      resident_f32             the same without an action upload (teacher-driven inside the kernel)
      roundtrip_f32            psk_craft_host_tick: additionally the states go up and come back
      resident_u8              the compact u8[n,404] frame instead of f32 (opt-in format)
    plus pcie_ceiling: a plain pinned D2H copy of the f32 frame's bytes, all ranks concurrently."""
    from psketch_b200.host import HostCraft
    env = HostCraft(tables, wl["grids"], wl["env"], wl["pos"], wl["task"], max_timesteps=40,
                    chunk_envs=args.e2e_chunk)
    steps = max(3, min(args.steps, 30))

    def timed(fn, reps, pre=3):
        """Wall time of `reps` calls after `pre` (>= 3) untimed ones, MAX over ranks.  fn=None, or an exception
        inside fn on ANY rank, gives inf on EVERY rank (the collectives are still executed, so no
        rank is left waiting): an optional form that fails is dropped, it does not take the run down."""
        ok = fn is not None
        try:
            for _ in range(pre if ok else 0):
                fn()
            torch.cuda.synchronize()
        except Exception as ex:  # noqa: BLE001
            ok, timed.error = False, repr(ex)
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        try:
            for _ in range(reps if ok else 0):
                fn()                    # returns after the D2H copies have landed
        except Exception as ex:  # noqa: BLE001
            ok, timed.error = False, repr(ex)
        wall = time.perf_counter() - t0 if ok else float("inf")
        if dist is not None:
            w = torch.tensor([wall], dtype=torch.float64, device=dev)
            dist.all_reduce(w, op=dist.ReduceOp.MAX)
            wall = float(w.item())
        return wall

    timed.error = None

    def timed_or_raise(fn, reps):
        wall = timed(fn, reps)
        if wall == float("inf"):
            raise RuntimeError("e2e leg failed: %s" % (timed.error or "on another rank"))
        return wall
    variants = {}
    before = int(env.stats[2])
    wall = timed_or_raise(env.tick, steps)
    assert int(env.stats[2]) - before == (steps + 3) * n
    variants["roundtrip_f32"] = {"value": n * steps * world / wall, "unit": UNIT,
                                 "h2d_bytes_per_step": env.last_h2d, "d2h_bytes_per_step": env.last_d2h}
    env.reset_resident()
    for name, fmt in (("resident_f32", "f32"), ("resident_u8", "u8")):
        before = int(env.stats[2])
        wall = timed_or_raise(lambda: env.tick_resident(features=fmt), steps)
        assert int(env.stats[2]) - before == (steps + 3) * n
        variants[name] = {"value": n * steps * world / wall, "unit": UNIT,
                          "h2d_bytes_per_step": env.last_h2d, "d2h_bytes_per_step": env.last_d2h}
    # host in the loop: the host's policy (here: follow the teacher action it was handed) picks the
    # actions, they go UP with every call, the step is applied, the new observation comes DOWN as an
    # f32[n,404] host array — over PCIe as f32, or as bytes widened by host threads (f32_wire_u8)
    for name, fmt in (("host_in_loop_f32", "f32"), ("host_in_loop_f32_wire_u8", "f32_wire_u8")):
        optional = fmt != "f32"         # the wire form may fail (then it is dropped); the f32 form may not
        step_fn, before = None, 0
        try:
            if fmt == "f32_wire_u8":
                # smaller chunks: the widening of the last chunk is the exposed tail of the pipeline
                env.close()
                local = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
                threads = args.e2e_host_threads or max(1, min(8, (os.cpu_count() or 2) // local))
                env = HostCraft(tables, wl["grids"], wl["env"], wl["pos"], wl["task"], max_timesteps=40,
                                chunk_envs=args.e2e_wire_chunk, host_threads=threads)
            env.reset_resident()
            env.features[:] = -1.0
            env.tick_resident(features=fmt, advance_first=True)        # first observation, no step yet
            acts = env.expert.copy()

            def step_fn(fmt=fmt, acts=acts):
                env.tick_resident(actions=acts, features=fmt, advance_first=True)
                acts[:] = env.expert                                    # the host "policy": np copy of n bytes

            before = int(env.stats[2])
        except Exception as ex:  # noqa: BLE001
            if not optional:
                raise
            step_fn, timed.error = None, repr(ex)
        # the wire form settles its split (chunks sent as f32 while the host threads widen the rest)
        # from measured rates over its first calls: those are untimed warm-up.  Both forms take the
        # same number of steps from the same reset, so that their final host frames can be compared
        pre = 12
        wall = timed(step_fn, steps, pre)
        if wall == float("inf"):
            if not optional:
                raise RuntimeError("e2e leg %s failed: %s" % (name, timed.error))
            variants[name] = {"value": 0.0, "unit": UNIT, "error": timed.error or "failed on another rank"}
            continue
        counted = int(env.stats[2]) - before == (steps + pre) * n
        variants[name] = {"value": n * steps * world / wall, "unit": UNIT,
                          "h2d_bytes_per_step": env.last_h2d, "d2h_bytes_per_step": env.last_d2h}
        if fmt == "f32":
            assert counted
            frame_f32 = env.features.copy()
            state_f32 = (env.expert.copy(), env.done.copy())
        else:   # both forms ran the same number of steps from the same reset: identical host frames
            same = bool(counted and np.array_equal(env.features, frame_f32) and
                        np.array_equal(env.expert, state_f32[0]))
            if dist is not None:         # every rank's frame must agree, not only rank 0's
                flag = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                same = bool(flag.item() > 0.5)
            variants[name]["host_threads"] = int(env.lib.psk_craft_host_threads(env.ctx))
            variants[name]["chunk_envs"] = args.e2e_wire_chunk
            variants[name]["chunks_sent_as_f32"] = "%d of %d (last call; split follows the measured PCIe / widening rates)" % (
                env.last_wire_direct, -(-n // env.chunk_envs))
            variants[name]["frame_equals_f32_path"] = same
            if not same:                 # never report a number for frames that differ
                variants[name]["measured_but_rejected"] = variants[name]["value"]
                variants[name]["value"] = 0.0
    # the reference's own operating point (configs/experiments/imitation.yaml: batch_size 32): latency of
    # one host-in-the-loop tick through the same C entry point, rank-local, not part of the headline
    try:
        w32 = load_workload(32)
        e32 = HostCraft(tables, w32["grids"], w32["env"], w32["pos"], w32["task"], max_timesteps=40, chunk_envs=128)
        e32.reset_resident()
        e32.tick_resident(features="f32", advance_first=True)
        a32 = e32.expert.copy()
        for i in range(20 + 400):
            if i == 20:
                t32 = time.perf_counter()
            e32.tick_resident(actions=a32, features="f32", advance_first=True)
            a32[:] = e32.expert
        us = (time.perf_counter() - t32) / 400 * 1e6
        variants["batch32_f32"] = {"us_per_tick": us, "env_steps_per_s_one_rank": 32 / us * 1e6,
                                   "note": "32 envs per call (the reference's batch size), host in the loop, "
                                           "one rank; latency-bound, not aggregated over ranks"}
        e32.close()
    except Exception as ex:  # noqa: BLE001
        variants["batch32_f32"] = {"error": repr(ex)}
    # PCIe ceiling for the f32 frame: the same bytes, pinned, nothing else
    frame = torch.empty((n, env.n_features), dtype=torch.float32, device=dev)
    host = torch.empty((n, env.n_features), dtype=torch.float32, pin_memory=True)
    wall = timed_or_raise(lambda: (host.copy_(frame, non_blocking=True), torch.cuda.synchronize()), steps)
    gbs = frame.numel() * 4 * steps / wall / 1e9
    ceiling = {"d2h_GBps_per_gpu": gbs, "env_steps_per_s": n * steps * world / wall,
               "how": "pinned cudaMemcpy D2H of one f32[%d,%d] frame per step, all %d ranks at once" % (n, env.n_features, world)}
    best = max(("host_in_loop_f32", "host_in_loop_f32_wire_u8"), key=lambda k: variants[k]["value"])
    head = dict(variants[best])
    head.update({"steps": steps, "form": best, "pcie_ceiling": ceiling,
                 "frac_of_pcie_ceiling": variants["host_in_loop_f32"]["value"] / ceiling["env_steps_per_s"],
                 "vs_f32_frame_over_pcie_ceiling": head["value"] / ceiling["env_steps_per_s"],
                 "how": "psk_craft_host_tick_resident (C ABI, host numpy buffers), host in the loop: per step "
                        "H2D the actions the host chose (u8[n]), fused step-then-observe tick in %d-env chunks over "
                        "3 streams, f32[n,404] features + teacher actions + done/success of the new states land in "
                        "host memory; the environments stay in HBM.  form = the faster of host_in_loop_f32 (the "
                        "f32 frame crosses PCIe; frac_of_pcie_ceiling is that form's) and host_in_loop_f32_wire_u8 "
                        "(the u8 frame crosses PCIe, host threads widen each chunk to f32 while the next is in "
                        "flight, and the last chunks_sent_as_f32 chunks cross as f32 into the caller's pinned frame "
                        "while the threads are still busy; same host frame, checked equal in this run).  e2e_variants: both, plus no action "
                        "upload, the state round trip of round 1, and the raw u8 frame" %
                        (args.e2e_wire_chunk if best.endswith("wire_u8") else args.e2e_chunk)})
    env.close()
    return {"headline": head, "variants": variants}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--unfused", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-chunk", type=int, default=16384)
    ap.add_argument("--e2e-host-threads", type=int, default=0,
                    help="widening threads per rank of the u8-on-the-wire form; 0 = min(8, cores / ranks on this box)")
    ap.add_argument("--e2e-wire-chunk", type=int, default=4096,
                    help="chunk size of the u8-on-the-wire e2e form (profiles/bench_runs/r2_e2e_wire_sweep.txt)")
    ap.add_argument("--ticks-per-launch", type=int, default=8,
                    help="teacher-driven rollouts run this many ticks per kernel launch (1 = one tick per launch)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned on rank 0 (features, teacher actions, done / "
                         "success flags; a fixed sample of envs beyond %d MB) as DIR/<name>.npy" % (DUMP_BYTES // 10**6))
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed kernel")
    ap.add_argument("--no-1m", action="store_true", help="skip the 1,048,576-env per-kernel table")
    ap.add_argument("--no-config3", action="store_true", help="skip BASELINE config 3 (world > 1)")
    ap.add_argument("--no-light", action="store_true", help="skip the Light-world secondary record")
    ap.add_argument("--policy", default="teacher", choices=["teacher", "random"],
                    help="who acts: the teacher (BASELINE config) or uniform random actions (off-policy variant)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
