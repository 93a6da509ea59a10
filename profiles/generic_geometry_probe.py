#!/usr/bin/env python
"""What the generic tier (psketch_b200/csrc/psk_craft_generic.cu) costs, at 65,536 envs.

Per geometry: CUDA-event times of each primitive (teacher, f32 / u8 features, step, satisfies), the
pipelined tick (psk_craft_tick with PSK_TICK_PIPELINE: teacher, features, advance) in us, and env-steps/s
of that tick.  At 8x8 / 3 and 16x16 / 3 the specialised kernels and the generic tier (tuning key
`generic` = 1) run the same states in the same process, interleaved round by round; there the fused tick
of the specialised path is reported as well.  The other geometries (9x9 / 3, 12x12 / 5, 20x13 with a 3x5
window, 64x64 / 9) have only the generic tier.

States: 1,024 random scenarios per geometry (boundary ring, 20 % of the interior filled with every kind,
the agent on a free cell), get / make tasks, reused round-robin by the 65,536 envs.  Every time is the
median over --rounds rounds of --reps launches each, after a warm-up.  Writes one JSON file with the
GPU's name and power limit read in the same run.

    python profiles/generic_geometry_probe.py --out profiles/bench_runs/r3_generic_geometry_probe.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from psketch_b200 import _lib  # noqa: E402
from psketch_b200.tables import CraftTables  # noqa: E402
from psketch_b200.vec import VecCraft  # noqa: E402

# (W, H, window_w, window_h, compare with the specialised kernels)
CASES = [(8, 8, 3, 3, True), (16, 16, 3, 3, True), (9, 9, 3, 3, False), (12, 12, 5, 5, False),
         (20, 13, 3, 5, False), (64, 64, 9, 9, False)]


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "nvidia-smi failed: %s" % e
    return info


def make_env(W, H, ww, wh, n, seed=0):
    tables = CraftTables(world_config=dict(WIDTH=W, HEIGHT=H, WINDOW_WIDTH=ww, WINDOW_HEIGHT=wh, N_WORKSHOPS=3,
                                           N_PRIMITIVES=2, N_WORLDS=1))
    rng = np.random.RandomState(seed)
    S, K = 1024, tables.K
    g = np.where(rng.rand(S, W, H) < 0.2, rng.randint(1, K, size=(S, W, H)), 0).astype(np.uint8)
    b = tables.cookbook.index["boundary"]
    g[:, 0, :] = g[:, W - 1, :] = g[:, :, 0] = g[:, :, H - 1] = b
    pos = np.stack([rng.randint(1, W - 1, S), rng.randint(1, H - 1, S)], 1)
    g[np.arange(S), pos[:, 0], pos[:, 1]] = 0
    tasks = [t.task_id for t in tables.task_manager.tasks if t.goal_name in ("get", "make")]
    idx = np.arange(n) % S
    task = rng.choice(tasks, size=n)
    env = VecCraft.from_instances(tables, g.reshape(S, -1), idx, pos[idx], task, max_timesteps=40)
    return env


def timed(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1000.0 / reps          # us per call


def ops(env, n):
    feats = torch.empty((n, env.n_features), dtype=torch.float32, device=env.device)
    feats8 = torch.empty((n, env.n_features), dtype=torch.uint8, device=env.device)
    act = torch.from_numpy(np.random.RandomState(1).randint(0, 6, n).astype(np.uint8)).to(env.device)
    out = {k: torch.empty(n, dtype=torch.uint8, device=env.device) for k in ("expert", "done", "success")}
    return {
        "expert": lambda: env.expert(),
        "features_f32": lambda: env.features(out=feats),
        "features_u8": lambda: env.features_u8(out=feats8),
        "step": lambda: env.step(act),
        "satisfies": lambda: env.satisfies(),
        "tick_pipeline": lambda: env.tick(features_out=feats, out=out, fused=False),
        "tick_fused": lambda: env.tick(features_out=feats, out=out, fused=True),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_runs", "r3_generic_geometry_probe.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    result = dict(gpu_info(), n_envs=a.n, reps=a.reps, rounds=a.rounds, unit="us per call (median of rounds)",
                  geometries=[])
    for W, H, ww, wh, compare in CASES:
        env = make_env(W, H, ww, wh, a.n)
        tiers = ["specialised", "generic"] if compare else ["generic"]
        samples = {t: {} for t in tiers}
        calls = ops(env, a.n)
        for rnd in range(a.rounds + 1):                   # round 0 is the warm-up
            for tier in tiers:
                with_generic = 1 if tier == "generic" else -1
                old = _lib.set_tuning(generic=with_generic)
                try:
                    for name, fn in calls.items():
                        if name == "tick_fused" and tier == "generic":
                            continue                      # the generic tier has no fused tick
                        env.reset()
                        t = timed(fn, a.reps if rnd else 3)
                        if rnd:
                            samples[tier].setdefault(name, []).append(t)
                    env.check_errors()
                finally:
                    _lib.set_tuning(**old)
        row = dict(geometry="%dx%d window %dx%d" % (W, H, ww, wh), n_features=env.n_features)
        for tier in tiers:
            med = {k: float(np.median(v)) for k, v in samples[tier].items()}
            med["env_steps_per_s_pipeline"] = a.n / (med["tick_pipeline"] * 1e-6)
            if "tick_fused" in med:
                med["env_steps_per_s_fused"] = a.n / (med["tick_fused"] * 1e-6)
            row[tier] = {k: round(v, 2) for k, v in med.items()}
        if compare:
            row["generic_over_specialised"] = {k: round(row["generic"][k] / row["specialised"][k], 2)
                                               for k in row["generic"] if k in row["specialised"]
                                               and not k.startswith("env_steps")}
        result["geometries"].append(row)
        print(json.dumps(row), flush=True)
        del env
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "geometries"}))


if __name__ == "__main__":
    main()
