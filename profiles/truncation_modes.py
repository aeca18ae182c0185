"""Cost of BatchedPhysicsEnv(track_truncation=True) and RolloutCollector(bootstrap_truncated=...), alternated in one
process.

Workloads (in3d, template auto-reset, seed 1234, episode statistics, as bench.py builds them):
  headline   Balance-v0, 2^20 envs, packed state, 30-step (config 3) and 1000-step episodes, tracking off / on;
             the boundary step (every env of a synchronised batch at its time limit) is timed on its own
  config5    Balance-v0, 2^18 envs, RolloutCollector (fused policy, CUDA graph), T = 32: bootstrap None on an env without
             tracking, None on a tracking env (the step's cost of the flag and the final observation alone), "current"
             and "final"
Per (workload, variant), in rounds that cycle through the variants: microseconds per env step from CUDA events.
Writes one JSON line per measurement and a header line with the card name and power limit, read in the same process.

    python profiles/truncation_modes.py OUT.jsonl [--rounds 3] [--window 300]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

DEV = "cuda:0"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"card": q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown",
            "torch_device": torch.cuda.get_device_name(0)}


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for t in range(n):
        fn(t)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / n          # microseconds per call


def headline(track, max_steps, window):
    from walker_gym_b200 import BatchedPhysicsEnv
    E = 1 << 20
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, in3d=True, auto_reset="template", seed=1234, track_stats=True,
                            max_steps=max_steps, track_truncation=track)
    g = torch.Generator(device=DEV).manual_seed(0)
    ring = [torch.rand(E, env.M, device=DEV, generator=g) * 2 - 1 for _ in range(16)]
    for t in range(50):
        env.step(ring[t % 16])
    us = timed(lambda t: env.step(ring[t % 16]), window)
    # the boundary step: every env one step before its time limit (the synchronised batch of bench.py config 3)
    steps = torch.full((E,), max_steps - 1, dtype=torch.int32, device=DEV)
    boundary = []
    for k in range(20):
        env.set_state(steps=steps)
        torch.cuda.synchronize()
        boundary.append(timed(lambda t: env.step(ring[k % 16]), 1))
    boundary.sort()
    return {"us_per_step": us, "boundary_us_median": boundary[len(boundary) // 2]}


def config5(bootstrap, track, rollouts):
    from walker_gym_b200 import BatchedPhysicsEnv
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    E, T = 1 << 18, 32
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, in3d=True, auto_reset="template", seed=1234, graph_safe=True,
                            obs_layout="row", act_layout="row", track_truncation=track)
    torch.manual_seed(0)
    pol = FeatureMajorMLP(env.obs_dim, env.M).to(DEV)
    col = RolloutCollector(env, pol, T, seed=5, bootstrap_truncated=bootstrap)
    for _ in range(3):
        col.collect()
    us = timed(lambda t: col.collect(), rollouts) / T
    return {"us_per_step": us}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--window", type=int, default=300)
    args = ap.parse_args()
    with open(args.out, "w") as f:
        f.write(json.dumps(dict(card(), header=True)) + "\n")
        for r in range(args.rounds):
            for max_steps in (30, 1000):
                for track in (False, True):
                    rec = dict(workload="headline", max_steps=max_steps, track_truncation=track, round=r)
                    rec.update(headline(track, max_steps, args.window))
                    f.write(json.dumps(rec) + "\n")
                    f.flush()
                    torch.cuda.empty_cache()
            for bootstrap, track in ((None, False), (None, True), ("current", True), ("final", True)):
                rec = dict(workload="config5", bootstrap_truncated=bootstrap, track_truncation=track, round=r)
                rec.update(config5(bootstrap, track, 30))
                f.write(json.dumps(rec) + "\n")
                f.flush()
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
