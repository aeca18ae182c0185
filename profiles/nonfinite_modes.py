"""Cost and effect of BatchedPhysicsEnv(nonfinite="keep" | "count" | "end"), alternated in one process.

Workloads (all in3d, template auto-reset, seed 1234, episode statistics, as bench.py builds them):
  headline   Balance-v0, 2^20 envs, packed state, 30-step and 1000-step episodes
  config4    quad_balance and quad_balance_chain, 2^20 envs, 8 substeps, 1000-step episodes
  config5    Balance-v0, 2^18 envs, RolloutCollector (fused policy, CUDA graph), T = 32 rollouts
Per (workload, mode), in rounds that cycle through the three modes: the time per env step from CUDA events over a
window after a preroll past the first 1000-step episode end (so the window is steady state), the share of
non-finite observation rows over the steps after the window, and episode_stats().  Writes one JSON line per
measurement and a header line with the card name and power limit, read in the same process.

    python profiles/nonfinite_modes.py OUT.jsonl [--rounds 2] [--window 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

MODES = ("keep", "count", "end")
DEV = "cuda:0"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"card": q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown",
            "torch_device": torch.cuda.get_device_name(0)}


def nonfinite_share(obs):
    return float((~torch.isfinite(obs).all(dim=-1)).float().mean())


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for t in range(n):
        fn(t)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / n          # microseconds per call


def env_run(body, E, mode, *, max_steps, k_sub, preroll, window, probe=20):
    from walker_gym_b200 import BatchedPhysicsEnv
    env = BatchedPhysicsEnv(body, E, DEV, in3d=True, auto_reset="template", seed=1234, track_stats=True, k_sub=k_sub,
                            max_steps=max_steps, nonfinite=mode)
    g = torch.Generator(device=DEV).manual_seed(0)
    ring = [torch.rand(E, env.M, device=DEV, generator=g) * 2 - 1 for _ in range(16)]
    for t in range(preroll):
        env.step(ring[t % 16])
    us = timed(lambda t: env.step(ring[t % 16]), window)
    share = 0.0
    for t in range(probe):
        obs, _, _, _ = env.step(ring[t % 16])
        share += nonfinite_share(obs) / probe
    return {"us_per_step": us, "us_per_env_step": us / E, "nonfinite_obs_share": share,
            "episode_stats": env.episode_stats(), "state_layout": env.state_layout}


def rollout_run(mode, *, E=1 << 18, T=32, rollouts=40, preroll=40):
    from walker_gym_b200 import BatchedPhysicsEnv
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, in3d=True, auto_reset="template", seed=1234, track_stats=True,
                            graph_safe=True, max_steps=1000, nonfinite=mode)
    torch.manual_seed(0)
    col = RolloutCollector(env, FeatureMajorMLP(env.obs_dim, env.M).to(DEV), T, seed=1234)
    for _ in range(preroll):
        col.collect()
    us = timed(lambda t: col.collect(), rollouts) / T
    out = col.collect()
    return {"us_per_step": us, "us_per_env_step": us / E, "nonfinite_obs_share": nonfinite_share(out["obs"]),
            "episode_stats": col.episode_stats(all_reduce=False), "horizon": T}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--window", type=int, default=200)
    args = ap.parse_args()
    work = [
        ("headline_ep30", lambda m: env_run("Balance-v0", 1 << 20, m, max_steps=30, k_sub=1, preroll=1100, window=args.window)),
        ("headline_ep1000", lambda m: env_run("Balance-v0", 1 << 20, m, max_steps=1000, k_sub=1, preroll=1100, window=args.window)),
        ("config4_quad_balance", lambda m: env_run("quad_balance", 1 << 20, m, max_steps=1000, k_sub=8, preroll=1100, window=args.window)),
        ("config4_quad_balance_chain", lambda m: env_run("quad_balance_chain", 1 << 20, m, max_steps=1000, k_sub=8, preroll=1100,
                                                         window=args.window)),
        ("config5_rollout", lambda m: rollout_run(m)),
    ]
    with open(args.out, "w") as f:
        f.write(json.dumps({"header": True, **card(), "time": time.strftime("%Y-%m-%dT%H:%M:%S")}) + "\n")
        for r in range(args.rounds):
            for name, fn in work:
                for mode in (MODES if r % 2 == 0 else MODES[::-1]):
                    rec = {"workload": name, "mode": mode, "round": r, **fn(mode)}
                    f.write(json.dumps(rec) + "\n")
                    f.flush()
                    print(json.dumps(rec), flush=True)
                    torch.cuda.empty_cache()
        f.write(json.dumps({"footer": True, **card()}) + "\n")


if __name__ == "__main__":
    main()
