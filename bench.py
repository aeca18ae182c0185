#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused walker-gym physics step on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference itself on the box's host cores

A *step* is one pass of the hot path (PhysicsEnv.step: act -> physics -> reward /
done / auto-reset -> observation) over every env of the batch: ONE kernel launch.
Workload (BASELINE.json config 3, the throughput config; weak scaling): Balance-v0
(gym/optimized_walker.py:176-199), in3d, 2^20 envs per GPU, U(-1,1) float32
actions resident on the device, template auto-reset after EPISODE_STEPS env-steps, reference semantics as written.
Rank 0 prints ONE JSON line.  Besides the headline it carries short sub-measurements of
the other BASELINE configs (`sub_configs`), the end-to-end number on host buffers (`e2e`)
next to the box's own device-to-host ceiling measured in the same run, the roofline of
the step kernel and the CPU baseline.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

POLICY_KERNELS = {2: "wg::policy_act_ws_kernel (warp-specialised tcgen05 / TMEM pipeline, TMA-staged observations)",
                  1: "wg::policy_act_tc_kernel (monolithic tcgen05 / TMEM kernel)", 0: "wg::policy_act_kernel (mma.sync TF32)"}
METRIC = "env-steps/sec (whole box)"
UNIT = "env-steps/s"
ENV_ID = "Balance-v0"
N_MASS, N_MUSCLE = 4, 2
OBS_DIM = 3 * 3 * N_MASS + N_MUSCLE
ROLLOUT_T = 32         # config 5: env-steps per RolloutCollector.collect (one CUDA-graph replay)
PREROLL = 256          # untimed env-steps before any timed window: the timed region is the steady state of the reset
#                        cycle, not the first steps after the initial template reset
EPISODE_STEPS = 30     # max_steps of every config 3 measurement and of its CPU arms: Balance-v0's as-written dynamics
#                        overflow float32 no sooner than ~34 env-steps after a reset, so every env stepped stays finite
#                        (with the reference's default of 1000, ~70 % of the envs hold inf / NaN in steady state)


def algorithmic_bytes(n_mass: int, n_muscle: int) -> int:
    """Per env-step (SURVEY 8d): state R+W 48N, muscle x R+W + action R 12M, steps R+W 8, reward 4, done 1;
    plus the materialised observation 36N + 4M."""
    return 48 * n_mass + 12 * n_muscle + 13 + 36 * n_mass + 4 * n_muscle


BYTES_PER_ENV_STEP = algorithmic_bytes(N_MASS, N_MUSCLE)     # 381


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of the cpu_baseline sample")
    ap.add_argument("--ref-seconds", type=float, default=8.0, help="reference arm: target duration of the timed region")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "reference", "port"],
                    help="reference arm: the reference itself (oracle/_ref, made by oracle/make_ref.py) or the C port")
    ap.add_argument("--policy", default="fused-fp32", choices=["fused-fp32", "fused-tf32", "torch"],
                    help="config 5: wg_policy_act (3xTF32 float32-grade / plain TF32 tensor-core MLP) or torch ops")
    ap.add_argument("--probe-stream", action="store_true",
                    help="measure the HBM rate of a pure streaming kernel with the step kernel's read:write mix and exit")
    ap.add_argument("--k-sub", type=int, default=0, help="physics substeps per env step (0 = the config's default)")
    ap.add_argument("--steps-per-launch", type=int, default=1, help="config 6: update_physics calls fused in one launch; config 3: env-steps per launch (wg_step_multi)")
    ap.add_argument("--pkg-body", default="box", help="config 6: body builder of gym/optimized_walker/walker.py")
    ap.add_argument("--config", type=int, default=3, choices=[3, 4, 5, 6],
                    help="BASELINE.json config: 3 = Balance-v0 throughput (headline, default), 4 = enlarged body "
                         "(4x masses/springs) with 8 substeps, 5 = PPO rollout collection (torch MLP policy + step kernel)")
    ap.add_argument("--body", default="balance", choices=["balance", "box", "legacy_box", "test", "intrian", "hat", "humanb", "box4", "leg", "leg2", "insect", "quad", "quad_chain", "balance2", "balance3"],
                    help="config 3 body: Balance-v0 (headline) or Box-v0, both from gym/optimized_walker.py:176-224")
    ap.add_argument("--obs-layout", default="row", choices=["row", "feature"],
                    help="observation layout written by the kernel: row-major [E,D] (default) or feature-major [D,E]")
    ap.add_argument("--generic", action="store_true", help="measure the run-time-topology kernel instead of the specialisation")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub_configs measurements (configs 3-strong, 4, 5, multi-step)")
    ap.add_argument("--no-affinity", action="store_true", help="do not bind the rank to CPUs next to its GPU")
    ap.add_argument("--strong-envs-per-gpu", type=int, default=0,
                    help="sub-config 3_strong: envs per GPU (default 2^20 / n_gpus, BASELINE config 3 as written)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed window, write rank 0's results of the last timed step (obs, reward, done) "
                         "as DIR/<name>.npy in float32; above 63 MB in all, every array keeps the same seeded sample of envs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config == 5 and args.steps % ROLLOUT_T:
        ap.error(f"--config 5 times whole {ROLLOUT_T}-step rollouts: --steps must be a multiple of {ROLLOUT_T}")
    if args.dump_outputs and (args.impl != "ours" or args.probe_stream or args.config != 3 or args.body != "balance"
                              or args.steps_per_launch > 1 or args.k_sub > 1):
        ap.error("--dump-outputs applies to the headline path (--config 3, --body balance, one env-step per launch)")
    return args


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_env_step():
    """dram read+write bytes per env-step of the step kernel from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            d = json.load(f)
            return float(d["dram_bytes_per_env_step"]), d.get("source", "profiles/ncu_traffic.json")
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------
# CPU arms
# ----------------------------------------------------------------------------------
def host_cpus():
    try:
        return sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))


def cpu_run(n_env: int, steps: int, warmup: int, seed: int = 0):
    """Step `n_env` Balance-v0 envs `steps` times with the oracle port (C restatement of the reference, OpenMP over
    envs); returns (env-steps/s, seconds, threads)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import walker_oracle as wo
    threads = wo.set_threads(len(host_cpus()))      # all host threads (torchrun would pin OMP_NUM_THREADS=1)
    body = wo.make_body(wo.BALANCE)
    prm = wo.make_params(in3d=True, auto_reset=2, seed=seed, max_steps=EPISODE_STEPS)
    st = wo.init_state(body, n_env)
    st.pop("old_a")
    wo.reset(body, prm, st, mode=2)
    rng = np.random.default_rng(seed)
    ring = [rng.uniform(-1, 1, (n_env, N_MUSCLE)).astype(np.float32) for _ in range(8)]
    # OpenMP pool spin-up on a scratch state (untimed): the first ~20 parallel regions of a fresh pool run 10-25x
    # slower than steady state (thread creation, scheduler spreading the threads over the cores); without this a
    # short --steps run would under-report the CPU arm.  Bounded at 3 s; the timed trajectory is not touched.
    scratch = wo.init_state(body, n_env)
    scratch.pop("old_a")
    wo.reset(body, prm, scratch, mode=2)
    t_spin = time.perf_counter()
    for _ in range(60):
        wo.step(body, prm, scratch, ring[0], want_info=False)
        if time.perf_counter() - t_spin > 3.0:
            break
    del scratch
    for t in range(warmup):
        prm.step_index = t + 1
        wo.step(body, prm, st, ring[t % 8], want_info=False)
    t0 = time.perf_counter()
    for t in range(steps):
        prm.step_index = warmup + t + 1
        wo.step(body, prm, st, ring[t % 8], want_info=False)
    dt = time.perf_counter() - t0
    return n_env * steps / dt, dt, threads


def cpu_baseline(target_seconds: float):
    n_env = 1 << 15
    rate, _, threads = cpu_run(n_env, 20, 3)
    steps = max(10, int(target_seconds * rate / n_env))
    rate, dt, threads = cpu_run(n_env, steps, 3)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{ENV_ID} in3d, {n_env} envs x {steps} steps, oracle/walker_oracle.c (C restatement of the "
                      f"reference, bit-exact vs its golden vectors), OpenMP over envs, {dt:.1f} s"}


def _ref_worker(idx, cpu, ref_root, n_warm, n_timed, barrier, out_q):
    """One process = one reference env (its Point registry is process-global, gym/optimized_engine.py:258-272), the
    loop of gym/performance_demo.py:241-262: random action, env.step, rebuild the env when the episode is done."""
    try:
        os.sched_setaffinity(0, {cpu})
    except OSError:
        pass
    import warnings
    import numpy as np
    warnings.filterwarnings("ignore")
    np.seterr(all="ignore")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness as rh
    engine, _, envmod = rh.load(ref_root)
    rng = np.random.default_rng(1000 + idx)
    acts = rng.uniform(-1.0, 1.0, size=(1024, N_MUSCLE)).astype(np.float32)

    def make():
        engine.Point.clear()
        np.random.seed(idx)
        env = envmod.make_env(ENV_ID, in3d=True)
        env.max_steps = EPISODE_STEPS
        return env

    env = make()
    done_steps = 0

    def run(n):
        nonlocal env, done_steps
        for t in range(n):
            _, _, done, _ = env.step(acts[(done_steps + t) & 1023])
            if done:
                env = make()                          # template auto-reset == make_env again
        done_steps += n

    run(n_warm)
    barrier.wait()
    t0 = time.perf_counter()
    run(n_timed)
    dt = time.perf_counter() - t0
    barrier.wait()
    out_q.put((idx, dt))


def reference_exec(steps: int, warmup: int, target_seconds: float):
    """The reference itself (unmodified modules, bytecode in oracle/_ref made by oracle/make_ref.py) on every host
    core: one env per process, `per_step` env.step calls per bench step and process."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness as rh
    ref_root = rh.COMPILED_REF if rh.available(rh.COMPILED_REF) else (rh.DEFAULT_REF if rh.available(rh.DEFAULT_REF) else None)
    if ref_root is None:
        return None
    cpus = host_cpus()
    Cn = len(cpus)
    per_step = max(1, int(round(target_seconds * 2000.0 / max(1, steps))))     # ~2.0-2.5 k env-steps/s/core measured
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(Cn + 1), ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(i, cpus[i], ref_root, warmup * per_step, steps * per_step, barrier, q),
                         daemon=True) for i in range(Cn)]
    for p in procs:
        p.start()
    barrier.wait(timeout=600)
    t0 = time.perf_counter()
    barrier.wait(timeout=1800)
    wall = time.perf_counter() - t0
    times = [q.get(timeout=60)[1] for _ in range(Cn)]
    for p in procs:
        p.join(timeout=30)
    total = Cn * steps * per_step
    return {"value": total / wall, "seconds": wall, "cores": Cn, "per_step": per_step, "total_env_steps": total,
            "slowest_worker_s": max(times), "fastest_worker_s": min(times), "ref_root": os.path.relpath(ref_root, ROOT)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_start = time.perf_counter()
    W, K = max(args.warmup, 3), args.steps
    ref = reference_exec(K, W, args.ref_seconds) if args.ref_kind in ("auto", "reference") else None
    # the C port beside it (>= 2 s of timed work): a far stronger CPU implementation of the same arithmetic, ours
    n_env = 1 << 15
    rate0, _, threads = cpu_run(n_env, 20, 3)
    port_steps = max(K, int(3.0 * rate0 / n_env))
    port_rate, port_dt, threads = cpu_run(n_env, port_steps, 3)
    port = {"value": port_rate, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_env} envs x {port_steps} steps, oracle/walker_oracle.c with OpenMP, {port_dt:.1f} s"}
    if ref is not None:
        value, dt, kind, cores = ref["value"], ref["seconds"], "reference", ref["cores"]
        sample = (f"the unmodified reference modules (bytecode in {ref['ref_root']}, oracle/make_ref.py) through their own "
                  f"make_env / PhysicsEnv.step, {ENV_ID} in3d: {cores} processes (one env each: the reference's Point "
                  f"registry is process-global), {ref['per_step']} env.step calls per bench step and process, "
                  f"{ref['total_env_steps']} env-steps in {dt:.1f} s; float32 U(-1,1) actions, make_env again on done "
                  f"(max_steps = {EPISODE_STEPS})")
        workload = (f"{ENV_ID} in3d=True, template auto-reset, U(-1,1) f32 actions; reference arm: one env per process on "
                    f"{cores} host cores, a bench step = {ref['per_step']} env.step calls per process (the GPU arm steps "
                    "2^20 envs per GPU per step)")
    else:
        value, dt, kind, cores, sample = port_rate, port_dt, "port", threads, port["sample"] + "; oracle/_ref absent"
        workload = (f"{ENV_ID} in3d=True, template auto-reset, U(-1,1) f32 actions; CPU sample of {n_env} envs per step "
                    "(the GPU arm steps 2^20 per GPU)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": 1e3 * dt / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "port": port,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "timed_region_s": dt, "wall_s": time.perf_counter() - t_start,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------
class Ctx:
    """Rank / device plumbing shared by the measurements."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.affinity = None
        self.allowed_cpus = host_cpus()
        if not args.no_affinity:
            from walker_gym_b200.host import bind_to_device
            self.affinity = bind_to_device(self.local, int(os.environ.get("LOCAL_WORLD_SIZE", self.world)))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, x: float):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(x)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def timed(self, fn, n: int, clocks: bool = False):
        """barrier + synchronize, n x fn(i) between two CUDA events on the current stream, barrier + synchronize;
        returns (ms, max over ranks) and, optionally, the NVML clock record of the region."""
        torch = self.torch
        self.barrier()
        sampler = ClockSampler(self.local) if clocks else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        self.barrier()
        rec = sampler.stop() if sampler else None
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        return (ms, rec) if clocks else ms

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def action_ring(ctx, E, M, n=16, seed=100):
    torch = ctx.torch
    g = torch.Generator(device=ctx.dev).manual_seed(seed + ctx.rank)
    return [(torch.rand(E, M, device=ctx.dev, generator=g) * 2 - 1) for _ in range(n)]


DUMP_BYTES = 63 * 10 ** 6      # a dump stays under 64 MB with its .npy headers


def dump_outputs(directory: str, outputs: dict, n_envs: int):
    """Write ``outputs`` ({name: (tensor, env axis)}) as ``directory/<name>.npy`` in float32.  If they do not fit in
    DUMP_BYTES, each keeps the envs of one fixed sample (seed 0, env order), so that two builds compare output for output."""
    import numpy as np
    import torch
    per_env = 4 * sum(t.numel() // n_envs for t, _ in outputs.values())
    keep = min(n_envs, DUMP_BYTES // per_env)
    idx = None
    if keep < n_envs:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n_envs, keep, replace=False)))
    os.makedirs(directory, exist_ok=True)
    for name, (t, axis) in outputs.items():
        t = t.float()
        if idx is not None:
            t = t.index_select(axis, idx.to(t.device))
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    ctx = Ctx(args)
    torch = ctx.torch
    from walker_gym_b200 import BatchedPhysicsEnv
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    W, K = max(args.warmup, 3), args.steps
    E = args.envs_per_gpu
    if args.generic:
        from walker_gym_b200 import _lib
        _lib.load().wg_force_generic(1)
    if args.config == 5:
        return run_rollout(args, ctx)
    if args.config == 6:
        return run_pkg(args, ctx)
    if args.config == 3 and args.steps_per_launch > 1:
        return run_multi(args, ctx)
    env_id = {"balance": ENV_ID, "box": "Box-v0", "legacy_box": "box", "quad": "quad_balance",
              "quad_chain": "quad_balance_chain"}.get(args.body, args.body)
    body, k_sub = env_id, 1
    if args.config == 4:          # the enlarged morphology: disconnected units (default), the connected chain, or walker.py's insect
        body, k_sub = (env_id if args.body in ("quad", "quad_chain", "insect") else "quad_balance"), 8
    if args.k_sub > 0:
        k_sub = args.k_sub

    max_steps = EPISODE_STEPS if args.config == 3 else 1000     # config 4: the reference's default
    env = BatchedPhysicsEnv(body, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                            track_stats=True, k_sub=k_sub, obs_layout=args.obs_layout, max_steps=max_steps)
    bytes_per_env_step = algorithmic_bytes(env.N, env.M)
    ring = action_ring(ctx, E, env.M)

    # early-episode window (labelled extra): the first steps after the template reset, every lane finite
    for t in range(3):
        env.step(ring[t % 16])
    ms_early = ctx.timed(lambda t: env.step(ring[t % 16]), 20)
    # steady state: >= PREROLL untimed env-steps whatever --warmup says, then the W warm-up steps of the contract
    for t in range(max(0, PREROLL - 23)):
        env.step(ring[t % 16])
    for t in range(W):
        env.step(ring[t % 16])
    ms, clocks = ctx.timed(lambda t: env.step(ring[t % 16]), K, clocks=True)
    if args.dump_outputs and rank == 0:
        # env.step returns views of these buffers: they hold the last timed step's results until the next step
        dump_outputs(args.dump_outputs, {"obs": (env.obs, 0 if args.obs_layout == "row" else 1),
                                         "reward": (env.reward, 0), "done": (env.done, 0)}, E)
    value = world * E * K / (ms * 1e-3)
    # a longer window right after the timed one
    long_n = 1000 if env.N <= 8 and k_sub == 1 else 100
    ms_long = ctx.timed(lambda t: env.step(ring[t % 16]), long_n)
    stats = env.episode_stats(all_reduce=True)       # the only collective: 8 doubles, off the timed path

    e2e = None
    if not args.no_e2e and args.obs_layout == "row":
        e2e = measure_e2e(ctx, env, args)
    sub = None
    if not args.no_sub and args.config == 3 and args.body == "balance" and not args.generic and args.obs_layout == "row":
        del ring
        sub = measure_sub_configs(ctx, args)

    if rank == 0:
        peak, peak_src = hbm_peak()
        per_launch_s = ms * 1e-3 / K
        achieved = E * bytes_per_env_step / per_launch_s / 1e9
        tr, tr_src = ncu_traffic_per_env_step() if (args.config == 3 and args.obs_layout == "row" and not args.generic
                                                    and args.body == "balance") else (None, None)
        kernel = {"balance": "wg::step_static_packed_kernel<TopoBalanceV0, in3d, row-major obs via TMA bulk store, packed "
                             "float4 state, L2 bulk prefetch, mass pattern [k,k,1,j] at compile time, programmatic dependent launch>",
                  "quad": "wg::step_units_kernel<TopoBalanceV0, in3d, P=4 lanes per env (one per Balance unit), row-major obs via TMA bulk store, MM=3>",
                  "quad_chain": "wg::step_units_kernel<TopoBalanceV0, ..., LINK=1> (4 linked Balance units, neighbour masses over warp shuffles)"
                  }.get(args.body if args.config == 3 or args.body in ("quad", "quad_chain") else "quad",
                        f"wg::step_static_packed_kernel<{args.body}, in3d, {env.state_layout} state>")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{body}" + (" (gym/optimized_walker.py create_balance_creature)" if args.body == "balance" else "") +
                                   f", in3d=True, {E} envs per GPU, 1 kernel launch per env-step, K_sub={k_sub}, template "
                                   f"auto-reset at max_steps = {max_steps}, reference semantics as written otherwise, U(-1,1) f32 actions from a 16-deep device ring; "
                                   f"{PREROLL} untimed pre-roll env-steps + {W} warm-up steps before the timed window (steady state)",
                       "baseline_config": args.config,
                       "envs_per_gpu": E, "global_envs": world * E, "state_layout": env.state_layout, "obs": (f"row-major [E,{env.obs_dim}] materialised" if args.obs_layout == "row"
                               else f"feature-major [{env.obs_dim},E] materialised"),
                       "l2": f"state+obs+actions per step = {E * bytes_per_env_step / 1e6:.0f} MB > 126 MB L2 "
                             "(inputs larger than L2, no flush needed)",
                       "parallelism": f"env-sharded x{world}, no data-path collective",
                       "cpu_affinity": ctx.affinity},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None if tr is None else tr * E, "traffic_source": tr_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": bytes_per_env_step,
                         "kernel": kernel, "kernel_us": per_launch_s * 1e6,
                         "window": f"{K} steps after {PREROLL} pre-roll + {W} warm-up steps",
                         "episode_period": {"steps": long_n, "kernel_us": ms_long * 1e3 / long_n,
                                            "frac": E * bytes_per_env_step / (ms_long * 1e-3 / long_n) / 1e9 / peak,
                                            "what": f"average over {long_n} env-steps right after the timed window (max_steps = {max_steps})"},
                         "early_episode": {"steps": 20, "kernel_us": ms_early * 1e3 / 20,
                                           "frac": E * bytes_per_env_step / (ms_early * 1e-3 / 20) / 1e9 / peak,
                                           "what": "the first steps after a template reset (every lane finite): NOT the headline"}},
            "e2e": e2e, "gpu_launches": K, "clocks": clocks, "sub_configs": sub,
            "episode_stats": {k: stats[k] for k in ("episodes", "return_mean", "length_mean")},
        }
        if args.config == 4:
            line["roofline"]["note"] = ("config 4 is fp32-issue bound, not HBM bound: 8 substeps x 20+ springs per env-step "
                                        "against 1485 bytes (SURVEY 7.5); the HBM fraction is reported for completeness")
        if not args.no_cpu_baseline and world == 1 and args.config == 3 and args.body == "balance":
            line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
        print(json.dumps(line), flush=True)
    ctx.close()


def measure_e2e(ctx, env, args):
    """End to end through the host-buffer path: every step uploads its pinned host actions and downloads observations,
    rewards and dones into pinned host memory.  Also measures, in the same run and with the same buffers, what the
    box's PCIe / host fabric gives plain device-to-host copies of those bytes: every rank at once (the ceiling of
    the e2e number at this rank count) and one rank at a time (the per-GPU link)."""
    torch = ctx.torch
    from walker_gym_b200 import HostStepPipeline
    from walker_gym_b200.host import pinned_empty
    E, dev, world = env.num_envs, ctx.dev, ctx.world
    Ke = args.e2e_steps
    h_act = pinned_empty((E, env.M))
    h_act.uniform_(-1, 1)
    slots = [(pinned_empty((E, env.obs_dim)), pinned_empty((E,)), pinned_empty((E,), dtype=torch.uint8)) for _ in range(2)]
    d_act = torch.empty(E, env.M, dtype=torch.float32, device=dev)
    d2h_bytes = E * (env.obs_dim * 4 + 4 + 1)
    h2d_bytes = E * env.M * 4

    # ---- the box's own ceiling for these bytes: plain cudaMemcpyAsync D2H of the result buffers, one stream per rank ----
    d_res = (torch.empty(E, env.obs_dim, device=dev), torch.empty(E, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))

    def d2h(i):
        for h, d in zip(slots[i & 1], d_res):
            h.copy_(d, non_blocking=True)
    for i in range(3):
        d2h(i)
    ms_all = ctx.timed(d2h, Ke)                              # every rank at once
    solo = []
    for r in range(world):                                   # one rank at a time
        ctx.barrier()
        if r == ctx.rank:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(Ke):
                d2h(i)
            e1.record()
            torch.cuda.synchronize()
            my_solo = d2h_bytes * Ke / (e0.elapsed_time(e1) * 1e-3) / 1e9
        ctx.barrier()
    solo = ctx.gather(my_solo)
    ceiling_gbs = world * d2h_bytes * Ke / (ms_all * 1e-3) / 1e9
    ceiling_steps = ceiling_gbs * 1e9 / d2h_bytes * E       # env-steps/s if the D2H wire were the only cost
    # the other direction, every rank at once (names the limiter: the links are symmetric, the host's write path is not)

    def h2d(i):
        for h, d in zip(slots[i & 1], d_res):
            d.copy_(h, non_blocking=True)
    for i in range(3):
        h2d(i)
    ms_h2d = ctx.timed(h2d, Ke)
    h2d_all_gbs = world * d2h_bytes * Ke / (ms_h2d * 1e-3) / 1e9
    # and what the host's own cores copy (rank 0, every allowed core, 512 MiB blocks), while the GPUs idle
    host_copy_gbs = None
    ctx.barrier()
    if ctx.rank == 0:
        try:
            saved = os.sched_getaffinity(0)
            os.sched_setaffinity(0, ctx.allowed_cpus)
            nthr = torch.get_num_threads()
            torch.set_num_threads(len(ctx.allowed_cpus))
            a = torch.empty(1 << 27, dtype=torch.float32)
            b = torch.empty(1 << 27, dtype=torch.float32)
            a.fill_(1.0); b.copy_(a)
            t0 = time.perf_counter()
            for _ in range(4):
                b.copy_(a)
            host_copy_gbs = 4 * 2 * a.numel() * 4 / (time.perf_counter() - t0) / 1e9
            del a, b
            torch.set_num_threads(nthr)
            os.sched_setaffinity(0, saved)
        except Exception:
            pass
    ctx.barrier()

    # ---- synchronous C-ABI call: upload, kernel, download back to back on one stream ----
    for _ in range(3):
        env.step_host(h_act, d_act, *slots[0])
    ms_sync = ctx.timed(lambda i: env.step_host(h_act, d_act, *slots[0]), Ke)
    sync_e2e = {"value": world * E * Ke / (ms_sync * 1e-3), "unit": UNIT, "steps": Ke,
                "what": "wg_step_host: upload, kernel and download back to back on one stream"}

    # ---- the same traffic double-buffered (HostStepPipeline): step t+1's upload + kernel overlap step t's download ----
    pipe = HostStepPipeline(env)
    for i in range(4):
        pipe.submit(h_act, *slots[i & 1])
    pipe.drain()

    def run_pipe(n, fn):
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        pipe.drain()                                         # blocks the host; the events bracket all pipeline work
        e1.record()
        ctx.barrier()
        return ctx.max_over_ranks(e0.elapsed_time(e1))
    ms_pipe = run_pipe(Ke, lambda i: pipe.submit(h_act, *slots[i & 1]))
    copy_value = world * E * Ke / (ms_pipe * 1e-3)
    # ---- zero-copy: the kernel writes its results into the mapped pinned buffers itself (no staging, no D2H copies) ----
    for i in range(4):
        pipe.submit_zero_copy(h_act, *slots[i & 1])
    pipe.drain()
    ms_zc = run_pipe(Ke, lambda i: pipe.submit_zero_copy(h_act, *slots[i & 1]))
    zc_value = world * E * Ke / (ms_zc * 1e-3)
    value, path = (zc_value, "zero_copy") if zc_value > copy_value else (copy_value, "copy_pipeline")
    e2e = {"value": value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "steps": Ke,
           "path": path,
           "what": "every step uploads its pinned host actions (wg_host_alloc by the CPU-bound rank) and delivers "
                   "observations, rewards and dones into pinned host memory; value = the faster of the two public paths "
                   "measured below (both move the same bytes over PCIe, which bounds them)",
           "copy_pipeline": {"value": copy_value, "unit": UNIT,
                             "what": "HostStepPipeline.submit: two streams and two device result slots overlap step t+1's "
                                     "upload + kernel with step t's cudaMemcpyAsync downloads"},
           "zero_copy": {"value": zc_value, "unit": UNIT,
                         "what": "HostStepPipeline.submit_zero_copy: the step kernel's TMA bulk stores write the observation "
                                 "rows (and reward / done) straight into the mapped pinned host buffers: no device staging, "
                                 "no download copy; the next step's upload overlaps the kernel"},
           "achieved_d2h_gbs": value * d2h_bytes / E / 1e9,
           "d2h_ceiling": {"all_ranks_gbs": ceiling_gbs, "env_steps_per_s": ceiling_steps, "per_rank_solo_gbs": solo,
                           "h2d_all_ranks_gbs": h2d_all_gbs, "host_memcpy_gbs": host_copy_gbs,
                           "what": f"plain cudaMemcpyAsync device->pinned host of the same {d2h_bytes} bytes per step, "
                                   f"{Ke} steps, one stream per rank: all {world} rank(s) at once / one rank at a time; "
                                   "h2d_all_ranks: the same buffers the other way, all ranks at once; host_memcpy: "
                                   "read+write rate of the host's own cores copying 512 MiB blocks (rank 0, GPUs idle)"},
           "frac_of_d2h_ceiling": value / ceiling_steps,
           "synchronous": sync_e2e}
    # the other usage mode: policy on the device -- observations stay in HBM, only reward/done go to the host
    Kd = max(Ke, 50)
    for i in range(4):
        pipe.submit(h_act, None, *slots[i & 1][1:])
    pipe.drain()
    ms_dp = run_pipe(Kd, lambda i: pipe.submit(h_act, None, *slots[i & 1][1:]))
    e2e["device_policy_mode"] = {"value": world * E * Kd / (ms_dp * 1e-3), "unit": UNIT,
                                 "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": E * 5, "steps": Kd,
                                 "what": "same pipeline with h_obs = None: observations stay on the device"}
    return e2e


def measure_sub_configs(ctx, args):
    """Short, driver-visible measurements of the other BASELINE configs with the same timing rules (pre-roll, CUDA
    events, max over ranks, clocks): each entry has kernel_us per env-step, env-steps/s for the whole job and the
    fraction of the measured HBM peak its algorithmic bytes amount to."""
    torch = ctx.torch
    from walker_gym_b200 import BatchedPhysicsEnv, StepGraph, _lib
    world, dev, rank = ctx.world, ctx.dev, ctx.rank
    peak, _ = hbm_peak()
    out = {}

    def entry(name, fn):
        try:
            out[name] = fn()
        except Exception as ex:                       # a sub-measurement must never take the headline down
            out[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()

    # ---- config 3 as written: 2^20 envs TOTAL, split over the GPUs (strong scaling), 1000-step rollout replayed from a
    # CUDA graph of 50 closed-loop steps so that the few-us kernel is not hidden behind Python + ctypes launch cost ----
    def strong():
        Es = args.strong_envs_per_gpu or (1 << 20) // world
        env = BatchedPhysicsEnv(ENV_ID, Es, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * Es,
                                track_stats=True, graph_safe=True, max_steps=EPISODE_STEPS)
        T = 50
        g = torch.Generator(device=dev).manual_seed(300 + rank)
        acts = torch.rand(T, Es, env.M, device=dev, generator=g) * 2 - 1
        sg = StepGraph(env, acts)
        for _ in range(max(3, PREROLL // T + 1)):
            sg.replay()
        n_rep = 20
        ms, clk = ctx.timed(lambda i: sg.replay(), n_rep, clocks=True)
        us = ms * 1e3 / (n_rep * T)
        b = algorithmic_bytes(env.N, env.M)
        # what a pure streaming kernel with the same read : write mix reaches at this (L2-resident) size, same replay
        lib = _lib.load()
        src = torch.zeros(32 * Es * 4, dtype=torch.float32, device=dev)
        dst = torch.zeros(32 * Es * 4, dtype=torch.float32, device=dev)
        pg = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            lib.wg_stream_probe(src.data_ptr(), dst.data_ptr(), Es, 7, 17, C.c_void_p(s.cuda_stream))
        torch.cuda.current_stream(dev).wait_stream(s)
        with torch.cuda.graph(pg):
            for _ in range(T):
                lib.wg_stream_probe(src.data_ptr(), dst.data_ptr(), Es, 7, 17,
                                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        for _ in range(3):
            pg.replay()
        ms_p = ctx.timed(lambda i: pg.replay(), n_rep)
        us_p = ms_p * 1e3 / (n_rep * T)
        return {"what": f"BASELINE config 3 as written: 2^20 envs in total = {Es} per GPU x {world} GPU(s), {n_rep * T}-step "
                        f"closed-loop rollout, {T} wg_step launches per CUDA-graph replay (StepGraph), template auto-reset "
                        f"at max_steps = {EPISODE_STEPS}",
                "scaling": "strong", "envs_per_gpu": Es, "steps": n_rep * T, "kernel_us": us,
                "value": world * Es / (us * 1e-6), "unit": UNIT,
                "frac_hbm": Es * b / (us * 1e-6) / 1e9 / peak,
                "stream_probe_us": us_p, "frac_of_stream_probe": us_p / us,
                "note": "at 131072 envs the 50 MB working set is L2-resident, so the HBM fraction can exceed 1; "
                        "frac_of_stream_probe compares with a pure streaming kernel of the same size and read : write mix",
                "clocks": clk}
    entry("3_strong", strong)

    def body_cfg(body, k_sub, steps, what, kernel):
        def run():
            E = args.envs_per_gpu
            env = BatchedPhysicsEnv(body, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                                    track_stats=True, k_sub=k_sub)
            ring = action_ring(ctx, E, env.M, n=4)
            for t in range(max(8, PREROLL // k_sub)):
                env.step(ring[t % 4])
            ms, clk = ctx.timed(lambda t: env.step(ring[t % 4]), steps, clocks=True)
            us = ms * 1e3 / steps
            b = algorithmic_bytes(env.N, env.M)
            return {"what": what, "envs_per_gpu": E, "steps": steps, "k_sub": k_sub, "kernel": kernel, "kernel_us": us,
                    "value": world * E / (us * 1e-6), "unit": UNIT, "algorithmic_bytes_per_env_step": b,
                    "frac_hbm": E * b / (us * 1e-6) / 1e9 / peak, "bound": "fp32 issue (8 substeps of bit-exact arithmetic per 1485+ bytes)",
                    "clocks": clk}
        return run
    entry("4_units", body_cfg("quad_balance", 8, 40, "BASELINE config 4 on four DISCONNECTED Balance units (N=16, S=20, M=8), 8 substeps",
                              "wg::step_units_kernel (one lane per unit)"))
    entry("4_connected", body_cfg("quad_balance_chain", 8, 40,
                                  "BASELINE config 4 on a CONNECTED enlarged body: four Balance units chained by bones (N=16, S=23, M=8), 8 substeps",
                                  "wg::step_units_kernel with link springs (neighbour masses over warp shuffles)"))

    # ---- T env-steps per launch (wg_step_multi) ----
    def multi():
        E, T = args.envs_per_gpu, 16
        env = BatchedPhysicsEnv(ENV_ID, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                                track_stats=True, state_layout="packed", max_steps=EPISODE_STEPS)
        g = torch.Generator(device=dev).manual_seed(500 + rank)
        ring = [(torch.rand(T, E, env.M, device=dev, generator=g) * 2 - 1) for _ in range(2)]
        res = (torch.empty(T, E, device=dev), torch.empty(T, E, dtype=torch.uint8, device=dev))
        for t in range(PREROLL // T):
            env.step_many(ring[t % 2], out=res)
        n = 20
        ms, clk = ctx.timed(lambda t: env.step_many(ring[t % 2], out=res), n, clocks=True)
        us = ms * 1e3 / (n * T)
        # the same launch with the actions generated in the kernel (sinusoidal CPG): no per-step HBM read at all
        from walker_gym_b200.actions import CPGActions
        cpg = CPGActions(amp=[0.8] * env.M, freq=[1.5 + 0.5 * m for m in range(env.M)], phase=[0.7 * m for m in range(env.M)])
        for t in range(4):
            env.step_many(cpg, n_steps=T, out=res)
        ms_g = ctx.timed(lambda t: env.step_many(cpg, n_steps=T, out=res), n)
        us_g = ms_g * 1e3 / (n * T)
        return {"what": f"{T} env-steps per launch (wg_step_multi, actions [T,E,M] known up front), Balance-v0, {E} envs per GPU",
                "steps": n * T, "kernel_us": us, "value": world * E / (us * 1e-6), "unit": UNIT,
                "in_kernel_cpg": {"kernel_us": us_g, "value": world * E / (us_g * 1e-6),
                                  "what": "actions generated in the kernel (CPGActions): the launch reads no action memory"},
                "bound": "fp32 / fp64 instruction issue (state read and written once per 16 env-steps)", "clocks": clk}
    entry("multi16", multi)

    # ---- config 5: PPO rollout collection, MLP policy + step kernel ----
    def rollout():
        from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
        E, T = 1 << 18, 32
        torch.manual_seed(7 + rank)
        env = BatchedPhysicsEnv(ENV_ID, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                                obs_layout="row", act_layout="row", graph_safe=True)
        pol = FeatureMajorMLP(env.obs_dim, env.M).to(dev)
        col = RolloutCollector(env, pol, T, fused=True, precision="fp32")
        for _ in range(max(3, PREROLL // T)):
            col.collect()
        n = 4
        ms, clk = ctx.timed(lambda i: col.collect(), n, clocks=True)
        us = ms * 1e3 / (n * T)
        return {"what": f"BASELINE config 5: PPO rollout collection, MLP {env.obs_dim}->64->64->{env.M} policy kernel (wg_policy_act, "
                        f"float32-grade) + step kernel + GAE, {E} envs per GPU, T={T} per CUDA-graph replay",
                "steps": n * T, "us_per_env_step": us, "value": world * E / (us * 1e-6), "unit": UNIT,
                "policy_kernel": POLICY_KERNELS[int(os.environ.get("WG_POLICY_TC", "2"))],
                "clocks": clk}
    entry("5", rollout)
    return out


def run_multi(args, ctx):
    """Next-row workload (SURVEY 8 f2): T env-steps per launch (wg_step_multi / BatchedPhysicsEnv.step_many) for
    actions known up front.  A bench step = one launch = --steps-per-launch env-steps of every env; value counts
    env-steps.  The state is read and written once per launch, so the kernel is bound by the instruction rate of
    the bit-exact arithmetic, not by HBM: the HBM fraction is reported for completeness."""
    torch, dist = ctx.torch, ctx.dist
    from walker_gym_b200 import BatchedPhysicsEnv
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    W, K, E, T = max(args.warmup, 3), args.steps, args.envs_per_gpu, args.steps_per_launch
    env_id = {"balance": ENV_ID, "box": "Box-v0", "legacy_box": "box"}.get(args.body, args.body)
    env = BatchedPhysicsEnv(env_id, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                            track_stats=True, k_sub=args.k_sub or 1, state_layout="packed", max_steps=EPISODE_STEPS)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    ring = [(torch.rand(T, E, env.M, device=dev, generator=g) * 2 - 1) for _ in range(4)]
    out = (torch.empty(T, E, device=dev), torch.empty(T, E, dtype=torch.uint8, device=dev))

    for t in range(max(W, PREROLL // T)):
        env.step_many(ring[t % 4], out=out)
    ms, clocks = ctx.timed(lambda t: env.step_many(ring[t % 4], out=out), K, clocks=True)
    stats = env.episode_stats(all_reduce=True)

    # ---- end to end through the host-buffer C-ABI call (wg_step_multi_host): pinned host actions [T,E,M] in,
    # last observation + per-step rewards / dones out, every launch ----
    e2e = None
    if not args.no_e2e:
        from walker_gym_b200.host import pinned_empty
        Ke = max(3, args.e2e_steps // 2)
        h_act = pinned_empty((T, E, env.M))
        h_act.uniform_(-1, 1)
        h_obs = pinned_empty((E, env.obs_dim))
        slots = [(torch.empty(T, E, env.M, device=dev), (torch.empty(T, E, device=dev), torch.empty(T, E, dtype=torch.uint8, device=dev)),
                  pinned_empty((T, E)), pinned_empty((T, E), dtype=torch.uint8)) for _ in range(2)]
        d_act, d_out, h_rew, h_done = slots[0]
        for _ in range(2):
            env.step_many_host(h_act, d_act, h_obs, h_rew, h_done, out=d_out)
        ms_sync = ctx.timed(lambda i: env.step_many_host(h_act, d_act, h_obs, h_rew, h_done, out=d_out), Ke)
        h2d, d2h = T * E * env.M * 4, E * env.obs_dim * 4 + T * E * 5
        e2e = {"value": world * E * T * Ke / (ms_sync * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": Ke, "what": f"wg_step_multi_host: one bench step = one {T}-env-step launch; uploads the pinned host action "
                                    "block, downloads the last observation and the per-step rewards / dones, back to back on one stream"}
        # open-loop mode: observations stay in HBM; HostStepPipeline.submit_many overlaps block i+1's upload and kernel
        # with block i's download (two streams, two staging slots; the kernels serialise: they share the env state)
        from walker_gym_b200 import HostStepPipeline
        pipe = HostStepPipeline(env)
        hres = [(slots[i][2], slots[i][3]) for i in range(2)]
        for i in range(2):
            pipe.submit_many(h_act, *hres[i & 1])
        pipe.drain()
        ctx.barrier()
        Kp = 2 * Ke
        t0 = time.perf_counter()
        for i in range(Kp):
            pipe.submit_many(h_act, *hres[i & 1])
        pipe.drain()
        ms_pipe = ctx.max_over_ranks((time.perf_counter() - t0) * 1e3)
        ctx.barrier()
        e2e["open_loop_mode"] = {"value": world * E * T * Kp / (ms_pipe * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                                 "d2h_bytes_per_step": T * E * 5, "steps": Kp,
                                 "what": "HostStepPipeline.submit_many (step_many on two streams with pinned-host copies around "
                                         "it): observations stay on the device, rewards / dones come back every launch; "
                                         "timed host-side across a full (host-blocking) drain"}
    if rank == 0:
        peak, peak_src = hbm_peak()
        bytes_per_launch_env = 48 * env.N + 8 * env.M + 8 + 36 * env.N + 4 * env.M + T * (4 * env.M + 5)
        per_launch_s = ms * 1e-3 / K
        achieved = E * bytes_per_launch_env / per_launch_s / 1e9
        line = {"metric": METRIC, "value": world * E * K * T / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{env_id}, in3d=True, {E} envs per GPU, {T} env-steps per launch (wg_step_multi: actions "
                                       f"[T,E,M] known up front, per-step reward / done, observation after the last step), "
                                       f"template auto-reset at max_steps = {EPISODE_STEPS}, U(-1,1) f32 actions from a 4-deep device ring of blocks",
                           "baseline_config": "next row f2", "envs_per_gpu": E, "global_envs": world * E,
                           "steps_per_launch": T, "us_per_env_step": per_launch_s * 1e6 / T,
                           "l2": f"state+obs+actions per launch = {E * bytes_per_launch_env / 1e6:.0f} MB > 126 MB L2"},
                "roofline": {"bound": "fp32 issue", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_env_launch": bytes_per_launch_env,
                             "kernel": "wg::step_multi_packed_kernel", "kernel_us": per_launch_s * 1e6},
                "e2e": e2e, "gpu_launches": K, "clocks": clocks,
                "episode_stats": {k: stats[k] for k in ("episodes", "return_mean", "length_mean")}}
        print(json.dumps(line), flush=True)
    ctx.close()


def run_pkg(args, ctx):
    """Next-row workload (SURVEY 8 f3): the package lineage's Environment.update_physics
    (gym/optimized_walker/env.py:135-184) on one of its own bodies, 2^20 independent copies per GPU.
    A step = one launch = --steps-per-launch updates of every env; value counts env-updates."""
    import numpy as np
    torch = ctx.torch
    import walker_gym_b200.optimized_walker as ow
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    W, K, E, T = max(args.warmup, 3), args.steps, args.envs_per_gpu, args.steps_per_launch
    env = ow.Environment(num_envs=E, device=str(dev), ground_level=-8.0)
    getattr(ow, args.pkg_body)(env)
    P, S = len(env._order), len(env.springs)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    env.vel.add_(torch.randn(env.vel.shape, device=dev, generator=g))
    for _ in range(W):
        env.update_physics(T)
    ms, clocks = ctx.timed(lambda i: env.update_physics(T), K, clocks=True)
    if rank == 0:
        peak, peak_src = hbm_peak()
        bytes_per_launch_env = 48 * P + 12 * P            # pos + vel read and written, old_a written
        per_launch_s = ms * 1e-3 / K
        achieved = E * bytes_per_launch_env / per_launch_s / 1e9
        line = {"metric": "env-updates/sec (whole box)", "value": world * E * K * T / (ms * 1e-3), "unit": "env-updates/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"package lineage Environment.update_physics, body {args.pkg_body} (P={P} points, "
                                       f"S={S} springs), {E} envs per GPU, {T} update(s) per launch, ground at -8, N(0,1) "
                                       "initial velocities", "baseline_config": "next row f3",
                           "l2": f"state per launch = {E * bytes_per_launch_env / 1e6:.0f} MB > 126 MB L2"},
                "roofline": {"bound": "hbm" if T == 1 else "fp32 issue", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_env_launch": bytes_per_launch_env,
                             "kernel": "wg::pkg_update_kernel", "kernel_us": per_launch_s * 1e6},
                "e2e": None, "gpu_launches": K, "clocks": clocks}
        if not args.no_cpu_baseline and world == 1:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import walker_oracle as wo
            threads = wo.set_threads(len(host_cpus()))
            n = 1 << 14
            system = {"points": [(float(p.m), tuple(map(float, p.pos)), (0.0, 0.0, 0.0), p.fixed) for p in env._order],
                      "springs": [(env._order.index(a), env._order.index(b), float(x), float(k), bool(st))
                                  for a, b, x, k, st in env.springs]}
            so, po, st = wo.make_l2_system(system), wo.make_l2_params(ground_level=-8.0), wo.l2_init_state(system, n)
            st["vel"] += np.random.default_rng(0).normal(0, 1, st["vel"].shape).astype(np.float32)
            wo.l2_step(so, po, st, 20)
            t0 = time.perf_counter()
            wo.l2_step(so, po, st, 2000)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n * 2000 / dt, "unit": "env-updates/s", "cores": threads, "kind": "port",
                                    "sample": f"{n} envs x 2000 updates, oracle wgo_l2_step (OpenMP), {dt:.1f} s"}
        print(json.dumps(line), flush=True)
    ctx.close()


def run_rollout(args, ctx):
    """BASELINE config 5: PPO rollout collection -- torch MLP policy (obs->64->64->M, tanh) + the step kernel,
    262144 envs per GPU, T=32 steps per CUDA-graph replay, episode-return statistics all-reduced over NCCL."""
    torch = ctx.torch
    from walker_gym_b200 import BatchedPhysicsEnv
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    E = args.envs_per_gpu if args.envs_per_gpu != (1 << 20) else (1 << 18)
    T = ROLLOUT_T
    torch.manual_seed(7 + rank)
    fused = args.policy != "torch"
    lay = "row" if (fused and args.obs_layout == "row") else "feature"
    env = BatchedPhysicsEnv(ENV_ID, E, dev, in3d=True, auto_reset="template", seed=1234, env_offset=rank * E,
                            obs_layout=lay, act_layout=lay, graph_safe=True)
    pol = FeatureMajorMLP(env.obs_dim, env.M).to(dev)
    col = RolloutCollector(env, pol, T, fused=fused, precision="tf32" if args.policy == "fused-tf32" else "fp32")
    n_roll = args.steps // T
    n_warm = max(3, args.warmup // T, PREROLL // T)
    for _ in range(n_warm):
        col.collect()
    ctx.barrier()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(n_roll):
        col.collect()
    stats = col.episode_stats(all_reduce=True)         # K3 + NCCL all-reduce of 8 doubles, once per timed region
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop()
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    steps = n_roll * T
    if rank == 0:
        line = {
            "metric": METRIC, "value": world * E * steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": n_warm * T, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"PPO rollout collection (BASELINE config 5): torch MLP policy {env.obs_dim}->64->64->{env.M} "
                                   f"(tanh, gaussian head, value head) + fused step kernel, {ENV_ID} in3d, {E} envs per GPU, "
                                   f"T={T} steps per CUDA-graph replay, GAE on device, {lay}-major obs/actions",
                       "policy": {"fused-fp32": "wg_policy_act: the torch module's weights evaluated by one CUDA kernel per step, "
                                                "error-compensated 3xTF32 products (float32-grade, 1e-5 vs torch fp32); kernel: "
                                                + POLICY_KERNELS[int(os.environ.get("WG_POLICY_TC", "2"))],
                                  "fused-tf32": "wg_policy_act with plain TF32 products and tanh.approx",
                                  "torch": "torch eager ops captured in the CUDA graph"}[args.policy],
                       "baseline_config": 5, "envs_per_gpu": E, "global_envs": world * E,
                       "parallelism": f"env-sharded x{world}; one NCCL all-reduce of 8 doubles (episode-return stats) per timed region"},
            "gpu_launches": n_roll * col.kernel_launches_per_rollout, "clocks": clocks,
            "episode_stats": {k: stats[k] for k in ("episodes", "return_mean", "length_mean")},
        }
        print(json.dumps(line), flush=True)
    ctx.close()


def probe_stream():
    """HBM rate of pure streaming kernels (wg_stream_probe) at several read : write mixes, 2^20 threads."""
    import torch
    from walker_gym_b200 import _lib
    lib, dev, n = _lib.load(), torch.device("cuda", 0), 1 << 20
    src = torch.zeros(32 * n * 4, dtype=torch.float32, device=dev)
    dst = torch.zeros(32 * n * 4, dtype=torch.float32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    out = {}
    for name, (R, W) in {"copy 16:16": (16, 16), "balance 7.5:16.8 (120 B read, 269 B written per env)": (7, 17),
                         "box 8:17.8": (8, 18), "read only 24:0": (24, 0), "write only 0:24": (0, 24)}.items():
        for _ in range(5):
            lib.wg_stream_probe(src.data_ptr(), dst.data_ptr(), n, R, W, stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            lib.wg_stream_probe(src.data_ptr(), dst.data_ptr(), n, R, W, stream)
        e1.record()
        torch.cuda.synchronize()
        out[name] = round(200 * n * 16 * (R + W) / (e0.elapsed_time(e1) * 1e-3) / 1e9, 1)
    print(json.dumps({"probe": "wg_stream_probe, 2^20 threads x 16-byte vectors, GB/s", "hbm_peak_measured": hbm_peak()[0], **out}))


def main():
    args = parse()
    if args.probe_stream:
        return probe_stream()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
