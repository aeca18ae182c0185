"""GPU: BatchedPhysicsEnv(nonfinite="keep" | "count" | "end") on every step-kernel family, against the C oracle.

"end" ends the episode of an env whose step reward is not finite (its state overflowed to inf / NaN), "count" keeps the
reference's dynamics and counts episodes with a non-finite return apart from the return statistics.  The oracle side
is tests/nonfinite_ref.py: the C oracle plus both rules restated in NumPy.  Equality is bit for bit (up to NaN
payload); large batches are followed on head / tail / first-wave slices, as in test_cuda_full_size.py.

A mutation this file catches: account_episode (wg_kernels.cuh) sending a finite return to nf_stats, or testing the
running return before adding the step's reward; epilogue_reduce ending episodes on a finite reward."""
import os

import numpy as np
import pytest

import golden_util as gu
import nonfinite_ref as nr
import walker_oracle as wo
from test_cuda_full_size import default_slices
from test_cuda_vs_oracle import spec_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def oracle_threads():
    old = int(wo.lib().wgo_get_max_threads())
    wo.set_threads(len(os.sched_getaffinity(0)))
    try:
        yield
    finally:
        wo.set_threads(old)


@pytest.fixture(autouse=True)
def clear_points():
    from walker_gym_b200 import Point
    Point.clear()
    yield
    Point.clear()


def _where(a, b):
    eq = (a == b) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == "f" else a == b
    bad = np.nonzero(~eq.reshape(eq.shape[0], -1).all(1))[0]
    return f"{bad.size} rows differ, first at slice row {bad[0] if bad.size else -1}"


class NFLock:
    """Oracle states of env slices [a, b) (env_offset = a) under one nonfinite mode, started from the env's initial
    template reset (Philox step index 0); step k of the env then has step index k + 1.  `gen`: take the actions from
    the in-kernel action source description (wo.gen_actions); `x64`: float64 actions (wo.step_x64)."""

    def __init__(self, env, spec, slices, *, mode, max_steps, seed, k_sub=1, gen=None, x64=False):
        import torch
        self.env, self.mode, self.gen, self.step_index = env, mode, gen, 1
        self.slices = list(slices)
        self.body = wo.make_body(spec)
        self.xb = wo.make_x64(spec) if x64 else None
        self.parts, self.last_obs = [], []
        for a, b in self.slices:
            prm = wo.make_params(in3d=env.in3d, auto_reset=2, max_steps=max_steps, k_sub=k_sub, seed=seed, env_offset=a)
            st = wo.init_state(self.body, b - a)
            if env.old_a is None:
                st.pop("old_a")
            if x64:
                st["mx64"], st["mx_weak"] = wo.init_x64(self.body, self.xb, b - a)
            prm.step_index = 0
            self.parts.append((a, b, prm, st, nr.new_stats(b - a)))
            self.last_obs.append(wo.reset(self.body, prm, st, mode=2))
        self.idx = torch.cat([torch.arange(a, b, device=DEV) for a, b in self.slices])
        self.rows = self.finite_rows = self.ended_nonfinite = self.done_count = 0
        self.check("obs at reset", env.obs, self.last_obs)

    def _split(self, t):
        out, k = [], 0
        for a, b in self.slices:
            out.append(t[k:k + b - a])
            k += b - a
        return out

    def check(self, what, got_dev, want_parts):
        got = self._split(got_dev[self.idx].cpu().numpy())
        for (a, b, *_), g, w in zip(self.parts, got, want_parts):
            g = g.astype(bool) if w.dtype == bool else g
            assert gu.same(g, w), f"{what}: slice [{a}, {b}) of {self.env.num_envs}: {_where(g, w)}"

    def step(self, action, obs=None, reward=None, done=None, what=""):
        """Step the oracle slices with the env's device actions [E, M] (None with `gen`) and compare the results the env
        returned for the same step (any may be None)."""
        acts = None if action is None else self._split(action[self.idx].cpu().numpy())
        outs = []
        for p, (a, b, prm, st, stats) in enumerate(self.parts):
            prm.step_index = self.step_index
            if self.gen is not None:
                act = wo.gen_actions(self.gen, st["steps"], self.body.n_muscle)
            else:
                act = acts[p]
            if self.xb is not None:
                out = nr.step(self.body, prm, st, None, mode=self.mode, stats=stats, xb=self.xb,
                              action64=np.ascontiguousarray(act, np.float64))
            else:
                out = nr.step(self.body, prm, st, act, mode=self.mode, stats=stats)
            d = out["done"].astype(bool)
            self.done_count += int(d.sum())
            self.ended_nonfinite += int((d & nr.nonfinite(out["reward"])).sum())
            self.rows += d.size
            self.finite_rows += int(np.isfinite(out["obs"]).all(1).sum())
            outs.append(out)
        for name, dev in (("obs", obs), ("reward", reward), ("done", done)):
            if dev is not None:
                want = [o[name].astype(bool) if name == "done" else o[name] for o in outs]
                self.check(f"{name} at step {self.step_index} {what}", dev, want)
        self.step_index += 1
        self.last_obs = [o["obs"] for o in outs]
        return outs

    def check_state(self, what="at the end"):
        env = self.env
        names = ["pos", "vel", "mx", "steps", "ep_ret", "fin_stats"] + (["nf_stats"] if env.nf_stats is not None else [])
        for a, b, prm, st, (ep, fin, nf) in self.parts:
            want = dict(st, ep_ret=ep, fin_stats=fin, nf_stats=nf)
            for k in names:
                g = getattr(env, k)[..., a:b].cpu().numpy()
                assert gu.same(g, want[k]), f"{k} {what}: slice [{a}, {b})"


def _env(body, E, mode, **kw):
    from walker_gym_b200 import BatchedPhysicsEnv
    args = dict(in3d=True, auto_reset="template", seed=1234, track_stats=True, max_steps=1000, nonfinite=mode)
    args.update(kw)
    return BatchedPhysicsEnv(body, E, DEV, **args)


def _act(env, g):
    import torch
    return torch.rand(env.num_envs, env.M, device=DEV, generator=g) * 2 - 1


def _assert_end_recovers(lock, overflows=True):
    if overflows:
        assert lock.ended_nonfinite > 0, "no episode ended on a non-finite reward: the test did not reach overflow"
    assert lock.finite_rows == lock.rows, "under 'end' every returned observation is finite"


# ---- "end" against the oracle, one test per kernel family --------------------------------------------------------------
def test_end_packed_balance_at_bench_shape():
    """Packed Balance-v0 (the headline kernel) at 2^20 envs, 1000-step episodes, 1010 steps: head, tail and first-wave
    slices every step, the state and both accumulators at the end."""
    import torch
    E = 1 << 20
    env = _env("Balance-v0", E, "end")
    assert env.state_layout == "packed"
    lock = NFLock(env, wo.BALANCE, default_slices(E, 8192), mode="end", max_steps=1000, seed=1234)
    g = torch.Generator(device=DEV).manual_seed(3)
    for t in range(1010):
        act = _act(env, g)
        obs, rew, done, _ = env.step(act)
        lock.step(act, obs, rew, done)
    lock.check_state()
    _assert_end_recovers(lock)
    assert bool(torch.isfinite(env.fin_stats).all()), "finite returns only in fin_stats"


# Balance-v0's spring graph with one more bone (2-3): no ahead-of-time kernel, so the packed layout compiles one at run time
JIT_SPEC = dict(wo.BALANCE, skeletons=list(wo.BALANCE["skeletons"]) + [(2, 3, {})])


def jit_creature():
    from walker_gym_b200 import Creature, Muscle, Point, Skeleton
    pts = [Point(m, list(p), [0, 0, 0]) for m, p, _ in JIT_SPEC["points"]]
    return Creature(pts, [Muscle(pts[i], pts[j]) for i, j, _ in JIT_SPEC["muscles"]],
                    [Skeleton(pts[i], pts[j]) for i, j, _ in JIT_SPEC["skeletons"]])


FAMILIES = {
    # name: (body, spec, env kwargs, k_sub, steps, setup)
    "box_packed": ("Box-v0", wo.BOX, {}, 1, 150, None),
    "balance_soa": ("Balance-v0", wo.BALANCE, {"state_layout": "soa"}, 1, 150, None),
    "balance_generic": ("Balance-v0", wo.BALANCE, {"state_layout": "soa"}, 1, 150, "generic"),
    "balance_x64": ("Balance-v0", wo.BALANCE, {"x64": True}, 1, 150, None),
    "jit_packed": (None, JIT_SPEC, {"state_layout": "packed"}, 1, 150, "jit"),
    "quad_units": ("quad_balance", spec_of("quad_balance"), {}, 8, 60, None),
    "quad_chain_units": ("quad_balance_chain", spec_of("quad_balance_chain"), {}, 8, 60, None),
    "quad_part": ("quad_balance", spec_of("quad_balance"), {}, 8, 60, "part"),
}


@pytest.fixture()
def knobs():
    from walker_gym_b200 import _lib
    lib = _lib.load()
    saved = []

    def set_(what):
        if what == "generic":
            saved.append(("generic", lib.wg_force_generic(1)))
        elif what == "part":
            saved.append((_lib.TUNE_PART, lib.wg_set_tuning(_lib.TUNE_PART, 4)))
    yield set_
    for k, v in reversed(saved):
        if k == "generic":
            lib.wg_force_generic(v)
        else:
            lib.wg_set_tuning(k, v)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_end_and_count_per_family(family, knobs):
    """Each family: 'end' against the oracle on a full batch of 4096 envs (+37 for a partial last CTA) through the
    overflow and the resets it causes; 'count' against 'keep' on the GPU: obs / reward / done bit-identical every step,
    and per env fin_stats[3] + nf_stats[0] and the length sums equal keep's fin_stats."""
    import torch
    from walker_gym_b200 import _lib
    body, spec, kw, k_sub, T, setup = FAMILIES[family]
    knobs(setup)
    E = 4096 + 37
    x64 = bool(kw.get("x64"))
    max_steps = 2 * T // 3            # episodes that overflowed finish (with a non-finite return) under keep / count
    mk = lambda mode: _env(body or jit_creature(), E, mode, k_sub=k_sub, max_steps=max_steps, **kw)     # noqa: E731
    env = mk("end")
    if setup == "jit":
        assert env.state_layout == "packed" and _lib.load().wg_packed_available(C_ref(env.topo)) == 2
    lock = NFLock(env, spec, [(0, E)], mode="end", max_steps=max_steps, seed=1234, k_sub=k_sub, x64=x64)
    keep, count = mk("keep"), mk("count")
    g = torch.Generator(device=DEV).manual_seed(11)
    for t in range(T):
        act = _act(env, g)
        if x64:
            act = act.double()
        outs = []
        for e in (env, keep, count):
            o, r, d, _ = e.step(act)
            outs.append((o.clone(), r.clone(), d.clone()))
        lock.step(act, *outs[0])
        for a, b, name in zip(outs[1], outs[2], ("obs", "reward", "done")):
            assert gu.same(b.cpu().numpy(), a.cpu().numpy()), f"count vs keep: {name} at step {t}"
    lock.check_state()
    overflows = family != "box_packed"
    _assert_end_recovers(lock, overflows)
    _assert_split_sums(keep, count, overflows)


def C_ref(x):
    import ctypes
    return ctypes.byref(x)


def _assert_split_sums(keep, count, overflows=True):
    kf, cf, cn = keep.fin_stats.cpu().numpy(), count.fin_stats.cpu().numpy(), count.nf_stats.cpu().numpy()
    assert np.array_equal(cf[3] + cn[0], kf[3]), "episode counts: finite + non-finite = keep"
    assert np.array_equal(cf[2] + cn[1], kf[2]), "episode lengths: finite + non-finite = keep"
    assert np.isfinite(cf).all()
    if overflows:
        assert cn[0].sum() > 0, "no non-finite episode finished: the test did not reach overflow"


def test_count_packed_balance_at_bench_shape():
    """'count' next to 'keep' at 2^20 envs for 1010 steps of 1000-step episodes: every step's obs / reward / done
    bit-identical, and the split of the episode statistics."""
    import torch
    E = 1 << 20
    keep, count = _env("Balance-v0", E, "keep"), _env("Balance-v0", E, "count")
    g = torch.Generator(device=DEV).manual_seed(5)
    bad = torch.zeros((), dtype=torch.int64, device=DEV)
    for t in range(1010):
        act = _act(keep, g)
        o1, r1, d1, _ = keep.step(act)
        o2, r2, d2, _ = count.step(act)
        same = lambda x, y: ((x == y) | (torch.isnan(x) & torch.isnan(y))).all()    # noqa: E731
        bad += (~(same(o1, o2) & same(r1, r2) & (d1 == d2).all())).to(torch.int64)
    assert int(bad) == 0, f"{int(bad)} steps differ between count and keep"
    _assert_split_sums(keep, count)
    s = count.episode_stats()
    assert s["episodes"] + s["nonfinite_episodes"] == keep.episode_stats()["episodes"]
    assert s["episodes"] == 0 or np.isfinite(s["return_mean"])


def test_end_quad_units_at_bench_shape():
    """Config 4's step_units_kernel, quad_balance and quad_balance_chain, at 2^20 envs and 8 substeps: 'end' against the
    oracle on head and tail slices for 60 steps (lanes overflow within 5-10 steps, so this crosses several ends)."""
    import torch
    E = 1 << 20
    for body in ("quad_balance", "quad_balance_chain"):
        env = _env(body, E, "end", k_sub=8)
        lock = NFLock(env, spec_of(body), [(0, 4096), (E - 4096, E)], mode="end", max_steps=1000, seed=1234, k_sub=8)
        g = torch.Generator(device=DEV).manual_seed(7)
        for t in range(60):
            act = _act(env, g)
            obs, rew, done, _ = env.step(act)
            lock.step(act, obs, rew, done, what=body)
        lock.check_state()
        _assert_end_recovers(lock)


def test_config4_as_benchmarked_stays_finite():
    """bench.py config 4 (quad_balance, 2^20 envs, 8 substeps, 1000-step episodes) under 'end' for 1010 steps: every
    returned observation is finite (one device-side accumulator, one sync at the end).  Under 'count' next to 'keep':
    the episode counts add up and the mean return of the finite episodes is finite."""
    import torch
    E = 1 << 20
    g = torch.Generator(device=DEV).manual_seed(9)
    end = _env("quad_balance", E, "end", k_sub=8)
    ok = torch.ones((), dtype=torch.bool, device=DEV)
    for t in range(1010):
        obs, _, _, _ = end.step(_act(end, g))
        ok &= torch.isfinite(obs).all()
    assert bool(ok), "a returned observation was not finite under nonfinite='end'"
    del end
    keep, count = _env("quad_balance", E, "keep", k_sub=8), _env("quad_balance", E, "count", k_sub=8)
    for t in range(1010):
        act = _act(keep, g)
        keep.step(act)
        count.step(act)
    sk, sc = keep.episode_stats(), count.episode_stats()
    assert sc["episodes"] + sc["nonfinite_episodes"] == sk["episodes"] > 0
    assert sc["episodes"] == 0 or np.isfinite(sc["return_mean"])


def test_end_step_many_tensor_and_cpg():
    """wg_step_multi (and its in-kernel CPG instance) under 'end': 16-step launches against the oracle.  The CPG alone
    does not overflow Balance-v0 within this horizon, so its run starts with two launches of random tensor actions;
    envs then overflow during the CPG launches, which must end them."""
    import torch
    from walker_gym_b200 import CPGActions
    E, T = 4096 + 37, 16
    for src in ("tensor", "cpg"):
        env = _env("Balance-v0", E, "end", state_layout="packed")
        cpg = CPGActions(amp=[0.8] * env.M, freq=[1.5 + 0.5 * m for m in range(env.M)], phase=[0.7 * m for m in range(env.M)])
        lock = NFLock(env, wo.BALANCE, [(0, E)], mode="end", max_steps=1000, seed=1234)
        g = torch.Generator(device=DEV).manual_seed(2)
        for k in range(10):
            gen = src == "cpg" and k >= 2
            if gen and lock.gen is None:
                lock.gen, lock.ended_nonfinite = cpg.describe(float(env.params.dt)), 0
            acts = torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1
            obs, rew, done = env.step_many(cpg if gen else acts, n_steps=T)
            for t in range(T):
                lock.step(None if gen else acts[t], None, rew[t], done[t], what=f"{src} launch {k}")
            lock.check(f"{src}: obs after launch {k}", obs, lock.last_obs)
        lock.check_state(src)
        _assert_end_recovers(lock)


def test_end_step_graph_replay():
    """StepGraph (a CUDA graph of 16 env.step calls) under 'end', replayed 8 times, against the oracle."""
    import torch
    from walker_gym_b200 import StepGraph
    E, T = 4096 + 37, 16
    env = _env("Balance-v0", E, "end", graph_safe=True)
    lock = NFLock(env, wo.BALANCE, [(0, E)], mode="end", max_steps=1000, seed=1234)
    g = torch.Generator(device=DEV).manual_seed(4)
    acts = torch.empty(T, E, env.M, device=DEV)
    sg = StepGraph(env, acts, keep_obs="all")
    for k in range(8):
        acts.copy_(torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1)
        sg.replay()
        for t in range(T):
            lock.step(acts[t], sg.obs[t], sg.rewards[t], sg.dones[t], what=f"replay {k}")
    lock.check_state()
    _assert_end_recovers(lock)


def test_rollout_collector_end_mode_fused_matches_two_launches():
    """RolloutCollector under a CUDA graph with nonfinite='end': fuse_step=True (one launch per env step, where the
    library has it) gives the bits of the two-launch path, including the split statistics."""
    import torch
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    E, T = (1 << 18) + 37, 32
    res = []
    for fuse in (False, True):
        env = _env("Balance-v0", E, "end", graph_safe=True, state_layout="packed")
        torch.manual_seed(0)
        pol = FeatureMajorMLP(env.obs_dim, env.M).to(DEV)
        col = RolloutCollector(env, pol, T, fuse_step=fuse, seed=5)
        for _ in range(3):
            out = col.collect()
        torch.cuda.synchronize()
        res.append(({k: v.clone() for k, v in out.items()}, env.fin_stats.clone(), env.nf_stats.clone(),
                    col.episode_stats(all_reduce=False)))
    (a, fa, na, sa), (b, fb, nb, sb) = res
    for k in a:
        assert gu.same(a[k].cpu().numpy(), b[k].cpu().numpy()), k
    assert gu.same(fa.cpu().numpy(), fb.cpu().numpy()) and gu.same(na.cpu().numpy(), nb.cpu().numpy())
    assert sa["nonfinite_episodes"] == sb["nonfinite_episodes"]
    assert bool(torch.isfinite(a["obs"]).all())


def test_stats_reduce_split_against_float64():
    """wg_stats_reduce_split at 2^20 + 37 envs: one kernel fills [fin sums, nf count, nf length, 0, 0]; rows 0-3 are the
    bits wg_stats_reduce gives."""
    import ctypes as C
    import torch
    from walker_gym_b200 import _lib
    lib = _lib.load()
    E = (1 << 20) + 37
    g = torch.Generator(device=DEV).manual_seed(1)
    fin = (torch.rand(4, E, device=DEV, generator=g) * 100).contiguous()
    nf = torch.floor(torch.rand(2, E, device=DEV, generator=g) * 50).contiguous()
    out, out_plain = torch.empty(8, dtype=torch.float64, device=DEV), torch.empty(8, dtype=torch.float64, device=DEV)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.wg_stats_reduce_split(fin.data_ptr(), nf.data_ptr(), E, out.data_ptr(), s) == 0
    assert lib.wg_stats_reduce(fin.data_ptr(), E, out_plain.data_ptr(), s) == 0
    want = torch.cat([fin.double().sum(1), nf.double().sum(1), torch.zeros(2, dtype=torch.float64, device=DEV)])
    o, w, p = out.cpu().numpy(), want.cpu().numpy(), out_plain.cpu().numpy()
    assert np.allclose(o, w, rtol=1e-12, atol=0), (o, w)
    assert o[4] == w[4] and o[5] == w[5] and o[6] == 0 and o[7] == 0      # integer-valued sums are exact
    assert np.array_equal(o[:4], p[:4]) and (p[4:] == 0).all()


def test_two_shards_sum_to_single_env():
    """Two env_offset shards of a 'count' job reduce to the statistics of the single env: counts exact, sums to float64
    rounding."""
    import torch
    from walker_gym_b200.dist import finalize_stats
    E, h = 8192 + 37, 4096
    whole = _env("Balance-v0", E, "count", max_steps=60)
    parts = [_env("Balance-v0", h, "count", max_steps=60), _env("Balance-v0", E - h, "count", max_steps=60, env_offset=h)]
    g = torch.Generator(device=DEV).manual_seed(8)
    for t in range(150):
        act = _act(whole, g)
        whole.step(act)
        parts[0].step(act[:h].contiguous())
        parts[1].step(act[h:].contiguous())
    vecs = []
    for p in parts:
        p.episode_stats()
        vecs.append(p._stats_out.clone())
    s1 = finalize_stats(vecs[0] + vecs[1], nonfinite=True)
    s0 = whole.episode_stats()
    assert s0["nonfinite_episodes"] > 0
    for k in ("episodes", "nonfinite_episodes"):
        assert s1[k] == s0[k], k
    for k in ("return_sum", "return_sqsum", "length_sum", "nonfinite_length_mean"):
        assert s1[k] == pytest.approx(s0[k], rel=1e-12), k


def test_rejections():
    """'end' with jitter resets, 'count' without statistics, and nf_stats without fin_stats at the ABI."""
    import ctypes as C
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv, _lib
    with pytest.raises(ValueError, match="jitter"):
        BatchedPhysicsEnv("Balance-v0", 64, DEV, auto_reset="jitter", nonfinite="end")
    with pytest.raises(ValueError, match="track_stats"):
        BatchedPhysicsEnv("Balance-v0", 64, DEV, track_stats=False, nonfinite="count")
    env = _env("Balance-v0", 64, "count", state_layout="soa")
    lib, b = _lib.load(), env._buf
    saved = b.fin_stats
    b.fin_stats = None
    try:
        rc = lib.wg_step(C.byref(env.topo), C.byref(env.params), C.byref(b), 64, None)
    finally:
        b.fin_stats = saved
    assert rc == -1 and b"nf_stats" in lib.wg_last_error_string()
    env.params.end_nonfinite, env.params.auto_reset = 1, 1
    rc = lib.wg_step(C.byref(env.topo), C.byref(env.params), C.byref(b), 64, None)
    assert rc == -1 and b"end_nonfinite" in lib.wg_last_error_string()
    torch.cuda.synchronize()
