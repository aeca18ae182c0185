"""GPU: the packed step kernel at the sizes and horizons bench.py measures, against the C oracle.

The other oracle tests run at sizes where every CTA of the step kernel is in the first wave and the horizon is a few
dozen steps.  Here: 2^20 envs for 1000 steps (BASELINE config 3 as benchmarked and at the reference's own max_steps),
the 7-CTA-per-SM instance that grids of (6, 7] waves run, 16 steps per launch, and programmatic dependent launch at
full size.  The oracle follows env slices [a, a + n) (built with env_offset = a, so env ids and Philox streams
coincide): the head, the tail (the last CTAs of the grid, where the L2-prefetch guard switches off and where PDL
overlaps a step with the next launch) and a slice across the end of the first wave.  Equality is bit for bit."""
import os
import re
import warnings

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SLICE = 1 << 14
PACKED_BLOCK = 128            # envs per CTA of step_static_packed_kernel (WG_PACKED_BLOCK)
MIN_BLOCKS = 6                # resident CTAs per SM it is compiled for (WG_PACKED_MIN_BLOCKS) for bodies of <= 4 masses
EPISODE_STEPS = 30            # bench.py's max_steps for config 3


def n_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def default_slices(E, n=SLICE, block=PACKED_BLOCK, per_sm=MIN_BLOCKS):
    """Head, tail, and a slice across the end of the first wave of CTAs (`per_sm` CTAs of `block` envs per SM) when it
    is clear of both."""
    wave = per_sm * n_sms() * block
    out = [(0, min(n, E))]
    if E > n:
        out.append((E - n, E))
    if n + n // 2 <= wave <= E - n - n // 2:
        out.append((wave - n // 2, wave + n // 2))
    return out


def _where(a, b):
    """First env (row of an [n, ...] pair) where a and b differ, as a string."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return f"shape {a.shape} vs {b.shape}"
    eq = (a == b) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == "f" else a == b
    bad = np.nonzero(~eq.reshape(eq.shape[0], -1).all(1))[0]
    return f"{bad.size} envs differ, first at slice row {bad[0]}" if bad.size else "equal"


class SliceLockstep:
    """One oracle state per env slice [a, a + n) of an env, built with env_offset = a; the env and the oracle start
    from the same initial reset (Philox step index 0), so step k of the run has step index k + 1.  The defaults are
    bench.py's config 3 (Balance-v0, one substep, template auto-reset, the packed kernel's 128-env CTAs); `block` is
    the step kernel's envs per CTA (failure messages name CTAs with it).  With `gen` (a wo.gen_actions description)
    the oracle takes each step's actions from the in-kernel action source instead of from the recorded device
    actions."""

    def __init__(self, env, slices, *, max_steps, seed, spec=wo.BALANCE, k_sub=1, auto_reset="template",
                 rand_sigma=0.1, in3d=True, block=PACKED_BLOCK, gen=None):
        import torch
        assert env.obs_layout == "row" and env.in3d == in3d and env.num_envs >= max(b for _, b in slices)
        self.env, self.slices, self.step_index = env, list(slices), 1
        self.block, self.gen = block, gen
        mode = {"jitter": 1, "template": 2}[auto_reset]
        self._prm_kw = dict(in3d=in3d, auto_reset=mode, max_steps=int(max_steps), k_sub=k_sub, rand_sigma=rand_sigma,
                            seed=seed)
        self.body = wo.make_body(spec)
        self.track = env.fin_stats is not None
        self.parts = []
        for a, b in self.slices:
            prm = wo.make_params(env_offset=a, **self._prm_kw)
            st = wo.init_state(self.body, b - a)
            if env.old_a is None:
                st.pop("old_a")
            prm.step_index = 0
            o = wo.reset(self.body, prm, st, mode=mode)
            ep = (np.zeros(b - a, np.float32), np.zeros((4, b - a), np.float32)) if self.track else (None, None)
            self.parts.append((a, b, prm, st, ep, o))
        self.idx = torch.cat([torch.arange(a, b, device=env.obs.device) for a, b in self.slices])
        self._pending = []
        self.nonfinite = 0               # obs rows of the slices seen non-finite so far
        self.done_count = 0
        self.obs_rows = 0                # obs rows compared so far, and how many of them were entirely finite
        self.finite_rows = 0
        self.check_obs(env.obs, "reset")

    def _split(self, t):
        out, k = [], 0
        for a, b in self.slices:
            out.append(t[k:k + b - a])
            k += b - a
        return out

    def _msg(self, a, what, where):
        E, b, B = self.env.num_envs, dict(self.slices)[a], self.block
        n_blocks = (E + B - 1) // B
        return f"{what}: slice [{a}, {b}) of {E} envs = CTAs [{a // B}, {(b - 1) // B}] of {n_blocks}: {where}"

    def restrict(self, slices):
        """Continue with sub-slices of a lockstep that follows the whole batch [0, E) (cheaper from here on)."""
        import torch
        (a0, b0, _, st, ep, o), = self.parts
        assert (a0, b0) == (0, self.env.num_envs)
        self.slices, self.parts = list(slices), []
        for a, b in self.slices:
            prm = wo.make_params(env_offset=a, **self._prm_kw)
            sub = {k: np.ascontiguousarray(v[..., a:b]) for k, v in st.items()}
            sep = (ep[0][a:b].copy(), np.ascontiguousarray(ep[1][:, a:b])) if self.track else (None, None)
            self.parts.append((a, b, prm, sub, sep, o[a:b]))
        self.idx = torch.cat([torch.arange(a, b, device=self.env.obs.device) for a, b in self.slices])

    def _count_obs(self, want):
        self.obs_rows += want.shape[0]
        self.finite_rows += int(np.isfinite(want).all(1).sum())

    def check_obs(self, obs, what):
        got = self._split(obs[self.idx].cpu().numpy())
        for (a, b, prm, st, ep, o), g in zip(self.parts, got):
            assert gu.same(g, o), self._msg(a, f"obs {what}", _where(g, o))
            self._count_obs(o)

    def record(self, action, obs=None, reward=None, done=None):
        """Gather the slice rows of the step the env has just been given -- its device actions [E, M] and results obs
        [E, D] / reward [E] / done [E] (each may be None) -- into device buffers.  No host synchronisation: steps
        recorded between two flush() calls run back to back on the device."""
        import torch
        self._pending.append({k: None if v is None else torch.index_select(v, 0, self.idx)
                              for k, v in (("action", action), ("obs", obs), ("reward", reward), ("done", done))})

    def flush(self, what=""):
        """Copy the recorded steps to the host, step every slice's oracle through them and compare bit for bit.
        Returns the host copies [(step index, {name: [slice rows]})]."""
        pending, self._pending = self._pending, []
        host = [{k: None if v is None else v.cpu().numpy() for k, v in r.items()} for r in pending]
        out_steps = []
        for got in host:
            acts = None if self.gen is not None else self._split(got["action"])
            split = {k: None if got[k] is None else self._split(got[k]) for k in ("obs", "reward", "done")}
            for p, (a, b, prm, st, ep, _) in enumerate(self.parts):
                prm.step_index = self.step_index
                act = acts[p] if acts is not None else wo.gen_actions(self.gen, st["steps"], self.body.n_muscle)
                out = wo.step(self.body, prm, st, act, want_info=False, ep_ret=ep[0], fin_stats=ep[1])
                self.parts[p] = (a, b, prm, st, ep, out["obs"])
                self.nonfinite += int((~np.isfinite(out["obs"]).all(1)).sum())
                self.done_count += int(out["done"].sum())
                if split["obs"] is not None:
                    self._count_obs(out["obs"])
                for k, want in (("obs", out["obs"]), ("reward", out["reward"]), ("done", out["done"].astype(bool))):
                    if split[k] is not None:
                        g = split[k][p].astype(bool) if k == "done" else split[k][p]
                        assert gu.same(g, want), self._msg(a, f"{k} at step {self.step_index} {what}", _where(g, want))
            out_steps.append((self.step_index, got))
            self.step_index += 1
        return out_steps

    def step(self, action, obs=None, reward=None, done=None, what=""):
        self.record(action, obs, reward, done)
        return self.flush(what)

    def check_state(self, what="at the end"):
        env = self.env
        names = ["pos", "vel", "mx", "steps"] + (["old_a"] if env.old_a is not None else []) + \
                (["ep_ret", "fin_stats"] if self.track else [])
        dev = {k: getattr(env, k) for k in names}
        for a, b, prm, st, ep, _ in self.parts:
            want = dict(st, ep_ret=ep[0], fin_stats=ep[1])
            for k in names:
                g = dev[k][..., a:b].cpu().numpy()
                assert gu.same(g, want[k]), self._msg(a, f"{k} {what}", _where(g.T if g.ndim == 2 else g,
                                                                                 want[k].T if want[k].ndim == 2 else want[k]))


def _env(E, **kw):
    from walker_gym_b200 import BatchedPhysicsEnv
    args = dict(in3d=True, auto_reset="template", seed=1234, track_stats=True, max_steps=EPISODE_STEPS)
    args.update(kw)
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, **args)
    assert env.state_layout == "packed" and env.obs_layout == "row"
    return env


@pytest.fixture(autouse=True)
def oracle_threads():
    """The oracle on every CPU of this process (its OpenMP team size is process-global: restored afterwards)."""
    old = int(wo.lib().wgo_get_max_threads())
    wo.set_threads(len(os.sched_getaffinity(0)))
    try:
        yield
    finally:
        wo.set_threads(old)


def _defaults_on():
    from walker_gym_b200 import _lib
    lib = _lib.load()
    val = {}
    for knob in (_lib.TUNE_PDL, _lib.TUNE_L2_PREFETCH):
        old = lib.wg_set_tuning(knob, 1)            # returns the value in effect before the call
        try:
            val[knob] = old
        finally:
            lib.wg_set_tuning(knob, old)
    assert val[_lib.TUNE_PDL] == 1 and val[_lib.TUNE_L2_PREFETCH] > 0, "PDL and the L2 prefetch are on by default"


def _assert_tail_covered(E, slices):
    """A slice covers the last 128 CTAs of the grid (and so its last env)."""
    n_blocks = (E + PACKED_BLOCK - 1) // PACKED_BLOCK
    assert any(b == E and a // PACKED_BLOCK <= n_blocks - 128 for a, b in slices), slices


class BackToBack:
    """Blocks of steps that run back to back on the device.  Each block starts behind a spin kernel (torch.cuda._sleep)
    that holds the stream while the host enqueues the whole block: producer kernel, step, gathers of the slice rows,
    next producer, next step, ... -- so every step is launched while the kernel before it is still in the queue or
    running, which is what programmatic dependent launch overlaps.  `queued` counts the blocks whose spin kernel was
    still running when the last launch of the block had been enqueued; the spin doubles after a block that was not."""

    def __init__(self, cycles=1 << 24):
        self.cycles, self.queued, self.blocks = cycles, 0, 0

    def run(self, n, launch):
        import torch
        torch.cuda._sleep(self.cycles)
        held = torch.cuda.Event()
        held.record()
        for t in range(n):
            launch(t)
        self.blocks += 1
        if not held.query():
            self.queued += 1
        else:
            self.cycles *= 2

    def check(self):
        assert self.blocks > 0 and self.queued >= self.blocks - 3, \
            f"only {self.queued} of {self.blocks} blocks ran back to back behind the spin kernel"


BLOCK = 25


def _run_back_to_back(env, lock, T, g, what=""):
    """T steps of U(-1, 1) actions (torch.rand: the producer kernel right before each step) in blocks of BLOCK."""
    import torch
    b2b = BackToBack()
    done_steps = []

    def launch(_):
        act = torch.rand(env.num_envs, env.M, device=DEV, generator=g) * 2 - 1
        obs, rew, done, _ = env.step(act)
        lock.record(act, obs, rew, done)
    for k in range(0, T, BLOCK):
        b2b.run(min(BLOCK, T - k), launch)
        done_steps += lock.flush(what)
    b2b.check()
    return done_steps


def test_config3_as_benchmarked_1000_steps():
    """bench.py config 3 (run_ours): Balance-v0, 2^20 envs, template auto-reset every EPISODE_STEPS, seed 1234, episode
    statistics, packed state, row-major obs, PDL and L2 prefetch on; 1000 steps of U(-1, 1) actions launched back to
    back, every step compared."""
    import torch
    _defaults_on()
    E = 1 << 20
    env = _env(E)
    slices = default_slices(E)
    assert len(slices) == 3
    _assert_tail_covered(E, slices)
    lock = SliceLockstep(env, slices, max_steps=EPISODE_STEPS, seed=1234)
    _run_back_to_back(env, lock, 1000, torch.Generator(device=DEV).manual_seed(3))
    lock.check_state()
    assert lock.done_count > 0


def test_reference_horizon_max_steps_1000():
    """The same at the reference's max_steps = 1000, for 1010 steps: lanes overflow to inf / NaN (the oracle's first
    non-finite lane appears near step 37); lanes that did not end early (non-finite ones never do) end at step
    1000, and their post-reset observations are finite again."""
    import torch
    E = 1 << 20
    env = _env(E, max_steps=1000)
    lock = SliceLockstep(env, default_slices(E), max_steps=1000, seed=1234)
    steps = _run_back_to_back(env, lock, 1010, torch.Generator(device=DEV).manual_seed(4))
    got = dict(steps)[1000]
    d = got["done"].astype(bool)
    assert d.sum() > 0 and np.isfinite(got["obs"][d]).all(), "the max_steps reset leads to finite states"
    lock.check_state()
    assert lock.nonfinite > 0, "the run reached non-finite states"


SEVEN_SIZES = ["2^17", "6*SMs*128+1", "7*SMs*128", "6*SMs*128"]


def seven_size(which):
    sms = n_sms()
    return {"2^17": 1 << 17, "6*SMs*128+1": 6 * sms * 128 + 1, "7*SMs*128": 7 * sms * 128, "6*SMs*128": 6 * sms * 128}[which]


_PROBE_BUILDERS = {}
_PROFILED = []


def register_probes(builder):
    """Adds builder() -> [(probe label, run)] to the one profiler session of this process (see kernel_names)."""
    _PROBE_BUILDERS[f"{builder.__module__}.{builder.__name__}"] = builder
    return builder


def kernel_names():
    """{probe label: name of the step or package-physics kernel that the probe's run launched}, or None when
    torch.profiler reports no kernel names.  One profiler session for the probes of every test module loaded in this
    process, on first use: a second session in the same process may see no device activity.  Every probe's objects
    are built before the session and each run launches exactly one such kernel, so the kernels are told apart by their
    launch order."""
    if _PROFILED:
        return _PROFILED[0]
    import torch
    from torch.profiler import ProfilerActivity, profile
    probes = [p for build in _PROBE_BUILDERS.values() for p in build()]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, run in probes:
            run()
            torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if re.search(r"step_\w*kernel|pkg_update\w*kernel", e.name)),
                key=lambda e: e.time_range.start)
    names = None
    if ev:
        assert len(ev) == len(probes), [e.name for e in ev]
        names = {label: e.name for (label, _), e in zip(probes, ev)}
    _PROFILED.append(names)
    return names


@register_probes
def _seven_cta_probes():
    import torch
    out = []
    for w in SEVEN_SIZES:
        e = _env(seven_size(w), graph_safe=True)
        a = torch.zeros(e.num_envs, e.M, device=DEV)
        out.append((f"step {w}", lambda e=e, a=a: e.step(a)))
    return out


@pytest.fixture(scope="module")
def step_kernel_minb():
    """{size id: MINB template argument of the step kernel one step at that size launched (0 = default)}, or None when
    torch.profiler reports no kernel names."""
    names = kernel_names()
    if names is None:
        return None
    out = {}
    for w in SEVEN_SIZES:   # demangled "...StepArgs<4, 5>, 7>(...)" (or "(int)7"), or mangled "...ELi7EEEvT3_"
        name = names[f"step {w}"]
        assert "step_static_packed_kernel" in name, (w, name)
        m = re.search(r"step_static_packed_kernel<.*,\s*(?:\(int\))?(\d+)\s*>\s*\(", name) or re.search(r"Li(\d+)EEEvT", name)
        out[w] = int(m.group(1)) if m else name
    return out


@pytest.mark.parametrize("which", SEVEN_SIZES)
def test_seven_cta_instance(which, step_kernel_minb):
    """launch_static_packed runs step_static_packed_kernel<..., MINB = 7> (72 registers) when the grid has (6, 7] CTAs
    per SM: 2^17 envs is bench.py's 3_strong shape on a 148-SM B200, built as 3_strong builds it (graph_safe, episode
    statistics, no old_a); the other sizes also keep old_a, so that its stores are checked too.  6*SMs*128 envs is the
    control on the 6-CTA side.  Eager steps against the oracle on every env for 100 steps, then a StepGraph of 32 steps
    replayed 32 times against the slices."""
    import torch
    from walker_gym_b200 import StepGraph
    sms = n_sms()
    E = seven_size(which)
    n_blocks = (E + PACKED_BLOCK - 1) // PACKED_BLOCK
    seven = 6 * sms < n_blocks <= 7 * sms
    if which in ("6*SMs*128+1", "7*SMs*128"):
        assert seven
    if which == "6*SMs*128":
        assert not seven
    env = _env(E, graph_safe=True, keep_old_a=which != "2^17")
    lock = SliceLockstep(env, [(0, E)], max_steps=EPISODE_STEPS, seed=1234)
    g = torch.Generator(device=DEV).manual_seed(E)
    # the kernel instance by name; torch.profiler without kernel names skips only that identification (a value
    # mutation of the MINB = 7 instance alone still fails the comparisons below)
    if step_kernel_minb is not None:
        assert step_kernel_minb[which] == (7 if seven else 0), (step_kernel_minb, E, n_blocks, sms)
    else:
        warnings.warn("torch.profiler reported no step kernel names: the MINB instance was not identified")
    _run_back_to_back(env, lock, 100, g)
    lock.check_state("after 100 eager steps")

    # the CUDA-graph path of 3_strong, continued from the same state, against the slices
    T = 32
    lock.restrict(default_slices(E))
    acts = torch.empty(T, E, env.M, device=DEV)
    sg = StepGraph(env, acts, keep_obs="all")
    assert int(env._counter.item()) == lock.step_index
    for r in range(32):
        acts.copy_(torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1)
        sg.replay()
        for t in range(T):
            lock.record(acts[t], sg.obs[t], sg.rewards[t], sg.dones[t])
        lock.flush(f"(graph replay {r})")
    lock.check_state("after 32 graph replays")
    assert lock.done_count > 0


def test_step_many_at_full_size():
    """wg_step_multi at 2^20 envs, 16 steps per launch, 63 launches, template auto-reset every EPISODE_STEPS: rewards and
    dones of every step, the observation after every launch and the state at the end, against the oracle slices."""
    import torch
    E, T = 1 << 20, 16
    env = _env(E, state_layout="packed")
    lock = SliceLockstep(env, default_slices(E), max_steps=EPISODE_STEPS, seed=1234)
    g = torch.Generator(device=DEV).manual_seed(6)
    res = (torch.empty(T, E, device=DEV), torch.empty(T, E, dtype=torch.uint8, device=DEV))
    for k in range(63):
        acts = torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1
        obs, rew, done = env.step_many(acts, out=res)
        for t in range(T):
            lock.record(acts[t], None, rew[t], done[t])
        lock.flush(f"(launch {k})")
        lock.check_obs(obs, f"after launch {k}")
    lock.check_state()
    assert lock.done_count > 0


def test_programmatic_dependent_launch_at_full_size():
    """With PDL on, at 2^20 envs, against the oracle on the head and tail slices:
    - 100 steps, each preceded immediately by a producer kernel that writes its actions (the dependency
      griddepcontrol.wait protects), enqueued back to back in blocks so that each step is launched behind a
      producer that has not run yet;
    - 4 replays of a StepGraph of 16 steps at 2^20 envs: step after step with nothing in between, so the CTAs of a
      step may be scheduled while the previous step's last wave is still writing the state."""
    import torch
    from walker_gym_b200 import StepGraph, _lib
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_PDL, 1)
    try:
        E = 1 << 20
        env = _env(E, max_steps=25, graph_safe=True)
        sl = default_slices(E)
        lock = SliceLockstep(env, [sl[0], sl[1]], max_steps=25, seed=1234)
        assert lock.slices[1][1] == E
        g = torch.Generator(device=DEV).manual_seed(11)
        base = torch.rand(E, env.M, device=DEV, generator=g) * 2 - 1
        acts = torch.empty(100, E, env.M, device=DEV)
        b2b = BackToBack()

        def launch(t):
            torch.mul(base, 1.0 - 0.015 * t, out=acts[t])
            obs, rew, done, _ = env.step(acts[t])
            lock.record(acts[t], obs, rew, done)
        for k in range(0, 100, BLOCK):
            b2b.run(BLOCK, lambda t: launch(k + t))
            lock.flush("(producer + step)")
        b2b.check()
        T = 16
        ga = torch.empty(T, E, env.M, device=DEV)
        sg = StepGraph(env, ga, keep_obs="all")
        for r in range(4):
            ga.copy_(torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1)
            sg.replay()
            for t in range(T):
                lock.record(ga[t], sg.obs[t], sg.rewards[t], sg.dones[t])
            lock.flush(f"(graph replay {r})")
        lock.check_state()
        assert lock.done_count > 0
    finally:
        lib.wg_set_tuning(_lib.TUNE_PDL, old)
