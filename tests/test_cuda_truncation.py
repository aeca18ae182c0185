"""GPU: BatchedPhysicsEnv(track_truncation=True) on every step-kernel family against the C oracle, wg_gae_trunc against
float64, and RolloutCollector(bootstrap_truncated="current").

The oracle side is tests/truncation_ref.py: the unchanged C oracle plus the truncation rule restated in NumPy.  Every env
starts from its template reset with a hand-built edge: every 5th env far below the fall threshold, every 3rd env one step
before its time limit (every 15th both: a fall on the time-limit step, which must count as terminated), so both kinds of
ending occur on the first step and the time limit keeps firing afterwards.  Equality is bit for bit (up to NaN payload),
and every run also steps a twin env without track_truncation whose obs / reward / done / state must be the same bits.

A mutation this file catches: epilogue_reduce setting trunc when a terminal clause coincides with the time limit, or
not at all; a family that does not write buf->truncated; the NF = false packed instance launched with truncated bound."""
import os

import numpy as np
import pytest

import golden_util as gu
import nonfinite_ref as nr
import truncation_ref as tr
import walker_oracle as wo
from test_cuda_full_size import default_slices
from test_cuda_nonfinite import JIT_SPEC, jit_creature
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


def _edge(st, max_steps, nonfinite_every=0):
    """The hand-built edges, in place on an oracle state [rows, E]."""
    st["pos"][1::3, ::5] = -1000.0
    st["steps"][::3] = max_steps - 1
    if nonfinite_every:
        st["vel"][0, ::nonfinite_every] = np.inf


class TLock:
    """Oracle states of env slices [a, b) (env_offset = a) from the env's initial template reset plus the hand-built
    edges, which are copied into the env (and its twin) with set_state."""

    def __init__(self, envs, spec, slices, *, max_steps, seed, k_sub=1, end_nonfinite=False, x64=False, nonfinite_every=0):
        import torch
        env = envs[0]
        self.env, self.end_nonfinite, self.step_index, self.gen = env, end_nonfinite, 1, None
        self.slices = list(slices)
        self.body = wo.make_body(spec)
        self.xb = wo.make_x64(spec) if x64 else None
        self.parts = []
        E = env.num_envs
        full = wo.init_state(self.body, E)
        prm0 = wo.make_params(in3d=env.in3d, auto_reset=2, max_steps=max_steps, k_sub=k_sub, seed=seed)
        prm0.step_index = 0
        wo.reset(self.body, prm0, full, mode=2)
        _edge(full, max_steps, nonfinite_every)
        for e in envs:
            e.set_state(pos=torch.from_numpy(full["pos"]).to(DEV), vel=torch.from_numpy(full["vel"]).to(DEV),
                        steps=torch.from_numpy(full["steps"]).to(DEV))
        for a, b in self.slices:
            prm = wo.make_params(in3d=env.in3d, auto_reset=2, max_steps=max_steps, k_sub=k_sub, seed=seed, env_offset=a)
            st = {k: np.ascontiguousarray(v[..., a:b]) for k, v in full.items()}
            st.pop("old_a")
            if x64:
                st["mx64"], st["mx_weak"] = wo.init_x64(self.body, self.xb, b - a)
            self.parts.append((a, b, prm, st, nr.new_stats(b - a)))
        self.idx = torch.cat([torch.arange(a, b, device=DEV) for a, b in self.slices])
        self.truncs = self.terms = self.final_rows = 0
        self.last_obs = None

    def _split(self, t):
        out, k = [], 0
        for a, b in self.slices:
            out.append(t[k:k + b - a])
            k += b - a
        return out

    def check(self, what, got_dev, want_parts, rows=None):
        got = self._split(got_dev[self.idx].cpu().numpy())
        for p, ((a, b, *_), g, w) in enumerate(zip(self.parts, got, want_parts)):
            g = g.astype(bool) if w.dtype == bool else g
            assert gu.same(g, w), f"{what}: slice [{a}, {b}) of {self.env.num_envs}"

    def step(self, action, obs=None, reward=None, done=None, truncated=None, what="", final_obs=None):
        """`final_obs`: the env's final_obs [E, D] (row-major view), compared on the rows whose done is set."""
        acts = None if action is None else self._split(action[self.idx].cpu().numpy())
        outs = []
        for p, (a, b, prm, st, stats) in enumerate(self.parts):
            prm.step_index = self.step_index
            act = wo.gen_actions(self.gen, st["steps"], self.body.n_muscle) if self.gen is not None else acts[p]
            if self.xb is not None:
                out = _step_x64(self.body, self.xb, prm, st, act)
            else:
                out = tr.step(self.body, prm, st, act, end_nonfinite=self.end_nonfinite, stats=stats)
            d, t = out["done"].astype(bool), out["truncated"].astype(bool)
            self.truncs += int(t.sum())
            self.terms += int((d & ~t).sum())
            outs.append(out)
        for name, dev in (("obs", obs), ("reward", reward), ("done", done), ("truncated", truncated)):
            if dev is not None:
                want = [o[name].astype(bool) if name in ("done", "truncated") else o[name] for o in outs]
                self.check(f"{name} at step {self.step_index} {what}", dev, want)
        if final_obs is not None:
            got = self._split(final_obs[self.idx].cpu().numpy())
            for (a, b, *_), g, o in zip(self.parts, got, outs):
                d = o["done"].astype(bool)
                self.final_rows += int(d.sum())
                assert gu.same(g[d], o["final_obs"][d]), f"final_obs at step {self.step_index} {what}: slice [{a}, {b})"
        self.step_index += 1
        self.last_obs = [o["obs"] for o in outs]
        return outs

    def check_state(self, what="at the end"):
        for a, b, prm, st, (ep, fin, _) in self.parts:
            want = dict(st, ep_ret=ep, fin_stats=fin)
            for k in ("pos", "vel", "mx", "steps") + (("ep_ret", "fin_stats") if self.xb is None else ()):
                g = getattr(self.env, k)[..., a:b].cpu().numpy()
                assert gu.same(g, want[k]), f"{k} {what}: slice [{a}, {b})"

    def both_kinds(self):
        assert self.truncs > 0, "no truncation happened"
        assert self.terms > 0, "no termination happened"


def _step_x64(body, xb, prm, st, act):
    """truncation_ref.step for float64 actions (wo.step_x64)."""
    max_steps, auto = int(prm.max_steps), int(prm.auto_reset)
    prm.max_steps, prm.auto_reset = tr.INT32_MAX, 0
    try:
        out = wo.step_x64(body, xb, prm, st, np.ascontiguousarray(act, np.float64), want_info=False)
    finally:
        prm.max_steps, prm.auto_reset = max_steps, auto
    term = out["done"].astype(bool)
    timelimit = st["steps"] >= max_steps
    done = term | timelimit
    out["final_obs"] = out["obs"].copy()
    if auto and done.any():
        obs_r = wo.reset(body, prm, st, mode=auto, mask=done.astype(np.uint8))
        out["obs"][done] = obs_r[done]
        st["mx64"][:, done] = np.array([xb.x0_d[m] for m in range(body.n_muscle)], np.float64)[:, None]
        st["mx_weak"][:, done] = 1
    out["done"], out["truncated"] = done.astype(np.uint8), (timelimit & ~term).astype(np.uint8)
    return out


def _env(body, E, *, track=True, **kw):
    from walker_gym_b200 import BatchedPhysicsEnv
    args = dict(in3d=True, auto_reset="template", seed=1234, track_stats=True, max_steps=1000, track_truncation=track)
    args.update(kw)
    return BatchedPhysicsEnv(body, E, DEV, **args)


def _act(env, g):
    import torch
    return torch.rand(env.num_envs, env.M, device=DEV, generator=g) * 2 - 1


def _same_dev(a, b):
    return gu.same(a.cpu().numpy(), b.cpu().numpy())


def _assert_twin(env, twin, what="at the end"):
    for k in ("pos", "vel", "mx", "steps", "ep_ret", "fin_stats"):
        x, y = getattr(env, k), getattr(twin, k)
        if x is not None:
            assert _same_dev(x, y), f"twin: {k} {what}"


FAMILIES = {
    # name: (body, spec, env kwargs, k_sub, steps, setup)
    "balance_packed": ("Balance-v0", wo.BALANCE, {}, 1, 40, None),
    "box_packed": ("Box-v0", wo.BOX, {}, 1, 40, None),
    "balance_soa": ("Balance-v0", wo.BALANCE, {"state_layout": "soa"}, 1, 40, None),
    "balance_soa_feature": ("Balance-v0", wo.BALANCE, {"state_layout": "soa", "obs_layout": "feature"}, 1, 40, None),
    "balance_tma": ("Balance-v0", wo.BALANCE, {"state_layout": "soa"}, 1, 40, "tma"),
    "balance_generic": ("Balance-v0", wo.BALANCE, {"state_layout": "soa"}, 1, 40, "generic"),
    "balance_x64": ("Balance-v0", wo.BALANCE, {"x64": True}, 1, 40, None),
    "jit_packed": (None, JIT_SPEC, {"state_layout": "packed"}, 1, 40, "jit"),
    "quad_units": ("quad_balance", spec_of("quad_balance"), {}, 8, 25, None),
    "quad_units_feature": ("quad_balance", spec_of("quad_balance"), {"obs_layout": "feature"}, 8, 25, None),
    "quad_chain_units": ("quad_balance_chain", spec_of("quad_balance_chain"), {}, 8, 25, None),
    "quad_part": ("quad_balance", spec_of("quad_balance"), {}, 8, 25, "part"),
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
        elif what == "tma":
            saved.append((_lib.TUNE_TMA, lib.wg_set_tuning(_lib.TUNE_TMA, 1)))
    yield set_
    for k, v in reversed(saved):
        if k == "generic":
            lib.wg_force_generic(v)
        else:
            lib.wg_set_tuning(k, v)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_truncation_per_family(family, knobs):
    """Each family on 4096 + 37 envs (4096 + 36 for the TMA kernel, which needs E % 4 == 0) with 9-step episodes:
    truncated / obs / reward / done every step against the oracle, the state at the end, and the twin's bits."""
    import torch
    body, spec, kw, k_sub, T, setup = FAMILIES[family]
    knobs(setup)
    E = 4096 + (36 if setup == "tma" else 37)
    max_steps = 9
    x64 = bool(kw.get("x64"))
    mk = lambda track: _env(body or jit_creature(), E, track=track, k_sub=k_sub, max_steps=max_steps, **kw)  # noqa: E731
    env, twin = mk(True), mk(False)
    assert twin.truncated is None and env.truncated is not None
    lock = TLock([env, twin], spec, [(0, E)], max_steps=max_steps, seed=1234, k_sub=k_sub, x64=x64)
    g = torch.Generator(device=DEV).manual_seed(11)
    for t in range(T):
        act = _act(env, g)
        if x64:
            act = act.double()
        o, r, d, info = env.step(act)
        o2, r2, d2, info2 = twin.step(act)
        assert "truncated" not in info2 and "final_obs" not in info2
        rm = (lambda x: x) if env.obs_layout == "row" else (lambda x: x.t())    # noqa: E731
        lock.step(act, rm(o), r, d, info["truncated"], final_obs=rm(info["final_obs"]))
        for a, b, name in ((o, o2, "obs"), (r, r2, "reward"), (d, d2, "done")):
            assert _same_dev(a, b), f"twin: {name} at step {t}"
    lock.check_state()
    _assert_twin(env, twin)
    lock.both_kinds()
    assert lock.final_rows > 0


def test_packed_balance_at_bench_shape():
    """The headline kernel at 2^20 envs with config 3's 30-step episodes, 100 steps, head / tail / first-wave slices;
    the twin runs the NF = false instance."""
    import torch
    E, T = 1 << 20, 100
    env, twin = _env("Balance-v0", E, max_steps=30), _env("Balance-v0", E, track=False, max_steps=30)
    assert env.state_layout == "packed"
    lock = TLock([env, twin], wo.BALANCE, default_slices(E, 8192), max_steps=30, seed=1234)
    g = torch.Generator(device=DEV).manual_seed(3)
    bad = torch.zeros((), dtype=torch.int64, device=DEV)
    for t in range(T):
        act = _act(env, g)
        o, r, d, info = env.step(act)
        lock.step(act, o, r, d, info["truncated"], final_obs=info["final_obs"])
        o2, r2, d2, _ = twin.step(act)
        same = lambda x, y: ((x == y) | (torch.isnan(x) & torch.isnan(y))).all()    # noqa: E731
        bad += (~(same(o, o2) & same(r, r2) & (d == d2).all())).to(torch.int64)
    assert int(bad) == 0, f"{int(bad)} steps differ from the twin"
    lock.check_state()
    _assert_twin(env, twin)
    lock.both_kinds()


@pytest.mark.parametrize("body", ["quad_balance", "quad_balance_chain"])
def test_quad_units_at_bench_shape(body):
    """Config 4's units kernels at 2^20 envs and 8 substeps, 12-step episodes, 30 steps on head and tail slices."""
    import torch
    E, T = 1 << 20, 30
    env, twin = _env(body, E, k_sub=8, max_steps=12), _env(body, E, track=False, k_sub=8, max_steps=12)
    lock = TLock([env, twin], spec_of(body), [(0, 4096), (E - 4096, E)], max_steps=12, seed=1234, k_sub=8)
    g = torch.Generator(device=DEV).manual_seed(7)
    for t in range(T):
        act = _act(env, g)
        o, r, d, info = env.step(act)
        lock.step(act, o, r, d, info["truncated"], what=body, final_obs=info["final_obs"])
        o2, r2, d2, _ = twin.step(act)
        assert _same_dev(o, o2) and _same_dev(r, r2) and _same_dev(d, d2), f"twin at step {t}"
    lock.check_state()
    lock.both_kinds()


@pytest.mark.parametrize("state_layout", ["packed", "soa"])
def test_with_nonfinite_end(state_layout):
    """nonfinite='end' with truncation: every 7th env starts with an infinite velocity (every 21st also one step before
    its time limit: a non-finite reward on the time-limit step counts as terminated), 60 steps of 40-step episodes."""
    import torch
    E, T = 4096 + 37, 60
    kw = dict(max_steps=40, nonfinite="end", state_layout=state_layout)
    env, twin = _env("Balance-v0", E, **kw), _env("Balance-v0", E, track=False, **kw)
    lock = TLock([env, twin], wo.BALANCE, [(0, E)], max_steps=40, seed=1234, end_nonfinite=True, nonfinite_every=7)
    g = torch.Generator(device=DEV).manual_seed(2)
    z = torch.zeros(E, env.M, device=DEV)
    o, r, d, info = env.step(z)
    first = lock.step(z, o, r, d, info["truncated"])[0]
    assert first["done"][::21].all() and not first["truncated"][::21].any()
    twin.step(z)
    for t in range(1, T):
        act = _act(env, g)
        o, r, d, info = env.step(act)
        lock.step(act, o, r, d, info["truncated"], final_obs=info["final_obs"])
        o2, r2, d2, _ = twin.step(act)
        assert _same_dev(o, o2) and _same_dev(r, r2) and _same_dev(d, d2), f"twin at step {t}"
    lock.check_state()
    _assert_twin(env, twin)
    lock.both_kinds()


def test_step_many_equals_steps():
    """step_many's truncated_out [T, E] is the per-step flag of T step calls, with tensor actions and with CPGActions;
    rewards / dones / obs agree as well."""
    import torch
    from walker_gym_b200 import CPGActions
    E, T = 4096 + 37, 16
    for src in ("tensor", "cpg"):
        many, single = _env("Balance-v0", E, max_steps=7, state_layout="packed"), _env("Balance-v0", E, max_steps=7,
                                                                                         state_layout="packed")
        lock = TLock([many, single], wo.BALANCE, [(0, E)], max_steps=7, seed=1234)
        cpg = CPGActions(amp=[0.8] * many.M, freq=[1.5, 2.0], phase=[0.0, 0.7])
        if src == "cpg":
            lock.gen = cpg.describe(float(many.params.dt))
        g = torch.Generator(device=DEV).manual_seed(4)
        for k in range(3):
            acts = torch.rand(T, E, many.M, device=DEV, generator=g) * 2 - 1
            trunc = torch.empty(T, E, dtype=torch.uint8, device=DEV)
            obs, rew, done = many.step_many(cpg if src == "cpg" else acts, n_steps=T, truncated_out=trunc)
            for t in range(T):
                if src == "cpg":
                    a = torch.from_numpy(wo.gen_actions(lock.gen, single.steps.cpu().numpy(), single.M)).to(DEV)
                else:
                    a = acts[t]
                o, r, d, info = single.step(a.contiguous())
                assert _same_dev(r, rew[t]) and _same_dev(d, done[t]), f"{src}: step {t} of launch {k}"
                assert _same_dev(info["truncated"].view(torch.uint8), trunc[t]), f"{src}: truncated at step {t} of launch {k}"
                lock.step(None if src == "cpg" else acts[t], None, rew[t], done[t], trunc[t], what=f"{src} launch {k}")
            assert _same_dev(obs, o), f"{src}: obs after launch {k}"
        lock.check_state(src)
        lock.both_kinds()


def test_step_graph_passes_truncation_through():
    """StepGraph of a tracking env: g.truncated [T, E] against the oracle over 4 replays."""
    import torch
    from walker_gym_b200 import StepGraph
    E, T = 4096 + 37, 8
    env = _env("Balance-v0", E, max_steps=5, graph_safe=True)
    lock = TLock([env], wo.BALANCE, [(0, E)], max_steps=5, seed=1234)
    acts = torch.empty(T, E, env.M, device=DEV)
    sg = StepGraph(env, acts, keep_obs="all")
    assert sg.truncated is not None
    g = torch.Generator(device=DEV).manual_seed(6)
    for k in range(4):
        acts.copy_(torch.rand(T, E, env.M, device=DEV, generator=g) * 2 - 1)
        sg.replay()
        for t in range(T):
            lock.step(acts[t], sg.obs[t], sg.rewards[t], sg.dones[t], sg.truncated[t], what=f"replay {k}")
    lock.check_state()
    lock.both_kinds()


def _gae_ref(rewards, values, dones, truncated, final, gamma, lam, clip):
    import torch
    san = lambda x: torch.nan_to_num(x.double(), nan=0.0, posinf=clip, neginf=-clip).clamp(-clip, clip)   # noqa: E731
    r = san(rewards)
    T, E = rewards.shape
    a = torch.zeros(E, dtype=torch.float64, device=DEV)
    want = torch.zeros(T, E, dtype=torch.float64, device=DEV)
    for t in range(T - 1, -1, -1):
        fv = torch.where(truncated[t], san(torch.where(truncated[t], final[t], 0.0)), 0.0)
        boot = torch.where(dones[t], fv, values[t + 1].double())
        delta = r[t] + gamma * boot - values[t].double()
        a = torch.where(dones[t], delta, delta + gamma * lam * a)
        want[t] = a
    return want


def test_gae_trunc_against_float64():
    """wg_gae_trunc against a float64 restatement; final_values rows of non-truncated steps poisoned with NaN / +-inf
    are ignored; a NaN or huge final value of a truncated step is sanitised; with no truncated step it is wg_gae."""
    import torch
    from walker_gym_b200.rollout import gae, gae_trunc
    T, E = 32, 3001
    g = torch.Generator(device=DEV).manual_seed(0)
    rewards = torch.randn(T, E, device=DEV, generator=g) * 50
    rewards[3, ::17] = float("nan")
    values = torch.randn(T + 1, E, device=DEV, generator=g)
    dones = torch.rand(T, E, device=DEV, generator=g) < 0.1
    truncated = dones & (torch.rand(T, E, device=DEV, generator=g) < 0.5)
    final = torch.randn(T, E, device=DEV, generator=g)
    final[~truncated] = float("nan")
    final[~truncated & (torch.rand(T, E, device=DEV, generator=g) < 0.5)] = float("inf")
    final[~truncated & (torch.rand(T, E, device=DEV, generator=g) < 0.3)] = float("-inf")
    nan_rows = truncated & (torch.rand(T, E, device=DEV, generator=g) < 0.2)
    final[nan_rows] = float("nan")
    final[truncated & ~nan_rows & (torch.rand(T, E, device=DEV, generator=g) < 0.1)] = 1e9
    assert nan_rows.any() and (truncated & (final == 1e9)).any()
    gamma, lam, clip = 0.99, 0.95, 1e3
    adv, ret = torch.zeros(T, E, device=DEV), torch.zeros(T, E, device=DEV)
    gae_trunc(rewards, values, dones.view(torch.uint8), truncated.view(torch.uint8), final, adv, ret, gamma, lam, clip)
    want = _gae_ref(rewards, values, dones, truncated, final, gamma, lam, clip)
    assert torch.isfinite(adv).all() and torch.isfinite(ret).all()
    scale = want.abs().max().item()
    assert (adv.double() - want).abs().max().item() < 1e-5 * scale
    assert (ret.double() - (want + values[:T].double())).abs().max().item() < 1e-5 * scale
    # the bootstrap matters: zeroing it (wg_gae) gives different advantages exactly where truncations are
    a0, r0 = torch.zeros(T, E, device=DEV), torch.zeros(T, E, device=DEV)
    gae(rewards, values, dones.view(torch.uint8), a0, r0, gamma, lam, clip)
    assert not torch.equal(a0, adv)
    # no truncated step: the bits of wg_gae
    none = torch.zeros(T, E, dtype=torch.uint8, device=DEV)
    a1, r1 = torch.zeros(T, E, device=DEV), torch.zeros(T, E, device=DEV)
    gae_trunc(rewards, values, dones.view(torch.uint8), none, final, a1, r1, gamma, lam, clip)
    assert torch.equal(a1, a0) and torch.equal(r1, r0)


def _gae_check(out, gamma=0.99, lam=0.95, clip=1e3):
    final = out["final_values"] if "final_values" in out else out["values"][:-1]
    want = _gae_ref(out["rewards"], out["values"], out["dones"], out["truncated"], final, gamma, lam, clip)
    scale = max(want.abs().max().item(), 1.0)
    assert (out["advantages"].double() - want).abs().max().item() < 1e-5 * scale


@pytest.mark.parametrize("mode", ["current", "final"])
@pytest.mark.parametrize("fused", [True, False])
def test_rollout_collector_bootstrap(fused, mode):
    """bootstrap_truncated='current' / 'final' with 6-step episodes over a 16-step horizon: graph replay gives the
    bits of the rollout without a graph; the advantages of both collectors (fused: wg_gae_trunc, torch ops: its
    restatement) are the float64 restatement's within the tolerance of the GAE tests; under 'final' the bootstrap
    values of truncated steps are the value pass over the final observation, not V(s_t)."""
    import torch
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    E, T = 4096 + 37, 16
    layout = "row" if fused else "feature"
    kw = dict(max_steps=6, graph_safe=True, obs_layout=layout, act_layout=layout, track_truncation=True)
    res = []
    for graph in (False, True):
        env = _env("Balance-v0", E, **kw)
        torch.manual_seed(0)
        pol = FeatureMajorMLP(env.obs_dim, env.M).to(DEV)
        col = RolloutCollector(env, pol, T, fused=fused, use_cuda_graph=graph, seed=5, bootstrap_truncated=mode,
                               fuse_step=True)
        assert not col.fused_step, "the fused policy + step kernel does not write the truncation flag"
        torch.manual_seed(1)
        outs = [{k: v.clone() for k, v in col.collect().items()} for _ in range(2)]
        torch.cuda.synchronize()
        res.append(outs)
        for out in outs:
            assert out["truncated"].any() and not (out["truncated"] & ~out["dones"]).any()
            assert ("final_values" in out) == (mode == "final")
            if mode == "final":
                tr_rows = out["truncated"]
                assert not torch.equal(out["final_values"][tr_rows], out["values"][:-1][tr_rows])
            _gae_check(out)
    if fused:                   # torch.randn of the torch-op collector is not replayed identically inside a graph
        for a, b in zip(*res):
            for k in a:
                if k == "final_values":         # specified on the done rows only (the others value stale rows)
                    assert _same_dev(a[k][a["dones"]], b[k][b["dones"]]), k
                else:
                    assert _same_dev(a[k], b[k]), k


def test_rollout_collector_none_is_unchanged():
    """bootstrap_truncated=None on a tracking env is the collector without the argument, bit for bit, and both equal
    the collector on an env without tracking."""
    import torch
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    E, T = 4096 + 37, 16
    res = []
    for track, arg in ((False, False), (True, False), (True, True)):
        env = _env("Balance-v0", E, track=track, max_steps=6, graph_safe=True, obs_layout="row", act_layout="row")
        torch.manual_seed(0)
        pol = FeatureMajorMLP(env.obs_dim, env.M).to(DEV)
        extra = dict(bootstrap_truncated=None) if arg else {}
        col = RolloutCollector(env, pol, T, seed=5, **extra)
        out = [{k: v.clone() for k, v in col.collect().items()} for _ in range(2)]
        assert "truncated" not in out[0]
        res.append(out)
    for other in res[1:]:
        for a, b in zip(res[0], other):
            for k in a:
                assert _same_dev(a[k], b[k]), k


def test_rejections():
    """A 4th out entry needs tracking, wrong shapes, final_obs in wg_step_multi, step_host of a tracking env, and
    wg_policy_step with the flag bound."""
    import ctypes as C
    import torch
    from walker_gym_b200 import _lib
    E = 256
    plain, env = _env("Balance-v0", E, track=False), _env("Balance-v0", E)
    o, r, d = torch.empty_like(env.obs), torch.empty_like(env.reward), torch.empty_like(env._done_u8)
    with pytest.raises(ValueError, match="track_truncation"):
        plain.step(None, out=(o, r, d, torch.empty(E, dtype=torch.uint8, device=DEV)))
    with pytest.raises(ValueError, match="out truncated"):
        env.step(None, out=(o, r, d, torch.empty(E + 1, dtype=torch.uint8, device=DEV)))
    with pytest.raises(ValueError, match="out truncated"):
        env.step(None, out=(o, r, d, torch.empty(E, dtype=torch.float32, device=DEV)))
    with pytest.raises(ValueError, match="truncated_out"):
        env.step_many(None, n_steps=4, truncated_out=torch.empty(3, E, dtype=torch.uint8, device=DEV))
    b = env._buf
    rc = _lib.load().wg_step_multi(C.byref(env.topo), C.byref(env.params), C.byref(b), E, 2, 2, None)
    assert rc == -1 and b"final_obs" in _lib.load().wg_last_error_string()
    tr_buf = torch.empty(E, dtype=torch.uint8, device=DEV)
    _, _, _, info = env.step(None, out=(o, r, d, tr_buf))
    assert info["truncated"] is tr_buf
    h = torch.zeros(E, env.M).pin_memory()
    with pytest.raises(ValueError, match="truncated"):
        env.step_host(h, torch.zeros(E, env.M, device=DEV))
    from walker_gym_b200.rollout import FeatureMajorMLP, FusedPolicy
    pol = FeatureMajorMLP(env.obs_dim, env.M).to(DEV)
    lib, b = _lib.load(), env._buf
    rc = lib.wg_policy_step(C.byref(FusedPolicy(pol)._struct()), C.byref(env.topo), C.byref(env.params), C.byref(b),
                            env.obs.data_ptr(), None, None, None, None, E, 1, 0, 0, 0, 0, None)
    assert rc == -2 and b"truncated" in lib.wg_last_error_string()
    torch.cuda.synchronize()
