"""GPU: float64-action stepping (wg_step_x64, the run-time-topology kernel with XArgs = X64Args) on rope-type muscles and
on the largest bodies the ABI admits, against the C oracle bit for bit (up to NaN payload and the sign of zero).

A muscle whose length is an np.float64 ("strong") evaluates its elastic term in double; the rope rule
(`if dx < 0 and string: f_size = 0`) holds there too, tested on the double dx.  The rope tests prove the rule fired:
while the actions keep every muscle strong, an oracle run with the muscles' rope flags cleared must end up elsewhere
in a stated share of envs.

The body-limit matrix: at 32 masses and 96 springs the per-block tile of the run-time-topology kernel (11 * N + M + 3
rows of 129 floats) reaches the device's opt-in shared memory per block.  Each case either matches the oracle or, in
x64 mode, is refused with ValueError when the env is built; the float32 cases are in
test_cuda_vs_oracle.py::test_maximum_and_minimum_body_sizes.  Every case names the kernel it ran through the shared
profiler session of test_cuda_full_size.py."""
import re

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo
from test_cuda_full_size import default_slices, kernel_names, n_sms, register_probes
from test_cuda_vs_oracle import _random_spec, rope_bodies, rope_creature

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GENERIC_BLOCK = 128                       # envs per CTA of step_generic_kernel (kBlock)
ROW_STATIC_SMEM = 1536                    # static shared memory of the row-major instances (ptxas -v, sm_100a)


@pytest.fixture(autouse=True)
def clear_points():
    from walker_gym_b200 import Point
    Point.clear()
    yield
    Point.clear()


def _rows_equal(a, b):
    """[n, ...] x [n, ...] -> [n] bool: row equal up to NaN payload and the sign of zero."""
    eq = (a == b) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == "f" else a == b
    return eq.reshape(eq.shape[0], -1).all(1)


class X64Lock:
    """Oracle states of env slices [a, b) (env_offset = a) in x64 mode, started from the env's initial reset (Philox
    step index 0, so step k has step index k + 1).  Each slice is stepped twice: with the body as built, and with the
    muscles' rope flags cleared (`diverged` marks the envs where the two runs' observations differed)."""

    def __init__(self, env, spec, slices, *, auto_reset, max_steps, seed, k_sub, integrator=0):
        self.env, self.slices, self.step_index = env, list(slices), 1
        self.body, self.xb = wo.make_body(spec), wo.make_x64(spec)
        self.plain = wo.make_body(spec)
        for m in range(self.plain.n_muscle):
            self.plain.sstring[m] = 0
        assert any(self.body.sstring[m] for m in range(self.body.n_muscle)), "the body has no rope-type muscle"
        self.parts = []
        for a, b in self.slices:
            pair = []
            for body in (self.body, self.plain):
                prm = wo.make_params(in3d=env.in3d, auto_reset=auto_reset, max_steps=max_steps, k_sub=k_sub, seed=seed,
                                     env_offset=a, integrator=integrator)
                st = wo.init_state(body, b - a)
                st["mx64"], st["mx_weak"] = wo.init_x64(body, self.xb, b - a)
                prm.step_index = 0
                obs = wo.reset(body, prm, st, mode=auto_reset)
                pair.append((prm, st))
            self.parts.append(pair)
            self._check(f"obs at reset [{a}, {b})", self._obs(a, b), obs)
        self.diverged = [np.zeros(b - a, bool) for a, b in self.slices]
        self.weak_seen = set()

    def _obs(self, a, b):
        o = self.env.obs
        return (o[a:b] if self.env.obs_layout == "row" else o[:, a:b].T).cpu().numpy()

    @staticmethod
    def _check(what, got, want):
        ok = _rows_equal(got, want) if got.ndim else np.array([gu.same(got, want)])
        bad = np.nonzero(~ok)[0]
        assert bad.size == 0, f"{what}: {bad.size} envs differ, first at slice row {bad[0]}"

    def step(self, act_rows, obs, reward, done, *, all_strong=False):
        """act_rows: the step's float64 actions as [E, M] (a view of the device tensor); compares everything the env
        returned and its whole state.  all_strong: assert that no muscle length was clamped."""
        env = self.env
        for (a, b), ((prm, st), (pprm, pst)), div in zip(self.slices, self.parts, self.diverged):
            act = np.ascontiguousarray(act_rows[a:b].cpu().numpy())
            prm.step_index = pprm.step_index = self.step_index
            out = wo.step_x64(self.body, self.xb, prm, st, act, want_info=False)
            pout = wo.step_x64(self.plain, self.xb, pprm, pst, act, want_info=False)
            div |= ~_rows_equal(out["obs"], pout["obs"])
            where = f"step {self.step_index}, slice [{a}, {b}) of {env.num_envs}"
            self._check(f"obs at {where}", (obs[a:b] if env.obs_layout == "row" else obs[:, a:b].T).cpu().numpy(), out["obs"])
            self._check(f"reward at {where}", reward[a:b].cpu().numpy(), out["reward"])
            self._check(f"done at {where}", done[a:b].cpu().numpy(), out["done"].astype(bool))
            for k in ("pos", "vel", "old_a", "mx", "mx64", "mx_weak"):
                self._check(f"{k} at {where}", getattr(env, k)[:, a:b].cpu().numpy().T, st[k].T)
            self._check(f"steps at {where}", env.steps[a:b].cpu().numpy(), st["steps"])
            self.weak_seen |= set(np.unique(st["mx_weak"]).tolist())
            if all_strong:     # after the step a muscle is weak only where a template auto-reset restored it
                reset = out["done"].astype(bool) & (prm.auto_reset == 2)
                assert ((st["mx_weak"] == 0) | reset[None]).all(), f"a muscle was clamped at {where}"
        self.step_index += 1

    def diverged_share(self):
        return float(np.concatenate(self.diverged).mean())


# (id, E, obs layout, act layout, auto-reset, k_sub, integrator)
ROPE_CASES = [
    ("ragged-row-template-k1", "ragged", "row", "row", "template", 1, 0),
    ("ragged-feature-jitter-k3", "ragged", "feature", "feature", "jitter", 3, 0),
    ("ragged-row-jitter-run2", "ragged", "row", "feature", "jitter", 1, 1),
    ("slices-feature-template-k3", "slices", "feature", "row", "template", 3, 0),
]
STRONG_STEPS, CLAMP_STEPS = 12, 12
STRONG_RANGE, CLAMP_RANGE = 0.5, 60.0     # +-0.5 a step never leaves [0.1, 1.5] * originx in 12 steps; +-60 clamps
MIN_DIVERGED = 0.5                        # share of envs where clearing the muscles' rope flags changes the run


@pytest.mark.parametrize("case", ROPE_CASES, ids=[c[0] for c in ROPE_CASES])
def test_rope_muscles_x64_match_oracle(case):
    """Rope-type muscles (and bones) of the two bodies of test_rope_type_springs_match_oracle, stepped with float64
    actions: first in a range that keeps every muscle strong (its length an np.float64: the double rope rule), then in
    one that clamps (weak: the float32 rule).  All envs of a ragged batch (2 * SMs * 128 + 1), or the head, tail and
    first-wave slices of 2^18 + 37 envs, bit for bit every step."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    _, size, obs_layout, act_layout, auto_reset, k_sub, integrator = case
    if size == "ragged":
        E = 2 * n_sms() * GENERIC_BLOCK + 1
        slices = [(0, E)]
    else:
        E = (1 << 18) + 37
        slices = default_slices(E, 8192, block=GENERIC_BLOCK, per_sm=2)
    ar = {"template": 2, "jitter": 1}[auto_reset]
    for b, body_s in enumerate(rope_bodies(np.random.default_rng(1000))):
        cr, spec = rope_creature(*body_s)
        env = BatchedPhysicsEnv(cr, E, DEV, in3d=True, auto_reset=auto_reset, max_steps=9, k_sub=k_sub, seed=5,
                                obs_layout=obs_layout, act_layout=act_layout, integrator=("run1", "run2")[integrator],
                                keep_old_a=True, x64=True)
        lock = X64Lock(env, spec, slices, auto_reset=ar, max_steps=9, seed=5, k_sub=k_sub, integrator=integrator)
        g = torch.Generator(device=DEV).manual_seed(17 + b)
        for t in range(STRONG_STEPS + CLAMP_STEPS):
            r = STRONG_RANGE if t < STRONG_STEPS else CLAMP_RANGE
            rows = (torch.rand(E, env.M, device=DEV, dtype=torch.float64, generator=g) * 2 - 1) * r
            act = rows if act_layout == "row" else rows.T.contiguous()
            obs, rew, done, _ = env.step(act)
            lock.step(rows, obs, rew, done, all_strong=t < STRONG_STEPS)
            if t == STRONG_STEPS - 1:
                share = lock.diverged_share()
                assert share >= MIN_DIVERGED, f"body {b}: the rope rule changed only {share:.1%} of the strong-muscle runs"
        assert lock.weak_seen == {0, 1}, f"body {b}: strong and weak muscles must both occur ({lock.weak_seen})"


def test_facade_rope_muscles_with_numpy_float64_actions():
    """PhysicsEnv on a user creature whose two muscles are rope-type, stepped 100 times with np.random.uniform actions
    (float64 ndarrays: the x64 path), against wo.step_x64 at E = 1: observation, reward, done, Point.pos, and the
    value and type of every Muscle.x."""
    from walker_gym_b200 import Creature, Muscle, PhysicsEnv, Point, Skeleton
    base = [(5, (-50, 100, 0)), (5, (50, 100, 0)), (1, (0, 0, 0)), (3, (0, 100, 0))]
    mus_s = [(0, 2, {"string": True}), (1, 2, {"string": True})]
    sks_s = [(0, 1, {}), (0, 3, {}), (1, 3, {})]
    pts = [Point(m, list(p), [0, 0, 0]) for m, p in base]
    cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in mus_s], [Skeleton(pts[i], pts[j], **kw) for i, j, kw in sks_s])
    spec = {"points": [(m, p, False) for m, p in base], "muscles": mus_s, "skeletons": sks_s}
    np.random.seed(11)
    env = PhysicsEnv(cr, in3d=True, device=DEV)               # reset(): 12 np.random.normal draws, point by point
    np.random.seed(11)
    nz = np.array([[np.random.normal(0, 0.1) for _ in range(3)] for _ in range(4)], np.float32)
    body, xb = wo.make_body(spec), wo.make_x64(spec)
    plain = wo.make_body(spec)
    plain.sstring[0] = plain.sstring[1] = 0
    prm = wo.make_params(in3d=True)
    st, pst = wo.init_state(body, 1), wo.init_state(plain, 1)
    for s in (st, pst):
        s["mx64"], s["mx_weak"] = wo.init_x64(body, xb, 1)
        wo.reset(body, prm, s, mode=1, noise=gu.soa(nz))
    diverged = False
    for t in range(100):
        a = np.random.uniform(-1, 1, 2)
        obs, rew, done, _ = env.step(a)
        out = wo.step_x64(body, xb, prm, st, a[None])
        pout = wo.step_x64(plain, xb, prm, pst, a[None])
        diverged = diverged or not gu.same(out["obs"], pout["obs"])
        assert obs.dtype == np.float64 and gu.same(obs[:-2], out["obs"][0, :-2].astype(np.float64)), t
        assert gu.same(obs[-2:], st["mx64"][:, 0]), t
        assert gu.same(np.float32(rew), out["reward"][0]) and done == bool(out["done"][0]), t
        assert gu.same(np.array([p.pos for p in env.creature.phys], np.float32), gu.aos(st["pos"], 4)[0]), t
        assert gu.same(np.array([float(m.x) for m in env.creature.muscles]), st["mx64"][:, 0]), t
        for m, w in zip(env.creature.muscles, st["mx_weak"][:, 0]):
            assert isinstance(m.x, np.float32 if w else np.float64), (t, type(m.x), w)
    assert diverged, "the rope rule never changed the run"


# ---- body limits ---------------------------------------------------------------------------------------------------
# (N, S, M): at N = 32 the largest and smallest muscle counts on each side of today's limits -- x64 23 / 24 (before its
# lengths left shared memory), float32 92 / 93 (row-major) and 95 / 96 (feature-major) -- and N = 16 with M = 68
LIMIT_BODIES = [(32, 96, 23), (32, 96, 24), (32, 96, 92), (32, 96, 93), (32, 96, 95), (32, 96, 96), (16, 96, 68)]
LIMIT_LAYOUTS = ["row", "feature"]


def tile_fits(N, M, layout):
    """Whether the run-time-topology kernel's tile fits a block on device 0 (opt-in limit less static shared memory)."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    return 4 * (11 * N + M + 3) * (GENERIC_BLOCK + 1) <= optin - (ROW_STATIC_SMEM if layout == "row" else 0)


def limit_creature(N, S, M):
    from walker_gym_b200 import Creature, DingPoint, Muscle, Point, Skeleton
    spec = _random_spec(np.random.default_rng(N * 1000 + M), N, S, M)
    Point.clear()
    pts = [DingPoint(m, list(p)) if f else Point(m, list(p), [0, 0, 0]) for m, p, f in spec["points"]]
    cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in spec["muscles"]],
                  [Skeleton(pts[i], pts[j], **kw) for i, j, kw in spec["skeletons"]])
    return cr, spec


def limit_env(N, S, M, layout, E=300, x64=True):
    from walker_gym_b200 import BatchedPhysicsEnv
    cr, spec = limit_creature(N, S, M)
    env = BatchedPhysicsEnv(cr, E, DEV, in3d=True, auto_reset="template", max_steps=5, k_sub=1, seed=3, obs_layout=layout,
                            keep_old_a=True, track_info=True, track_contacts=True, initial_reset=False, x64=x64)
    return env, spec


@register_probes
def _x64_limit_probes():
    """One x64 step of every limit case that builds (refused ones have no env); everything built before the session."""
    import torch
    out = []
    for N, S, M in LIMIT_BODIES:
        for layout in LIMIT_LAYOUTS:
            if not tile_fits(N, M, layout):
                continue
            env, _ = limit_env(N, S, M, layout, E=256)
            a = torch.zeros(env.num_envs, env.M, device=DEV, dtype=torch.float64)
            out.append((f"x64 {N}-{S}-{M} {layout}", lambda env=env, a=a: env.step(a)))
    return out


def _set_part(value):
    from walker_gym_b200 import _lib
    return _lib.load().wg_set_tuning(_lib.TUNE_PART, value)


@register_probes
def _float32_limit_probes():
    """One float32 step of each of test_maximum_and_minimum_body_sizes' limit cases, under its WG_TUNE_PART."""
    import torch
    from test_cuda_vs_oracle import BODY_LIMIT_CASES
    out = []
    for N, S, M, parts, k_sub, layout in BODY_LIMIT_CASES:
        env, _ = limit_env(N, S, M, layout, E=256, x64=False)
        a = torch.zeros(env.num_envs, env.M, device=DEV)

        def run(env=env, a=a, parts=parts):
            saved = _set_part(parts)
            try:
                env.step(a)
            finally:
                _set_part(saved)
        out.append((f"float32 {N}-{S}-{M} parts={parts} {layout}", run))
    return out


def test_float32_body_limit_kernels():
    """float32, k_sub = 1, partition automatic or off: the one-thread-per-env step_generic_kernel where its tile fits a
    block, step_part_kernel with two lanes per env where it does not (instead of a failed cudaFuncSetAttribute)."""
    from test_cuda_vs_oracle import BODY_LIMIT_CASES
    names = kernel_names()
    if names is None:
        pytest.skip("torch.profiler reports no kernel names")
    for N, S, M, parts, _, layout in BODY_LIMIT_CASES:
        name = names[f"float32 {N}-{S}-{M} parts={parts} {layout}"]
        if tile_fits(N, M, layout):
            assert "step_generic_kernel" in name and "X64Args" not in name, (N, M, parts, layout, name)
        else:
            assert "step_part_kernel" in name, (N, M, parts, layout, name)
            assert re.search(r"step_part_kernel<[^,]+,\s*(?:\(int\))?2\s*,|step_part_kernelILb[01]ELi2E", name), name


@pytest.mark.parametrize("layout", LIMIT_LAYOUTS)
@pytest.mark.parametrize("N,S,M", LIMIT_BODIES)
def test_x64_body_limits(N, S, M, layout):
    """x64 mode at the largest admitted bodies, float masses and a DingPoint, k_sub = 1: a body whose tile fits steps
    bit for bit with the oracle through step_generic_kernel<..., X64Args>; one that does not is refused when the env is
    built, with ValueError naming the shared-memory limit, never with a CUDA error at step time."""
    import torch
    if not tile_fits(N, M, layout):
        with pytest.raises(ValueError, match="shared memory per block"):
            limit_env(N, S, M, layout)
        return
    env, spec = limit_env(N, S, M, layout)
    names = kernel_names()
    if names is not None:
        name = names[f"x64 {N}-{S}-{M} {layout}"]
        assert "step_generic_kernel" in name and "X64Args" in name, name
    E = env.num_envs
    body, xb = wo.make_body(spec), wo.make_x64(spec)
    prm = wo.make_params(in3d=True, auto_reset=2, max_steps=5, seed=3)
    st = wo.init_state(body, E)
    st["mx64"], st["mx_weak"] = wo.init_x64(body, xb, E)
    rng = np.random.default_rng(N + M)
    for t in range(9):
        a = rng.uniform(-40, 40, (E, M))
        prm.step_index = env.step_count
        obs, rew, done, _ = env.step(torch.from_numpy(a).to(DEV))
        out = wo.step_x64(body, xb, prm, st, a)
        o = obs.cpu().numpy()
        assert gu.same(o if layout == "row" else o.T, out["obs"]), t
        assert gu.same(rew.cpu().numpy(), out["reward"]) and gu.same(done.cpu().numpy(), out["done"].astype(bool)), t
        for k in ("pos", "vel", "old_a", "mx", "mx64", "mx_weak", "steps"):
            assert gu.same(getattr(env, k).cpu().numpy(), st[k]), (k, t)
    assert 0 < st["mx_weak"].mean() < 1
