"""GPU: the config 4 and config 6 kernels of bench.py at the shapes it runs, against the C oracle.

Config 4 (4_units / 4_connected) steps quad_balance and quad_balance_chain with step_units_kernel at 2^20 envs and 8
substeps: one lane per Balance unit, 256 threads per CTA, so EB = 256 / R envs per CTA, EW = 32 / R envs per warp and
3 CTAs per SM; the linked form fetches the neighbour unit's link endpoint over warp shuffles.  With 8 substeps a lane
overflows to inf / NaN within 5-10 steps of a template reset and stays there until it is reset again (a jitter reset
keeps positions and velocities, so it never brings a lane back), and once every element of a row is NaN comparing it
proves nothing: every test here counts the slice rows it compared while they were entirely finite.

Config 6 runs the package lineage's Environment.update_physics at 2^20 envs: the run-time-topology kernel (box), the
point-partitioned kernel (insect, humanb; 128 / LP envs per CTA), the register-resident kernels (leg2, balance3) and
the run-time-topology kernel with more than 48 KB of shared memory.  The oracle follows env slices; equality is bit
for bit (up to NaN payload)."""
import ctypes as C
import os
import re
import warnings

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo
from test_cuda_full_size import EPISODE_STEPS, SliceLockstep, _run_back_to_back, default_slices, register_probes
from test_cuda_full_size import kernel_names as profiled_kernel_names
from test_cuda_vs_oracle import spec_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
UNITS_THREADS = 256            # threads per CTA of step_units_kernel (WG_UNITS_BLOCK)
UNITS_CTAS_PER_SM = 768 // 256  # WG_UNITS_THREADS_PER_SM / UNITS_THREADS
BENCH_BODIES = ["quad_balance", "quad_balance_chain"]
GROUND = -8.0                  # bench.py config 6: ow.Environment(ground_level=-8)
PKG_BLOCK = 128                # threads per CTA of the package-physics kernels (kBlock)


def units_geometry(R):
    """(envs per CTA, envs per warp) of step_units_kernel for bodies of R units."""
    return UNITS_THREADS // R, 32 // R


def units_spec(R, linked):
    """R Balance-v0 units side by side (quad_balance for R = 4), chained by link bones when `linked`."""
    from walker_gym_b200 import BODIES
    base = BODIES["balance_v0"]
    pts, mus, sks = [], [], []
    for u in range(R):
        off = 150.0 * (u - (R - 1) / 2)
        pts += [(float(m), (p[0] + off, p[1], p[2]), False) for m, p in base["points"]]
        mus += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["muscles"]]
    for u in range(R):
        sks += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["skeletons"]]
    if linked:
        sks += [(4 * u + 1, 4 * (u + 1), {}) for u in range(R - 1)]
    return {"points": pts, "muscles": mus, "skeletons": sks}


def units_env(R, linked, E, **kw):
    """R units in the SoA state layout, which the units kernel steps (R = 2 also has a run-time-compiled packed kernel)."""
    from walker_gym_b200 import BatchedPhysicsEnv, Creature, Muscle, Point, Skeleton
    spec = units_spec(R, linked)
    pts = [Point(m, list(p), [0, 0, 0]) for m, p, _ in spec["points"]]
    cr = Creature(pts, [Muscle(pts[i], pts[j]) for i, j, _ in spec["muscles"]],
                  [Skeleton(pts[i], pts[j]) for i, j, _ in spec["skeletons"]])
    env = BatchedPhysicsEnv(cr, E, DEV, state_layout="soa", **kw)
    assert env.state_layout == "soa" and env.obs_layout == "row"
    return env, spec


def bench_env(body, E, **kw):
    """As bench.py's body_cfg builds it: in3d, template auto-reset, seed 1234, episode statistics, 8 substeps, the
    reference's max_steps of 1000, row-major observations."""
    from walker_gym_b200 import BatchedPhysicsEnv
    args = dict(in3d=True, auto_reset="template", seed=1234, track_stats=True, k_sub=8)
    args.update(kw)
    env = BatchedPhysicsEnv(body, E, DEV, **args)
    assert env.state_layout == "soa" and env.obs_layout == "row"
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


@pytest.fixture(autouse=True)
def clear_points():
    """Creature and Environment constructors register points process-wide: start and leave with an empty registry."""
    import walker_gym_b200.optimized_walker as ow
    from walker_gym_b200 import Point
    Point.clear()
    ow.Point.clear()
    yield
    Point.clear()
    ow.Point.clear()


def _set_part(value):
    from walker_gym_b200 import _lib
    return _lib.load().wg_set_tuning(_lib.TUNE_PART, value)


@pytest.fixture()
def part_knob():
    """Sets WG_TUNE_PART (lanes per env of the package-physics kernels) for one test; automatic (-1) afterwards."""
    saved = _set_part(-1)
    yield _set_part
    _set_part(saved)


# ---- kernel instances by name ----------------------------------------------------------------------------------------
def template_ints(name, kernel):
    """The integer (and bool) template arguments of `kernel` in a demangled ("kernel<wg::T, true, 4, -1>(...)", ints
    maybe written "(int)-1") or mangled ("...kernelINS_1TELb1ELi4ELin1EEEv...") kernel name, in order; type arguments
    are left out.  None when the name is not an instance of `kernel`."""
    i = name.find(kernel + "<")
    if i >= 0:
        out = []
        for a in name[i + len(kernel) + 1:name.index(">(", i)].split(","):
            a = re.sub(r"^\(\w+\)", "", a.strip())
            if a in ("true", "false"):
                out.append(int(a == "true"))
            elif re.fullmatch(r"-?\d+", a):
                out.append(int(a))
        return out
    m = re.search(r"\d" + re.escape(kernel) + r"I(.*?)EEv", name)
    if m:
        return [int(v.replace("n", "-")) for v in re.findall(r"L[ib](n?\d+)E", m.group(1))]
    return None


def _pkg_env(build, E):
    import walker_gym_b200.optimized_walker as ow
    env = ow.Environment(num_envs=E, device=DEV, ground_level=GROUND)
    build(env)
    return env


def _random_pkg_body(env, seed=4, P=32, S=96):
    """A random system at the ABI limits (DingPoints, rope-type springs, explicit rest lengths) in an Environment."""
    from test_cuda_pkg import random_system
    system = random_system(np.random.default_rng(seed), P, S)
    pts = [(env.add_ding_point if ding else env.add_point)(m, pos, v) for m, pos, v, ding in system["points"]]
    for i, j, x, k, string in system["springs"]:
        env.add_spring(pts[i], pts[j], x=x, k=k, string=string)


def _pkg_builders():
    import walker_gym_b200.optimized_walker as ow
    return {"box": ow.box, "insect": ow.insect, "humanb": ow.humanb, "leg2": ow.leg2, "balance3": ow.balance3,
            "random32": _random_pkg_body}


# (probe, R, linked) of the config 4 tests and (probe, body, WG_TUNE_PART) of the config 6 tests
UNIT_PROBES = [(f"units R={R} {'linked' if ln else 'disconnected'}", R, ln) for R in (2, 4, 8) for ln in (False, True)]
PKG_PROBES = [("pkg box", "box", -1), ("pkg insect", "insect", -1), ("pkg humanb", "humanb", -1),
              ("pkg insect LP=8", "insect", 8), ("pkg leg2", "leg2", -1), ("pkg balance3", "balance3", -1),
              ("pkg random32 parts=0", "random32", 0)]


@register_probes
def _bench_shape_probes():
    """One step / update of every kernel instance these tests claim, everything built here (before the session)."""
    import torch
    from walker_gym_b200 import Point
    probes = []

    def step(env):
        a = torch.zeros(env.num_envs, env.M, device=DEV)
        return lambda: env.step(a)
    for body in BENCH_BODIES:
        probes.append((body, step(bench_env(body, 4096))))
    for label, R, linked in UNIT_PROBES:
        probes.append((label, step(units_env(R, linked, 1000, in3d=True, auto_reset="template", k_sub=8)[0])))
    Point.clear()

    def update(env, part):
        def run():
            saved = _set_part(part)
            try:
                env.update_physics(1)
            finally:
                _set_part(saved)
        return run
    builders = _pkg_builders()
    for label, body, part in PKG_PROBES:
        probes.append((label, update(_pkg_env(builders[body], 1000), part)))
    return probes


@pytest.fixture(scope="module")
def kernel_names():
    return profiled_kernel_names()


def assert_units_instance(kernel_names, probe, R, linked):
    """The probe ran step_units_kernel<TopoBalanceV0 (the Balance-v0 mass pattern), in3d, R, row-major, 3, 256, LA, LB>:
    (LA, LB) = (1, 0) for the linked form, no link arguments (-1, -1) for disconnected units."""
    if kernel_names is None:
        warnings.warn("torch.profiler reported no kernel names: the step kernel instance was not identified")
        return
    name = kernel_names[probe]
    args = template_ints(name, "step_units_kernel")
    assert args is not None, f"{probe} ran {name}, not step_units_kernel"
    in3d, P, rowmajor, mm, kb, la, lb = args
    assert (in3d, P, rowmajor, kb) == (1, R, 1, UNITS_THREADS), name
    assert (la, lb) == ((1, 0) if linked else (-1, -1)), name
    assert "TopoBalanceV0" in name and mm == 3, name


def assert_pkg_instance(kernel_names, probe, kernel, lp=None, topo=None):
    if kernel_names is None:
        warnings.warn("torch.profiler reported no kernel names: the update_physics kernel instance was not identified")
        return
    name = kernel_names[probe]
    assert re.search(r"\b" + kernel + r"\b", name) or re.search(r"\d" + kernel + r"[IE]", name), \
        f"{probe} ran {name}, not {kernel}"
    if lp is not None:
        assert template_ints(name, kernel) == [lp], name
    if topo is not None:
        assert topo in name, name


def test_template_ints_reads_both_name_forms():
    assert template_ints("void wg::step_units_kernel<wg::TopoBalanceV0, true, 4, true, 3, 256, -1, -1>"
                         "(wg::UnitsArgs<wg::TopoBalanceV0, 3>)", "step_units_kernel") == [1, 4, 1, 3, 256, -1, -1]
    assert template_ints("void wg::step_units_kernel<wg::TopoBalanceV0, true, (int)4, true, (int)3, (int)256, (int)1, "
                         "(int)0>(wg::UnitsArgs<wg::TopoBalanceV0, 3>)", "step_units_kernel") == [1, 4, 1, 3, 256, 1, 0]
    assert template_ints("_ZN2wg17step_units_kernelINS_11TopoBalanceELb0ELi2ELb0ELi0ELi256ELin1ELin1EEEvNS_9UnitsArgsIT_"
                         "XT3_EEE", "step_units_kernel") == [0, 2, 0, 0, 256, -1, -1]
    assert template_ints("_ZN2wg22pkg_update_part_kernelILi4EEEvNS_11PkgPartArgsE", "pkg_update_part_kernel") == [4]
    assert template_ints("void wg::pkg_update_part_kernel<8>(wg::PkgPartArgs)", "pkg_update_part_kernel") == [8]
    assert template_ints("void wg::pkg_update_kernel(wg::PkgArgs)", "pkg_update_part_kernel") is None


# ---- config 4: step_units_kernel -------------------------------------------------------------------------------------
def _assert_units_tail(E, R, slices):
    """A slice ends at the last env and covers the whole last CTA."""
    EB, _ = units_geometry(R)
    last_cta = (E - 1) // EB
    assert any(b == E and a <= last_cta * EB for a, b in slices), (E, slices)


def check_episode_stats(env):
    """episode_stats() (stats_reduce_kernel: one CTA looping over every env) against a float64 sum of the host copy of
    fin_stats: episode count and length sum exactly, return sums to rtol 1e-12, NaN exactly where a float64 sum is NaN.
    Returns the host fin_stats."""
    fin = env.fin_stats.cpu().numpy()
    want = fin.astype(np.float64).sum(1)
    got = env.episode_stats()
    assert got["episodes"] == int(want[3]) and got["length_sum"] == want[2], (got, want)
    for k, q in (("return_sum", 0), ("return_sqsum", 1)):
        if np.isfinite(want[q]):
            np.testing.assert_allclose(got[k], want[q], rtol=1e-12, err_msg=k)
        else:
            assert np.isnan(got[k]) == np.isnan(want[q]) and (np.isnan(want[q]) or got[k] == want[q]), (k, got[k], want[q])
    return fin


@pytest.mark.parametrize("body", BENCH_BODIES)
def test_config4_as_benchmarked_reference_horizon(body, kernel_names):
    """bench.py 4_units / 4_connected: 2^20 envs as body_cfg builds them, 1010 steps of U(-1, 1) actions launched back to
    back, against head, tail and first-wave-boundary slices of 8192 envs, every step; the state at the end with ep_ret
    and fin_stats.  Lanes run through inf / NaN until the max_steps reset at step 1000, whose post-reset observations
    are finite; episode_stats over the NaN returns that leaves behind."""
    import torch
    R, linked = 4, body == "quad_balance_chain"
    EB, EW = units_geometry(R)
    assert_units_instance(kernel_names, body, R, linked)
    E = 1 << 20
    env = bench_env(body, E)
    assert env.params.max_steps == 1000 and env.old_a is None
    slices = default_slices(E, 8192, block=EB, per_sm=UNITS_CTAS_PER_SM)
    assert len(slices) == 3
    _assert_units_tail(E, R, slices)
    lock = SliceLockstep(env, slices, max_steps=1000, seed=1234, spec=spec_of(body), k_sub=8, block=EB)
    steps = _run_back_to_back(env, lock, 1010, torch.Generator(device=DEV).manual_seed(41 + linked))
    got = dict(steps)[1000]
    d = got["done"].astype(bool)
    assert d.sum() > 0 and np.isfinite(got["obs"][d]).all(), "the max_steps reset leads to finite states"
    lock.check_state()
    assert lock.done_count > 0 and lock.nonfinite > 0 and lock.finite_rows > 0
    fin = check_episode_stats(env)
    assert np.isnan(fin[0]).any(), "some lanes ended their episode with a NaN return"


SHORT = [(4, "template"), (4, "jitter"), (8, "template")]


@pytest.mark.parametrize("max_steps,mode", SHORT)
@pytest.mark.parametrize("body", BENCH_BODIES)
def test_config4_short_episodes_at_full_size(body, max_steps, mode, kernel_names):
    """The config 4 bodies at 2^20 envs for 200 steps with episodes short enough that the comparisons see finite
    states.  max_steps 4: every lane is reset (template, or jitter: Philox noise keyed per global mass and env id, here
    up to env id 2^20 - 1) before it can overflow; with template resets at least 95 % of the compared rows are finite.
    A jitter reset keeps positions and velocities, so after the first one the lanes overflow regardless: there the
    test asserts that every lane's observation after the first reset (step 4) was finite when compared.  max_steps 8:
    the finite -> inf / NaN transition inside every episode and the reset out of it."""
    import torch
    R, linked = 4, body == "quad_balance_chain"
    EB, _ = units_geometry(R)
    assert_units_instance(kernel_names, body, R, linked)
    E = 1 << 20
    env = bench_env(body, E, max_steps=max_steps, auto_reset=mode)
    slices = default_slices(E, 4096, block=EB, per_sm=UNITS_CTAS_PER_SM)
    _assert_units_tail(E, R, slices)
    lock = SliceLockstep(env, slices, max_steps=max_steps, seed=1234, spec=spec_of(body), k_sub=8, auto_reset=mode,
                         block=EB)
    steps = dict(_run_back_to_back(env, lock, 200, torch.Generator(device=DEV).manual_seed(max_steps + len(mode))))
    lock.check_state()
    assert lock.done_count > 0
    frac = lock.finite_rows / lock.obs_rows
    if mode == "template" and max_steps == 4:
        assert frac >= 0.95, f"only {frac:.3f} of the compared rows were finite"
    if mode == "jitter":
        d = steps[4]["done"].astype(bool)
        assert d.all() and np.isfinite(steps[4]["obs"]).all(), "every lane reset at step 4 with a finite observation"
    if max_steps == 8:
        assert lock.nonfinite > 0 and frac >= 0.5, (lock.nonfinite, frac)
    check_episode_stats(env)


TAILS = ["last warp holds 1 env", "last CTA holds 1 warp", "whole CTAs"]


def grid_edge_size(R, tail):
    EB, EW = units_geometry(R)
    return {"last warp holds 1 env": (1 << 20) + 2 * EW + 1, "last CTA holds 1 warp": (1 << 20) + EW,
            "whole CTAs": (1 << 20) - 3 * EB}[tail]


@pytest.mark.parametrize("tail", TAILS)
@pytest.mark.parametrize("linked", [False, True])
@pytest.mark.parametrize("R", [2, 4, 8])
def test_units_kernel_grid_edges(R, linked, tail, kernel_names):
    """step_units_kernel for R = 2, 4, 8 units, disconnected and linked, at E near 2^20 with a ragged last CTA: its last
    warp holding exactly one env (E = 1 mod EW: the element-by-element observation store, and for the linked form the
    link shuffles under a partial mask), exactly one full warp (E = EW mod EB), or whole CTAs.  50 steps with template
    resets every 6 steps (every lane finite when compared), against the head and the tail slice."""
    import torch
    EB, EW = units_geometry(R)
    E = grid_edge_size(R, tail)
    last = E - (E - 1) // EB * EB                  # envs in the last CTA
    if tail == "last warp holds 1 env":
        assert E % EW == 1 and last == 2 * EW + 1
    elif tail == "last CTA holds 1 warp":
        assert E % EB == EW and last == EW
    else:
        assert E % EB == 0 and last == EB
    probe = f"units R={R} {'linked' if linked else 'disconnected'}"
    assert_units_instance(kernel_names, probe, R, linked)
    env, spec = units_env(R, linked, E, in3d=True, auto_reset="template", max_steps=6, k_sub=8, seed=77 + R,
                          track_stats=True)
    D = env.obs_dim
    assert (EW * D * 4) % 16 == 0, "full warps store their observation rows with one bulk copy"
    n = 2048
    slices = [(0, n), (E - n, E)]
    _assert_units_tail(E, R, slices)
    lock = SliceLockstep(env, slices, max_steps=6, seed=77 + R, spec=spec, k_sub=8, block=EB)
    _run_back_to_back(env, lock, 50, torch.Generator(device=DEV).manual_seed(E))
    lock.check_state()
    assert lock.done_count > 0 and lock.finite_rows >= 0.95 * lock.obs_rows, (lock.finite_rows, lock.obs_rows)


@pytest.mark.parametrize("body", BENCH_BODIES)
def test_units_kernel_unaligned_observation_buffer(body, kernel_names):
    """step(out=...) with a contiguous observation buffer 4 bytes off a 16-byte boundary: no warp can use the bulk
    store, every observation row leaves through the element-by-element path, at 2^20 envs.  Same bits as the env's
    own (aligned) buffer, which takes the bulk path, for every step."""
    import torch
    R, linked = 4, body == "quad_balance_chain"
    EB, EW = units_geometry(R)
    assert_units_instance(kernel_names, body, R, linked)
    E = 1 << 20
    a = bench_env(body, E, max_steps=4)
    b = bench_env(body, E, max_steps=4)
    D = a.obs_dim
    assert (EW * D * 4) % 16 == 0 and a.obs.data_ptr() % 16 == 0
    flat = torch.full((E * D + 4,), 7.0, device=DEV)
    obs_u = flat[1:1 + E * D].view(E, D)
    assert obs_u.is_contiguous() and obs_u.data_ptr() % 16 == 4
    rew_u, done_u = torch.empty(E, device=DEV), torch.empty(E, dtype=torch.uint8, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(5)
    finite = 0
    for t in range(12):
        act = torch.rand(E, a.M, device=DEV, generator=g) * 2 - 1
        a.step(act, out=(obs_u, rew_u, done_u))
        ob, rb, db, _ = b.step(act)
        assert torch.equal(obs_u.view(torch.int32), ob.view(torch.int32)), f"obs at step {t}"
        assert torch.equal(rew_u.view(torch.int32), rb.view(torch.int32)) and torch.equal(done_u, db.view(torch.uint8)), t
        finite += int(torch.isfinite(ob).all(1).sum())
    assert finite >= 0.95 * 12 * E
    assert float(flat[0]) == 7.0 and float(flat[-3]) == 7.0, "nothing written outside the buffer"
    assert torch.equal(a.pos.view(torch.int32), b.pos.view(torch.int32))


def test_episode_stats_with_a_ragged_batch():
    """stats_reduce_kernel at E = 2^20 + 37 (one CTA strides over every env: the last stride is partial), finite
    returns: against the float64 sum of the host copy of fin_stats."""
    import torch
    E = (1 << 20) + 37
    env = bench_env("quad_balance", E, max_steps=4)
    g = torch.Generator(device=DEV).manual_seed(9)
    for _ in range(13):
        env.step(torch.rand(E, env.M, device=DEV, generator=g) * 2 - 1)
    fin = check_episode_stats(env)
    assert fin[3].sum() == 3 * E and np.isfinite(fin).all()


def test_step_many_in_kernel_cpg_at_full_size():
    """bench.py multi16's second half: step_many(CPGActions(...), n_steps=16) at 2^20 envs, actions computed in the
    kernel from each env's step counter, template auto-reset every EPISODE_STEPS (which restarts the gait).  40 launches;
    the oracle takes the same actions from wo.gen_actions: rewards and dones of every step, the observation after every
    launch, the state at the end."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv, CPGActions
    E, T = 1 << 20, 16
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, in3d=True, auto_reset="template", seed=1234, track_stats=True,
                            state_layout="packed", max_steps=EPISODE_STEPS)
    cpg = CPGActions(amp=[0.8] * env.M, freq=[1.5 + 0.5 * m for m in range(env.M)], phase=[0.7 * m for m in range(env.M)])
    desc = cpg.describe(float(env.params.dt))
    lock = SliceLockstep(env, default_slices(E, 8192), max_steps=EPISODE_STEPS, seed=1234, gen=desc)
    res = (torch.empty(T, E, device=DEV), torch.empty(T, E, dtype=torch.uint8, device=DEV))
    for k in range(40):
        obs, rew, done = env.step_many(cpg, n_steps=T, out=res)
        for t in range(T):
            lock.record(None, None, rew[t], done[t])
        lock.flush(f"(launch {k})")
        lock.check_obs(obs, f"after launch {k}")
    lock.check_state()
    assert lock.done_count > 0 and lock.finite_rows == lock.obs_rows


# ---- config 6: package physics ---------------------------------------------------------------------------------------
def pkg_system(env):
    """The oracle's system of an Environment (as bench.py builds it for its CPU baseline)."""
    return {"points": [(float(p.m), tuple(map(float, p.pos)), (0.0, 0.0, 0.0), p.fixed) for p in env._order],
            "springs": [(env._order.index(a), env._order.index(b), float(x), float(k), bool(st))
                        for a, b, x, k, st in env.springs]}


class PkgSlices:
    """The oracle (wo.l2_step) on env slices [a, b) of a batched Environment, started from the device state; every
    update_physics launch is compared bit for bit: pos, vel and old_a.  `block` = envs per CTA of the kernel (for
    failure messages).  ground_points counts oracle points lying on the ground after each launch."""

    def __init__(self, env, slices, block):
        self.env, self.block = env, block
        self.so, self.po = wo.make_l2_system(pkg_system(env)), wo.make_l2_params(ground_level=GROUND)
        self.parts = []
        for a, b in slices:
            self.parts.append((a, b, {k: np.ascontiguousarray(getattr(env, k)[:, a:b].cpu().numpy())
                                      for k in ("pos", "vel", "old_a")}))
        self.updates, self.ground_points = 0, 0

    def restrict(self, slices):
        (a0, b0, st), = self.parts
        assert (a0, b0) == (0, self.env.num_envs)
        self.parts = [(a, b, {k: np.ascontiguousarray(v[:, a:b]) for k, v in st.items()}) for a, b in slices]

    def update(self, T):
        self.env.update_physics(T)
        for _, _, st in self.parts:
            wo.l2_step(self.so, self.po, st, T)
        self.updates += T
        E, B = self.env.num_envs, self.block
        for a, b, st in self.parts:
            for k in ("pos", "vel", "old_a"):
                g = getattr(self.env, k)[:, a:b].cpu().numpy()
                assert gu.same(g, st[k]), (f"{k} after {self.updates} updates ({T} per launch): slice [{a}, {b}) of {E} "
                                           f"envs = CTAs [{a // B}, {(b - 1) // B}] of {(E + B - 1) // B}")
            self.ground_points += int((st["pos"][1::3] == np.float32(GROUND)).sum())


def _perturbed_pkg_env(body, E, seed=7):
    """bench.py run_pkg's state: the body in E copies, velocities + N(0, 1) from a seeded generator."""
    import torch
    env = _pkg_env(_pkg_builders()[body], E)
    g = torch.Generator(device=DEV).manual_seed(seed)
    env.vel.add_(torch.randn(env.vel.shape, device=DEV, generator=g))
    return env


@pytest.mark.parametrize("T", [1, 16])
def test_config6_as_benchmarked(T, kernel_names):
    """bench.py config 6 (run_pkg): box at 2^20 envs, ground at -8, velocities + N(0, 1), update_physics(T) launches
    to 200+ updates.  The whole batch after the first launch, then head, middle and tail slices after every launch;
    points reach the ground."""
    import torch
    assert_pkg_instance(kernel_names, "pkg box", "pkg_update_kernel")
    E = 1 << 20
    env = _perturbed_pkg_env("box", E)
    ps = PkgSlices(env, [(0, E)], PKG_BLOCK)
    ps.update(T)
    n = 8192
    ps.restrict([(0, n), (E // 2 - n // 2, E // 2 + n // 2), (E - n, E)])
    while ps.updates < 200:
        ps.update(T)
    on_ground = float((env.pos[1::3] == GROUND).float().mean())
    assert ps.ground_points > 0 and on_ground > 0.005, (ps.ground_points, on_ground)
    assert torch.isfinite(env.pos).all()


PARTS = [("insect", -1, 4, "pkg insect"), ("humanb", -1, 2, "pkg humanb"), ("insect", 8, 8, "pkg insect LP=8")]


@pytest.mark.parametrize("body,knob,LP,probe", PARTS)
def test_config6_partitioned_kernel_ragged_grid(body, knob, LP, probe, part_knob, kernel_names):
    """pkg_update_part_kernel<LP> (128 / LP envs per CTA) as --pkg-body insect / humanb select it (LP 4 / 2 by the
    automatic rule) and insect with LP forced to 8, at E = 2^20 + 37 so the last CTA is partial (nvalid < EB):
    update_physics(1), (16) and (200) against the head and tail slices, old_a included."""
    EB = PKG_BLOCK // LP
    E = (1 << 20) + 37
    assert 0 < E % EB < EB
    part_knob(knob)
    assert_pkg_instance(kernel_names, probe, "pkg_update_part_kernel", lp=LP)
    env = _perturbed_pkg_env(body, E)
    n = 4096
    ps = PkgSlices(env, [(0, n), (E - n, E)], EB)
    for T in (1, 16, 200):
        ps.update(T)
    assert ps.ground_points > 0


@pytest.mark.parametrize("body,topo", [("leg2", "PkgLeg2"), ("balance3", "PkgChain4")])
def test_config6_register_resident_kernels_ragged_grid(body, topo, kernel_names):
    """pkg_update_static_kernel for leg2 and balance3 (a DingPoint pivot) at E = 2^20 + 37: a partial last CTA,
    update_physics(1), (16) and (200) against the head and tail slices."""
    from walker_gym_b200 import _lib
    assert_pkg_instance(kernel_names, f"pkg {body}", "pkg_update_static_kernel", topo=topo)
    E = (1 << 20) + 37
    assert E % PKG_BLOCK
    env = _perturbed_pkg_env(body, E)
    assert _lib.load().wg_pkg_kernel_variant(C.byref(env.system())) > 0
    n = 4096
    ps = PkgSlices(env, [(0, n), (E - n, E)], PKG_BLOCK)
    for T in (1, 16, 200):
        ps.update(T)
    if body == "leg2":
        assert ps.ground_points > 0


def test_config6_generic_kernel_above_48k_shared_memory(part_knob, kernel_names):
    """The run-time-topology kernel on a random 32-point, 96-spring system (DingPoints, rope-type springs) with the
    point partition off: 9 * 32 rows of 129 floats = 148.6 KB of dynamic shared memory per CTA, launched after
    cudaFuncSetAttribute; E = 2^20 + 37, head and tail slices."""
    part_knob(0)
    assert_pkg_instance(kernel_names, "pkg random32 parts=0", "pkg_update_kernel")
    assert 4 * 9 * 32 * (PKG_BLOCK + 1) > 48 * 1024
    E = (1 << 20) + 37
    env = _perturbed_pkg_env("random32", E)
    assert len(env._order) == 32 and len(env.springs) == 96
    n = 2048
    ps = PkgSlices(env, [(0, n), (E - n, E)], PKG_BLOCK)
    for T in (1, 16, 40):
        ps.update(T)
    assert ps.ground_points > 0
