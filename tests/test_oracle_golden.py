"""CPU: the C oracle must reproduce the reference's recorded outputs bit for bit."""
import os

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo


def replay_trajectory(g, stepper):
    """Replay a golden trajectory; returns the name of the first mismatching field or None."""
    spec, kw = g["spec"], g["env_kwargs"]
    body = stepper.make_body(spec)
    N, M = body.n_mass, body.n_muscle
    in3d = bool(kw.get("in3d", False))
    d = 3 if in3d else 2
    prm_kw = dict(kw)
    if g["max_steps"] is not None:
        prm_kw["max_steps"] = g["max_steps"]
    if g["k_sub"] is not None:
        prm_kw["k_sub"] = g["k_sub"]
    if g.get("integrator"):
        prm_kw["integrator"] = g["integrator"]
    auto = 1 if g["reset_on_done"] else 0
    prm = stepper.make_params(auto_reset=auto, **prm_kw)
    st = stepper.init_state(body, 1)
    draws = g["reset_noise"].astype(np.float32)
    cursor = 0

    def next_noise():
        nonlocal cursor
        nz = np.zeros((N, 3), np.float32)
        nz[:, :d] = draws[cursor:cursor + N * d].reshape(N, d)
        cursor += N * d
        return gu.soa(nz)

    obs0 = stepper.reset(body, prm, st, mode=1, noise=next_noise())
    if "init_pos" in g:
        st["pos"][:] = gu.soa(g["init_pos"])
        st["vel"][:] = gu.soa(g["init_vel"])
    else:
        if not gu.same(obs0[0], g["obs"][0]):
            return "obs0"
    T = len(g["actions"])
    for t in range(T):
        nz = next_noise() if (auto and g["done"][t]) else None
        if nz is None and auto:
            nz = np.zeros((N * 3, 1), np.float32)
        out = stepper.step(body, prm, st, g["actions"][t:t + 1], noise=nz)
        checks = {
            "pos": gu.same(gu.aos(st["pos"], N)[0], g["pos"][t + 1]),
            "vel": gu.same(gu.aos(st["vel"], N)[0], g["vel"][t + 1]),
            "old_a": gu.same(gu.aos(st["old_a"], N)[0], g["old_a"][t + 1]),
            "x": gu.same(st["mx"][:, 0], g["x"][t + 1]),
            "obs": gu.same(out["obs"][0], g["obs"][t + 1]),
            "reward": gu.same(out["reward"][0], g["reward"][t]),
            "done": bool(out["done"][0]) == bool(g["done"][t]),
            "contact_pre": gu.same(gu.mask_bits(out["contact_pre"], N)[0], g["contact_pre"][t]),
            "energy": gu.same(out["energy"][0], g["energy"][t]),
            "centroid": gu.same(out["centroid"][:, 0], g["centroid"][t]),
            "steps": int(st["steps"][0]) == int(g["steps"][t]),
        }
        bad = [k for k, ok in checks.items() if not ok]
        if bad:
            return f"step {t}: {bad}"
    return None


@pytest.mark.parametrize("name", gu.trajectory_names())
def test_oracle_matches_reference_trajectory(name):
    g = gu.load(name)
    assert replay_trajectory(g, wo) is None


def replay_batch(g, stepper):
    spec, kw = g["spec"], g["env_kwargs"]
    body = stepper.make_body(spec)
    N = body.n_mass
    prm = stepper.make_params(**kw)
    E = g["init_pos"].shape[0]
    st = stepper.init_state(body, E)
    st["pos"][:] = gu.soa(g["init_pos"])
    st["vel"][:] = gu.soa(g["init_vel"])
    out = stepper.step(body, prm, st, g["actions"])
    checks = {
        "pos": gu.same(gu.aos(st["pos"], N), g["pos"]),
        "vel": gu.same(gu.aos(st["vel"], N), g["vel"]),
        "old_a": gu.same(gu.aos(st["old_a"], N), g["old_a"]),
        "x": gu.same(st["mx"].T, g["x"]),
        "obs": gu.same(out["obs"], g["obs"]),
        "reward": gu.same(out["reward"], g["reward"]),
        "done": gu.same(out["done"].astype(bool), g["done"]),
        "contact_pre": gu.same(gu.mask_bits(out["contact_pre"], N), g["contact_pre"]),
        "energy": gu.same(out["energy"], g["energy"]),
        "centroid": gu.same(out["centroid"].T, g["centroid"]),
    }
    return [k for k, ok in checks.items() if not ok]


@pytest.mark.parametrize("name", gu.batch_names())
def test_oracle_matches_reference_batch(name):
    assert replay_batch(gu.load(name), wo) == []


def test_golden_cover_the_branches():
    """The fixtures must actually exercise contact, every done clause, NaN and resets."""
    assert gu.load("done_fall")["done"].any()
    assert gu.load("done_stopped")["done"].any()
    assert gu.load("done_maxsteps")["done"].any()
    assert not np.isfinite(gu.load("box3d_overflow")["pos"]).all()
    assert gu.load("balance3d_s0")["contact_pre"].any()
    assert gu.load("autoreset_jitter")["done"].sum() >= 3


def replay_l2(g, stepper, chunk=1):
    """Replay an L2 (package lineage) trajectory; `chunk` steps per call."""
    sysm = stepper.make_l2_system(g["system"])
    prm = stepper.make_l2_params(**g["env_kwargs"])
    st = stepper.l2_init_state(g["system"], 1)
    P = len(g["system"]["points"])
    T = g["pos"].shape[0] - 1
    t = 0
    while t < T:
        n = min(chunk, T - t)
        stepper.l2_step(sysm, prm, st, n)
        t += n
        ok = (gu.same(st["pos"].reshape(P, 3), g["pos"][t]) and gu.same(st["vel"].reshape(P, 3), g["vel"][t])
              and gu.same(st["old_a"].reshape(P, 3), g["old_a"][t]))
        if not ok:
            return f"step {t}"
    return None


@pytest.mark.parametrize("chunk", [1, 7])
@pytest.mark.parametrize("name", gu.l2_names())
def test_oracle_matches_reference_package_physics(name, chunk):
    """L2: Environment.update_physics of gym/optimized_walker/env.py, bit for bit."""
    assert replay_l2(gu.load_l2(name), wo, chunk) is None


# ---- float64 actions: the tolerance protocol (SURVEY 7.2) ---------------------------------------------------------
def rel_err(a, b):
    """max |a - b| / max |b| over finite reference entries (the north_star's "relative" state error)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    fin = np.isfinite(b)
    if not fin.any():
        return 0.0
    return float(np.abs(a[fin] - b[fin]).max() / max(np.abs(b[fin]).max(), 1e-30))


def replay_f64_teacher_forced(g, stepper):
    """The reference was driven with float64 ndarray actions, which silently turns Muscle.x and the muscle spring
    term into float64 (SURVEY 7.7); the library computes in float32 on float32(action).  Every step is re-seeded
    from the reference's state (x rounded to float32) and advanced once: the float32 state (positions, velocities,
    muscle lengths) and the reward within 1e-5 relative (north_star's single-step tolerance), the accelerations --
    differences of large spring forces, and with them the observation that carries them -- within 1e-4, force-phase
    contact and done flags exact.  Returns (worst state error, worst acceleration/observation error, flag mismatches)."""
    spec, kw = g["spec"], g["env_kwargs"]
    body = stepper.make_body(spec)
    N = body.n_mass
    prm = stepper.make_params(**kw)
    st = stepper.init_state(body, 1)
    worst, worst_acc, flags = 0.0, 0.0, 0
    for t in range(len(g["actions"])):
        st["pos"][:] = gu.soa(g["pos"][t])
        st["vel"][:] = gu.soa(g["vel"][t])
        st["mx"][:, 0] = g["x"][t].astype(np.float32)
        st["steps"][:] = 0 if t == 0 else int(g["steps"][t - 1])
        out = stepper.step(body, prm, st, g["actions"][t:t + 1].astype(np.float32))
        if not np.isfinite(g["pos"][t + 1]).all():
            break
        worst = max(worst, rel_err(gu.aos(st["pos"], N)[0], g["pos"][t + 1]), rel_err(gu.aos(st["vel"], N)[0], g["vel"][t + 1]),
                    rel_err(st["mx"][:, 0], g["x"][t + 1]), rel_err(out["reward"][0], g["reward"][t]))
        worst_acc = max(worst_acc, rel_err(gu.aos(st["old_a"], N)[0], g["old_a"][t + 1]), rel_err(out["obs"][0], g["obs"][t + 1]))
        flags += int(bool(out["done"][0]) != bool(g["done"][t]))
        flags += int(not gu.same(gu.mask_bits(out["contact_pre"], N)[0], g["contact_pre"][t]))
    return worst, worst_acc, flags


def replay_f64_free_running(g, stepper, T):
    """Free-running T steps on float32(action) against the reference's float64-action trajectory."""
    body = stepper.make_body(g["spec"])
    N = body.n_mass
    prm = stepper.make_params(**g["env_kwargs"])
    st = stepper.init_state(body, 1)
    st["pos"][:] = gu.soa(g["pos"][0])
    st["vel"][:] = gu.soa(g["vel"][0])
    worst = 0.0
    for t in range(T):
        stepper.step(body, prm, st, g["actions"][t:t + 1].astype(np.float32))
        worst = max(worst, rel_err(gu.aos(st["pos"], N)[0], g["pos"][t + 1]))
    return worst


TOLERANCE_FIXTURES = ["f64act_balance3d", "f64act_box2d", "f64act_box3d_physical_sign"]


@pytest.mark.parametrize("name", TOLERANCE_FIXTURES)
def test_oracle_float64_actions_teacher_forced(name):
    worst, worst_acc, flags = replay_f64_teacher_forced(gu.load(name), wo)
    assert flags == 0 and worst < 1e-5 and worst_acc < 1e-4, (worst, worst_acc, flags)


def test_oracle_float64_actions_free_running_100_steps():
    """With physically signed springs (stable dynamics) the 100-step free-running trajectory stays within the
    north_star's 1e-3 even though the reference ran its muscles in float64."""
    assert replay_f64_free_running(gu.load("f64act_box3d_physical_sign"), wo, 100) < 1e-3


def replay_x64(g, stepper):
    """Bit-exact replay of a float64-action trajectory in x64 mode (Muscle.x as double + type bit): positions,
    velocities, accelerations, the float64 muscle lengths, observation (the reference's float64 observation rounded to
    float32), reward, done, contact.  Returns the first mismatch or None."""
    spec, kw = g["spec"], g["env_kwargs"]
    body, xb = stepper.make_body(spec), stepper.make_x64(spec)
    N = body.n_mass
    in3d = bool(kw.get("in3d", False))
    d = 3 if in3d else 2
    prm_kw = dict(kw)
    if g["max_steps"] is not None:
        prm_kw["max_steps"] = g["max_steps"]
    if g["k_sub"] is not None:
        prm_kw["k_sub"] = g["k_sub"]
    auto = 1 if g["reset_on_done"] else 0
    prm = stepper.make_params(auto_reset=auto, **prm_kw)
    st = stepper.init_state(body, 1)
    st["mx64"], st["mx_weak"] = stepper.init_x64(body, xb, 1)
    draws = g["reset_noise"].astype(np.float32)
    cursor = 0

    def next_noise():
        nonlocal cursor
        nz = np.zeros((N, 3), np.float32)
        nz[:, :d] = draws[cursor:cursor + N * d].reshape(N, d)
        cursor += N * d
        return gu.soa(nz)

    stepper.reset(body, prm, st, mode=1, noise=next_noise())
    for t in range(len(g["actions"])):
        nz = next_noise() if (auto and g["done"][t]) else (np.zeros((N * 3, 1), np.float32) if auto else None)
        out = stepper.step_x64(body, xb, prm, st, g["actions"][t:t + 1], noise=nz)
        checks = {
            "pos": gu.same(gu.aos(st["pos"], N)[0], g["pos"][t + 1]),
            "vel": gu.same(gu.aos(st["vel"], N)[0], g["vel"][t + 1]),
            "old_a": gu.same(gu.aos(st["old_a"], N)[0], g["old_a"][t + 1]),
            "x": gu.same(st["mx64"][:, 0], g["x"][t + 1]),
            "obs": gu.same(out["obs"][0], g["obs"][t + 1].astype(np.float32)),
            "reward": gu.same(out["reward"][0], np.float32(g["reward"][t])),
            "done": bool(out["done"][0]) == bool(g["done"][t]),
            "contact_pre": gu.same(gu.mask_bits(out["contact_pre"], N)[0], g["contact_pre"][t]),
            "steps": int(st["steps"][0]) == int(g["steps"][t]),
        }
        bad = [k for k, ok in checks.items() if not ok]
        if bad:
            return f"step {t}: {bad}"
    return None


@pytest.mark.parametrize("name", gu.f64_names())
def test_oracle_x64_mode_matches_reference_bit_for_bit(name):
    """The reference driven with float64 ndarray actions -- its own demo loop -- reproduced exactly: NumPy promotes
    the muscle spring term to double while Muscle.x is an np.float64 and drops back to float32 when regulation()
    replaced it by a limit object."""
    assert replay_x64(gu.load(name), wo) is None


def test_x64_fixtures_exercise_the_type_switch():
    g = gu.load("f64act_clamps_custom3d")
    body, xb = wo.make_body(g["spec"]), wo.make_x64(g["spec"])
    lo = np.array([xb.mlo_d[m] for m in range(body.n_muscle)])
    hi = np.array([xb.mhi_d[m] for m in range(body.n_muscle)])
    clamped = (g["x"][1:] == lo) | (g["x"][1:] == hi)
    assert clamped[:, :3].any(axis=0).all() and (~clamped[:, :3]).any(axis=0).all()    # both types occur per acted muscle
    assert (g["x"][1:, 3] == g["x"][0, 3]).all()                                       # the un-acted muscle never moves
    assert gu.load("f64act_autoreset_box3d")["done"].sum() >= 3


def test_getstat_options_and_actdisp_against_the_reference_recording():
    """Creature.actdisp (discrete +-stride actions) driving PhysicsEnv.step and Creature.getstat with non-default
    options, recorded from the reference itself (tests/golden/make_golden.py main_getstat): the oracle stepped with
    actions +-float32(stride) reproduces the trajectory, and its getstat restatement every recorded variant."""
    import json
    z = np.load(os.path.join(gu.GOLDEN_DIR, "getstat_actdisp_custom3d.npz"))
    spec = json.loads(str(z["spec"]))
    spec = {"points": [(m, tuple(p), bool(f)) for m, p, f in spec["points"]],
            "muscles": [(i, j, dict(kw)) for i, j, kw in spec["muscles"]],
            "skeletons": [(i, j, dict(kw)) for i, j, kw in spec["skeletons"]]}
    strides = np.array([np.float32(kw.get("stride", 2)) for _, _, kw in spec["muscles"]], np.float32)
    oracle_spec = {"points": spec["points"], "skeletons": spec["skeletons"],
                   "muscles": [(i, j, {k: v for k, v in kw.items() if k != "stride"}) for i, j, kw in spec["muscles"]]}
    body = wo.make_body(oracle_spec)
    prm = wo.make_params(in3d=True)
    st = wo.init_state(body, 1)
    N = body.n_mass
    noise = np.zeros((3 * N, 1), np.float32)
    k = 0
    for n in range(N):                                   # PhysicsEnv.reset draws x, y, z per point, in order
        for c in range(3):
            noise[n * 3 + c, 0] = z["reset_noise"][k]
            k += 1
    wo.reset(body, prm, st, mode=1, noise=noise)
    variants = json.loads(str(z["variants"]))
    for t in range(z["disp"].shape[0]):
        act = np.where(z["disp"][t].astype(bool), strides, -strides).astype(np.float32)[None]
        out = wo.step(body, prm, st, act)
        assert gu.same(gu.aos(st["pos"], N)[0], z["pos"][t]) and gu.same(gu.aos(st["vel"], N)[0], z["vel"][t]), t
        assert gu.same(st["mx"][:, 0], z["x"][t]) and gu.same(out["reward"][0], z["reward"][t]), t
        for v, kw in enumerate(variants):
            assert gu.same(wo.getstat(body, st, st["old_a"], **kw)[0], z[f"stat{v}"][t]), (t, v)


def test_rope_type_springs_follow_point_resilience():
    """`string=True` (extension of Muscle / Skeleton; semantics of Point.resilience, gym/optimized_engine.py:134-138):
    while the spring is shorter than its rest length the elastic term is f_size = 0 and only the damping term acts;
    once it is longer it is the ordinary spring.  Checked against the reference's own arithmetic written out in NumPy
    (float32 arrays, python-scalar constants) for one spring, and: a body whose springs never get shorter than their
    rest lengths steps identically with and without the flag.  (The reference's L1 classes have no such flag, so there is
    no reference recording for it: parity of this option is pinned to this restatement only.)"""
    def spec(string, x):
        return {"points": [(2.0, (0.0, 50.0, 0.0), False), (3.0, (30.0, 90.0, 0.0), False)], "muscles": [],
                "skeletons": [(0, 1, {"x": x, "k": 700, "dampk": 12, "string": string})]}
    for x, slack in ((80.0, True), (20.0, False)):            # current distance is 50: shorter / longer than x
        outs = []
        for string in (False, True):
            body = wo.make_body(spec(string, x))
            prm = wo.make_params(in3d=True, g=0, ground_high=-1000)
            st = wo.init_state(body, 1)
            st["vel"][:, 0] = np.array([1, -2, 0.5, -3, 4, 0.25], np.float32)
            v0 = st["vel"].copy()
            wo.step(body, prm, st, np.zeros((1, 0), np.float32))
            outs.append(st["old_a"].copy())
        p1, p2 = np.array([0, 50, 0], np.float32), np.array([30, 90, 0], np.float32)
        v1, v2 = v0[:3, 0], v0[3:, 0]
        L = np.linalg.norm(p1 - p2)
        direction = (p2 - p1) / L
        dk = np.dot(v1 - v2, direction)
        damp = dk * 12 * direction
        for string, got in zip((False, True), outs):
            f_size = 0 if (string and L - x < 0) else -(L - x) * 700
            force = f_size * direction
            a1 = np.zeros(3, np.float32); a1 += force / 2.0; a1 += (-damp) / 2.0
            a2 = np.zeros(3, np.float32); a2 += (-force) / 3.0; a2 += damp / 3.0
            assert gu.same(got[:3, 0], a1) and gu.same(got[3:, 0], a2), (x, string)
        assert gu.same(outs[0], outs[1]) == (not slack)

    # A rope-type muscle driven with float64 actions (wo.step_x64).  Its length is then an np.float64 ("strong") and the
    # elastic term is NumPy float64 arithmetic: dx = np.float64(L) - x, f_size = -dx * float(k), a float64 force array,
    # and Point.forced rounds `acc + force / m` once.  A length that regulation() clamped holds the float32 limit
    # ("weak") and is back on the float32 arithmetic above.  The rope rule holds on both.
    def muscle_spec(string, p2, x0, k):
        return {"points": [(2.0, (0.0, 50.0, 0.0), False), (3.0, p2, False)], "skeletons": [],
                "muscles": [(0, 1, {"x": x0, "k": k, "dampk": 12, "string": string})]}

    def restated(string, p2, x0, k, a):
        p1, p2 = np.array([0, 50, 0], np.float32), np.array(p2, np.float32)
        v1, v2 = np.array([1, -2, 0.5], np.float32), np.array([-3, 4, 0.25], np.float32)
        L = np.linalg.norm(p1 - p2)
        direction = (p2 - p1) / L if L > 0 else p2 - p1         # coincident endpoints: no division (the oracle's guard)
        x = np.float64(x0) + np.float64(a)                       # Muscle.x += a
        lo, hi = x0 * 0.1, x0 * 1.5                              # originx a python float: python float limits
        weak = bool(lo > x or hi < x)
        if weak:
            x = lo if lo > x else hi                             # max() / min() return the limit object
            dx = L - x                                           # np.float32 - python float: float32
            f_size = np.float32(0) if (string and dx < 0) else -dx * np.float32(k)
            force = f_size * direction                           # float32
        else:
            dx = np.float64(L) - x
            f_size = np.float64(0) if (string and dx < 0) else -dx * float(k)
            force = np.float64(f_size) * direction.astype(np.float64)
        damp = np.dot(v1 - v2, direction) * np.float32(12) * direction
        a1 = np.zeros(3, np.float32); a1 += force / 2.0; a1 += (-damp) / np.float32(2.0)
        a2 = np.zeros(3, np.float32); a2 += (-force) / 3.0; a2 += damp / np.float32(3.0)
        return weak, np.concatenate([a1, a2])

    cases = [  # (what, p2, x0, k, action, weak, slack); the endpoints are 50 apart unless p2 coincides with p1
        ("strong slack", (30.0, 90.0, 0.0), 40.0, 700, 15.0, False, True),
        ("strong taut", (30.0, 90.0, 0.0), 40.0, 700, -5.5, False, False),
        ("strong slack, negative k", (30.0, 90.0, 0.0), 40.0, -700, 15.0, False, True),
        ("weak slack", (30.0, 90.0, 0.0), 40.0, 700, 80.0, True, True),      # clamped to x0 * 1.5 = 60 > 50
        ("weak taut", (30.0, 90.0, 0.0), 40.0, 700, -80.0, True, False),     # clamped to x0 * 0.1 = 4 < 50
        ("L == x", (30.0, 90.0, 0.0), 40.0, 700, 10.0, False, False),        # dx = 0: f_size = -0 * k either way
        ("coincident endpoints", (0.0, 50.0, 0.0), 40.0, 700, 3.0, False, True),
    ]
    for what, p2, x0, k, a, weak, slack in cases:
        outs = []
        for string in (False, True):
            spec = muscle_spec(string, p2, x0, k)
            body, xb = wo.make_body(spec), wo.make_x64(spec)
            prm = wo.make_params(in3d=True, g=0, ground_high=-1000)
            st = wo.init_state(body, 1)
            st["mx64"], st["mx_weak"] = wo.init_x64(body, xb, 1)
            st["vel"][:, 0] = np.array([1, -2, 0.5, -3, 4, 0.25], np.float32)
            wo.step_x64(body, xb, prm, st, np.array([[a]], np.float64))
            want_weak, want = restated(string, p2, x0, k, a)
            assert want_weak == weak and int(st["mx_weak"][0, 0]) == int(weak), (what, string)
            assert gu.same(st["old_a"][:, 0], want), (what, string, st["old_a"][:, 0], want)
            outs.append(st["old_a"].copy())
        # the flag changes the step exactly when the muscle is slack and its direction is defined
        assert gu.same(outs[0], outs[1]) == (not slack or what == "coincident endpoints"), what
