"""CPU: the package lineage (gym/optimized_walker/{core,env,walker}.py) -- oracle against the reference-built
bodies, the host mirror's body tables against the reference's, env_state.pkl / state.pkl compatibility."""
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo

BODY_NAMES = ("test", "leg2", "box", "balance1", "balance2", "balance3", "humanb", "insect")


def body_record(name):
    z = np.load(os.path.join(gu.GOLDEN_DIR, "l2_bodies.npz"))
    return {k.split("__", 1)[1]: z[k] for k in z.files if k.startswith(name + "__")}


def system_of(rec):
    return {"points": [(float(m), tuple(map(float, p)), (0.0, 0.0, 0.0), bool(d))
                       for m, p, d in zip(rec["mass"], rec["pos0"], rec["ding"])],
            "springs": [(int(i), int(j), float(x), float(k), bool(s))
                        for i, j, x, k, s in zip(rec["si"], rec["sj"], rec["sx"], rec["sk"], rec["sstring"])]}


def replay_body(rec, stepper, chunk):
    system = system_of(rec)
    sysm, prm, st = stepper.make_l2_system(system), stepper.make_l2_params(), stepper.l2_init_state(system, 1)
    P, T, t = len(rec["mass"]), rec["pos"].shape[0] - 1, 0
    while t < T:
        n = min(chunk, T - t)
        stepper.l2_step(sysm, prm, st, n)
        t += n
        if not (gu.same(st["pos"].reshape(P, 3), rec["pos"][t]) and gu.same(st["vel"].reshape(P, 3), rec["vel"][t])):
            return f"step {t}"
    return None


@pytest.mark.parametrize("name", BODY_NAMES)
def test_oracle_matches_reference_bodies(name):
    """120 update_physics calls on every body the reference ships, bit for bit (mass-0 DingPoints included)."""
    assert replay_body(body_record(name), wo, 5) is None


def build(name, **kw):
    import walker_gym_b200.optimized_walker as ow
    ow.Point.clear()
    env = ow.Environment(**kw)
    return env, getattr(ow, name)(env)


@pytest.mark.parametrize("name", BODY_NAMES)
def test_host_body_tables_match_the_reference(name):
    """The transcribed builders produce the reference's points, springs (order, k, float32 rest length) and muscles."""
    rec = body_record(name)
    env, creature = build(name)
    s = env.system()
    P, S = len(rec["mass"]), len(rec["si"])
    assert (s.n_point, s.n_spring) == (P, S)
    assert [s.mass[n] for n in range(P)] == list(rec["mass"])
    assert [bool(s.fixed[n]) for n in range(P)] == list(rec["ding"])
    assert gu.same(np.array([p.pos for p in env._order], np.float32), rec["pos0"])
    assert [s.si[q] for q in range(S)] == list(rec["si"]) and [s.sj[q] for q in range(S)] == list(rec["sj"])
    assert gu.same(np.array([s.srest[q] for q in range(S)], np.float32), rec["sx"])
    assert [s.sk[q] for q in range(S)] == [np.float32(k) for k in rec["sk"]]
    assert [bool(s.sstring[q]) for q in range(S)] == list(rec["sstring"])
    mus = creature.skeleton.muscles
    idx = {id(p): n for n, p in enumerate(env._order)}
    assert [idx[id(m.point1)] for m in mus] == list(rec["muscle_i"])
    assert [idx[id(m.point2)] for m in mus] == list(rec["muscle_j"])
    assert gu.same(np.array([m.x for m in mus], np.float32), rec["muscle_x"])
    assert np.array_equal(np.array([[m.amp, m.freq, m.phase, m.power] for m in mus], np.float64).reshape(-1, 4),
                          rec["muscle_par"])


def test_muscle_pattern_generator_matches_the_reference():
    """Muscle.act: t += dt; state = (sin(2 pi f t + phase) + 1) / 2 (walker.py:56-70), without touching the device."""
    rec = body_record("humanb")
    env, creature = build("humanb")
    creature.act(env.time_step)                    # first call: positions are still the template on both sides
    assert np.array_equal(np.array([m.state for m in creature.skeleton.muscles]), rec["muscle_state"][0])
    for p in env._order:
        p.zero()
    for t in range(1, 20):
        for m in creature.skeleton.muscles:       # t / state only
            m.t += env.time_step
            m.state = (np.sin(2 * np.pi * m.freq * m.t + m.phase) + 1) / 2
        assert np.array_equal(np.array([m.state for m in creature.skeleton.muscles]), rec["muscle_state"][t])
    c2 = build("test")[1]
    c2.act(0.01)                                   # books the push on the descriptors' pending a
    p1, p2 = c2.skeleton.points
    assert c2.age == 1 and p1.a[0] != 0 and p1.a[0] == -p2.a[0]


def test_params_are_float32_at_the_point_of_use():
    env, _ = build("box", gravity=(0.5, -30, 0.1), air_resistance=0.2, time_step=0.02)
    p, o = env.params(), wo.make_l2_params(gravity=(0.5, -30, 0.1), air_resistance=0.2, time_step=0.02)
    assert [p.gravity[c] for c in range(3)] == [o.gravity[c] for c in range(3)]
    for k in ("damping", "drag_c", "ground_level", "restitution", "friction", "dt", "min_dist", "ground"):
        assert getattr(p, k) == getattr(o, k), k


def test_env_state_written_by_the_reference_loads(tmp_path):
    import walker_gym_b200.optimized_walker as ow
    env = ow.Environment()
    env.load_state(os.path.join(gu.GOLDEN_DIR, "env_state_ref.pkl"))
    assert len(env.points) == 2 and len(env.ding_points) == 1 and len(env.springs) == 3
    assert isinstance(env.ding_points[0], ow.DingPoint) and env.ding_points[0].fixed
    assert env.time_step == 0.02 and env.friction == 0.3 and env.gravity.dtype == np.float32
    assert env.springs[2][2] == 70.0 and env.springs[1][4] is True
    assert env.springs[0][0] is env.ding_points[0] and env.springs[0][1] is env.points[0]   # identity preserved
    # round trip through our writer
    out = tmp_path / "env_state.pkl"
    env.save_state(str(out))
    env2 = ow.Environment()
    env2.load_state(str(out))
    for a, b in zip(env.points + env.ding_points, env2.points + env2.ding_points):
        assert gu.same(a.pos, b.pos) and gu.same(a.v, b.v) and a.m == b.m and a.fixed == b.fixed
    assert [s[2:] for s in env.springs] == [s[2:] for s in env2.springs]


def test_env_state_rejects_foreign_classes(tmp_path):
    import pickle
    import walker_gym_b200.optimized_walker as ow
    bad = tmp_path / "bad.pkl"
    bad.write_bytes(pickle.dumps({"points": [subprocess.Popen], "ding_points": []}, protocol=4))
    with pytest.raises(pickle.UnpicklingError):
        ow.Environment().load_state(str(bad))


@pytest.mark.reference
def test_reference_reads_env_state_we_write(tmp_path):
    """The reference's own Environment.load_state accepts a file written by save_state."""
    import ref_harness_l2 as r2
    if not r2.available():
        pytest.skip("reference checkout not present")
    env, _ = build("leg2", ground_level=-30)
    out = tmp_path / "env_state.pkl"
    env.save_state(str(out))
    code = ("import sys\nfrom unittest import mock\nsys.modules['pygame'] = mock.MagicMock()\n"
            f"sys.path.insert(0, {os.path.join(r2.DEFAULT_REF, 'gym')!r})\nfrom optimized_walker.env import Environment\n"
            f"e = Environment(); e.load_state({str(out)!r})\n"
            "e.update_physics()\n"
            "print(len(e.points), len(e.springs), e.ground_level, type(e.points[0]).__module__)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["7", "6", "-30", "optimized_walker.core"]


def test_snapshot_schema_of_the_package_lineage(tmp_path):
    import walker_gym_b200.optimized_walker as ow
    ow.Point.clear()
    ow.Point(2, (1, 2, 3), (0, 1, 0))
    ow.DingPoint(0, (0, 5, 0), (0, 0, 0))
    ow.Point.fps = 17
    f = tmp_path / "state.pkl"
    ow.Point.snapshot(str(f))
    ow.Point.clear()
    ow.Point.load_snapshot(str(f))
    assert len(ow.Point.points) == 2 and ow.Point.fps == 17 and ow.Point.points[1].fixed
    assert gu.same(ow.Point.points[0].pos, np.array([1, 2, 3], np.float32))


def test_update_physics_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    env, _ = build("box")
    with pytest.raises(Exception):
        env.update_physics()
    assert gu.same(env.points[0].pos, np.array([-5, 5, -5], np.float32))      # nothing was computed on the host
