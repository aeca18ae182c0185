"""CPU: the nonfinite option restated on the C oracle (tests/nonfinite_ref.py), and what needs no GPU of its API.

- The restatement with the rules inert is the oracle itself: stepping with auto-reset off and resetting the done envs
  with wo.reset gives the bits of the oracle's in-step auto-reset, and the NumPy accounting gives its fin_stats.
- Balance-v0 and quad_balance (8 substeps), 4096 envs x 1010 steps of 1000-step episodes with template resets: under
  "end" no returned observation holds inf / NaN; under "count" obs / reward / done are those of "keep", and the
  per-env episode counts and lengths of fin_stats + nf_stats are keep's.
- Argument validation of BatchedPhysicsEnv, the C ABI and finalize_stats."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_util as gu
import nonfinite_ref as nr
import walker_oracle as wo


@pytest.fixture(autouse=True)
def oracle_threads():
    old = int(wo.lib().wgo_get_max_threads())
    wo.set_threads(len(os.sched_getaffinity(0)))
    try:
        yield
    finally:
        wo.set_threads(old)


def _spec(name):
    from test_cuda_vs_oracle import spec_of
    return spec_of(name)


def _start(spec, E, *, k_sub=1, max_steps=1000, seed=1234):
    body = wo.make_body(spec)
    prm = wo.make_params(in3d=True, auto_reset=2, max_steps=max_steps, k_sub=k_sub, seed=seed)
    st = wo.init_state(body, E)
    st.pop("old_a")
    prm.step_index = 0
    obs = wo.reset(body, prm, st, mode=2)
    return body, prm, st, obs


def test_restatement_with_inert_rules_is_the_oracle():
    """Balance-v0, 4096 envs, 30 steps of 10-step episodes (no lane overflows this early): the composed 'end' step and the
    NumPy accounting equal wo.step with its own auto-reset and fin_stats, bit for bit."""
    E = 4096
    body, prm, st, _ = _start(wo.BALANCE, E, max_steps=10)
    _, prm2, st2, _ = _start(wo.BALANCE, E, max_steps=10)
    stats = nr.new_stats(E)
    ep, fin = np.zeros(E, np.float32), np.zeros((4, E), np.float32)
    rng = np.random.default_rng(0)
    for t in range(30):
        act = rng.uniform(-1, 1, (E, 2)).astype(np.float32)
        prm.step_index = prm2.step_index = t + 1
        a = nr.step(body, prm, st, act, mode="end", stats=stats)
        b = wo.step(body, prm2, st2, act, want_info=False, ep_ret=ep, fin_stats=fin)
        assert not nr.nonfinite(b["reward"]).any()
        for k in ("obs", "reward", "done"):
            assert gu.same(a[k], b[k]), f"{k} at step {t}"
        for k in ("pos", "vel", "mx", "steps"):
            assert gu.same(st[k], st2[k]), f"{k} at step {t}"
    assert gu.same(stats[0], ep) and gu.same(stats[1], fin) and not stats[2].any()
    assert fin[3].sum() == 3 * E


def test_accounting_matches_the_oracle_through_overflow():
    """keep-mode accounting in NumPy equals the oracle's own fin_stats also when returns are inf / NaN (60 steps of
    50-step episodes: most lanes overflow near step 34 and end at step 50 with a non-finite return)."""
    E = 4096
    body, prm, st, _ = _start(wo.BALANCE, E, max_steps=50)
    stats = nr.new_stats(E)
    ep, fin = np.zeros(E, np.float32), np.zeros((4, E), np.float32)
    rng = np.random.default_rng(1)
    for t in range(60):
        act = rng.uniform(-1, 1, (E, 2)).astype(np.float32)
        prm.step_index = t + 1
        before = st["steps"].copy()
        out = wo.step(body, prm, st, act, want_info=False, ep_ret=ep, fin_stats=fin)
        nr.account("keep", out["done"], out["reward"], before, *stats, 2)
    assert gu.same(stats[0], ep) and gu.same(stats[1], fin)
    assert nr.nonfinite(fin[0]).any(), "some returns overflowed"


@pytest.mark.parametrize("name,k_sub", [("balance_v0", 1), ("quad_balance", 8)])
def test_end_and_count_at_1010_steps(name, k_sub):
    """4096 envs x 1010 steps, 1000-step episodes, template resets, the same actions under all three modes."""
    E, T = 4096, 1010
    spec = wo.BALANCE if name == "balance_v0" else _spec(name)
    runs = {m: list(_start(spec, E, k_sub=k_sub)) + [nr.new_stats(E)] for m in nr.MODES}
    assert np.isfinite(runs["end"][3]).all()
    M = runs["keep"][0].n_muscle
    rng = np.random.default_rng(2)
    ended_nonfinite = 0
    for t in range(T):
        act = rng.uniform(-1, 1, (E, M)).astype(np.float32)
        out = {}
        for m, (body, prm, st, _, stats) in runs.items():
            prm.step_index = t + 1
            out[m] = nr.step(body, prm, st, act, mode=m, stats=stats)
        assert np.isfinite(out["end"]["obs"]).all(), f"end: non-finite observation at step {t}"
        ended_nonfinite += int((out["end"]["done"].astype(bool) & nr.nonfinite(out["end"]["reward"])).sum())
        for k in ("obs", "reward", "done"):
            assert gu.same(out["count"][k], out["keep"][k]), f"count vs keep: {k} at step {t}"
    assert ended_nonfinite > 0
    (_, kf, kn), (_, cf, cn) = runs["keep"][4], runs["count"][4]
    assert not kn.any()
    assert np.array_equal(cf[3] + cn[0], kf[3]) and np.array_equal(cf[2] + cn[1], kf[2])
    assert cn[0].sum() > 0 and np.isfinite(cf).all() and not np.isfinite(kf[0]).all()
    _, ef, en = runs["end"][4]
    assert np.isfinite(ef).all() and en[0].sum() > 0


def test_env_rejects_bad_combinations_without_a_gpu():
    from walker_gym_b200 import BatchedPhysicsEnv
    with pytest.raises(ValueError, match="jitter"):
        BatchedPhysicsEnv("Balance-v0", 8, "cuda", auto_reset="jitter", nonfinite="end")
    with pytest.raises(ValueError, match="track_stats"):
        BatchedPhysicsEnv("Balance-v0", 8, "cuda", track_stats=False, nonfinite="count")
    with pytest.raises(ValueError, match="nonfinite"):
        BatchedPhysicsEnv("Balance-v0", 8, "cuda", nonfinite="drop")


def test_abi_rejects_bad_combinations_without_a_gpu():
    from walker_gym_b200 import _lib, create_balance_creature, make_params
    from walker_gym_b200.topology import topology_from_creature
    lib = _lib.load()
    topo = topology_from_creature(create_balance_creature())
    buf = _lib.WgBuffers()
    dummy = (C.c_float * 64)()
    buf.pos = buf.vel = buf.mx = buf.steps = buf.ep_ret = C.addressof(dummy)
    prm = make_params(in3d=True, auto_reset=1, end_nonfinite=True)
    assert lib.wg_step(C.byref(topo), C.byref(prm), C.byref(buf), 4, None) == -1
    assert b"end_nonfinite" in lib.wg_last_error_string()
    prm = make_params(in3d=True, auto_reset=2)
    prm.end_nonfinite = 2
    assert lib.wg_step(C.byref(topo), C.byref(prm), C.byref(buf), 4, None) == -1
    prm.end_nonfinite = 0
    buf.nf_stats = C.addressof(dummy)
    assert lib.wg_step(C.byref(topo), C.byref(prm), C.byref(buf), 4, None) == -1
    assert b"nf_stats" in lib.wg_last_error_string()
    assert lib.wg_stats_reduce_split(None, C.addressof(dummy), 4, C.addressof(dummy), None) == -1


def test_finalize_stats_keys():
    from walker_gym_b200.dist import finalize_stats
    vec = [10.0, 60.0, 30.0, 2.0, 3.0, 120.0, 0.0, 0.0]
    keep = finalize_stats(vec)
    assert set(keep) == {"episodes", "return_mean", "return_std", "length_mean", "return_sum", "return_sqsum", "length_sum"}
    split = finalize_stats(vec, nonfinite=True)
    assert {k: split[k] for k in keep} == keep
    assert split["nonfinite_episodes"] == 3 and split["nonfinite_length_mean"] == 40.0
    empty = finalize_stats([0.0] * 8, nonfinite=True)
    assert empty["nonfinite_episodes"] == 0 and np.isnan(empty["nonfinite_length_mean"])
