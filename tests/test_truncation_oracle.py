"""CPU: time-limit truncation restated on the C oracle (tests/truncation_ref.py), and what needs no GPU of its API.

- The restatement (oracle stepped without a time limit and without auto-reset, the time limit and the resets applied
  after it) is the oracle's own auto-reset run, bit for bit: obs, reward, done, state and the episode accumulators, for
  Balance-v0 and quad_balance, template and jitter resets, short and 1000-step limits.
- A hand-built step on which the time limit and a fall coincide counts as terminated.
- Argument validation of the C ABI and of BatchedPhysicsEnv / RolloutCollector options."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_util as gu
import nonfinite_ref as nr
import truncation_ref as tr
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
    if name == "balance_v0":
        return wo.BALANCE
    from test_cuda_vs_oracle import spec_of
    return spec_of(name)


def _start(spec, E, *, auto, k_sub=1, max_steps=1000, seed=1234):
    body = wo.make_body(spec)
    prm = wo.make_params(in3d=True, auto_reset=auto, max_steps=max_steps, k_sub=k_sub, seed=seed)
    st = wo.init_state(body, E)
    prm.step_index = 0
    wo.reset(body, prm, st, mode=2)
    return body, prm, st


@pytest.mark.parametrize("name,k_sub,auto,max_steps,E,T", [
    ("balance_v0", 1, 2, 10, 4096, 45),
    ("balance_v0", 1, 1, 10, 4096, 45),
    ("quad_balance", 8, 2, 7, 1024, 30),
    ("quad_balance", 8, 1, 7, 1024, 30),
    ("balance_v0", 1, 2, 1000, 256, 1005),
])
def test_restatement_is_the_oracle(name, k_sub, auto, max_steps, E, T):
    spec = _spec(name)
    body, prm, st = _start(spec, E, auto=auto, k_sub=k_sub, max_steps=max_steps)
    _, prm2, st2 = _start(spec, E, auto=auto, k_sub=k_sub, max_steps=max_steps)
    for s in (st, st2):                   # every 5th env starts far below fall_thresh: it falls on its first step
        s["pos"][1::3, ::5] = -1000.0
    stats = nr.new_stats(E)
    ep, fin = np.zeros(E, np.float32), np.zeros((4, E), np.float32)
    rng = np.random.default_rng(0)
    truncs = terms = 0
    for t in range(T):
        act = rng.uniform(-1, 1, (E, body.n_muscle)).astype(np.float32)
        prm.step_index = prm2.step_index = t + 1
        a = tr.step(body, prm, st, act, stats=stats)
        b = wo.step(body, prm2, st2, act, want_info=False, ep_ret=ep, fin_stats=fin)
        for k in ("obs", "reward", "done"):
            assert gu.same(a[k], b[k]), f"{k} at step {t}"
        for k in ("pos", "vel", "old_a", "mx", "steps"):
            assert gu.same(st[k], st2[k]), f"{k} at step {t}"
        assert not (a["truncated"].astype(bool) & ~a["done"].astype(bool)).any()
        truncs += int(a["truncated"].sum())
        terms += int((a["done"].astype(bool) & ~a["truncated"].astype(bool)).sum())
    assert gu.same(stats[0], ep) and gu.same(stats[1], fin)
    assert truncs > 0
    assert terms >= E // 5, "the seeded falls did not terminate"


def test_time_limit_and_fall_on_the_same_step_count_as_terminated():
    """Env 0 falls on its time-limit step, env 1 reaches the time limit upright, env 2 falls mid-episode, env 3 goes on."""
    E, max_steps = 4, 10
    body, prm, st = _start(wo.BALANCE, E, auto=2, max_steps=max_steps)
    st["pos"][1::3, 0] = -1000.0          # every mass far below fall_thresh (ground - 50)
    st["pos"][1::3, 2] = -1000.0
    st["steps"][:] = [max_steps - 1, max_steps - 1, 3, 3]
    prm.step_index = 1
    out = tr.step(body, prm, st, np.zeros((E, body.n_muscle), np.float32))
    assert list(out["done"]) == [1, 1, 1, 0]
    assert list(out["truncated"]) == [0, 1, 0, 0]


def test_end_nonfinite_on_the_time_limit_step_counts_as_terminated():
    """A non-finite reward on the time-limit step under the 'end' rule is a termination."""
    E, max_steps = 2, 10
    body, prm, st = _start(wo.BALANCE, E, auto=2, max_steps=max_steps)
    st["vel"][0, :] = np.inf
    st["steps"][:] = max_steps - 1
    prm.step_index = 1
    out = tr.step(body, prm, st, np.zeros((E, body.n_muscle), np.float32), end_nonfinite=True)
    assert nr.nonfinite(out["reward"]).all()
    assert list(out["done"]) == [1, 1] and list(out["truncated"]) == [0, 0]


def test_abi_without_a_gpu():
    """wg_buffers gained two trailing fields and the version is 5; final_obs needs obs; the host paths refuse them;
    wg_gae_trunc validates."""
    from walker_gym_b200 import _lib, create_balance_creature, make_params
    from walker_gym_b200.topology import topology_from_creature
    lib = _lib.load()
    assert lib.wg_abi_version() == 5 and _lib.ABI_VERSION == 5
    names = [f[0] for f in _lib.WgBuffers._fields_]
    assert names[-3:] == ["nf_stats", "truncated", "final_obs"]
    assert _lib.WgBuffers.truncated.offset == _lib.WgBuffers.nf_stats.offset + 8
    assert _lib.WgBuffers.final_obs.offset == _lib.WgBuffers.truncated.offset + 8
    assert C.sizeof(_lib.WgBuffers) == _lib.WgBuffers.final_obs.offset + 8
    assert hasattr(lib, "wg_gae_trunc")
    topo = topology_from_creature(create_balance_creature())
    buf = _lib.WgBuffers()
    dummy = (C.c_float * 64)()
    buf.pos = buf.vel = buf.mx = buf.steps = buf.truncated = C.addressof(dummy)
    prm = make_params(in3d=True, auto_reset=2)
    assert lib.wg_step_host(C.byref(topo), C.byref(prm), C.byref(buf), 4, None, None, None, None, None) == -1
    assert b"truncated" in lib.wg_last_error_string()
    assert lib.wg_step_multi_host(C.byref(topo), C.byref(prm), C.byref(buf), 4, 2, 2, None, None, None, None, None) == -1
    assert b"truncated" in lib.wg_last_error_string()
    buf.truncated, buf.final_obs = None, C.addressof(dummy)
    assert lib.wg_step(C.byref(topo), C.byref(prm), C.byref(buf), 4, None) == -1
    assert b"final_obs needs obs" in lib.wg_last_error_string()
    buf.obs = C.addressof(dummy)
    assert lib.wg_step_host(C.byref(topo), C.byref(prm), C.byref(buf), 4, None, None, None, None, None) == -1
    assert b"final_obs" in lib.wg_last_error_string()
    p = C.addressof(dummy)
    assert lib.wg_gae_trunc(p, p, p, None, p, p, p, 2, 4, 0.99, 0.95, 10.0, None) == -1
    assert lib.wg_gae_trunc(p, p, p, p, p, p, p, -1, 4, 0.99, 0.95, 10.0, None) == -1
    assert lib.wg_gae_trunc(p, p, p, p, p, p, p, 0, 4, 0.99, 0.95, 10.0, None) == 0


def test_collector_option_validation_without_a_gpu():
    from walker_gym_b200.rollout import RolloutCollector

    class FakeEnv:
        truncated = None
    with pytest.raises(ValueError, match="bootstrap_truncated must be"):
        RolloutCollector(FakeEnv(), None, 4, bootstrap_truncated="next")
    for mode in ("current", "final"):
        with pytest.raises(ValueError, match="track_truncation"):
            RolloutCollector(FakeEnv(), None, 4, bootstrap_truncated=mode)
