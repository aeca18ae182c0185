"""Test helper: the ``nonfinite`` option of BatchedPhysicsEnv restated on top of the C oracle.

The oracle implements the reference's step as written.  The option adds two rules, both restated here in NumPy:
  - with ``mode="end"``, a step whose reward is not finite (``!(|reward| <= FLT_MAX)``) also sets ``done``; the env is
    then reset like any other done env.  The oracle steps with auto-reset off and ``wo.reset`` resets the done envs
    with the same Philox step index (a template reset does not depend on ``old_a``, so the observation is the one the
    in-step reset writes);
  - with ``mode="count"`` or ``"end"``, a finished episode whose return is not finite goes into ``nf_stats`` [2][E]
    (count, length sum) instead of ``fin_stats`` [4][E] (return, return^2, length, count).
The accumulators are summed in float32 in step order, as the kernels sum them."""
import numpy as np

import walker_oracle as wo

F32_MAX = np.float32(np.finfo(np.float32).max)
MODES = ("keep", "count", "end")


def nonfinite(x):
    """!(|x| <= FLT_MAX), elementwise: the kernels' test."""
    with np.errstate(invalid="ignore"):
        return ~(np.abs(x) <= F32_MAX)


def new_stats(E):
    """(ep_ret [E], fin_stats [4, E], nf_stats [2, E]) all zero, float32."""
    return np.zeros(E, np.float32), np.zeros((4, E), np.float32), np.zeros((2, E), np.float32)


def account(mode, done, reward, steps_before, ep_ret, fin_stats, nf_stats, auto_reset):
    """One step of episode accounting, in place; the lengths of episodes that end now are steps_before + 1."""
    with np.errstate(invalid="ignore", over="ignore"):
        r = (ep_ret + reward).astype(np.float32)
        ended = done.astype(bool)
        apart = ended & nonfinite(r) if mode != "keep" else np.zeros_like(ended)
        fin = ended & ~apart
        length = (steps_before + 1).astype(np.float32)
        fin_stats[0, fin] += r[fin]
        fin_stats[1, fin] += r[fin] * r[fin]
        fin_stats[2, fin] += length[fin]
        fin_stats[3, fin] += np.float32(1)
        nf_stats[0, apart] += np.float32(1)
        nf_stats[1, apart] += length[apart]
        ep_ret[:] = np.where(ended & bool(auto_reset), np.float32(0), r)


def step(body, prm, st, action, *, mode="keep", stats=None, xb=None, action64=None):
    """One env-step of every env of ``st`` (in place) under ``mode``; ``stats`` = new_stats(E) or None.
    ``xb`` / ``action64``: x64 mode (wo.step_x64).  Returns dict(obs, reward, done)."""
    assert mode in MODES
    auto = int(prm.auto_reset)
    assert not (mode == "end" and auto == 1), "end needs a template reset (or none)"
    steps_before = st["steps"].copy()
    if mode == "end":
        prm.auto_reset = 0
    try:
        if xb is None:
            out = wo.step(body, prm, st, action, want_info=False)
        else:
            out = wo.step_x64(body, xb, prm, st, action64, want_info=False)
    finally:
        prm.auto_reset = auto
    done = out["done"].astype(bool)
    if mode == "end":
        done |= nonfinite(out["reward"])
        if auto and done.any():
            obs_r = wo.reset(body, prm, st, mode=auto, mask=done.astype(np.uint8))
            out["obs"][done] = obs_r[done]
            if xb is not None:                      # a fresh Muscle: x = originx, float32-typed
                M = body.n_muscle
                st["mx64"][:, done] = np.array([xb.x0_d[m] for m in range(M)], np.float64)[:, None]
                st["mx_weak"][:, done] = 1
        out["done"] = done.astype(np.uint8)
    if stats is not None:
        account(mode, done, out["reward"], steps_before, *stats, auto)
    return out
