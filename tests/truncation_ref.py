"""Test helper: time-limit truncation (``BatchedPhysicsEnv(track_truncation=True)``) restated on top of the C oracle.

The oracle implements the reference's step as written, whose ``_is_done`` stops at the time limit.  The restatement
  1. steps the oracle with ``max_steps = INT32_MAX`` and auto-reset off: the dynamics do not depend on ``max_steps``, so
     this gives the step's results and the terminal-only ``done`` (the fall, all masses stopped after step 100);
  2. adds ``nonfinite_ref``'s "end" rule to the terminal set when it is on;
  3. sets ``timelimit = steps_after >= max_steps``, ``done = terminal | timelimit``,
     ``truncated = timelimit & ~terminal``;
  4. keeps the observation of step 1 as ``final_obs`` (the pre-reset observation of the done envs), then resets the
     done envs with ``wo.reset`` at the same Philox index.
The episode accumulators are those of ``nonfinite_ref.account``."""
import numpy as np

import nonfinite_ref as nr
import walker_oracle as wo

INT32_MAX = (1 << 31) - 1


def step(body, prm, st, action, *, end_nonfinite=False, stats=None):
    """One env-step of every env of ``st`` (in place); ``stats`` = nonfinite_ref.new_stats(E) or None.
    Returns dict(obs, reward, done, truncated, final_obs) with done / truncated as uint8; final_obs rows of envs that
    are not done are this step's observation too, but only the done rows are specified."""
    max_steps, auto = int(prm.max_steps), int(prm.auto_reset)
    steps_before = st["steps"].copy()
    prm.max_steps, prm.auto_reset = INT32_MAX, 0
    try:
        out = wo.step(body, prm, st, action, want_info=False)
    finally:
        prm.max_steps, prm.auto_reset = max_steps, auto
    term = out["done"].astype(bool)
    if end_nonfinite:
        term |= nr.nonfinite(out["reward"])
    timelimit = st["steps"] >= max_steps
    done = term | timelimit
    out["final_obs"] = out["obs"].copy()
    if auto and done.any():
        obs_r = wo.reset(body, prm, st, mode=auto, mask=done.astype(np.uint8))
        out["obs"][done] = obs_r[done]
    out["done"] = done.astype(np.uint8)
    out["truncated"] = (timelimit & ~term).astype(np.uint8)
    if stats is not None:
        nr.account("end" if end_nonfinite else "keep", done, out["reward"], steps_before, *stats, auto)
    return out
