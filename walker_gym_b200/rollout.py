"""PPO rollout collection around the fused step kernel (BASELINE.json config 5, SURVEY 8 f1).

The caller of the hot path: a small torch MLP policy acts on the observation, the
CUDA kernel steps every env, and the trajectory (obs, action, log-prob, value,
reward, done) is written into preallocated device buffers.  Everything stays on
the device.  To keep the per-step launch overhead off the critical path the whole
T-step rollout (policy kernels + step kernel per step) is captured once into a
CUDA graph and replayed; the env runs in ``graph_safe`` mode so the in-kernel
Philox jitter keeps advancing across replays.  The policy consumes the
observation feature-major ([D, E]) -- the layout the kernel writes straight from
registers with coalesced stores -- and emits feature-major actions ([M, E]).
Returns/advantages (GAE) are computed on the device; episode-return statistics
are reduced by the K3 kernel and all-reduced across ranks (NCCL), once per rollout.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional

import torch

from . import _lib
from .batched import BatchedPhysicsEnv


class FusedPolicy:
    """``FeatureMajorMLP`` evaluated by ``wg_policy_act``: one CUDA kernel per env step instead of ~25 torch
    kernels.  Reads the module's parameters in place (no copies: an optimiser step is visible to the next call).
    ``precision="fp32"`` uses error-compensated 3xTF32 tensor-core products (float32-grade), ``"tf32"`` plain TF32."""

    def __init__(self, module: "FeatureMajorMLP", precision: str = "fp32"):
        if precision not in ("fp32", "tf32"):
            raise ValueError("precision must be 'fp32' or 'tf32'")
        hidden, obs_dim = module.l1.weight.shape
        act_dim = module.mu.weight.shape[0]
        if hidden != 64 or tuple(module.l2.weight.shape) != (64, 64) or not 1 <= obs_dim <= 64 or not 1 <= act_dim <= 7:
            raise ValueError("the fused policy kernel needs hidden == 64, obs_dim <= 64 and act_dim <= 7")
        self.module, self.obs_dim, self.act_dim = module, int(obs_dim), int(act_dim)
        self.lib = _lib.load()
        self.precision = precision

    def _struct(self) -> "_lib.WgMlpPolicy":
        m, p = self.module, _lib.WgMlpPolicy()
        tensors = dict(w1=m.l1.weight, b1=m.l1.bias, w2=m.l2.weight, b2=m.l2.bias, w_mu=m.mu.weight, b_mu=m.mu.bias,
                       w_v=m.v.weight, b_v=m.v.bias, log_std=m.log_std)
        for name, t in tensors.items():
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device.type != "cuda":
                raise ValueError(f"policy parameter {name} must be a contiguous float32 CUDA tensor")
            setattr(p, name, t.data_ptr())
        p.obs_dim, p.act_dim = self.obs_dim, self.act_dim
        p.obs_scale, p.obs_clip = float(m.obs_scale), float(m.obs_clip)
        p.precision = 0 if self.precision == "fp32" else 1
        return p

    def act(self, obs_fm: torch.Tensor, *, action=None, logp=None, value=None, mean=None, sample: bool = True,
            seed: int = 0, step_index: int = 0, step_counter: Optional[torch.Tensor] = None, env_offset: int = 0,
            act_layout: str = "feature", obs_layout: str = "feature") -> None:
        """obs [D, E] (or [E, D] with obs_layout="row") -> any of action [M, E] (or [E, M] with act_layout="row"),
        logp [E], value [E], mean [M, E]."""
        D, E = obs_fm.shape if obs_layout == "feature" else obs_fm.shape[::-1]
        if D != self.obs_dim or obs_fm.dtype != torch.float32 or not obs_fm.is_contiguous():
            raise ValueError(f"obs must be a contiguous float32 [{self.obs_dim}, E] (feature) or [E, {self.obs_dim}] (row) tensor")
        for t, n in ((action, self.act_dim * E), (logp, E), (value, E), (mean, self.act_dim * E)):
            if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n):
                raise ValueError("outputs must be contiguous float32 tensors of the documented shapes")
        pol = self._struct()
        ptr = lambda t: None if t is None else t.data_ptr()          # noqa: E731
        with torch.cuda.device(obs_fm.device):
            rc = self.lib.wg_policy_act(C.byref(pol), obs_fm.data_ptr(), 1 if obs_layout == "feature" else 0,
                                        ptr(action), 1 if act_layout == "feature" else 0,
                                        ptr(logp), ptr(value), ptr(mean), E, 1 if sample else 0,
                                        seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, step_index & 0xFFFFFFFF,
                                        ptr(step_counter), env_offset & 0xFFFFFFFF,
                                        C.c_void_p(torch.cuda.current_stream(obs_fm.device).cuda_stream))
        _lib.check(rc, "wg_policy_act")


def gae_trunc(rewards, values, dones, truncated, final_values, advantages, returns, gamma: float, lam: float,
              reward_clip: float) -> None:
    """``wg_gae_trunc``: ``gae`` whose truncated steps (truncated [T, E], 1-byte) bootstrap from final_values [T, E]
    instead of 0.  final_values is read only where a step is both done and truncated."""
    T, E = rewards.shape
    if values.shape != (T + 1, E) or dones.shape != (T, E) or truncated.shape != (T, E) or final_values.shape != (T, E) \
            or dones.element_size() != 1 or truncated.element_size() != 1:
        raise ValueError("gae_trunc: shape mismatch")
    with torch.cuda.device(rewards.device):
        rc = _lib.load().wg_gae_trunc(rewards.data_ptr(), values.data_ptr(), dones.data_ptr(), truncated.data_ptr(),
                                      final_values.data_ptr(), advantages.data_ptr(), returns.data_ptr(), T, E, gamma, lam,
                                      reward_clip, C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream))
    _lib.check(rc, "wg_gae_trunc")


def gae(rewards, values, dones, advantages, returns, gamma: float, lam: float, reward_clip: float) -> None:
    """``wg_gae``: rewards [T, E], values [T+1, E], dones [T, E] (1-byte) -> advantages, returns [T, E]."""
    T, E = rewards.shape
    if values.shape != (T + 1, E) or dones.shape != (T, E) or dones.element_size() != 1:
        raise ValueError("gae: shape mismatch")
    with torch.cuda.device(rewards.device):
        rc = _lib.load().wg_gae(rewards.data_ptr(), values.data_ptr(), dones.data_ptr(), advantages.data_ptr(),
                                returns.data_ptr(), T, E, gamma, lam, reward_clip,
                                C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream))
    _lib.check(rc, "wg_gae")


class FeatureMajorMLP(torch.nn.Module):
    """obs [D, E] -> (action mean [M, E], value [E]); two tanh hidden layers of ``hidden`` units."""

    def __init__(self, obs_dim: int, act_dim: int, hidden: int = 64, obs_scale: float = 1e-2, obs_clip: float = 10.0):
        super().__init__()
        self.obs_scale, self.obs_clip = obs_scale, obs_clip
        self.l1 = torch.nn.Linear(obs_dim, hidden)
        self.l2 = torch.nn.Linear(hidden, hidden)
        self.mu = torch.nn.Linear(hidden, act_dim)
        self.v = torch.nn.Linear(hidden, 1)
        self.log_std = torch.nn.Parameter(torch.full((act_dim, 1), -0.5))

    def forward(self, obs_fm: torch.Tensor):
        # exploded envs produce inf/NaN observations (SURVEY 0.5): sanitise before the first layer
        x = torch.nan_to_num(obs_fm * self.obs_scale, nan=0.0, posinf=self.obs_clip, neginf=-self.obs_clip)
        x = x.clamp_(-self.obs_clip, self.obs_clip)
        h = torch.tanh(torch.addmm(self.l1.bias[:, None], self.l1.weight, x))
        h = torch.tanh(torch.addmm(self.l2.bias[:, None], self.l2.weight, h))
        mean = torch.addmm(self.mu.bias[:, None], self.mu.weight, h)
        value = torch.addmm(self.v.bias[:, None], self.v.weight, h)[0]
        return mean, value


class RolloutCollector:
    """Collect ``horizon`` steps from a ``BatchedPhysicsEnv`` under a policy.

    The env must be built with ``graph_safe=True`` for CUDA-graph rollouts.  The fused collector (default for a
    ``FeatureMajorMLP``) takes either layout; row-major observations (``obs_layout="row"``, the step kernel's fastest
    path) and row-major actions are the fastest combination.  The torch-op collector needs feature-major both.
    ``collect()`` returns views of device buffers: obs [T+1, D, E] (or [T+1, E, D]), actions [T, M, E] (or [T, E, M]),
    logp/values/rewards [T(+1), E], dones [T, E].

    ``bootstrap_truncated``: what the returns of an episode that hit ``max_steps`` bootstrap from.  ``None`` (default):
    nothing -- every ``done`` is treated as termination, which biases the returns of time-limited episodes towards zero.
    ``"final"``: the value of the state the episode ended in -- after each step a value-only policy pass over
    ``env.final_obs`` fills ``final_values[t]`` -- the exact time-limit correction, at one extra value pass per step.
    ``"current"``: the value V(s_t) of the state the truncated step started from (legged_gym / rsl_rl's approximation; no
    extra policy pass).  Both need ``BatchedPhysicsEnv(track_truncation=True)``; ``collect()`` then adds ``truncated``
    [T, E] and, for ``"final"``, ``final_values`` [T, E] (rows of steps that are not done hold whatever the value pass made
    of stale observations; GAE never reads them)."""

    def __init__(self, env: BatchedPhysicsEnv, policy: torch.nn.Module, horizon: int, *, gamma: float = 0.99,
                 lam: float = 0.95, use_cuda_graph: bool = True, reward_clip: float = 1e3, fused: Optional[bool] = None,
                 precision: str = "fp32", seed: int = 0, fuse_step: bool = False,
                 bootstrap_truncated: Optional[str] = None):
        if bootstrap_truncated not in (None, "current", "final"):
            raise ValueError("bootstrap_truncated must be None, 'current' or 'final'")
        if bootstrap_truncated is not None and env.truncated is None:
            raise ValueError("bootstrap_truncated needs BatchedPhysicsEnv(track_truncation=True)")
        self.bootstrap_truncated = bootstrap_truncated
        row = env.obs_layout == "row" or env.act_layout == "row"
        if row and fused is False:
            raise ValueError("the torch-op collector needs obs_layout='feature' and act_layout='feature'")
        if use_cuda_graph and env._counter is None:
            raise ValueError("CUDA-graph rollouts need BatchedPhysicsEnv(graph_safe=True)")
        self.env, self.policy, self.T = env, policy, int(horizon)
        self.gamma, self.lam, self.reward_clip = gamma, lam, reward_clip
        E, D, M, dev = env.num_envs, env.obs_dim, env.M, env.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs = torch.zeros((self.T + 1, D, E) if env.obs_layout == "feature" else (self.T + 1, E, D), **f32)
        self.actions = torch.zeros((self.T, M, E) if env.act_layout == "feature" else (self.T, E, M), **f32)
        self.logp = torch.zeros(self.T, E, **f32)
        self.values = torch.zeros(self.T + 1, E, **f32)
        self.rewards = torch.zeros(self.T, E, **f32)
        self.dones = torch.zeros(self.T, E, dtype=torch.bool, device=dev)
        self.truncated = torch.zeros(self.T, E, dtype=torch.bool, device=dev) if bootstrap_truncated else None
        self.final_values = torch.zeros(self.T, E, **f32) if bootstrap_truncated == "final" else None
        self.advantages = torch.zeros(self.T, E, **f32)
        self.returns = torch.zeros(self.T, E, **f32)
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._use_graph = use_cuda_graph
        # fused: the policy runs in wg_policy_act and GAE in wg_gae (2 launches per env step); otherwise torch ops.
        # In fused mode ``rewards`` holds the raw env rewards (wg_gae sanitises them on the fly).
        can_fuse = isinstance(policy, FeatureMajorMLP) and policy.l1.weight.shape[0] == 64 and D <= 64 and 1 <= M <= 7
        if (fused or row) and not can_fuse:
            raise ValueError("the fused collector needs a FeatureMajorMLP with hidden=64, obs_dim <= 64, 1 <= act_dim <= 7")
        self.fused = can_fuse if fused is None else bool(fused)
        self._fp = FusedPolicy(policy, precision) if self.fused else None
        self.seed = int(seed)
        # fuse_step=True: one launch per env step where the library has the env step fused into the policy pipeline
        # (wg_policy_step: Balance-v0, 3-D, packed state, row-major observations / actions, no truncation flag; probed
        # with an empty call).
        # Bit-identical to the two launches but measured SLOWER on B200 (71 vs 53 us per 2^18-env step: the output warps
        # that carry the step run its long straight-line body almost alone on their schedulers), hence off by default --
        # see DESIGN.md, K5.
        self.fused_step = bool(self.fused and fuse_step and not env.x64 and env.state_layout == "packed"
                               and env.obs_layout == "row" and env.act_layout == "row" and self._policy_step(0, probe=True))
        self.kernel_launches_per_rollout = ((self.T if self.fused_step else 2 * self.T) + 2 +
                                            (self.T if bootstrap_truncated == "final" else 0)) if self.fused else self.T   # ours only

    def _policy_step(self, t: int, probe: bool = False) -> bool:
        """``wg_policy_step``: policy evaluation of ``obs[t]`` + ``env.step`` with the sampled action in ONE launch; results
        in ``actions[t]``, ``logp[t]``, ``values[t]``, ``obs[t + 1]``, ``rewards[t]``, ``dones[t]``.  False = the library has
        no fused kernel for this env / policy (the caller makes the two calls)."""
        env, fp = self.env, self._fp
        lib, b = fp.lib, env._buf
        pol = fp._struct()
        p = (lambda x: x.data_ptr())
        saved = (b.action, b.act_dim, b.noise, b.obs, b.reward, b.done)
        b.action, b.act_dim, b.noise = None, 0, None
        if not probe:
            b.obs, b.reward, b.done = p(self.obs[t + 1]), p(self.rewards[t]), p(self.dones.view(torch.uint8)[t])
            env._stamp()
        try:
            with torch.cuda.device(env.device):
                rc = lib.wg_policy_step(C.byref(pol), C.byref(env.topo), C.byref(env.params), C.byref(b),
                                        p(self.obs[0 if probe else t]), p(self.actions[0 if probe else t]),
                                        p(self.logp[0 if probe else t]), p(self.values[0 if probe else t]), None,
                                        0 if probe else env.num_envs, 1, self.seed & 0xFFFFFFFF, (self.seed >> 32) & 0xFFFFFFFF,
                                        (t if env._counter is not None else env.step_count) & 0xFFFFFFFF,
                                        int(env.params.env_offset) & 0xFFFFFFFF, env._stream())
        finally:
            b.action, b.act_dim, b.noise, b.obs, b.reward, b.done = saved
        if rc == -2:
            return False
        _lib.check(rc, "wg_policy_step")
        if not probe:
            env._advance()
        return True

    @torch.no_grad()
    def _rollout_fused(self) -> None:
        env, fp = self.env, self._fp
        dones_u8 = self.dones.view(torch.uint8)
        kw = dict(seed=self.seed, step_counter=env._counter, env_offset=int(env.params.env_offset),
                  obs_layout=env.obs_layout, act_layout=env.act_layout)
        self.obs[0].copy_(env.obs)
        with env.deferred_steps(self.T):             # graph-safe mode: one counter update per rollout, not per step
            for t in range(self.T):
                env._step_offset = t
                if self.fused_step and self._policy_step(t):
                    continue
                fp.act(self.obs[t], action=self.actions[t], logp=self.logp[t], value=self.values[t], sample=True,
                       step_index=t if env._counter is not None else env.step_count, **kw)
                out = (self.obs[t + 1], self.rewards[t], dones_u8[t])
                env.step(self.actions[t], out=out if self.truncated is None else out + (self.truncated[t],))
                if self.final_values is not None:        # "final": the value of the state each ended episode ended in
                    fp.act(env.final_obs, value=self.final_values[t], sample=False, **kw)
        fp.act(self.obs[self.T], value=self.values[self.T], sample=False, **kw)
        env.obs.copy_(self.obs[self.T])                  # keep env.obs current for the next rollout / other callers
        if self.truncated is None:
            gae(self.rewards, self.values, dones_u8, self.advantages, self.returns, self.gamma, self.lam, self.reward_clip)
        else:                                            # a truncated step bootstraps from V(final state) or V(s_t)
            fv = self.final_values if self.final_values is not None else self.values[: self.T]
            gae_trunc(self.rewards, self.values, dones_u8, self.truncated.view(torch.uint8), fv,
                      self.advantages, self.returns, self.gamma, self.lam, self.reward_clip)

    @torch.no_grad()
    def _rollout(self) -> None:
        if self.fused:
            return self._rollout_fused()
        env, pol = self.env, self.policy
        self.obs[0].copy_(env.obs)
        for t in range(self.T):
            mean, value = pol(self.obs[t])
            std = pol.log_std.exp()
            eps = torch.randn_like(mean)
            act = torch.addcmul(mean, std, eps, out=self.actions[t])
            self.logp[t] = (-0.5 * eps * eps - pol.log_std - 0.5 * math.log(2 * math.pi)).sum(0)
            self.values[t] = value
            obs, rew, done, info = env.step(act)
            if self.truncated is not None:
                self.truncated[t] = info["truncated"]
            if self.final_values is not None:
                self.final_values[t] = pol(env.final_obs)[1]
            self.obs[t + 1].copy_(obs)
            r = torch.nan_to_num(rew, nan=0.0, posinf=self.reward_clip, neginf=-self.reward_clip)
            self.rewards[t] = r.clamp_(-self.reward_clip, self.reward_clip)
            self.dones[t] = done
        self.values[self.T] = pol(self.obs[self.T])[1]
        # GAE(lambda) on the device
        adv = torch.zeros_like(self.values[0])
        for t in range(self.T - 1, -1, -1):
            nonterminal = (~self.dones[t]).to(torch.float32)
            if self.truncated is None:
                delta = self.rewards[t] + self.gamma * self.values[t + 1] * nonterminal - self.values[t]
            else:                                        # a truncated step bootstraps from V(final state) or V(s_t)
                fv = self.final_values[t] if self.final_values is not None else self.values[t]
                final = torch.nan_to_num(fv, nan=0.0).clamp(-self.reward_clip, self.reward_clip)
                boot = torch.where(self.dones[t], torch.where(self.truncated[t], final, 0.0), self.values[t + 1])
                delta = self.rewards[t] + self.gamma * boot - self.values[t]
            adv = delta + self.gamma * self.lam * nonterminal * adv
            self.advantages[t] = adv
        torch.add(self.advantages, self.values[: self.T], out=self.returns)

    def collect(self) -> Dict[str, torch.Tensor]:
        if not self._use_graph:
            self._rollout()
        else:
            if self._graph is None:
                # warm-up outside capture (allocator, cuBLAS handles) on a snapshot: the env, its device step counter and
                # the finished-episode accumulators are restored, so the first collect() advances the env by exactly
                # `horizon` steps and its statistics hold only what was returned
                snap = self.env.state_dict()
                s = torch.cuda.Stream(device=self.env.device)
                s.wait_stream(torch.cuda.current_stream(self.env.device))
                with torch.cuda.stream(s):
                    self._rollout()
                torch.cuda.current_stream(self.env.device).wait_stream(s)
                self.env.load_state_dict(snap)
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._rollout()
            self._graph.replay()
        out = {"obs": self.obs, "actions": self.actions, "logp": self.logp, "values": self.values,
               "rewards": self.rewards, "dones": self.dones, "advantages": self.advantages, "returns": self.returns}
        if self.truncated is not None:
            out["truncated"] = self.truncated
        if self.final_values is not None:
            out["final_values"] = self.final_values
        return out

    def episode_stats(self, all_reduce: bool = True) -> dict:
        """Finished-episode return statistics of all ranks: K3 reduction + one NCCL all-reduce of 8 doubles.  Also the
        point where the tcgen05 policy kernel's diagnostic flag is read (it synchronises the device anyway): a kernel
        that ever gave up on one of its bounded barrier waits produced garbage, and that must not go unnoticed."""
        if self.fused and _lib.load().wg_policy_tc_status() != 0:
            raise _lib.WalkerGymError("a tcgen05 policy kernel gave up waiting on one of its barriers (wg_policy_tc_status)")
        return self.env.episode_stats(all_reduce=all_reduce)
