"""``BatchedPhysicsEnv``: millions of independent walkers stepped by one CUDA kernel.

The per-env semantics are those of the reference's ``PhysicsEnv``
(gym/optimized_env.py:8-269); this class only adds the env axis.  PyTorch is
used for device memory and streams; every operation on the step path is a call
into ``libwalkergym_b200.so`` through its C ABI.

Layouts (float32, E = num_envs, N masses, M muscles, D = obs dim):
  pos, vel : [3N, E]   row n*3+c, env fastest (coalesced per mass component)
  mx       : [M, E]    current muscle rest lengths (Muscle.x)
  steps    : int32 [E]
  action   : [E, M]    row-major, what a policy emits
  obs      : [E, D] (obs_layout="row") or [D, E] (obs_layout="feature")
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Union

import numpy as np
import torch

from . import _lib
from ._lib import WgBuffers, WgParams
from .topology import topology_from_creature
from .walker import Creature, create_balance_creature, create_box_creature, make_creature, BODIES

AUTO_RESET = {None: 0, False: 0, "none": 0, "jitter": 1, "reference": 1, "template": 2, True: 2}
NONFINITE = ("keep", "count", "end")


def creature_from_id(env_id: str) -> Creature:
    """The ids ``make_env`` accepts (gym/optimized_env.py:273-294), case-insensitive,
    plus the names of the in-tree body tables."""
    key = env_id.lower()
    if key == "balance-v0":
        return create_balance_creature()
    if key == "box-v0":
        return create_box_creature()
    if key in BODIES:
        return make_creature(key)
    raise ValueError(f"Unknown environment ID: {key}")


def make_params(*, in3d=False, g=100, dampk=0, ground_high=0, ground_k=1000, ground_damp=100, friction=100,
                rand_sigma=0.1, time_step=0.01, max_steps=1000, k_sub=1, auto_reset=0, seed=0,
                step_index=0, env_offset=0, integrator="run1", end_nonfinite=False) -> WgParams:
    """PhysicsEnv's constructor arguments -> ``wg_params``.  Scalars are converted
    the way NumPy converts the reference's python numbers at their point of use.
    ``end_nonfinite``: a step whose reward is not finite also sets ``done`` (not in the reference)."""
    p = WgParams()
    p.g = float(g)
    p.dampk = np.float32(dampk)
    p.ground = np.float32(ground_high)
    p.fall_thresh = np.float32(ground_high - 50)
    p.ground_k, p.ground_damp, p.friction = np.float32(ground_k), np.float32(ground_damp), np.float32(friction)
    p.dt, p.sigma = np.float32(time_step), np.float32(rand_sigma)
    p.dt2 = np.float32(time_step ** 2)            # python `t ** 2`, cast where NumPy would cast it
    if integrator not in ("run1", "run2", 0, 1):
        raise ValueError("integrator must be 'run1' (Point.run1) or 'run2' (Point.run2)")
    p.integrator = 1 if integrator in ("run2", 1) else 0
    p.in3d, p.max_steps, p.k_sub, p.auto_reset = int(bool(in3d)), int(max_steps), int(k_sub), int(auto_reset)
    p.seed_lo, p.seed_hi = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    p.step_index, p.env_offset = int(step_index) & 0xFFFFFFFF, int(env_offset) & 0xFFFFFFFF
    p.end_nonfinite = int(bool(end_nonfinite))
    return p


class BatchedPhysicsEnv:
    def __init__(self, creature: Union[Creature, str], num_envs: int, device: Union[str, torch.device] = "cuda",
                 in3d: bool = False, g=100, dampk=0, ground_high=0, ground_k=1000, ground_damp=100,
                 friction=100, rand_sigma=0.1, *, max_steps: int = 1000, time_step: float = 0.01, k_sub: int = 1,
                 auto_reset="template", obs_layout: str = "row", act_layout: str = "row", seed: int = 0,
                 env_offset: int = 0, graph_safe: bool = False, integrator: str = "run1",
                 state_layout: str = "auto", x64: bool = False,
                 track_info: bool = False, track_stats: bool = True, track_contacts: bool = False,
                 keep_old_a: bool = False, initial_reset: bool = True, nonfinite: str = "keep"):
        """``nonfinite`` decides what happens to an env whose state overflowed to inf / NaN (Balance-v0 as written does
        so a few dozen steps after a reset; such an env then steps NaN arithmetic until ``max_steps``):
          "keep"  -- the reference's semantics: nothing special; its episode return enters the statistics (and makes
                     their mean NaN);
          "count" -- the same dynamics, observations, rewards and dones, bit for bit; a finished episode whose return
                     is not finite is counted apart (``episode_stats()["nonfinite_episodes"]``) instead of entering the
                     return statistics;
          "end"   -- as "count", and a step whose reward is not finite also sets ``done``, so the template auto-reset
                     (or the caller, with ``auto_reset="none"``) restarts the env.  Not with ``auto_reset="jitter"``:
                     a jitter reset keeps the overflowed positions."""
        if nonfinite not in NONFINITE:
            raise ValueError(f"nonfinite must be one of {NONFINITE}")
        if nonfinite != "keep" and not track_stats:
            raise ValueError(f"nonfinite={nonfinite!r} needs track_stats=True (it splits the episode statistics)")
        if nonfinite == "end" and AUTO_RESET.get(auto_reset) == 1:
            raise ValueError("nonfinite='end' needs auto_reset='template' or 'none': a jitter reset keeps the "
                             "overflowed positions and cannot bring the env back")
        self.nonfinite = nonfinite
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.WalkerGymError("walker_gym_b200 runs on CUDA devices only (no CPU fallback)")
        if isinstance(creature, str):
            creature = creature_from_id(creature)
        self.creature = creature
        self.topo = topology_from_creature(creature)
        self.num_envs = E = int(num_envs)
        self.in3d = bool(in3d)
        if auto_reset not in AUTO_RESET:
            raise ValueError(f"auto_reset must be one of {sorted(map(str, AUTO_RESET))}")
        if obs_layout not in ("row", "feature"):
            raise ValueError("obs_layout must be 'row' ([E, D]) or 'feature' ([D, E])")
        if act_layout not in ("row", "feature"):
            raise ValueError("act_layout must be 'row' ([E, A]) or 'feature' ([A, E])")
        self.act_layout = act_layout
        self.params = make_params(in3d=in3d, g=g, dampk=dampk, ground_high=ground_high, ground_k=ground_k,
                                  ground_damp=ground_damp, friction=friction, rand_sigma=rand_sigma,
                                  time_step=time_step, max_steps=max_steps, k_sub=k_sub,
                                  auto_reset=AUTO_RESET[auto_reset], seed=seed, env_offset=env_offset,
                                  integrator=integrator, end_nonfinite=nonfinite == "end")
        self.N, self.M = self.topo.n_mass, self.topo.n_muscle
        self.obs_dim = self.lib.wg_obs_dim(C.byref(self.topo), int(self.in3d))
        self.obs_layout = obs_layout
        self.step_count = 0        # global step index: the Philox counter word of the in-kernel jitter
        dev, f32 = self.device, torch.float32
        tmpl = torch.tensor(list(self.topo.tmpl_pos[: 3 * self.N]), dtype=f32, device=dev)
        x0 = torch.tensor([np.float32(m.x) for m in creature.muscles], dtype=f32, device=dev).reshape(self.M)
        # state layout: "soa" = separate [rows, E] tensors; "packed" = one [tiles, R4, 128, 4] tensor moved with
        # 16-byte accesses (bodies with a specialised kernel only); "auto" picks packed when it is available
        if state_layout not in ("auto", "soa", "packed"):
            raise ValueError("state_layout must be 'auto', 'soa' or 'packed'")
        # x64: float64 actions with the reference's NumPy promotion semantics (wg_step_x64): muscle lengths are kept
        # as doubles plus a type bit; a compatibility path on the run-time-topology kernel, SoA state only
        self.x64 = bool(x64)
        if self.x64 and state_layout == "packed":
            raise ValueError("x64 mode uses state_layout='soa'")
        if self.x64:
            state_layout = "soa"
        avail = self.lib.wg_packed_available(C.byref(self.topo))       # 1 ahead-of-time kernel, 2 compiled at run time
        can_pack = avail == 1 or (avail == 2 and (E >= 4096 or state_layout == "packed"))   # small batches: not worth ~1 s
        if can_pack and state_layout != "soa":
            # bodies without an ahead-of-time kernel: compile one for this spring graph now (NVRTC, ~1 s); on failure
            # keep the SoA layout and the run-time-topology kernel
            rc = self.lib.wg_jit_prepare(C.byref(self.topo), int(self.in3d), 0 if obs_layout == "row" else 1)
            if rc != 0:
                if state_layout == "packed":
                    _lib.check(rc, "wg_jit_prepare")
                can_pack = False
        if state_layout == "packed" and not can_pack:
            raise ValueError("state_layout='packed' needs a body with a specialised kernel (Balance / Box topology)")
        self.state_layout = "packed" if (state_layout == "packed" or (state_layout == "auto" and can_pack)) else "soa"
        self._R = 6 * self.N + self.M + 2
        if self.state_layout == "packed":
            n_floats = self.lib.wg_packed_state_floats(C.byref(self.topo), E)
            self._T, self._R4 = (E + 127) // 128, (self._R + 3) // 4
            assert n_floats == self._T * self._R4 * 512
            self.state = torch.zeros(self._T, self._R4, 128, 4, dtype=f32, device=dev)
            self._pos = self._vel = self._mx = self._steps = self._ep_ret = None
            self.set_state(pos=tmpl[:, None].expand(3 * self.N, E), mx=x0[:, None].expand(self.M, E))
        else:
            self.state = None
            self._pos = tmpl[:, None].repeat(1, E).contiguous()
            self._vel = torch.zeros(3 * self.N, E, dtype=f32, device=dev)
            self._mx = x0[:, None].repeat(1, E).contiguous() if self.M else torch.zeros(0, E, dtype=f32, device=dev)
            self._steps = torch.zeros(E, dtype=torch.int32, device=dev)
            self._ep_ret = torch.zeros(E, dtype=f32, device=dev) if track_stats else None
        self.obs = torch.zeros((E, self.obs_dim) if obs_layout == "row" else (self.obs_dim, E), dtype=f32, device=dev)
        self.reward = torch.zeros(E, dtype=f32, device=dev)
        self._done_u8 = torch.zeros(E, dtype=torch.uint8, device=dev)
        self.done = self._done_u8.view(torch.bool)
        self.old_a = torch.zeros(3 * self.N, E, dtype=f32, device=dev) if keep_old_a else None
        self.energy = torch.zeros(E, dtype=f32, device=dev) if track_info else None
        self.centroid = torch.zeros(3, E, dtype=f32, device=dev) if track_info else None
        self.contact_pre = torch.zeros(E, dtype=torch.int32, device=dev) if track_contacts else None
        self.contact_post = torch.zeros(E, dtype=torch.int32, device=dev) if track_contacts else None
        self.fin_stats = torch.zeros(4, E, dtype=f32, device=dev) if track_stats else None
        # [0] count, [1] length sum of finished episodes whose return is not finite ("count" / "end" only)
        self.nf_stats = torch.zeros(2, E, dtype=f32, device=dev) if nonfinite != "keep" else None
        self._stats_out = torch.zeros(8, dtype=torch.float64, device=dev)
        # graph_safe: the Philox step index lives in a device scalar advanced by a device op, so a
        # captured CUDA graph that replays step() keeps drawing fresh reset jitter
        self._counter = torch.zeros(1, dtype=torch.int32, device=dev) if graph_safe else None
        if self.x64:
            from .topology import x64_from_creature
            self._x64 = x64_from_creature(creature)
            self._x0_d = torch.tensor([self._x64.x0_d[m] for m in range(self.M)], dtype=torch.float64, device=dev)
            self.mx64 = self._x0_d[:, None].repeat(1, E).contiguous()
            self.mx_weak = torch.ones(self.M, E, dtype=torch.uint8, device=dev)
        else:
            self._x64 = self.mx64 = self.mx_weak = None
        self._step_offset, self._defer_advance = 0, False
        self._buf = WgBuffers()
        self._bind()
        if initial_reset:
            self.reset()           # PhysicsEnv.__init__ ends with self.reset() (gym/optimized_env.py:51)

    # ---- plumbing ----------------------------------------------------------------
    @staticmethod
    def _p(t: Optional[torch.Tensor]):
        return None if t is None else t.data_ptr()

    def _bind(self) -> None:
        b = self._buf
        b.pos, b.vel, b.old_a, b.mx, b.steps = map(self._p, (self._pos, self._vel, self.old_a, self._mx, self._steps))
        b.state_packed = self._p(self.state)
        if self.M == 0 and self.state is None:
            b.mx = self._p(self._steps)    # never dereferenced (M == 0); keeps validation simple
        b.obs, b.reward, b.done = self._p(self.obs), self._p(self.reward), self._p(self._done_u8)
        b.obs_layout = 0 if self.obs_layout == "row" else 1
        b.contact_pre, b.contact_post = self._p(self.contact_pre), self._p(self.contact_post)
        b.energy, b.centroid = self._p(self.energy), self._p(self.centroid)
        b.ep_ret, b.fin_stats, b.nf_stats = self._p(self._ep_ret), self._p(self.fin_stats), self._p(self.nf_stats)
        b.action, b.act_dim, b.noise = None, 0, None
        b.act_layout = 0 if self.act_layout == "row" else 1
        b.step_counter = self._p(self._counter)
        b.mx64, b.mx_weak, b.action64 = self._p(self.mx64), self._p(self.mx_weak), None

    def _advance(self) -> None:
        if self._counter is not None:
            if not self._defer_advance:
                self._counter.add_(1)
        else:
            self.step_count += 1

    def _stamp(self) -> None:
        self.params.step_index = (self._step_offset if self._counter is not None else self.step_count) & 0xFFFFFFFF

    def deferred_steps(self, n: int):
        """Context manager for a block of ``n`` steps in graph-safe mode: the caller sets ``_step_offset`` to the step's
        position in the block before each step, the device counter is advanced once by ``n`` at the end instead of by
        one tiny kernel per step.  The Philox indices are the ones per-step advancing would have produced."""
        env = self

        class _Block:
            def __enter__(self_inner):
                env._defer_advance = env._counter is not None
                return env

            def __exit__(self_inner, *exc):
                if env._defer_advance:
                    env._defer_advance, env._step_offset = False, 0
                    env._counter.add_(n)
                return False
        return _Block()

    # ---- state access (layout independent) --------------------------------------------------------
    def _var(self, k: int) -> torch.Tensor:
        """Packed layout: strided view [tiles, 128] of per-env scalar k."""
        return self.state[:, k >> 2, :, k & 3]

    def _gather(self, k0: int, n: int, dtype=torch.float32) -> torch.Tensor:
        out = torch.stack([self._var(k0 + i).reshape(-1)[: self.num_envs] for i in range(n)]) if n else \
            torch.zeros(0, self.num_envs, dtype=torch.float32, device=self.device)
        return out.view(dtype) if dtype != torch.float32 else out

    @property
    def pos(self) -> torch.Tensor:
        """[3N, E] positions, row n*3+c.  A live tensor in the soa layout, a snapshot copy in the packed one
        (write through ``set_state``)."""
        return self._pos if self.state is None else self._gather(0, 3 * self.N)

    @property
    def vel(self) -> torch.Tensor:
        return self._vel if self.state is None else self._gather(3 * self.N, 3 * self.N)

    @property
    def mx(self) -> torch.Tensor:
        return self._mx if self.state is None else self._gather(6 * self.N, self.M)

    @property
    def steps(self) -> torch.Tensor:
        return self._steps if self.state is None else self._gather(6 * self.N + self.M, 1, torch.int32)[0]

    @property
    def ep_ret(self):
        if self.state is None:
            return self._ep_ret
        return self._gather(6 * self.N + self.M + 1, 1)[0]

    def set_state(self, pos=None, vel=None, mx=None, steps=None, ep_ret=None) -> None:
        """Overwrite (parts of) the state of all envs from [rows, E] / [E] tensors, in either layout."""
        def put(k0, t, rows):
            if t is None:
                return
            t = torch.as_tensor(t, device=self.device)
            t = t.reshape(rows, self.num_envs)
            if t.dtype == torch.int32:
                t = t.view(torch.float32)
            pad = self._T * 128 - self.num_envs
            for i in range(rows):
                row = t[i].to(torch.float32) if t.dtype != torch.float32 else t[i]
                if pad:
                    row = torch.cat([row, row.new_zeros(pad)])
                self._var(k0 + i).copy_(row.reshape(self._T, 128))
        if self.state is None:
            for dst, src in ((self._pos, pos), (self._vel, vel), (self._mx, mx), (self._steps, steps), (self._ep_ret, ep_ret)):
                if src is not None and dst is not None:
                    dst.copy_(torch.as_tensor(src, device=self.device).reshape(dst.shape))
            if self.x64 and mx is not None:
                # x64 mode steps from the double muscle lengths: a float32 length is a float32-typed ("weak") muscle,
                # a float64 tensor is taken as np.float64 lengths (gym/optimized_walker.py:33)
                src = torch.as_tensor(mx, device=self.device).reshape(self.mx64.shape)
                self.mx64.copy_(src.to(torch.float64))
                self.mx_weak.fill_(0 if src.dtype == torch.float64 else 1)
            return
        put(0, pos, 3 * self.N)
        put(3 * self.N, vel, 3 * self.N)
        put(6 * self.N, mx, self.M)
        if steps is not None:
            put(6 * self.N + self.M, torch.as_tensor(steps, device=self.device).to(torch.int32), 1)
        put(6 * self.N + self.M + 1, ep_ret, 1)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _on_device_or_mapped(self, t: torch.Tensor, mapped_ok: bool) -> bool:
        """On the env's device, or (results only) pinned host memory, which CUDA maps into the device's address
        space: the kernel then writes it over PCIe directly ("zero-copy")."""
        return t.device == self.obs.device or (mapped_ok and t.device.type == "cpu" and t.is_pinned())

    def _check_f32(self, t: torch.Tensor, shape, what: str, mapped_ok: bool = False) -> torch.Tensor:
        if not self._on_device_or_mapped(t, mapped_ok) or t.dtype != torch.float32 or not t.is_contiguous() \
                or tuple(t.shape) != tuple(shape):
            raise ValueError(f"{what} must be a contiguous float32 tensor of shape {tuple(shape)} on {self.obs.device}"
                             + (" (or pinned host memory)" if mapped_ok else ""))
        return t

    @property
    def kernel_variant(self) -> int:
        """0 = generic run-time-topology kernel, >0 = register-resident specialisation."""
        return self.lib.wg_kernel_variant(C.byref(self.topo))

    # ---- gym surface -------------------------------------------------------------
    def reset(self, mask: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None,
              mode: Optional[str] = None) -> torch.Tensor:
        """``PhysicsEnv.reset`` for every env (or those in ``mask``).

        mode "jitter" is the reference's reset (velocities += N(0, sigma), steps = 0;
        positions persist, gym/optimized_env.py:53-68); "template" first restores the
        creation-time body, which is what calling ``make_env`` again does.  Default:
        the env's ``auto_reset`` mode, or "jitter" if auto-reset is off.
        ``noise``: optional [3N, E] jitter (already scaled) instead of the Philox stream."""
        m = AUTO_RESET[mode] if mode is not None else (self.params.auto_reset or 1)
        if m not in (1, 2):
            raise ValueError("reset mode must be 'jitter' or 'template'")
        self._buf.noise = self._p(self._check_f32(noise, (3 * self.N, self.num_envs), "noise")) if noise is not None else None
        mptr = None
        if mask is not None:
            if mask.dtype == torch.bool:
                mask = mask.view(torch.uint8)
            if mask.dtype != torch.uint8 or mask.numel() != self.num_envs or not mask.is_contiguous():
                raise ValueError("mask must be a contiguous bool/uint8 tensor of length num_envs")
            mptr = mask.data_ptr()
        self._stamp()
        with torch.cuda.device(self.device):
            rc = self.lib.wg_reset(C.byref(self.topo), C.byref(self.params), C.byref(self._buf),
                                   self.num_envs, m, mptr, self._stream())
        self._buf.noise = None
        _lib.check(rc, "wg_reset")
        if self.x64 and m == 2:                 # a fresh creature: every Muscle holds its originx again
            sel = slice(None) if mask is None else mask.view(torch.bool)
            self.mx64[:, sel] = self._x0_d[:, None]
            self.mx_weak[:, sel] = 1
        self._advance()
        return self.obs

    def step(self, action: Optional[torch.Tensor], noise: Optional[torch.Tensor] = None, out=None):
        """``PhysicsEnv.step`` for every env, one kernel launch.

        ``action``: float32 [E, A] (or [A, E] with ``act_layout="feature"``); only the first
        min(A, M) columns drive muscles (Creature.act, gym/optimized_walker.py:164-167);
        ``None`` applies no action.
        Returns ``(obs, reward, done, info)``: views of buffers that the next call overwrites.
        With auto-reset on, ``obs`` of a done env is its post-reset observation while
        ``reward``/``done`` describe the step that ended the episode.
        ``out=(obs, reward, done)``: write this step's results straight into caller-owned tensors (e.g. slot t
        of a trajectory buffer) instead of the env's own buffers; ``done`` is uint8/bool.  The tensors may also be
        PINNED HOST memory (``walker_gym_b200.host.pinned_empty`` / ``tensor.pin_memory()``): the kernel then writes
        observation rows, rewards and dones over PCIe itself, with no device staging buffer and no separate copy."""
        b = self._buf
        res_obs, res_rew, res_done = self.obs, self.reward, self.done
        # validate everything before touching the bound buffers: a rejected call must leave the env as it was
        if out is not None:
            res_obs, res_rew, res_done = out
            self._check_f32(res_obs, self.obs.shape, "out obs", mapped_ok=True)
            self._check_f32(res_rew, (self.num_envs,), "out reward", mapped_ok=True)
            if res_done.element_size() != 1 or res_done.numel() != self.num_envs or not res_done.is_contiguous() \
                    or not self._on_device_or_mapped(res_done, True):
                raise ValueError("out done must be a contiguous 1-byte tensor of length num_envs on the env's device "
                                 "(or pinned host memory)")
        act_ptr, act64_ptr, act_dim = None, None, 0
        if action is not None:
            env_axis = 0 if self.act_layout == "row" else 1
            if action.dim() != 2 or action.shape[env_axis] != self.num_envs:
                raise ValueError(f"action must have shape [{self.num_envs}, A] (row) or [A, {self.num_envs}] (feature)")
            if self.x64:
                if action.dtype != torch.float64 or not action.is_contiguous() or action.device != self.obs.device:
                    raise ValueError("x64 mode takes contiguous float64 actions on the env's device")
                act64_ptr = action.data_ptr()
            else:
                self._check_f32(action, action.shape, "action")
                act_ptr = action.data_ptr()
            act_dim = int(action.shape[1 - env_axis])
        noise_ptr = self._p(self._check_f32(noise, (3 * self.N, self.num_envs), "noise")) if noise is not None else None
        b.action, b.action64, b.act_dim, b.noise = act_ptr, act64_ptr, act_dim, noise_ptr
        if out is not None:
            b.obs, b.reward, b.done = res_obs.data_ptr(), res_rew.data_ptr(), res_done.data_ptr()
        self._stamp()
        try:
            with torch.cuda.device(self.device):
                if self.x64:
                    rc = self.lib.wg_step_x64(C.byref(self.topo), C.byref(self._x64), C.byref(self.params), C.byref(b),
                                              self.num_envs, self._stream())
                else:
                    rc = self.lib.wg_step(C.byref(self.topo), C.byref(self.params), C.byref(b), self.num_envs, self._stream())
        finally:
            b.noise = None
            b.obs, b.reward, b.done = self._p(self.obs), self._p(self.reward), self._p(self._done_u8)
        _lib.check(rc, "wg_step_x64" if self.x64 else "wg_step")
        self._advance()
        info = {}
        if self.energy is not None:
            info = {"steps": self.steps, "centroid_position": self.centroid, "total_energy": self.energy}
        return res_obs, res_rew, res_done, info

    def step_many(self, actions: Optional[torch.Tensor], n_steps: Optional[int] = None, out=None, _host=None):
        """``n_steps`` consecutive ``PhysicsEnv.step`` calls in ONE launch (``wg_step_multi``) for actions known up
        front: scripted gaits / open-loop controllers (the phase-table gait sketched at gym/walker.py:356-366), action repeat, replays.

        ``actions``: float32 [T, E, M]; or [E, M] with ``n_steps`` = T: the same action at every step (action repeat /
        frame skip: ``Creature.act`` runs T times with it); or ``None`` with ``n_steps``: T steps without an action; or
        an in-kernel action source (``walker_gym_b200.actions.ScriptedActions`` / ``CPGActions``) with ``n_steps``:
        the action of every step is computed on chip from the env's own step counter (no action memory is read).
        Returns ``(obs, rewards [T, E], dones [T, E])``: ``obs`` is the observation after the last step (the env's own
        buffer), rewards / dones are per step.  Bit-identical to T ``step`` calls; needs ``state_layout="packed"``,
        row-major observations and actions, a body with an ahead-of-time packed kernel, and no per-step info buffers.
        ``out=(rewards, dones)``: caller-owned result tensors (dones 1 byte per element)."""
        if self.state is None or self.x64 or self.obs_layout != "row" or self.act_layout != "row":
            raise ValueError("step_many needs state_layout='packed', obs_layout='row', act_layout='row' and float32 actions")
        E = self.num_envs
        n_act = 1
        gen = None
        from .actions import ActionSource
        if isinstance(actions, ActionSource):
            # an in-kernel action source (scripted table / CPG): every step's action is computed on chip from the env's
            # own step counter; the launch reads no action memory
            if n_steps is None:
                raise ValueError("n_steps is required with an in-kernel action source")
            gen = actions.struct(self.M, float(self.params.dt))
            actions, T = None, int(n_steps)
        elif actions is not None and actions.dim() == 2:
            if n_steps is None:
                raise ValueError("n_steps is required with a single [E, M] action block (action repeat)")
            if actions.shape[0] != E or actions.shape[1] != self.M:
                raise ValueError(f"actions must have shape [{E}, {self.M}] or [T, {E}, {self.M}]")
            self._check_f32(actions, actions.shape, "actions")
            T = int(n_steps)
        elif actions is not None:
            if actions.dim() != 3 or actions.shape[1] != E or actions.shape[2] != self.M:
                raise ValueError(f"actions must have shape [T, {E}, {self.M}]")
            self._check_f32(actions, actions.shape, "actions")
            T = n_act = int(actions.shape[0])
            if n_steps is not None and int(n_steps) != T:
                raise ValueError("n_steps disagrees with actions.shape[0]")
        elif n_steps is None:
            raise ValueError("n_steps is required when actions is None")
        else:
            T = n_act = int(n_steps)
        if T < 1:
            raise ValueError("step_many needs at least one step")
        if out is None:
            rew = torch.empty(T, E, dtype=torch.float32, device=self.obs.device)
            done = torch.empty(T, E, dtype=torch.bool, device=self.obs.device)
        else:
            rew, done = out
            self._check_f32(rew, (T, E), "out rewards")
            if done.element_size() != 1 or tuple(done.shape) != (T, E) or not done.is_contiguous():
                raise ValueError("out dones must be a contiguous 1-byte tensor of shape [T, E]")
        b = self._buf
        saved = (b.old_a, b.contact_pre, b.contact_post, b.energy, b.centroid)
        b.old_a = b.contact_pre = b.contact_post = b.energy = b.centroid = None
        b.action, b.act_dim, b.noise = self._p(actions), (self.M if actions is not None else 0), None
        b.reward, b.done = rew.data_ptr(), done.data_ptr()
        b.action_gen = C.pointer(gen) if gen is not None else None
        self._stamp()
        try:
            with torch.cuda.device(self.device):
                if _host is None:
                    rc = self.lib.wg_step_multi(C.byref(self.topo), C.byref(self.params), C.byref(b), E, T, n_act, self._stream())
                else:
                    rc = self.lib.wg_step_multi_host(C.byref(self.topo), C.byref(self.params), C.byref(b), E, T, n_act,
                                                     *[self._p(t) for t in _host], self._stream())
        finally:
            b.old_a, b.contact_pre, b.contact_post, b.energy, b.centroid = saved
            b.reward, b.done = self._p(self.reward), self._p(self._done_u8)
            b.action_gen = None
        _lib.check(rc, "wg_step_multi" if _host is None else "wg_step_multi_host")
        if self._counter is not None:
            if not self._defer_advance:
                self._counter.add_(T)
        else:
            self.step_count += T
        return self.obs, rew, done

    def step_many_host(self, h_actions: torch.Tensor, d_actions: torch.Tensor, h_obs: Optional[torch.Tensor] = None,
                       h_rewards: Optional[torch.Tensor] = None, h_dones: Optional[torch.Tensor] = None,
                       n_steps: Optional[int] = None, out=None):
        """End-to-end ``step_many`` on HOST buffers (``wg_step_multi_host``): copies the pinned host ``h_actions``
        ([T, E, M], or [E, M] with ``n_steps`` for action repeat) into the device staging tensor ``d_actions`` of the
        same shape, runs the T-step launch and copies the last observation, the [T, E] rewards and dones back into the
        pinned host tensors, all asynchronously on the current stream.  ``out``: device (rewards, dones) staging."""
        if h_actions.device.type != "cpu" or h_actions.dtype != torch.float32 or not h_actions.is_contiguous() \
                or tuple(h_actions.shape) != tuple(d_actions.shape):
            raise ValueError("h_actions must be a contiguous float32 host tensor with d_actions' shape")
        T = int(n_steps) if h_actions.dim() == 2 and n_steps is not None else int(h_actions.shape[0])
        for t, name, n, size in ((h_obs, "h_obs", self.obs.numel(), 4), (h_rewards, "h_rewards", T * self.num_envs, 4),
                                 (h_dones, "h_dones", T * self.num_envs, 1)):
            if t is not None and (t.device.type != "cpu" or not t.is_contiguous() or t.numel() != n or t.element_size() != size):
                raise ValueError(f"{name} must be a contiguous host tensor of {n} elements of {size} byte(s)")
        return self.step_many(d_actions, n_steps=n_steps, out=out, _host=(h_actions, h_obs, h_rewards, h_dones))

    def step_host(self, h_action: torch.Tensor, d_action: torch.Tensor, h_obs: Optional[torch.Tensor] = None,
                  h_reward: Optional[torch.Tensor] = None, h_done: Optional[torch.Tensor] = None) -> None:
        """End-to-end step on HOST buffers (``wg_step_host``): copies the pinned host
        ``h_action`` [E, A] into the device staging tensor ``d_action``, launches the
        step, and copies obs / reward / done back into the pinned host tensors, all
        asynchronously on the current stream."""
        for t, name in ((h_action, "h_action"), (h_obs, "h_obs"), (h_reward, "h_reward"), (h_done, "h_done")):
            if t is not None and (t.device.type != "cpu" or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous host tensor (pinned for async copies)")
        if h_action.dtype != torch.float32 or h_action.dim() != 2 or h_action.shape[0] != self.num_envs:
            raise ValueError(f"h_action must be float32 [{self.num_envs}, A]")
        self._check_f32(d_action, h_action.shape, "d_action")
        if h_obs is not None and (h_obs.dtype != torch.float32 or h_obs.numel() != self.obs.numel()):
            raise ValueError("h_obs must be float32 with as many elements as obs")
        if h_reward is not None and (h_reward.dtype != torch.float32 or h_reward.numel() != self.num_envs):
            raise ValueError("h_reward must be float32 [E]")
        if h_done is not None and (h_done.element_size() != 1 or h_done.numel() != self.num_envs):
            raise ValueError("h_done must be a 1-byte dtype of length E")
        b = self._buf
        if self.act_layout != "row":
            raise ValueError("step_host needs act_layout='row'")
        b.action, b.act_dim, b.noise = d_action.data_ptr(), int(d_action.shape[1]), None
        self._stamp()
        with torch.cuda.device(self.device):
            rc = self.lib.wg_step_host(C.byref(self.topo), C.byref(self.params), C.byref(b), self.num_envs,
                                       h_action.data_ptr(), self._p(h_obs), self._p(h_reward), self._p(h_done),
                                       self._stream())
        _lib.check(rc, "wg_step_host")
        self._advance()

    def getstat(self, in3d: Optional[bool] = None, pk=1, vk=1, ak=1, mk=1, midform: bool = True, conmid: bool = False,
                out: Optional[torch.Tensor] = None, layout: str = "row") -> torch.Tensor:
        """``Creature.getstat`` (gym/optimized_walker.py:129-162) with its options for every env: a float32 tensor
        [E, D'] (or [D', E] with ``layout="feature"``), D' = 3*d*N + M (+3 with ``conmid``).  With the defaults this is
        the observation ``step`` returns.  ``Point.old_a`` comes from the env's ``old_a`` buffer (``keep_old_a=True``)
        or from the last observation (which needs ``in3d`` <= the env's dimensionality)."""
        in3d = self.in3d if in3d is None else bool(in3d)
        Dp = 3 * (3 if in3d else 2) * self.N + self.M + (3 if conmid else 0)
        shape = (self.num_envs, Dp) if layout == "row" else (Dp, self.num_envs)
        if layout not in ("row", "feature"):
            raise ValueError("layout must be 'row' or 'feature'")
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        else:
            self._check_f32(out, shape, "out")
        with torch.cuda.device(self.device):
            rc = self.lib.wg_getstat(C.byref(self.topo), C.byref(self._buf), self.obs.data_ptr(), int(self.in3d), int(in3d),
                                     float(np.float32(pk)), float(np.float32(vk)), float(np.float32(ak)), float(np.float32(mk)),
                                     int(bool(midform)), int(bool(conmid)), out.data_ptr(), 0 if layout == "row" else 1,
                                     self.num_envs, self._stream())
        _lib.check(rc, "wg_getstat")
        return out

    def step_disp(self, disp: torch.Tensor, **kw):
        """``Creature.actdisp`` (gym/optimized_walker.py:169-172; ``Muscle.actdisp`` :37-43) + ``PhysicsEnv.step``:
        ``disp`` is a bool / uint8 tensor [E, A]; muscle m lengthens by its ``stride`` where disp is true and shortens
        by it where false, then ``regulation()`` -- i.e. ``x += +-stride``, the same float32 addition ``act`` performs."""
        if disp.dim() != 2 or disp.shape[0] != self.num_envs or disp.device != self.obs.device:
            raise ValueError(f"disp must be a bool / uint8 tensor [{self.num_envs}, A] on the env's device")
        if self.act_layout != "row" or self.x64:
            raise ValueError("step_disp needs act_layout='row' and float32 muscle state")
        A = min(int(disp.shape[1]), self.M)
        if getattr(self, "_stride", None) is None:
            self._stride = torch.tensor([np.float32(m.stride) for m in self.creature.muscles], dtype=torch.float32, device=self.device)
        action = torch.where(disp[:, :A].to(torch.bool), self._stride[:A], -self._stride[:A]).contiguous()
        return self.step(action, **kw)

    def get_action_space(self):
        return {"shape": (self.M,), "type": "continuous", "low": -1.0, "high": 1.0}

    def get_observation_space(self):
        return {"shape": (self.obs_dim,), "type": "continuous", "low": -np.inf, "high": np.inf}

    # ---- episode statistics (K3) ---------------------------------------------------
    def episode_stats(self, all_reduce: bool = False, clear: bool = False) -> dict:
        """Sum of finished-episode returns / squared returns / lengths / count over
        this shard; with ``all_reduce`` the 8-double vector is summed across ranks
        (NCCL) -- the only collective anywhere near the step path.  With ``nonfinite``
        "count" / "end" the return statistics cover the finite episodes and the dict adds
        ``nonfinite_episodes`` and ``nonfinite_length_mean``."""
        if self.fin_stats is None:
            raise RuntimeError("construct the env with track_stats=True")
        with torch.cuda.device(self.device):
            if self.nf_stats is None:
                rc = self.lib.wg_stats_reduce(self.fin_stats.data_ptr(), self.num_envs, self._stats_out.data_ptr(),
                                              self._stream())
            else:
                rc = self.lib.wg_stats_reduce_split(self.fin_stats.data_ptr(), self.nf_stats.data_ptr(), self.num_envs,
                                                    self._stats_out.data_ptr(), self._stream())
        _lib.check(rc, "wg_stats_reduce")
        from .dist import all_reduce_stats, finalize_stats
        out = all_reduce_stats(self._stats_out) if all_reduce else self._stats_out
        stats = finalize_stats(out, nonfinite=self.nf_stats is not None)
        if clear:
            self.fin_stats.zero_()
            if self.nf_stats is not None:
                self.nf_stats.zero_()
        return stats

    # ---- checkpoint / state.pkl ------------------------------------------------------
    def state_dict(self) -> dict:
        """A complete snapshot (copies, in either layout): state, observation, host and device step counters
        (``graph_safe``), the float64 muscle state of x64 mode, episode accumulators."""
        def snap(t):
            return t.clone() if t is not None else None
        d = {"pos": snap(self.pos), "vel": snap(self.vel), "mx": snap(self.mx), "steps": snap(self.steps),
             "obs": snap(self.obs), "step_count": self.step_count}
        if self.ep_ret is not None:
            d["ep_ret"] = snap(self.ep_ret)
        for k in ("old_a", "fin_stats", "nf_stats", "mx64", "mx_weak"):
            if getattr(self, k) is not None:
                d[k] = snap(getattr(self, k))
        if self._counter is not None:
            d["counter"] = snap(self._counter)
        return d

    def load_state_dict(self, d: dict) -> None:
        self.set_state(**{k: d[k] for k in ("pos", "vel", "mx", "steps", "ep_ret") if k in d})
        for k, v in d.items():
            if k == "step_count":
                self.step_count = int(v)
            elif k == "counter":
                if self._counter is None:
                    raise ValueError("the checkpoint comes from a graph_safe env (device step counter); this env has none")
                self._counter.copy_(torch.as_tensor(v, device=self.device).reshape(1))
            elif k in ("obs", "old_a", "fin_stats", "nf_stats", "mx64", "mx_weak") and getattr(self, k, None) is not None:
                getattr(self, k).copy_(v)       # after set_state: the saved float64 muscle state wins over its float32 view

    def save_state(self, path: str, env_index: int = 0) -> None:
        """Write env ``env_index`` as a reference-compatible ``state.pkl``
        (gym/engine.py:199-204): the reference's ``Point.backup`` can load it."""
        from .engine import Point
        from .state_io import save_points
        pos = self.pos[:, env_index].reshape(self.N, 3).cpu().numpy()
        vel = self.vel[:, env_index].reshape(self.N, 3).cpu().numpy()
        old = self.old_a[:, env_index].reshape(self.N, 3).cpu().numpy() if self.old_a is not None else np.zeros((self.N, 3), np.float32)
        saved, pts = list(Point.points), []
        try:
            for n, p in enumerate(self.creature.phys):
                q = type(p).__new__(type(p))
                q.__dict__.update(p.__dict__)
                q.pos, q.v, q.old_a, q.a = pos[n].copy(), vel[n].copy(), old[n].copy(), np.zeros(3, np.float32)
                pts.append(q)
        finally:
            Point.points = saved
        save_points(path, pts, {})

    def load_state(self, path: str, env_index: Optional[int] = None) -> None:
        """Load point positions/velocities from a reference ``state.pkl`` into one env
        (or broadcast to all envs when ``env_index`` is None)."""
        from .state_io import load_points
        pts, _ = load_points(path)
        if len(pts) != self.N:
            raise ValueError(f"snapshot has {len(pts)} points, this body has {self.N}")
        pos = torch.tensor(np.stack([p.pos for p in pts]).reshape(-1), dtype=torch.float32, device=self.device)
        vel = torch.tensor(np.stack([p.v for p in pts]).reshape(-1), dtype=torch.float32, device=self.device)
        cur_pos, cur_vel = self.pos.clone(), self.vel.clone()
        if env_index is None:
            cur_pos.copy_(pos[:, None].expand_as(cur_pos))
            cur_vel.copy_(vel[:, None].expand_as(cur_vel))
        else:
            cur_pos[:, env_index] = pos
            cur_vel[:, env_index] = vel
        self.set_state(pos=cur_pos, vel=cur_vel)


class HostStepPipeline:
    """Double-buffered end-to-end stepping on HOST buffers: step t+1's action upload and kernel overlap step t's
    result download (two CUDA streams, two sets of device result buffers), so sustained throughput is bounded by the
    slower direction of the PCIe link instead of the sum of upload + kernel + download.

        pipe = HostStepPipeline(env)
        for t in range(T):
            pipe.submit(h_action[t], h_obs[t], h_reward[t], h_done[t])     # pinned host tensors; any result may be None
        pipe.drain()                                                        # all results are in the host tensors

    Only ``drain()`` (all steps) and ``wait_slot(age)`` (one step) guarantee that results are in the host tensors: both
    block the host.  ``submit`` never blocks; it orders the new step behind whatever the caller queued on its stream."""

    def __init__(self, env: BatchedPhysicsEnv):
        if env.act_layout != "row" or env.x64:
            raise ValueError("HostStepPipeline needs act_layout='row' and float32 actions")
        self.env = env
        dev = env.device
        self.s_step, self.s_copy = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        self.d_act = None
        self.obs = [torch.empty_like(env.obs) for _ in range(2)]
        self.rew = [torch.empty_like(env.reward) for _ in range(2)]
        self.done = [torch.empty_like(env._done_u8) for _ in range(2)]
        self.ev_step = [torch.cuda.Event() for _ in range(2)]
        self.ev_copy = [torch.cuda.Event() for _ in range(2)]
        self.t = 0
        self._many_key, self.m_act, self.m_rew, self.m_done, self._obs_copy = None, None, None, None, None
        self.s_up, self.ev_up = torch.cuda.Stream(device=dev), [torch.cuda.Event() for _ in range(2)]     # submit_many uploads
        self.s_step.wait_stream(torch.cuda.current_stream(dev))

    def submit(self, h_action, h_obs=None, h_reward=None, h_done=None) -> None:
        env, k = self.env, self.t & 1
        if self.d_act is None or self.d_act[0].shape != h_action.shape:
            self.d_act = [torch.empty(h_action.shape, dtype=torch.float32, device=env.device) for _ in range(2)]
        # whatever the caller queued on its stream (reset / step / set_state between drains) happens before this step
        self.s_step.wait_stream(torch.cuda.current_stream(env.device))
        with torch.cuda.stream(self.s_step):
            if self.t >= 2:
                self.s_step.wait_event(self.ev_copy[k])           # slot k's previous results have left the device
            self.d_act[k].copy_(h_action, non_blocking=True)
            env.step(self.d_act[k], out=(self.obs[k], self.rew[k], self.done[k]))
            self.ev_step[k].record(self.s_step)
        with torch.cuda.stream(self.s_copy):
            self.s_copy.wait_event(self.ev_step[k])
            if h_obs is not None:
                h_obs.copy_(self.obs[k], non_blocking=True)
            if h_reward is not None:
                h_reward.copy_(self.rew[k], non_blocking=True)
            if h_done is not None:
                h_done.copy_(self.done[k].view(h_done.dtype) if h_done.dtype != torch.uint8 else self.done[k], non_blocking=True)
            self.ev_copy[k].record(self.s_copy)
        self.t += 1

    def submit_zero_copy(self, h_action, h_obs, h_reward, h_done) -> None:
        """The same step with the results written by the kernel itself into the pinned (device-mapped) host tensors:
        no device result buffers, no download copies.  The action upload of step t+1 (its own stream) overlaps step
        t's kernel; the kernels serialise (they share the env state) and run at the PCIe write rate.  Results of a
        step are readable after ``wait_slot`` / ``drain``."""
        env, k = self.env, self.t & 1
        if self.d_act is None or self.d_act[0].shape != h_action.shape:
            self.d_act = [torch.empty(h_action.shape, dtype=torch.float32, device=env.device) for _ in range(2)]
        self.s_step.wait_stream(torch.cuda.current_stream(env.device))
        with torch.cuda.stream(self.s_up):
            if self.t >= 2:
                self.s_up.wait_event(self.ev_step[k])             # the kernel that read slot k's actions has finished
            else:
                self.s_up.wait_stream(torch.cuda.current_stream(env.device))
            self.d_act[k].copy_(h_action, non_blocking=True)
            self.ev_up[k].record(self.s_up)
        with torch.cuda.stream(self.s_step):
            self.s_step.wait_event(self.ev_up[k])
            env.step(self.d_act[k], out=(h_obs, h_reward, h_done))
            self.ev_step[k].record(self.s_step)
            self.ev_copy[k].record(self.s_step)                   # wait_slot waits on ev_copy
        self.t += 1

    def submit_many(self, h_actions, h_rewards=None, h_dones=None, h_obs=None, n_steps=None) -> None:
        """The same pipeline for T-step launches (``step_many``): pinned host ``h_actions`` [T, E, M] (or [E, M] with
        ``n_steps``: action repeat) up, per-step ``h_rewards`` / ``h_dones`` [T, E] and, optionally, the observation
        after the last step down.  Block i+1's upload and kernel overlap block i's download; asking for ``h_obs``
        makes the next kernel wait for that copy (the env has one observation buffer)."""
        env, k = self.env, self.t & 1
        T = int(n_steps) if h_actions.dim() == 2 else int(h_actions.shape[0])
        key = (tuple(h_actions.shape), T)
        if self._many_key != key:
            self.drain()
            torch.cuda.current_stream(env.device).synchronize()
            dev, E = env.device, env.num_envs
            self.m_act = [torch.empty(h_actions.shape, dtype=torch.float32, device=dev) for _ in range(2)]
            self.m_rew = [torch.empty(T, E, dtype=torch.float32, device=dev) for _ in range(2)]
            self.m_done = [torch.empty(T, E, dtype=torch.uint8, device=dev) for _ in range(2)]
            self._many_key = key
        self.s_step.wait_stream(torch.cuda.current_stream(env.device))    # caller-stream work precedes this block
        with torch.cuda.stream(self.s_up):                       # the upload also overlaps the previous block's kernel
            if self.t >= 2:
                self.s_up.wait_event(self.ev_step[k])             # the kernel that read slot k's actions has finished
            else:
                self.s_up.wait_stream(torch.cuda.current_stream(env.device))
            self.m_act[k].copy_(h_actions, non_blocking=True)
            self.ev_up[k].record(self.s_up)
        with torch.cuda.stream(self.s_step):
            if self.t >= 2:
                self.s_step.wait_event(self.ev_copy[k])           # slot k's previous results have left the device
            self.s_step.wait_event(self.ev_up[k])
            if self._obs_copy is not None:
                self.s_step.wait_event(self._obs_copy)            # the previous block's observation has left the device
                self._obs_copy = None
            env.step_many(self.m_act[k], n_steps=n_steps, out=(self.m_rew[k], self.m_done[k]))
            self.ev_step[k].record(self.s_step)
        with torch.cuda.stream(self.s_copy):
            self.s_copy.wait_event(self.ev_step[k])
            if h_obs is not None:
                h_obs.copy_(env.obs, non_blocking=True)
                self._obs_copy = torch.cuda.Event()
                self._obs_copy.record(self.s_copy)
            if h_rewards is not None:
                h_rewards.copy_(self.m_rew[k], non_blocking=True)
            if h_dones is not None:
                h_dones.copy_(self.m_done[k].view(h_dones.dtype) if h_dones.dtype != torch.uint8 else self.m_done[k], non_blocking=True)
            self.ev_copy[k].record(self.s_copy)
        self.t += 1

    def drain(self) -> None:
        """Block the HOST until every submitted step has finished and its results are in the host tensors; work the
        caller queues on its stream afterwards is ordered behind the pipeline."""
        cur = torch.cuda.current_stream(self.env.device)
        cur.wait_stream(self.s_up)
        cur.wait_stream(self.s_step)
        cur.wait_stream(self.s_copy)
        self.s_up.synchronize()
        self.s_step.synchronize()
        self.s_copy.synchronize()

    def wait_slot(self, age: int = 1) -> None:
        """Block the host until the results of the step submitted ``age`` submits ago (1 = the latest) are in its
        host tensors -- the closed-loop pattern: submit(t), wait_slot(2) -> step t-1's results are readable while
        step t is in flight."""
        if 1 <= age <= 2 and self.t >= age:
            self.ev_copy[(self.t - age) & 1].synchronize()


class StepGraph:
    """T closed-loop ``env.step`` calls captured once in a CUDA graph and replayed.

    For shards so small that one step kernel takes a few microseconds (BASELINE config 3 as written: 2^20 envs split
    over 8 GPUs = 131072 per GPU, about 9 us per step) the Python + ctypes cost of a launch (~15 us) would dominate;
    a graph replay launches T steps with one host call.  The env must be built with ``graph_safe=True`` (the Philox
    step index of the in-kernel reset jitter then lives in a device counter that the graph advances by T per replay).

        g = StepGraph(env, actions)        # actions: device float32 [T, E, M]; overwrite in place between replays
        g.replay()                          # T steps; g.obs [T, E, D] (or the last one only), g.rewards / g.dones [T, E]
    """

    def __init__(self, env: BatchedPhysicsEnv, actions: torch.Tensor, keep_obs: str = "last"):
        if env._counter is None:
            raise ValueError("StepGraph needs BatchedPhysicsEnv(graph_safe=True)")
        if keep_obs not in ("last", "all"):
            raise ValueError("keep_obs must be 'last' or 'all'")
        if actions.dim() != 3 or actions.device != env.obs.device or actions.dtype != torch.float32:
            raise ValueError("actions must be a device float32 tensor [T, E, A] (or [T, A, E] with act_layout='feature')")
        self.env, self.actions, self.T = env, actions, int(actions.shape[0])
        E, dev = env.num_envs, env.device
        n_obs = self.T if keep_obs == "all" else 1
        self.obs = torch.empty((n_obs,) + tuple(env.obs.shape), dtype=torch.float32, device=dev)
        self.rewards = torch.empty(self.T, E, dtype=torch.float32, device=dev)
        self.dones = torch.empty(self.T, E, dtype=torch.uint8, device=dev)
        snap = env.state_dict()                                   # warm-up outside capture, on a snapshot
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            self._steps()
        torch.cuda.current_stream(dev).wait_stream(s)
        env.load_state_dict(snap)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._steps()
        env.load_state_dict(snap)                                 # capture does not execute, but keep the contract explicit

    def _steps(self) -> None:
        env = self.env
        with env.deferred_steps(self.T):
            for t in range(self.T):
                env._step_offset = t
                env.step(self.actions[t], out=(self.obs[t if self.obs.shape[0] > 1 else 0], self.rewards[t], self.dones[t]))

    def replay(self) -> None:
        self.graph.replay()
