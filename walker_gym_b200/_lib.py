"""ctypes binding of ``libwalkergym_b200.so`` (C ABI: ``include/walker_gym_b200.h``).

The library is the product: there is no CPU or PyTorch fallback.  If the
shared object is missing, or was built for another ABI version, importing the
binding raises -- it never degrades silently.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_MASS, MAX_SPRING = 32, 96
ABI_VERSION = 5
GEN_MAX_ROWS, GEN_MAX_MUSCLE = 32, 16

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WG_LIB_PATH", os.path.join(_HERE, "libwalkergym_b200.so"))   # override: tuning experiments


class WgTopology(C.Structure):
    """``wg_topology``: replaces Creature(phys, muscles, skeletons) (gym/optimized_walker.py:108-115)."""
    _fields_ = [
        ("n_mass", C.c_int32), ("n_spring", C.c_int32), ("n_muscle", C.c_int32), ("reserved", C.c_int32),
        ("mass", C.c_double * MAX_MASS),
        ("fixed", C.c_uint8 * MAX_MASS),
        ("tmpl_pos", C.c_float * (MAX_MASS * 3)),
        ("si", C.c_int32 * MAX_SPRING), ("sj", C.c_int32 * MAX_SPRING),
        ("sk", C.c_float * MAX_SPRING), ("sdamp", C.c_float * MAX_SPRING), ("srest", C.c_float * MAX_SPRING),
        ("mlo", C.c_float * MAX_SPRING), ("mhi", C.c_float * MAX_SPRING),
        ("sstring", C.c_uint8 * MAX_SPRING),
    ]


class WgParams(C.Structure):
    """``wg_params``: replaces PhysicsEnv's constructor arguments (gym/optimized_env.py:15-44)."""
    _fields_ = [
        ("g", C.c_double),
        ("dampk", C.c_float), ("ground", C.c_float), ("fall_thresh", C.c_float),
        ("ground_k", C.c_float), ("ground_damp", C.c_float), ("friction", C.c_float),
        ("dt", C.c_float), ("dt2", C.c_float), ("sigma", C.c_float),
        ("in3d", C.c_int32), ("max_steps", C.c_int32), ("k_sub", C.c_int32), ("auto_reset", C.c_int32),
        ("integrator", C.c_int32),
        ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32), ("step_index", C.c_uint32), ("env_offset", C.c_uint32),
        ("end_nonfinite", C.c_int32), ("reserved1", C.c_int32),          # 1 = a non-finite reward ends the episode
    ]


class WgActionGen(C.Structure):
    """``wg_action_gen``: in-kernel action source of wg_step_multi (scripted table gym/walker.py:356-366, or a CPG
    after gym/optimized_walker/walker.py:56-90)."""
    _fields_ = [("mode", C.c_int32), ("n_rows", C.c_int32), ("hold", C.c_int32), ("reserved", C.c_int32),
                ("table", C.c_float * (GEN_MAX_ROWS * GEN_MAX_MUSCLE)), ("amp", C.c_float * GEN_MAX_MUSCLE),
                ("phase0", C.c_uint32 * GEN_MAX_MUSCLE), ("dphase", C.c_uint32 * GEN_MAX_MUSCLE)]


class WgBuffers(C.Structure):
    _fields_ = [
        ("pos", C.c_void_p), ("vel", C.c_void_p), ("old_a", C.c_void_p), ("mx", C.c_void_p), ("steps", C.c_void_p),
        ("action", C.c_void_p), ("act_dim", C.c_int32), ("obs_layout", C.c_int32),
        ("act_layout", C.c_int32), ("reserved0", C.c_int32),
        ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("contact_pre", C.c_void_p), ("contact_post", C.c_void_p),
        ("energy", C.c_void_p), ("centroid", C.c_void_p),
        ("ep_ret", C.c_void_p), ("fin_stats", C.c_void_p), ("noise", C.c_void_p),
        ("step_counter", C.c_void_p), ("state_packed", C.c_void_p),
        ("mx64", C.c_void_p), ("mx_weak", C.c_void_p), ("action64", C.c_void_p),      # x64 mode (wg_step_x64)
        ("action_gen", C.POINTER(WgActionGen)),                                         # wg_step_multi: in-kernel action source
        ("nf_stats", C.c_void_p),                                                       # [2][E] non-finite episodes
        ("truncated", C.c_void_p),                                                      # [E] uint8: done by the time limit alone
        ("final_obs", C.c_void_p),                                                      # like obs: pre-reset observation of done envs
    ]


class WgX64(C.Structure):
    """``wg_x64``: the double-typed objects of a Muscle once a float64 action made its length an np.float64."""
    _fields_ = [("sk_d", C.c_double * MAX_SPRING), ("x0_d", C.c_double * MAX_SPRING),
                ("mlo_d", C.c_double * MAX_SPRING), ("mhi_d", C.c_double * MAX_SPRING)]


class WgPkgSystem(C.Structure):
    """``wg_pkg_system``: Environment.points / ding_points / springs (gym/optimized_walker/env.py:39-41)."""
    _fields_ = [("n_point", C.c_int32), ("n_spring", C.c_int32),
                ("mass", C.c_double * MAX_MASS), ("fixed", C.c_uint8 * MAX_MASS),
                ("si", C.c_int32 * MAX_SPRING), ("sj", C.c_int32 * MAX_SPRING),
                ("srest", C.c_float * MAX_SPRING), ("sk", C.c_float * MAX_SPRING), ("sstring", C.c_uint8 * MAX_SPRING)]


class WgPkgParams(C.Structure):
    """``wg_pkg_params``: Environment constructor arguments (gym/optimized_walker/env.py:10-37)."""
    _fields_ = [("gravity", C.c_float * 3), ("damping", C.c_float), ("drag_c", C.c_float),
                ("ground_level", C.c_float), ("restitution", C.c_float), ("friction", C.c_float), ("dt", C.c_float),
                ("min_dist", C.c_float), ("ground", C.c_int32)]


class WgMlpPolicy(C.Structure):
    """``wg_mlp_policy``: device pointers to torch.nn.Linear weights of a D -> 64 -> 64 -> (M, 1) tanh MLP."""
    _fields_ = [("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w_mu", C.c_void_p), ("b_mu", C.c_void_p), ("w_v", C.c_void_p), ("b_v", C.c_void_p),
                ("log_std", C.c_void_p), ("obs_dim", C.c_int32), ("act_dim", C.c_int32),
                ("obs_scale", C.c_float), ("obs_clip", C.c_float), ("precision", C.c_int32), ("reserved", C.c_int32)]


TUNE_TMA, TUNE_PART, TUNE_L2_PREFETCH, TUNE_JIT, TUNE_POLICY_TC, TUNE_PDL = 0, 1, 2, 3, 4, 5

EXPORTS = ("wg_abi_version", "wg_last_error_string", "wg_obs_dim", "wg_kernel_variant", "wg_force_generic",
           "wg_set_tuning", "wg_packed_state_floats", "wg_packed_available", "wg_jit_prepare",
           "wg_step", "wg_step_multi", "wg_step_x64", "wg_reset", "wg_stats_reduce", "wg_stats_reduce_split", "wg_step_host", "wg_step_multi_host", "wg_pkg_update_physics", "wg_pkg_kernel_variant",
           "wg_policy_act", "wg_policy_step", "wg_gae", "wg_gae_trunc", "wg_stream_probe", "wg_host_alloc", "wg_host_free", "wg_getstat", "wg_policy_tc_status",
           "wg_selftest_div_smallint", "wg_selftest_forced_list", "wg_selftest_sqrt", "wg_selftest_div3")

_lib = None


class WalkerGymError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raise if it is absent (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WalkerGymError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  walker_gym_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise WalkerGymError(f"{LIB_PATH} does not export {name}")
    lib.wg_abi_version.restype = C.c_int
    if lib.wg_abi_version() != ABI_VERSION:
        raise WalkerGymError(f"ABI mismatch: library {lib.wg_abi_version()} != binding {ABI_VERSION}")
    lib.wg_last_error_string.restype = C.c_char_p
    P = C.POINTER
    lib.wg_obs_dim.argtypes = [P(WgTopology), C.c_int]
    lib.wg_kernel_variant.argtypes = [P(WgTopology)]
    lib.wg_packed_available.argtypes = [P(WgTopology)]
    lib.wg_packed_available.restype = C.c_int
    lib.wg_jit_prepare.argtypes = [P(WgTopology), C.c_int, C.c_int]
    lib.wg_jit_prepare.restype = C.c_int
    lib.wg_force_generic.argtypes = [C.c_int]
    lib.wg_set_tuning.argtypes = [C.c_int, C.c_int]
    lib.wg_set_tuning.restype = C.c_int
    lib.wg_packed_state_floats.argtypes = [P(WgTopology), C.c_int64]
    lib.wg_packed_state_floats.restype = C.c_int64
    lib.wg_step.argtypes = [P(WgTopology), P(WgParams), P(WgBuffers), C.c_int64, C.c_void_p]
    lib.wg_step_multi.argtypes = [P(WgTopology), P(WgParams), P(WgBuffers), C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    lib.wg_step_multi.restype = C.c_int
    lib.wg_step_multi_host.argtypes = [P(WgTopology), P(WgParams), P(WgBuffers), C.c_int64, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.wg_step_multi_host.restype = C.c_int
    lib.wg_step_x64.argtypes = [P(WgTopology), P(WgX64), P(WgParams), P(WgBuffers), C.c_int64, C.c_void_p]
    lib.wg_step_x64.restype = C.c_int
    lib.wg_reset.argtypes = [P(WgTopology), P(WgParams), P(WgBuffers), C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
    lib.wg_stats_reduce.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.wg_stats_reduce_split.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.wg_step_host.argtypes = [P(WgTopology), P(WgParams), P(WgBuffers), C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.wg_pkg_update_physics.argtypes = [P(WgPkgSystem), P(WgPkgParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int64, C.c_int32, C.c_void_p]
    lib.wg_pkg_kernel_variant.argtypes = [P(WgPkgSystem)]
    lib.wg_pkg_kernel_variant.restype = C.c_int
    lib.wg_policy_act.argtypes = [P(WgMlpPolicy), C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int64, C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32,
                                  C.c_void_p]
    lib.wg_policy_step.argtypes = [P(WgMlpPolicy), P(WgTopology), P(WgParams), P(WgBuffers), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                   C.c_void_p]
    lib.wg_policy_step.restype = C.c_int
    lib.wg_stream_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    lib.wg_stream_probe.restype = C.c_int
    lib.wg_gae.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64,
                           C.c_float, C.c_float, C.c_float, C.c_void_p]
    lib.wg_gae_trunc.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int32, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_void_p]
    lib.wg_getstat.argtypes = [P(WgTopology), P(WgBuffers), C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                               C.c_float, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p]
    lib.wg_getstat.restype = C.c_int
    lib.wg_host_alloc.argtypes = [P(C.c_void_p), C.c_uint64, C.c_int]
    lib.wg_host_free.argtypes = [C.c_void_p]
    lib.wg_selftest_div_smallint.argtypes = [C.c_float, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.wg_selftest_forced_list.argtypes = [C.c_double, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.wg_selftest_sqrt.argtypes = [C.c_void_p, C.c_void_p]
    lib.wg_selftest_div3.argtypes = [C.c_int, C.c_int, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    for name in ("wg_host_alloc", "wg_host_free", "wg_getstat", "wg_policy_tc_status", "wg_selftest_div_smallint", "wg_selftest_forced_list",
                 "wg_selftest_sqrt", "wg_selftest_div3"):
        getattr(lib, name).restype = C.c_int
    for name in ("wg_obs_dim", "wg_kernel_variant", "wg_force_generic", "wg_step", "wg_reset",
                 "wg_stats_reduce", "wg_stats_reduce_split", "wg_step_host", "wg_pkg_update_physics", "wg_policy_act", "wg_gae", "wg_gae_trunc"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().wg_last_error_string().decode("utf-8", "replace")
        exc = ValueError if rc == -1 else WalkerGymError
        raise exc(f"{what} failed ({rc}): {msg}")
