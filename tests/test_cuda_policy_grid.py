"""GPU: the persistent policy pipelines (wg_policy_act) and the fused policy + env step (wg_policy_step) on grids where
every CTA processes several tiles, as BASELINE config 5 (2^18 envs) does.

A persistent CTA b of a grid of G handles tiles b, b + G, b + 2G, ... (ordinal i = tile // G); the mbarrier parities,
the double-buffer halves, the look-ahead copies and, in the fused kernel, the second output-warp group only run for
i >= 1.  Every env's mean / value is compared with torch float32 and float64 and reported per tile; a tile evaluated
alone (where it is the first tile of CTA 0) must give the same bits as in the large call; and the fused kernel's
trajectory must equal the two-launch one bit for bit and the C oracle's physics."""
import math

import numpy as np
import pytest
import torch

import golden_util as gu
import walker_oracle as wo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TILE = 128                    # envs per tile of all three implementations (kPolBlock, kTcTile)
SMEM_PER_CTA = 227 * 1024


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(params=[2, 1, 0], ids=["tcgen05-pipeline", "tcgen05-monolithic", "mma.sync"])
def policy_impl(request):
    """The three implementations behind WG_TUNE_POLICY_TC (2 = warp-specialised tcgen05 pipeline, the default)."""
    from walker_gym_b200 import _lib
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_POLICY_TC, request.param)
    try:
        yield request.param
    finally:
        lib.wg_set_tuning(_lib.TUNE_POLICY_TC, old)
    assert lib.wg_policy_tc_status() == 0, "a tcgen05 policy kernel gave up waiting on one of its barriers"


def _tc_smem_bytes(D):
    """Dynamic shared memory of the monolithic tcgen05 kernel (TcSmem<K1>::bytes, wg_policy_tc.cuh)."""
    k1 = ((D + 1 + 7) // 8) * 8
    K1 = next(k for k in (24, 32, 40, 48, 72) if k1 <= k)
    W1, W2, WH = 64 * K1, 64 * 72, 9 * 64
    o_zs = 2 * W1 + 2 * W2 + WH + 4
    o_st = o_zs + 4 * 2 * TILE + 9 * TILE + 32
    return 4 * (o_st + 2 * ((TILE * D + 3) // 4) * 4) + 64


def policy_grid(impl, D, E):
    """CTAs the launch code of each implementation starts (wg_inst_policy.cu)."""
    n_tiles = (E + TILE - 1) // TILE
    per_sm = {2: 1, 1: 2 if 2 * _tc_smem_bytes(D) <= SMEM_PER_CTA else 1, 0: 2}[impl]
    return min(n_tiles, per_sm * n_sms())


def make_policy(D, M, seed=0):
    from walker_gym_b200.rollout import FeatureMajorMLP
    torch.manual_seed(seed)
    pol = FeatureMajorMLP(D, M).to(DEV)
    with torch.no_grad():                 # larger weights than the default init: exercises tanh away from 0
        for lin in (pol.l1, pol.l2, pol.mu, pol.v):
            lin.weight.mul_(2.0)
            lin.bias.uniform_(-0.5, 0.5)
        pol.log_std.copy_(torch.linspace(-1.0, 0.2, M)[:, None])
    return pol


def reference(pol, obs_fm):
    """torch float32 (TF32 off) and float64 evaluations of the module on feature-major observations."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            mean, value = pol(obs_fm)
            p64 = {k: v.double() for k, v in pol.state_dict().items()}
            x = torch.nan_to_num(obs_fm.double() * pol.obs_scale, nan=0.0, posinf=pol.obs_clip, neginf=-pol.obs_clip)
            x = x.clamp(-pol.obs_clip, pol.obs_clip)
            h = torch.tanh(p64["l1.weight"] @ x + p64["l1.bias"][:, None])
            h = torch.tanh(p64["l2.weight"] @ h + p64["l2.bias"][:, None])
            mean64 = p64["mu.weight"] @ h + p64["mu.bias"][:, None]
            value64 = (p64["v.weight"] @ h + p64["v.bias"][:, None])[0]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return mean, value, mean64, value64


SIZES = ["2*SMs*128+1", "3*SMs*128-77", "2^18", "2^18+37"]


def size_of(which):
    """Envs of each grid under test, from the SM count of device 0."""
    s = n_sms()
    return {"2*SMs*128+1": 2 * s * TILE + 1, "3*SMs*128-77": 3 * s * TILE - 77, "2^18": 1 << 18, "2^18+37": (1 << 18) + 37}[which]


def per_tile_check(err, bound, grid, what):
    """err [E] (float64, NaN = failure) against bound (a number or [E]); the message names the first failing env's tile,
    its CTA and its ordinal."""
    E = err.shape[0]
    n_tiles = (E + TILE - 1) // TILE
    ok = err <= bound
    if bool(ok.all()):
        return
    bad_env = (~ok).nonzero()[:, 0]
    tiles = torch.unique(bad_env // TILE)
    e = int(bad_env[0])
    t = e // TILE
    b = float(bound[e]) if torch.is_tensor(bound) else bound
    raise AssertionError(f"{what}: {bad_env.numel()} envs in {tiles.numel()} of {n_tiles} tiles exceed their bound; first env "
                         f"{e} (error {float(err[e]):.3g}, bound {b:.3g}) in tile {t} = CTA {t % grid}, ordinal {t // grid} of a grid of {grid}; "
                         f"bad tiles {tiles[:8].tolist()}")


def plant_specials(obs_fm, tiles, E):
    """NaN, +inf, -inf and 5000 entries in chosen tiles (feature-major [D, E])."""
    D = obs_fm.shape[0]
    for t in tiles:
        b = t * TILE
        n_in = min(TILE, E - b)
        for k, (row, v) in enumerate(((3, float("nan")), (17, float("inf")), (40, float("-inf")), (77, 5000.0))):
            obs_fm[k % D, b + min(row, n_in - 1)] = v


@pytest.mark.parametrize("which", SIZES)
@pytest.mark.parametrize("D,M", [(38, 2), (64, 7), (9, 3)])
def test_policy_multi_tile_grids(D, M, which, policy_impl):
    """Every env of a multi-tile grid, both observation layouts, both precisions: mean / value vs torch float32 (2e-5
    fp32, 2e-2 tf32) and, in fp32, vs float64 (at most max(4 x torch's own error, 5e-6)); sampled actions' logp vs the
    log-density recomputed from the action (a per-env bound from the mean's error and float32 rounding); and bit-exact
    position independence of chosen tiles."""
    from walker_gym_b200.rollout import FusedPolicy
    E = size_of(which)
    n_tiles = (E + TILE - 1) // TILE
    grid = policy_grid(policy_impl, D, E)
    last = n_tiles - 1
    ragged = E % TILE != 0
    # the shape each size claims to cover
    if which == "2*SMs*128+1":
        assert E - last * TILE == 1 and last // grid == (2 if grid == n_sms() else 1)
    elif which == "3*SMs*128-77":
        assert ragged and last // grid == (2 if grid == n_sms() else 1)
    else:
        assert n_tiles // grid >= 3, (n_tiles, grid)
        assert ragged == (which == "2^18+37")
    pol = make_policy(D, M, seed=D + M)
    g = torch.Generator(device=DEV).manual_seed(E + D)
    obs = torch.randn(D, E, device=DEV, generator=g) * 150.0          # obs_scale 1e-2 -> O(1) inputs, some clipped at +-10
    special = sorted({0, grid, last})                                  # ordinal 0, ordinal 1, the last (ragged) tile
    plant_specials(obs, special, E)
    obs_row = obs.t().contiguous()
    mean_t, value_t, mean64, value64 = reference(pol, obs)
    std64 = pol.log_std.detach().double().exp()
    ls64 = pol.log_std.detach().double()
    err_torch_m = (mean_t.double() - mean64).abs().max().item()
    err_torch_v = (value_t.double() - value64).abs().max().item()
    # tiles evaluated alone: ordinals 0, 1, 2 and the last of CTA 0, the ragged tile, the last CTA's last tile
    n0 = (n_tiles - 1) // grid
    alone = sorted({i * grid for i in (0, 1, 2, n0) if i * grid < n_tiles} | {last} |
                   {grid - 1 + ((n_tiles - grid) // grid) * grid})
    for precision, tol in (("fp32", 2e-5), ("tf32", 2e-2)):
        fp = FusedPolicy(pol, precision)
        for layout in ("feature", "row"):
            x = obs if layout == "feature" else obs_row
            what = f"{precision} {layout} E={E}"
            mean, value = torch.full((M, E), 7.0, device=DEV), torch.full((E,), 7.0, device=DEV)
            action = torch.zeros(M, E, device=DEV)
            fp.act(x, action=action, value=value, mean=mean, sample=False, obs_layout=layout)
            assert torch.equal(action, mean), what
            err_m = (mean - mean_t).abs().amax(0).double()
            err_v = (value - value_t).abs().double()
            per_tile_check(torch.nan_to_num(torch.maximum(err_m, err_v), nan=math.inf), tol, grid, f"{what}: vs torch float32")
            if precision == "fp32":
                e64 = torch.nan_to_num((mean.double() - mean64).abs().amax(0), nan=math.inf)
                per_tile_check(e64, max(4 * err_torch_m, 5e-6), grid, f"{what}: mean vs float64 (torch's error {err_torch_m:.3g})")
                e64 = torch.nan_to_num((value.double() - value64).abs(), nan=math.inf)
                per_tile_check(e64, max(4 * err_torch_v, 5e-6), grid, f"{what}: value vs float64 (torch's error {err_torch_v:.3g})")
            # sampled: the same mean / value, and logp = log N(action; mean, std)
            so = dict(action=torch.zeros(M, E, device=DEV), logp=torch.zeros(E, device=DEV),
                      value=torch.zeros(E, device=DEV), mean=torch.zeros(M, E, device=DEV))
            fp.act(x, sample=True, seed=77, step_index=9, obs_layout=layout, **so)
            assert torch.equal(so["mean"], mean) and torch.equal(so["value"], value), what
            ref_mean = mean64 if precision == "fp32" else so["mean"].double()       # tf32 means are 2e-2 from float64
            eps = (so["action"].double() - ref_mean) / std64
            want = (-0.5 * eps * eps - ls64 - 0.5 * math.log(2 * math.pi)).sum(0)
            # per-env bound: d logp = sum eps * d eps, with d eps from the kernel mean's error, the float32 rounding of the
            # action, and the approximate exp of log_std (relative 4e-7); plus float32 rounding of the kernel's sum
            dm = (so["mean"].double() - ref_mean).abs()
            de = (dm + so["action"].double().abs() * 2.0 ** -23) / std64 + eps.abs() * 4e-7
            bound = 2 * (eps.abs() * de).sum(0) + 1e-5 * M
            per_tile_check(torch.nan_to_num((so["logp"].double() - want).abs(), nan=math.inf), bound, grid, f"{what}: logp")
            # position independence: tile t alone (env_offset = its first env) runs at ordinal 0 of CTA 0
            for t in alone:
                a, b = t * TILE, min(E, (t + 1) * TILE)
                xs = x[:, a:b].contiguous() if layout == "feature" else x[a:b]
                o = {k: torch.zeros(v.shape[:-1] + (b - a,), device=DEV) for k, v in so.items()}
                fp.act(xs, sample=True, seed=77, step_index=9, obs_layout=layout, env_offset=a, **o)
                for k in o:
                    assert torch.equal(o[k].view(torch.int32), so[k][..., a:b].view(torch.int32)), \
                        f"{what}: {k} of tile {t} (CTA {t % grid}, ordinal {t // grid}) alone differs from the large call"
    torch.cuda.synchronize()


# ---------------- the fused policy + env step (wg_policy_step) ----------------
MAX_STEPS = 45          # lanes go non-finite before the first max_steps reset, which then runs inside the fused kernel
T_ROLL = 32
SEED = 21


def _collector(E, fuse_step, graph):
    from walker_gym_b200 import BatchedPhysicsEnv
    from walker_gym_b200.rollout import RolloutCollector
    env = BatchedPhysicsEnv("Balance-v0", E, DEV, in3d=True, auto_reset="template", max_steps=MAX_STEPS, seed=SEED,
                            obs_layout="row", act_layout="row", graph_safe=True, state_layout="packed")
    pol = make_policy(env.obs_dim, env.M, seed=5)
    col = RolloutCollector(env, pol, T_ROLL, use_cuda_graph=graph, fused=True, seed=9, fuse_step=fuse_step)
    assert col.fused_step == fuse_step
    return env, col


def _same_dev(a, b):
    """Bit equality on the device up to NaN payload and the sign of zero (gu.same's rule)."""
    if a.dtype in (torch.bool, torch.uint8):
        return torch.equal(a, b)
    return a.shape == b.shape and bool(((a == b) | (a.isnan() & b.isnan())).all())


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("which", ["2^18+37", "3*SMs*128"])
def test_fused_policy_step_at_scale(which, graph):
    """RolloutCollector(fuse_step=True) -- one launch per env step, the env step in the output warps -- against the two
    launches (wg_policy_act + the step kernel) on every slot of 4 rollouts of 32 steps, bit for bit.  The grid has one
    CTA per SM and several tiles per CTA, so both output-warp groups (even and odd ordinals) step envs; lanes go
    non-finite and are auto-reset inside the fused kernel.  Eagerly, the head and tail 4096 envs are also replayed
    through the C oracle from the recorded actions."""
    sms = n_sms()
    E = {"2^18+37": (1 << 18) + 37, "3*SMs*128": 3 * sms * TILE}[which]
    n_tiles = (E + TILE - 1) // TILE
    grid = min(n_tiles, sms)
    assert n_tiles >= 2 * grid, "odd ordinals exist: the second output group steps envs"
    if which == "3*SMs*128":
        assert n_tiles == 3 * grid
    env_f, col_f = _collector(E, True, graph)
    env_r, col_r = _collector(E, False, graph)
    n_slice = 1 << 12
    lock = None
    if not graph:
        body = wo.make_body(wo.BALANCE)
        lock = []
        for a in (0, E - n_slice):
            prm = wo.make_params(in3d=True, auto_reset=2, max_steps=MAX_STEPS, seed=SEED, env_offset=a)
            st = wo.init_state(body, n_slice)
            st.pop("old_a")
            prm.step_index = 0
            o = wo.reset(body, prm, st, mode=2)
            assert gu.same(env_f.obs[a:a + n_slice].cpu().numpy(), o)
            lock.append((a, prm, st))
    nonfinite_before_reset = 0
    step = 1
    for c in range(4):
        out_f = {k: v.clone() for k, v in col_f.collect().items()}
        out_r = col_r.collect()
        for k in ("obs", "actions", "rewards", "dones", "values", "logp", "advantages"):
            for t in range(out_f[k].shape[0]):
                assert _same_dev(out_f[k][t], out_r[k][t]), f"collect {c}: {k}[{t}] of the fused launch differs"
        for t in range(T_ROLL):
            if step + t < MAX_STEPS:
                nonfinite_before_reset += int((~torch.isfinite(out_f["obs"][t + 1]).all(1)).sum())
        if lock is not None:
            for t in range(T_ROLL):
                for a, prm, st in lock:
                    prm.step_index = step + t
                    act = out_f["actions"][t][a:a + n_slice].cpu().numpy()
                    o = wo.step(body, prm, st, act, want_info=False)
                    tile = (a + n_slice - 1) // TILE
                    where = f"collect {c} step {t}, envs [{a}, {a + n_slice}) (last tile {tile}: CTA {tile % grid}, ordinal {tile // grid})"
                    assert gu.same(out_f["obs"][t + 1][a:a + n_slice].cpu().numpy(), o["obs"]), f"obs, {where}"
                    assert gu.same(out_f["rewards"][t][a:a + n_slice].cpu().numpy(), o["reward"]), f"reward, {where}"
                    assert gu.same(out_f["dones"][t][a:a + n_slice].cpu().numpy(), o["done"].astype(bool)), f"done, {where}"
        step += T_ROLL
    assert nonfinite_before_reset > 0, "some lanes go non-finite before the first max_steps reset (raise MAX_STEPS)"
    assert int(out_f["dones"].sum()) > 0
    assert col_f.episode_stats(all_reduce=False)["episodes"] == col_r.episode_stats(all_reduce=False)["episodes"] > 0
