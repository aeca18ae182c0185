"""GPU: BatchedPhysicsEnv (public API -> C ABI -> CUDA) against the C oracle on the
same seeded inputs, at sizes the oracle finishes in seconds, plus size-independent
properties at BASELINE.json's full size.  Equality is exact (float32 bit patterns up
to NaN payload / sign of zero): the kernel evaluates the reference's operations in
the reference's order."""
import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def spec_of(name):
    from walker_gym_b200 import BODIES
    b = BODIES[name]
    ding = set(b.get("ding", ()))
    return {"points": [(m, tuple(p), n in ding) for n, (m, p) in enumerate(b["points"])],
            "muscles": b["muscles"], "skeletons": b["skeletons"]}


def make_pair(name, E, *, env_kw=None, auto_reset=None, max_steps=1000, k_sub=1, seed=7, obs_layout="row", **extra):
    """Build the CUDA env and the oracle state from the same template (no jitter yet)."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    env_kw = dict(env_kw or {})
    env = BatchedPhysicsEnv(name, E, "cuda:0", auto_reset=auto_reset, max_steps=max_steps, k_sub=k_sub, seed=seed,
                            obs_layout=obs_layout, keep_old_a=True, track_info=True, track_contacts=True,
                            initial_reset=False, **env_kw, **extra)
    body = wo.make_body(spec_of(name))
    ar = {None: 0, "jitter": 1, "template": 2}[auto_reset]
    prm = wo.make_params(max_steps=max_steps, k_sub=k_sub, auto_reset=ar, seed=seed,
                         env_offset=extra.get("env_offset", 0), **env_kw)
    st = wo.init_state(body, E)
    return env, body, prm, st


def assert_state_equal(env, st, N, what=""):
    assert gu.same(env.pos.cpu().numpy(), st["pos"]), f"pos {what}"
    assert gu.same(env.vel.cpu().numpy(), st["vel"]), f"vel {what}"
    assert gu.same(env.old_a.cpu().numpy(), st["old_a"]), f"old_a {what}"
    assert gu.same(env.mx.cpu().numpy(), st["mx"]), f"mx {what}"
    assert gu.same(env.steps.cpu().numpy(), st["steps"]), f"steps {what}"


def run_lockstep(env, body, prm, st, T, rng, *, noise_reset=True, ep=None):
    import torch
    E, M, N = env.num_envs, env.M, env.N
    if noise_reset:
        nz = (rng.standard_normal((3 * N, E)) * 0.1).astype(np.float32)
        o_c = env.reset(noise=torch.from_numpy(nz).cuda(), mode="jitter")
        o_o = wo.reset(body, prm, st, mode=1, noise=nz)
        assert gu.same(o_c.cpu().numpy().reshape(o_o.shape) if env.obs_layout == "row" else o_c.cpu().numpy().T, o_o), "reset obs"
    for t in range(T):
        act = rng.uniform(-1, 1, (E, M)).astype(np.float32)
        prm.step_index = env.step_count
        obs, rew, done, info = env.step(torch.from_numpy(act).cuda())
        out = wo.step(body, prm, st, act, ep_ret=None if ep is None else ep[0], fin_stats=None if ep is None else ep[1])
        o = obs.cpu().numpy()
        assert gu.same(o if env.obs_layout == "row" else o.T, out["obs"]), f"obs @ step {t}"
        assert gu.same(rew.cpu().numpy(), out["reward"]), f"reward @ step {t}"
        assert gu.same(done.cpu().numpy(), out["done"].astype(bool)), f"done @ step {t}"
        assert gu.same(env.contact_pre.cpu().numpy().astype(np.uint32), out["contact_pre"]), f"contact_pre @ step {t}"
        assert gu.same(env.contact_post.cpu().numpy().astype(np.uint32), out["contact_post"]), f"contact_post @ step {t}"
        assert gu.same(info["total_energy"].cpu().numpy(), out["energy"]), f"energy @ step {t}"
        assert gu.same(info["centroid_position"].cpu().numpy(), out["centroid"]), f"centroid @ step {t}"
        assert_state_equal(env, st, N, f"@ step {t}")


# ---- BASELINE config 2: optimized_walker bodies, 4096 envs, 100-step free-running trajectories ----
@pytest.mark.parametrize("name", ["balance_v0", "box_v0"])
@pytest.mark.parametrize("in3d", [True, False])
def test_config2_4096_envs_100_steps_bit_exact(name, in3d):
    env, body, prm, st = make_pair(name, 4096, env_kw=dict(in3d=in3d))
    assert env.kernel_variant > 0
    run_lockstep(env, body, prm, st, 100, np.random.default_rng(1))


@pytest.mark.parametrize("E", [1, 2, 31, 129, 255, 4097])
@pytest.mark.parametrize("name", ["balance_v0", "humanb"])
def test_ragged_batch_sizes(name, E):
    env, body, prm, st = make_pair(name, E, env_kw=dict(in3d=True))
    run_lockstep(env, body, prm, st, 12, np.random.default_rng(E))


@pytest.mark.parametrize("name", ["test", "leg2", "box", "box2", "balance", "balance2", "balance3", "intrian",
                                  "humanb", "insect", "box4", "leg", "hat", "quad_balance", "quad_balance_chain"])
def test_every_walker_py_body(name):
    """BASELINE config 1 bodies (gym/walker.py tables) under the L1 semantics."""
    env, body, prm, st = make_pair(name, 64, env_kw=dict(in3d=True))
    run_lockstep(env, body, prm, st, 40, np.random.default_rng(3))


def test_config4_enlarged_body_8_substeps():
    env, body, prm, st = make_pair("quad_balance", 1024, env_kw=dict(in3d=True), k_sub=8)
    assert env.kernel_variant == 3
    run_lockstep(env, body, prm, st, 25, np.random.default_rng(4))


@pytest.mark.parametrize("layout", ["row", "feature"])
@pytest.mark.parametrize("mode", ["template", "jitter"])
@pytest.mark.parametrize("name", ["balance_v0", "hat"])
def test_auto_reset_with_in_kernel_philox_noise(name, mode, layout):
    """done -> reset -> obs inside the kernel, jitter from the Philox stream both sides implement."""
    env, body, prm, st = make_pair(name, 1000, env_kw=dict(in3d=True, rand_sigma=0.25), auto_reset=mode,
                                   max_steps=9, obs_layout=layout, track_stats=True)
    E = env.num_envs
    ep = (np.zeros(E, np.float32), np.zeros((4, E), np.float32))
    run_lockstep(env, body, prm, st, 30, np.random.default_rng(5), noise_reset=False, ep=ep)
    assert gu.same(env.ep_ret.cpu().numpy(), ep[0])
    assert gu.same(env.fin_stats.cpu().numpy(), ep[1])
    stats = env.episode_stats()
    assert stats["episodes"] == int(ep[1][3].sum()) == 3 * E
    np.testing.assert_allclose(stats["return_sum"], ep[1][0].astype(np.float64).sum(), rtol=1e-12)
    np.testing.assert_allclose(stats["length_sum"], ep[1][2].astype(np.float64).sum(), rtol=1e-12)


def test_philox_reset_matches_oracle_and_is_normal():
    import torch
    env, body, prm, st = make_pair("box_v0", 1 << 16, env_kw=dict(in3d=True, rand_sigma=1.0))
    prm.step_index = env.step_count
    o_c = env.reset(mode="template")
    o_o = wo.reset(body, prm, st, mode=2)
    assert gu.same(o_c.cpu().numpy(), o_o)
    v = env.vel.cpu().numpy().ravel().astype(np.float64)
    assert abs(v.mean()) < 5e-3 and abs(v.std() - 1.0) < 5e-3
    assert abs(((v - v.mean()) ** 4).mean() / v.var() ** 2 - 3.0) < 0.05      # kurtosis of a normal


def test_sharding_is_invisible():
    """SURVEY 8e: shard k of the batch equals the same envs run in one piece, bit for bit."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    E, T = 8192, 30
    kw = dict(in3d=True, auto_reset="template", max_steps=11, seed=123, track_stats=True)
    whole = BatchedPhysicsEnv("balance_v0", E, "cuda:0", **kw)
    halves = [BatchedPhysicsEnv("balance_v0", E // 2, "cuda:0", env_offset=k * E // 2, **kw) for k in range(2)]
    g = torch.Generator(device="cuda:0").manual_seed(0)
    for t in range(T):
        act = torch.rand(E, 2, device="cuda:0", generator=g) * 2 - 1
        whole.step(act)
        for k, h in enumerate(halves):
            h.step(act[k * E // 2:(k + 1) * E // 2].contiguous())
    for name in ("pos", "vel", "mx", "fin_stats"):
        cat = torch.cat([getattr(h, name) for h in halves], dim=1)
        assert gu.same(getattr(whole, name).cpu().numpy(), cat.cpu().numpy()), name
    assert gu.same(whole.obs.cpu().numpy(), torch.cat([h.obs for h in halves], 0).cpu().numpy())
    a, b0, b1 = whole.episode_stats(), halves[0].episode_stats(), halves[1].episode_stats()
    assert a["episodes"] == b0["episodes"] + b1["episodes"] > 0
    np.testing.assert_allclose(a["return_sum"], b0["return_sum"] + b1["return_sum"], rtol=1e-9)


def test_full_size_properties_1m_envs():
    """BASELINE config 3 size (2^20 envs): determinism, agreement of both kernels and both
    observation layouts, and a 2^14-env slice checked against the oracle."""
    import ctypes as C
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv, _lib
    E, T = 1 << 20, 20
    kw = dict(in3d=True, auto_reset="template", max_steps=7, seed=5)
    a = BatchedPhysicsEnv("balance_v0", E, "cuda:0", **kw)
    b = BatchedPhysicsEnv("balance_v0", E, "cuda:0", obs_layout="feature", state_layout="soa", **kw)
    lib = _lib.load()
    g = torch.Generator(device="cuda:0").manual_seed(1)
    for t in range(T):
        act = torch.rand(E, 2, device="cuda:0", generator=g) * 2 - 1
        a.step(act)
        old = lib.wg_force_generic(1)           # b runs the generic shared-memory kernel
        try:
            b.step(act)
        finally:
            lib.wg_force_generic(old)
    for name in ("pos", "vel", "mx", "steps", "reward"):
        assert torch.equal(getattr(a, name).view(torch.int32), getattr(b, name).view(torch.int32)) or \
            gu.same(getattr(a, name).cpu().numpy(), getattr(b, name).cpu().numpy()), name
    assert gu.same(a.obs.cpu().numpy(), b.obs.t().contiguous().cpu().numpy())
    # oracle on the first 2^14 envs of the same run (env ids and Philox streams coincide)
    Es = 1 << 14
    env, body, prm, st = make_pair("balance_v0", Es, env_kw=dict(in3d=True), auto_reset="template", max_steps=7, seed=5)
    g = torch.Generator(device="cuda:0").manual_seed(1)
    prm.step_index = 0
    wo.reset(body, prm, st, mode=2)
    for t in range(T):
        act = torch.rand(E, 2, device="cuda:0", generator=g) * 2 - 1
        prm.step_index = t + 1
        wo.step(body, prm, st, act[:Es].cpu().numpy())
    assert gu.same(a.pos[:, :Es].cpu().numpy(), st["pos"])
    assert gu.same(a.vel[:, :Es].cpu().numpy(), st["vel"])


@pytest.mark.parametrize("E", [4, 128, 132, 4096, 4100, 65536])
@pytest.mark.parametrize("name", ["balance_v0", "box_v0"])
def test_tma_pipelined_kernel_matches_oracle(name, E):
    """Persistent TMA kernel (WG_TUNE_TMA): full tiles, partial last tile, multi-tile CTAs, auto-reset."""
    from walker_gym_b200 import _lib
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_TMA, 1)
    try:
        env, body, prm, st = make_pair(name, E, env_kw=dict(in3d=True), auto_reset="template", max_steps=6, track_stats=True,
                                       state_layout="soa")
        ep = (np.zeros(E, np.float32), np.zeros((4, E), np.float32))
        run_lockstep(env, body, prm, st, 15, np.random.default_rng(E), noise_reset=False, ep=ep)
        assert gu.same(env.fin_stats.cpu().numpy(), ep[1])
    finally:
        lib.wg_set_tuning(_lib.TUNE_TMA, old)


def test_feature_major_actions_and_graph_safe_counter():
    """act_layout='feature' reads [M, E] actions; graph_safe keeps the Philox step index on the device.
    Both must give the same bits as the plain path."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    E, T = 2048, 25
    kw = dict(in3d=True, auto_reset="template", max_steps=6, seed=9)
    a = BatchedPhysicsEnv("box_v0", E, "cuda:0", **kw)
    b = BatchedPhysicsEnv("box_v0", E, "cuda:0", act_layout="feature", obs_layout="feature", graph_safe=True, **kw)
    g = torch.Generator(device="cuda:0").manual_seed(2)
    for t in range(T):
        act = torch.rand(E, 4, device="cuda:0", generator=g) * 2 - 1
        a.step(act)
        b.step(act.t().contiguous())
    assert gu.same(a.pos.cpu().numpy(), b.pos.cpu().numpy()) and gu.same(a.vel.cpu().numpy(), b.vel.cpu().numpy())
    assert gu.same(a.obs.cpu().numpy(), b.obs.t().contiguous().cpu().numpy())
    assert int(b._counter.item()) == T + 1 and a.step_count == T + 1


def test_rollout_collector_cuda_graph_and_eager():
    """PPO rollout collection (config 5): eager and CUDA-graph-replayed rollouts agree on everything that
    does not depend on torch's RNG stream, and the episode statistics go through the K3 reduction."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    from walker_gym_b200.rollout import FeatureMajorMLP, RolloutCollector
    E, T = 4096, 16
    outs = []
    for use_graph in (False, True):
        torch.manual_seed(0)
        torch.cuda.manual_seed(0)
        env = BatchedPhysicsEnv("Balance-v0", E, "cuda:0", in3d=True, auto_reset="template", max_steps=10, seed=4,
                                obs_layout="feature", act_layout="feature", graph_safe=True)
        pol = FeatureMajorMLP(env.obs_dim, env.M).to("cuda:0")
        col = RolloutCollector(env, pol, T, use_cuda_graph=use_graph)
        # the capture warm-up of the first graph collect() runs on a snapshot that is restored (env state, device step
        # counter, finished-episode accumulators): the first collect() is one rollout from the initial state
        batch = col.collect()
        torch.cuda.synchronize()
        outs.append({k: v.clone() for k, v in batch.items()})
        stats = col.episode_stats(all_reduce=False)
        assert batch["obs"].shape == (T + 1, env.obs_dim, E) and batch["actions"].shape == (T, env.M, E)
        assert stats["episodes"] == E and torch.isfinite(batch["advantages"]).all()
        assert int(env._counter.item()) == T + 1            # reset + exactly one rollout, graph or not
    assert torch.equal(outs[0]["dones"], outs[1]["dones"]) and int(outs[0]["dones"].sum()) == E
    assert torch.equal(outs[0]["obs"][0], outs[1]["obs"][0])
    for o in outs:
        assert torch.isfinite(o["rewards"]).all() and torch.isfinite(o["logp"]).all()


@pytest.mark.parametrize("name", ["box2", "humanb"])
def test_config1_single_walker_1000_steps(name):
    """BASELINE config 1: one gym/walker.py body, 1000 steps of random actions; the CPU side is the oracle
    (the legacy walker.py/engine.py/env.py trio is not executable as shipped, SURVEY 0.2; L1 semantics apply)."""
    env, body, prm, st = make_pair(name, 1, env_kw=dict(in3d=True))
    run_lockstep(env, body, prm, st, 1000, np.random.default_rng(0))
    assert int(env.steps.item()) == 1000 and bool(env.done.item())


def test_run2_integrator_batched():
    env, body, prm, st = make_pair("box_v0", 512, env_kw=dict(in3d=True), integrator="run2")
    prm.integrator = 1
    run_lockstep(env, body, prm, st, 40, np.random.default_rng(8))


@pytest.mark.parametrize("parts", [2, 4, 8])
@pytest.mark.parametrize("name,layout", [("quad_balance", "row"), ("insect", "feature"), ("humanb", "row"),
                                         ("balance3", "row"), ("leg", "feature")])
def test_mass_partitioned_kernel_matches_oracle(name, layout, parts):
    """P lanes per env (WG_TUNE_PART): crossing springs are evaluated by both owners; bits must not change.
    Covers disjoint units, a connected body, DingPoints / float masses, auto-reset and ragged tails."""
    from walker_gym_b200 import _lib
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_PART, parts)
    try:
        env, body, prm, st = make_pair(name, 1000 + parts, env_kw=dict(in3d=True, rand_sigma=0.3), auto_reset="template",
                                       max_steps=7, k_sub=2, obs_layout=layout, track_stats=True)
        E = env.num_envs
        ep = (np.zeros(E, np.float32), np.zeros((4, E), np.float32))
        run_lockstep(env, body, prm, st, 16, np.random.default_rng(parts), noise_reset=False, ep=ep)
        assert gu.same(env.fin_stats.cpu().numpy(), ep[1])
    finally:
        lib.wg_set_tuning(_lib.TUNE_PART, old)


def test_partition_off_uses_one_thread_per_env():
    from walker_gym_b200 import _lib
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_PART, 0)
    try:
        env, body, prm, st = make_pair("quad_balance", 256, env_kw=dict(in3d=True), k_sub=3)
        run_lockstep(env, body, prm, st, 6, np.random.default_rng(1))
    finally:
        lib.wg_set_tuning(_lib.TUNE_PART, old)


@pytest.mark.parametrize("state_layout", ["soa", "packed"])
@pytest.mark.parametrize("E", [1, 127, 128, 129, 1000, 4096])
@pytest.mark.parametrize("name,in3d,layout", [("balance_v0", True, "row"), ("box_v0", True, "feature"),
                                               ("balance", False, "row"), ("box2", False, "feature"),
                                               ("box", True, "row"), ("test", False, "row"), ("intrian", True, "feature"),
                                               ("hat", True, "row"), ("humanb", True, "row"), ("box4", False, "feature"),
                                               ("leg2", True, "row"), ("leg", True, "feature"),
                                               ("balance2", True, "row"), ("balance3", True, "feature"),
                                               ("balance3", False, "row")])
def test_state_layouts_match_oracle(name, in3d, layout, E, state_layout):
    """Both state layouts -- separate SoA rows and the packed [tile][k/4][128][4] float4 layout -- against the
    oracle: full and ragged tiles, 2-D and 3-D, unit and integer masses, auto-reset with episode statistics."""
    env, body, prm, st = make_pair(name, E, env_kw=dict(in3d=in3d), auto_reset="template", max_steps=5,
                                   obs_layout=layout, track_stats=True, state_layout=state_layout)
    assert env.state_layout == state_layout
    ep = (np.zeros(E, np.float32), np.zeros((4, E), np.float32))
    run_lockstep(env, body, prm, st, 12, np.random.default_rng(E), noise_reset=True, ep=ep)
    assert gu.same(env.ep_ret.cpu().numpy(), ep[0]) and gu.same(env.fin_stats.cpu().numpy(), ep[1])


def test_packed_layout_rejected_for_bodies_without_a_specialised_kernel():
    from walker_gym_b200 import BatchedPhysicsEnv
    with pytest.raises(ValueError):
        BatchedPhysicsEnv("insect", 64, "cuda:0", state_layout="packed")
    assert BatchedPhysicsEnv("insect", 64, "cuda:0").state_layout == "soa"
    for name in ("Balance-v0", "Box-v0", "box", "test", "intrian", "hat", "humanb", "box4", "leg", "leg2",
                 "balance2", "balance3"):          # the last two: mass 0.1 / a DingPoint on the Balance spring graph
        assert BatchedPhysicsEnv(name, 64, "cuda:0").state_layout == "packed", name


def _random_spec(rng, N, S, M):
    pts = [(float(rng.choice([1, 1, 2, 3, 5, 0.5, 0.25, 7.5])), tuple(float(v) for v in rng.uniform(-150, 150, 3)), bool(n == 5))
           for n in range(N)]
    pairs = [(i, j) for i in range(N) for j in range(i + 1, N)]
    rng.shuffle(pairs)
    mus = [(i, j, {"k": float(rng.choice([500, 1000, -700]))}) for i, j in pairs[:M]]
    sks = [(j, i, {"dampk": float(rng.choice([5, 20]))}) for i, j in pairs[M:S]]
    return {"points": pts, "muscles": mus, "skeletons": sks}


# (N, S, M, WG_TUNE_PART, k_sub, obs layout).  The second list: one substep with the partition automatic (-1: off at
# k_sub 1) or off, so the one-thread-per-env kernel is asked for, at the muscle counts around its shared-memory limit
# (tile of 11 * N + M + 3 rows of 129 floats: at N = 32 on a B200 up to M = 92 with row-major, 95 with feature-major
# observations); beyond it the step runs the mass-partitioned kernel with two lanes per env.  Which kernel ran is
# checked in test_cuda_x64_bodies.py::test_float32_body_limit_kernels.
BODY_SIZE_CASES = [(32, 96, 10, -1, 2, "row"), (32, 96, 10, 8, 2, "row"), (32, 96, 10, 0, 2, "row"), (9, 30, 5, 2, 2, "row"),
                   (1, 0, 0, -1, 2, "row"), (2, 1, 1, -1, 2, "row"), (17, 16, 0, 4, 2, "row")]
BODY_LIMIT_CASES = [(N, 96, M, parts, 1, layout) for N, M in ((32, 92), (32, 93), (32, 95), (32, 96), (16, 68))
                    for parts in (-1, 0) for layout in ("row", "feature")]


@pytest.mark.parametrize("N,S,M,parts,k_sub,layout", BODY_SIZE_CASES + BODY_LIMIT_CASES,
                         ids=[f"{N}-{S}-{M}-{p}" for N, S, M, p, _, _ in BODY_SIZE_CASES] +
                             [f"{N}-{S}-{M}-{p}-k{k}-{lay}" for N, S, M, p, k, lay in BODY_LIMIT_CASES])
def test_maximum_and_minimum_body_sizes(N, S, M, parts, k_sub, layout):
    """The ABI limits (32 masses, 96 springs) and the degenerate ends (a single free mass, no muscles)
    on the generic and the mass-partitioned kernels, with float masses and a DingPoint."""
    import ctypes as C
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv, Creature, DingPoint, Muscle, Point, Skeleton, _lib
    rng = np.random.default_rng(N * 100 + S)
    spec = _random_spec(rng, N, S, M)
    Point.clear()
    pts = [DingPoint(m, list(p)) if f else Point(m, list(p), [0, 0, 0]) for m, p, f in spec["points"]]
    cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in spec["muscles"]],
                  [Skeleton(pts[i], pts[j], **kw) for i, j, kw in spec["skeletons"]])
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_PART, parts)
    try:
        E = 300
        env = BatchedPhysicsEnv(cr, E, "cuda:0", in3d=True, auto_reset="template", max_steps=5, k_sub=k_sub, seed=3,
                                obs_layout=layout, keep_old_a=True, track_info=True, track_contacts=True, initial_reset=False)
        body = wo.make_body(spec)
        prm = wo.make_params(in3d=True, auto_reset=2, max_steps=5, k_sub=k_sub, seed=3)
        st = wo.init_state(body, E)
        run_lockstep(env, body, prm, st, 9, rng, noise_reset=False)
    finally:
        lib.wg_set_tuning(_lib.TUNE_PART, old)
        Point.clear()


def test_empty_batch_is_a_no_op():
    import ctypes as C
    from walker_gym_b200 import _lib, create_box_creature, make_params
    from walker_gym_b200.topology import topology_from_creature
    lib = _lib.load()
    topo, prm, buf = topology_from_creature(create_box_creature()), make_params(in3d=True), _lib.WgBuffers()
    import torch
    z = torch.zeros(16, device="cuda:0")
    buf.pos = buf.vel = buf.mx = buf.steps = z.data_ptr()
    assert lib.wg_step(C.byref(topo), C.byref(prm), C.byref(buf), 0, None) == 0
    assert lib.wg_reset(C.byref(topo), C.byref(prm), C.byref(buf), 0, 1, None, None) == 0


def test_huge_batch_64bit_indexing():
    """2^26 + 3 Box-v0 envs in one launch: the observation buffer has more than 2^31 elements, so every index
    that is not 64-bit would wrap.  The batch repeats a pattern of 4096 distinct envs (no auto-reset, so nothing
    depends on the env id): the last full pattern -- beyond the 2^31-element mark -- and the ragged tail must equal
    the first pattern bit for bit, and the first pattern must equal the oracle."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    Pn, E, T = 4096, (1 << 26) + 3, 3
    reps = (E + Pn - 1) // Pn
    env = BatchedPhysicsEnv("Box-v0", E, "cuda:0", in3d=True, auto_reset=None, track_stats=False, initial_reset=False)
    assert env.state_layout == "packed" and env.obs.numel() > 2 ** 31
    rng = np.random.default_rng(42)
    body = wo.make_body(spec_of("box_v0"))
    prm = wo.make_params(in3d=True, auto_reset=0)
    st = wo.init_state(body, Pn)
    st["pos"] += rng.normal(0, 1.0, st["pos"].shape).astype(np.float32)
    st["vel"] += rng.normal(0, 1.0, st["vel"].shape).astype(np.float32)
    tile = lambda a: torch.from_numpy(a).to("cuda:0").repeat(1, reps)[:, :E]          # noqa: E731
    env.set_state(pos=tile(st["pos"]), vel=tile(st["vel"]))
    acts = [rng.uniform(-1, 1, (Pn, 4)).astype(np.float32) for _ in range(T)]
    for t in range(T):
        a = torch.from_numpy(acts[t]).to("cuda:0").repeat(reps, 1)[:E].contiguous()
        obs, rew, done, _ = env.step(a)
        out = wo.step(body, prm, st, acts[t], want_info=False)
    torch.cuda.synchronize()
    first = obs[:Pn]
    last_full = obs[(reps - 2) * Pn:(reps - 1) * Pn]
    tail = obs[(reps - 1) * Pn:]
    assert (reps - 2) * Pn * env.obs_dim > 2 ** 31
    assert torch.equal(first.view(torch.int32), last_full.view(torch.int32))
    assert torch.equal(first[: tail.shape[0]].view(torch.int32), tail.view(torch.int32)) and tail.shape[0] == E - (reps - 1) * Pn
    assert torch.equal(rew[:Pn].view(torch.int32), rew[(reps - 2) * Pn:(reps - 1) * Pn].view(torch.int32))
    assert gu.same(first.cpu().numpy(), out["obs"]) and gu.same(rew[:Pn].cpu().numpy(), out["reward"])
    assert gu.same(env.pos[:, (reps - 2) * Pn:(reps - 1) * Pn].cpu().numpy(), st["pos"])


@pytest.mark.parametrize("seed", range(16))
def test_fuzz_random_bodies_and_parameters(seed):
    """Seeded fuzz: random topology (1..32 masses, up to 96 springs), float / integer / unit masses, a DingPoint,
    signed k, random environment parameters (gravity, global damping, ground height/spring/damper/friction, dt),
    2-D or 3-D, run1 / run2, 1..4 substeps, both observation layouts, jitter or template auto-reset, and whichever
    kernel the dispatcher picks (generic or mass-partitioned) -- bit for bit against the oracle."""
    from walker_gym_b200 import BatchedPhysicsEnv, Creature, DingPoint, Muscle, Point, Skeleton
    rng = np.random.default_rng(1234 + seed)
    N = int(rng.integers(1, 33))
    S = int(rng.integers(0, min(96, N * (N - 1) // 2) + 1))
    M = int(rng.integers(0, min(S, 12) + 1))
    spec = _random_spec(rng, N, S, M)
    if rng.random() < 0.5:                                     # integer-only masses: the exact small-integer division path
        spec["points"] = [(float(rng.integers(1, 9)), p, f) for _, p, f in spec["points"]]
    in3d = bool(rng.random() < 0.6)
    env_kw = dict(in3d=in3d, g=float(rng.choice([100, 9.8, 0, 250.5])), dampk=float(rng.choice([0, 0, 0.5, 3])),
                  ground_high=float(rng.choice([0, -20, 35.5])), ground_k=float(rng.choice([1000, 0, 321])),
                  ground_damp=float(rng.choice([100, 0, 12.5])), friction=float(rng.choice([100, 0, 7])),
                  rand_sigma=float(rng.choice([0.1, 1.0])), time_step=float(rng.choice([0.01, 0.003])))
    k_sub = int(rng.integers(1, 5))
    integrator = "run2" if rng.random() < 0.3 else "run1"
    auto = str(rng.choice(["template", "jitter"]))
    layout = str(rng.choice(["row", "feature"]))
    Point.clear()
    try:
        pts = [DingPoint(m, list(p)) if f else Point(m, list(p), [0, 0, 0]) for m, p, f in spec["points"]]
        cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in spec["muscles"]],
                      [Skeleton(pts[i], pts[j], **kw) for i, j, kw in spec["skeletons"]])
        E = int(rng.integers(1, 700))
        env = BatchedPhysicsEnv(cr, E, "cuda:0", auto_reset=auto, max_steps=4, k_sub=k_sub, seed=seed, obs_layout=layout,
                                integrator=integrator, keep_old_a=True, track_info=True, track_contacts=True,
                                initial_reset=False, **env_kw)
        body = wo.make_body(spec)
        prm = wo.make_params(auto_reset={"jitter": 1, "template": 2}[auto], max_steps=4, k_sub=k_sub, seed=seed,
                             integrator=1 if integrator == "run2" else 0, **env_kw)
        st = wo.init_state(body, E)
        run_lockstep(env, body, prm, st, 10, rng, noise_reset=True)
    finally:
        Point.clear()


def _custom_creature(masses, ding=()):
    from walker_gym_b200 import Creature, DingPoint, Muscle, Point, Skeleton
    Point.clear()
    pos = [(-30, 40, 5), (35, 60, -3), (0, 5, 0), (10, 90, 2), (-60, 20, 0)]
    pts = [DingPoint(m, list(p)) if n in ding else Point(m, list(p), [0, 0, 0]) for n, (m, p) in enumerate(zip(masses, pos))]
    mus = [Muscle(pts[0], pts[2], k=800, dampk=15, minl=0.3, maxl=1.2), Muscle(pts[1], pts[2], k=1200, dampk=25), Muscle(pts[4], pts[0], k=-300)]
    sks = [Skeleton(pts[0], pts[1], k=500), Skeleton(pts[1], pts[3], k=2000, dampk=5), Skeleton(pts[4], pts[2], x=61.5)]
    spec = {"points": [(m, p, n in ding) for n, (m, p) in enumerate(zip(masses, pos))],
            "muscles": [(0, 2, {"k": 800, "dampk": 15, "minl": 0.3, "maxl": 1.2}), (1, 2, {"k": 1200, "dampk": 25}), (4, 0, {"k": -300})],
            "skeletons": [(0, 1, {"k": 500}), (1, 3, {"k": 2000, "dampk": 5}), (4, 2, {"x": 61.5})]}
    return Creature(pts, mus, sks), spec


@pytest.mark.parametrize("masses,ding,in3d,layout", [((1, 1, 1, 1, 1), (), True, "row"), ((2, 5, 1, 3, 4), (), False, "feature"),
                                                      ((2, 2, 1, 3, 2), (), True, "row"), ((2, 3, 1, 3, 1), (), True, "row"),
                                                      ((2.5, 0.1, 7, 1, 3), (3,), True, "row")])
def test_runtime_specialised_kernel_for_user_bodies(masses, ding, in3d, layout):
    """A user-built creature gets the packed-state kernel compiled for its spring graph at run time (NVRTC): unit,
    integer and arbitrary masses with a DingPoint; bit for bit against the oracle, and switched off it falls back to
    the run-time-topology kernel with the same bits."""
    from walker_gym_b200 import BatchedPhysicsEnv, Point, _lib
    lib = _lib.load()
    try:
        cr, spec = _custom_creature(masses, ding)
        E = 4100
        kw = dict(in3d=in3d, auto_reset="template", max_steps=6, k_sub=2, seed=4, obs_layout=layout, keep_old_a=True,
                  track_info=True, track_contacts=True, initial_reset=False)
        env = BatchedPhysicsEnv(cr, E, "cuda:0", **kw)
        assert env.state_layout == "packed" and env.kernel_variant == 0          # no ahead-of-time kernel: compiled now
        body = wo.make_body(spec)
        prm = wo.make_params(in3d=in3d, auto_reset=2, max_steps=6, k_sub=2, seed=4)
        st = wo.init_state(body, E)
        run_lockstep(env, body, prm, st, 14, np.random.default_rng(0), noise_reset=True)
        old = lib.wg_set_tuning(_lib.TUNE_JIT, 0)
        try:
            env2 = BatchedPhysicsEnv(cr, E, "cuda:0", **kw)
            assert env2.state_layout == "soa"
            with pytest.raises(ValueError):
                BatchedPhysicsEnv(cr, E, "cuda:0", state_layout="packed", **kw)
        finally:
            lib.wg_set_tuning(_lib.TUNE_JIT, old)
    finally:
        Point.clear()


def test_runtime_specialised_soa_kernel_for_mid_size_user_bodies():
    """9..16 masses: no packed layout, but the SoA step kernel is compiled for the body's spring graph at run time
    (NVRTC); bit for bit against the oracle, and against the run-time-topology kernel when the compiler is switched off."""
    from walker_gym_b200 import BatchedPhysicsEnv, Creature, Muscle, Point, Skeleton, _lib
    lib = _lib.load()
    rng = np.random.default_rng(77)
    spec = _random_spec(rng, 11, 18, 5)
    spec["points"] = [(float(rng.integers(1, 4)), p, False) for _, p, _ in spec["points"]]      # integer masses, no DingPoint
    Point.clear()
    try:
        pts = [Point(m, list(p), [0, 0, 0]) for m, p, _ in spec["points"]]
        cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in spec["muscles"]],
                      [Skeleton(pts[i], pts[j], **kw) for i, j, kw in spec["skeletons"]])
        E = 4200
        kw = dict(in3d=True, auto_reset="template", max_steps=5, k_sub=2, seed=8, keep_old_a=True, track_info=True,
                  track_contacts=True, initial_reset=False)
        res = []
        for jit in (1, 0):
            old = lib.wg_set_tuning(_lib.TUNE_JIT, jit)
            try:
                env = BatchedPhysicsEnv(cr, E, "cuda:0", **kw)
                assert env.state_layout == "soa"
                body = wo.make_body(spec)
                prm = wo.make_params(in3d=True, auto_reset=2, max_steps=5, k_sub=2, seed=8)
                st = wo.init_state(body, E)
                run_lockstep(env, body, prm, st, 12, np.random.default_rng(5), noise_reset=True)
                res.append(env.pos.clone())
            finally:
                lib.wg_set_tuning(_lib.TUNE_JIT, old)
        assert gu.same(res[0].cpu().numpy(), res[1].cpu().numpy())
    finally:
        Point.clear()


@pytest.mark.parametrize("R,masses,in3d,layout,auto", [(2, (5, 5, 1, 3), True, "row", "template"), (8, (5, 5, 1, 3), False, "feature", "jitter"),
                                                       (4, (1, 1, 1, 1), False, "row", "template"), (4, (2, 3, 4, 5), True, "feature", "jitter"),
                                                       (8, (5, 5, 1, 3), True, "row", "template")])
def test_units_kernel_for_bodies_of_identical_disconnected_units(R, masses, in3d, layout, auto):
    """R Balance units in one env (R = 2, 4, 8), one lane per unit: the Balance-v0 mass pattern (mode 3), unit masses
    and other integer masses; 2-D and 3-D, both observation layouts, both auto-reset modes, substeps, ragged batches."""
    from walker_gym_b200 import BODIES, BatchedPhysicsEnv, Creature, Muscle, Point, Skeleton
    base = BODIES["balance_v0"]
    pts_s, mus_s, sks_s = [], [], []
    for u in range(R):
        off = 150.0 * (u - (R - 1) / 2)
        pts_s += [(float(masses[n]), (p[0] + off, p[1], p[2]), False) for n, (_, p) in enumerate(base["points"])]
        mus_s += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["muscles"]]
    for u in range(R):
        sks_s += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["skeletons"]]
    spec = {"points": pts_s, "muscles": mus_s, "skeletons": sks_s}
    Point.clear()
    try:
        pts = [Point(m, list(p), [0, 0, 0]) for m, p, _ in pts_s]
        cr = Creature(pts, [Muscle(pts[i], pts[j]) for i, j, _ in mus_s], [Skeleton(pts[i], pts[j]) for i, j, _ in sks_s])
        E = 1003
        env = BatchedPhysicsEnv(cr, E, "cuda:0", in3d=in3d, auto_reset=auto, max_steps=6, k_sub=3, seed=R, obs_layout=layout,
                                keep_old_a=True, track_info=True, track_contacts=True, initial_reset=False)
        body = wo.make_body(spec)
        prm = wo.make_params(in3d=in3d, auto_reset={"jitter": 1, "template": 2}[auto], max_steps=6, k_sub=3, seed=R)
        st = wo.init_state(body, E)
        run_lockstep(env, body, prm, st, 14, np.random.default_rng(R), noise_reset=True)
    finally:
        Point.clear()


@pytest.mark.parametrize("R,masses,in3d,layout,auto,link", [
    (4, (5, 5, 1, 3), True, "row", "template", {}), (2, (5, 5, 1, 3), False, "feature", "jitter", {"k": 700, "dampk": 15}),
    (8, (5, 5, 1, 3), True, "row", "jitter", {"k": 3000}), (4, (1, 1, 1, 1), False, "row", "template", {"x": 80.0}),
    (4, (2, 3, 4, 5), True, "feature", "template", {})])
def test_linked_units_kernel_for_a_connected_chain_of_units(R, masses, in3d, layout, auto, link):
    """The same units CONNECTED by link bones (unit u's mass 1 -- unit u+1's mass 0, after every unit's own bones in
    the skeleton list): one lane per unit, the far endpoint of a link over warp shuffles, both owners evaluate the link.
    Bit-identical to the oracle's one-env-at-a-time evaluation: mass patterns, 2-D / 3-D, layouts, reset modes,
    substeps, ragged batch, custom link constants."""
    from walker_gym_b200 import BODIES, BatchedPhysicsEnv, Creature, Muscle, Point, Skeleton, _lib
    base = BODIES["balance_v0"]
    pts_s, mus_s, sks_s = [], [], []
    for u in range(R):
        off = 150.0 * (u - (R - 1) / 2)
        pts_s += [(float(masses[n]), (p[0] + off, p[1], p[2]), False) for n, (_, p) in enumerate(base["points"])]
        mus_s += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["muscles"]]
    for u in range(R):
        sks_s += [(4 * u + i, 4 * u + j, {}) for i, j, _ in base["skeletons"]]
    sks_s += [(4 * u + 1, 4 * (u + 1), dict(link)) for u in range(R - 1)]
    spec = {"points": pts_s, "muscles": mus_s, "skeletons": sks_s}
    Point.clear()
    try:
        pts = [Point(m, list(p), [0, 0, 0]) for m, p, _ in pts_s]
        cr = Creature(pts, [Muscle(pts[i], pts[j]) for i, j, _ in mus_s], [Skeleton(pts[i], pts[j], **kw) for i, j, kw in sks_s])
        E = 1003
        kw = dict(in3d=in3d, auto_reset=auto, max_steps=6, k_sub=3, seed=R, obs_layout=layout, keep_old_a=True,
                  track_info=True, track_contacts=True, initial_reset=False)
        env = BatchedPhysicsEnv(cr, E, "cuda:0", **kw)
        body = wo.make_body(spec)
        prm = wo.make_params(in3d=in3d, auto_reset={"jitter": 1, "template": 2}[auto], max_steps=6, k_sub=3, seed=R)
        st = wo.init_state(body, E)
        run_lockstep(env, body, prm, st, 14, np.random.default_rng(R), noise_reset=True)
        # and against the run-time-topology kernel on the same inputs (kernel agreement at a glance)
        lib = _lib.load()
        a, b = BatchedPhysicsEnv(cr, E, "cuda:0", **kw), BatchedPhysicsEnv(cr, E, "cuda:0", **kw)
        import torch
        g = torch.Generator(device="cuda:0").manual_seed(5)
        for t in range(6):
            act = torch.rand(E, a.M, device="cuda:0", generator=g) * 2 - 1
            oa = a.step(act)[0].clone()
            lib.wg_force_generic(1)
            try:
                ob = b.step(act)[0].clone()
            finally:
                lib.wg_force_generic(0)
            assert gu.same(oa.cpu().numpy(), ob.cpu().numpy()), t
    finally:
        Point.clear()


def test_config4_connected_enlarged_body_8_substeps():
    """BASELINE config 4 on ONE connected creature (quad_balance_chain: N=16, S=23, M=8), 8 substeps."""
    env, body, prm, st = make_pair("quad_balance_chain", 1024, env_kw=dict(in3d=True), k_sub=8, auto_reset="template", max_steps=12)
    run_lockstep(env, body, prm, st, 30, np.random.default_rng(4), noise_reset=False)


@pytest.mark.parametrize("mode", ["graph_safe_packed", "graph_safe_soa", "x64"])
def test_state_dict_round_trip_is_a_complete_snapshot(mode):
    """state_dict() is a snapshot (copies) that carries the device step counter of graph_safe envs and the float64
    muscle state of x64 envs: restore + replay reproduces the same trajectory bit for bit, auto-reset jitter included."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    E, T = 3000, 9
    x64 = mode == "x64"
    kw = dict(in3d=True, auto_reset="template", max_steps=4, seed=21)
    if x64:
        env = BatchedPhysicsEnv("Box-v0", E, DEV, x64=True, **kw)
    else:
        env = BatchedPhysicsEnv("Balance-v0", E, DEV, graph_safe=True,
                                state_layout="packed" if mode.endswith("packed") else "soa", **kw)
    g = torch.Generator(device=DEV).manual_seed(3)
    dt = torch.float64 if x64 else torch.float32
    acts = [(torch.rand(E, env.M, device=DEV, generator=g, dtype=dt) * (160 if x64 else 2) - (80 if x64 else 1)) for _ in range(2 * T)]
    for t in range(T):
        env.step(acts[t])
    sd = env.state_dict()
    before = {k: v.clone() for k, v in sd.items() if torch.is_tensor(v)}

    def run():
        out = []
        for t in range(T, 2 * T):
            obs, rew, done, _ = env.step(acts[t])
            out.append((obs.clone(), rew.clone(), done.clone()))
        return out, env.pos.clone(), env.vel.clone(), env.mx.clone()
    first = run()
    for k, v in before.items():                              # a snapshot: stepping did not change the dict's tensors
        assert torch.equal(sd[k].view(torch.uint8), v.view(torch.uint8)), k
    env.load_state_dict(sd)
    second = run()
    for (o1, r1, d1), (o2, r2, d2) in zip(first[0], second[0]):
        assert gu.same(o1.cpu().numpy(), o2.cpu().numpy()) and gu.same(r1.cpu().numpy(), r2.cpu().numpy())
        assert torch.equal(d1, d2)
    for a, b in zip(first[1:], second[1:]):
        assert gu.same(a.cpu().numpy(), b.cpu().numpy())
    if x64:
        assert "mx64" in sd and "mx_weak" in sd and 0 < float(sd["mx_weak"].float().mean()) < 1
    else:
        assert int(sd["counter"].item()) == T + 1


def test_rejected_step_leaves_the_bound_buffers_alone():
    """step(out=...) validates action / noise before it rebinds the result pointers: after a ValueError the next plain
    step() writes the env's own buffers."""
    import torch
    from walker_gym_b200 import BatchedPhysicsEnv
    E = 513
    env = BatchedPhysicsEnv("Box-v0", E, DEV, in3d=True, seed=1)
    ref = BatchedPhysicsEnv("Box-v0", E, DEV, in3d=True, seed=1)
    out = (torch.full((E, env.obs_dim), 7.0, device=DEV), torch.full((E,), 7.0, device=DEV), torch.zeros(E, dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError):
        env.step(torch.zeros(E + 1, env.M, device=DEV), out=out)
    with pytest.raises(ValueError):
        env.step(torch.zeros(E, env.M, device=DEV), noise=torch.zeros(3, device=DEV), out=out)
    a = torch.rand(E, env.M, device=DEV) * 2 - 1
    obs, rew, done, _ = env.step(a)
    obs_r, rew_r, done_r, _ = ref.step(a)
    assert obs.data_ptr() == env.obs.data_ptr() and gu.same(obs.cpu().numpy(), obs_r.cpu().numpy())
    assert gu.same(rew.cpu().numpy(), rew_r.cpu().numpy()) and float(out[0].min()) == 7.0 and float(out[1].min()) == 7.0


def rope_bodies(rng):
    """Balance-v0's graph (which has every specialisation) with two rope-type springs, and a random 9-mass body with a
    mix of rope-type muscles and bones: [(points [(m, pos)], muscles [(i, j, kw)], skeletons [(i, j, kw)])]."""
    base = [(5, (-50, 100, 0)), (5, (50, 100, 0)), (1, (0, 0, 0)), (3, (0, 100, 0))]
    bodies = [(base, [(0, 2, {"string": True}), (1, 2, {})], [(0, 1, {}), (0, 3, {"string": True, "x": 60.0}), (1, 3, {})])]
    pts9 = [(float(rng.integers(1, 6)), tuple(rng.uniform(-80, 80, 3).round(1))) for _ in range(9)]
    pts9 = [(m, (p[0], abs(p[1]) + 5, p[2])) for m, p in pts9]
    mus9 = [(int(i), int((i + 1 + rng.integers(0, 7)) % 9), {"string": bool(rng.integers(0, 2))}) for i in range(5)]
    sks9 = [(int(i), int((i + 1) % 9), {"string": bool(rng.integers(0, 2)), "k": float(rng.choice([300, 1000, -500]))}) for i in range(9)]
    bodies.append((pts9, [(i, j, kw) for i, j, kw in mus9 if i != j], [(i, j, kw) for i, j, kw in sks9 if i != j]))
    return bodies


def rope_creature(pts_s, mus_s, sks_s):
    """(Creature, oracle spec) of one rope_bodies() entry; clears the Point registry first."""
    from walker_gym_b200 import Creature, Muscle, Point, Skeleton
    spec = {"points": [(m, p, False) for m, p in pts_s], "muscles": mus_s, "skeletons": sks_s}
    Point.clear()
    pts = [Point(m, list(p), [0, 0, 0]) for m, p in pts_s]
    cr = Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in mus_s], [Skeleton(pts[i], pts[j], **kw) for i, j, kw in sks_s])
    return cr, spec


@pytest.mark.parametrize("E,layout,parts", [(1000, "row", -1), (777, "feature", -1), (515, "row", 4)])
def test_rope_type_springs_match_oracle(E, layout, parts):
    """Rope-type springs (`string=True`, Point.resilience semantics, gym/optimized_engine.py:134-138) as a per-spring
    flag of the run-time-topology kernels: random bodies with a mix of rope-type muscles and bones, bit-exact against
    the oracle; a body with such springs never takes a compile-time specialisation."""
    from walker_gym_b200 import BatchedPhysicsEnv, Point, _lib
    rng = np.random.default_rng(E)
    lib = _lib.load()
    old = lib.wg_set_tuning(_lib.TUNE_PART, parts)
    try:
        for body_s in rope_bodies(rng):
            cr, spec = rope_creature(*body_s)
            env = BatchedPhysicsEnv(cr, E, "cuda:0", in3d=True, auto_reset="template", max_steps=9, k_sub=2, seed=5,
                                    obs_layout=layout, keep_old_a=True, track_info=True, track_contacts=True, initial_reset=False)
            assert env.kernel_variant == 0 and env.state_layout == "soa"
            body = wo.make_body(spec)
            prm = wo.make_params(in3d=True, auto_reset=2, max_steps=9, k_sub=2, seed=5)
            st = wo.init_state(body, E)
            run_lockstep(env, body, prm, st, 20, rng, noise_reset=True)
    finally:
        lib.wg_set_tuning(_lib.TUNE_PART, old)
        Point.clear()
