"""GPU: the step kernels wg_jit.cu compiles at run time (NVRTC) for user-built bodies, against the C oracle.

A body with no ahead-of-time kernel gets, once the batch is large enough to pay for the compilation, a kernel compiled
for its spring graph: the packed-state kernel (1..8 masses, 1..16 springs; state_layout="auto" at E >= 4096), the SoA
kernel (up to 16 masses, 32 springs; wg_step at E >= 4096) or the T-steps-per-launch kernel (step_many).  Its mass
pattern picks the instance: MM 0 (every mass 1), MM 3 on TopoJitP (unit, power-of-two or odd small-integer masses, the
pattern of equal masses baked into the code) or MM 2 (any other mass, or a DingPoint).

Seeded random graphs of each mass class run at the batch sizes that select these kernels, bit for bit against the
oracle (up to NaN payload and the sign of zero).  A fallback (the run-time-topology kernel) gives the same bits, so every
case also names the kernel instance it ran, through the profiler session shared with test_cuda_full_size.py."""
import os
import re
import tempfile

import numpy as np
import pytest

import golden_util as gu
import walker_oracle as wo
from test_cuda_full_size import SliceLockstep, kernel_names, n_sms, register_probes
from test_cuda_vs_oracle import run_lockstep, spec_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
JIT_MIN_ENVS = 4096            # batch size from which the compiled kernels are chosen (batched.py, wg_step)
PACKED_BLOCK = 128             # envs per CTA of the packed kernels

SMALL = (2.0, 3.0, 4.0, 5.0, 7.0, 0.5)      # powers of two and odd integers: exact division, mass mode 1
GENERAL = (7.5, 0.1, 2.5, 1.3)              # neither: mass mode 2


@pytest.fixture(autouse=True)
def clear_points():
    from walker_gym_b200 import Point
    Point.clear()
    yield
    Point.clear()


# ---- bodies --------------------------------------------------------------------------------------------------------
def mass_mode(masses, fixed):
    """The MM template argument wg_jit.cu compiles for these masses (mass_mode + mode_of, wg_launch.cuh / wg_jit.cu)."""
    def kind(m):
        m = float(np.float32(m))
        if m == 1.0:
            return 0
        if np.frexp(m)[0] == 0.5:
            return 1
        return 2 if 3 <= m <= 2047 and m == int(m) and int(m) % 2 == 1 else 3
    kinds = [kind(m) for m in masses]
    if any(fixed) or 3 in kinds:
        return 2
    return 3 if any(kinds) else 0


def random_spec(seed, N, S, M, mass_class, feature=""):
    """A seeded random body of N masses and S springs (the first M muscles) for the oracle and creature().
    mass_class: "unit" (every mass 1), "classes" (odd small integers / powers of two with repeats, a unit mass, a spring
    between two equal non-unit masses and one with a unit endpoint), "general" (one mass that is neither) or "ding"
    (small integers and one DingPoint).  feature: "isolated" (the last mass has no spring) or "hub" (mass 0 has degree
    >= 5)."""
    rng = np.random.default_rng(seed)
    linked = N - 1 if feature == "isolated" else N
    pairs = [(i, j) for i in range(linked) for j in range(i + 1, linked)]
    order = rng.permutation(len(pairs))
    chosen = [pairs[k] for k in order]
    if feature == "hub":
        hub = [p for p in chosen if p[0] == 0][:5]
        chosen = hub + [p for p in chosen if p not in hub]
    chosen = chosen[:S]
    assert len(chosen) == S, (N, S, feature)
    springs = [(j, i) if rng.random() < 0.5 else (i, j) for i, j in chosen]       # both endpoint orders
    perm = rng.permutation(S)
    springs = [springs[k] for k in perm]
    masses = [1.0] * N
    fixed = [False] * N
    if mass_class == "classes":
        a, b = springs[0]
        masses = [float(rng.choice(SMALL + (1.0,))) for _ in range(N)]
        masses[a] = masses[b] = float(rng.choice(SMALL))
        other = next(n for i, j in springs[1:] for n in (i, j) if n not in (a, b))
        masses[other] = 1.0
    elif mass_class == "general":
        masses = [float(rng.choice(SMALL + (1.0,))) for _ in range(N)]
        masses[int(rng.integers(N))] = float(rng.choice(GENERAL))
    elif mass_class == "ding":
        masses = [float(rng.choice(SMALL + (1.0,))) for _ in range(N)]
        masses[int(rng.integers(N))] = float(rng.choice(SMALL))
        fixed[int(rng.integers(N))] = True
    pts = [(masses[n], tuple(float(v) for v in rng.uniform(-150, 150, 3).round(2)), fixed[n]) for n in range(N)]
    mus = [(i, j, {"k": float(rng.choice([500, 1000, -700, 1500])), "dampk": float(rng.choice([5, 20, 15])),
                   "minl": float(rng.choice([0.1, 0.3])), "maxl": float(rng.choice([1.2, 1.5]))}) for i, j in springs[:M]]
    sks = [(i, j, dict({"k": float(rng.choice([500, 1000, 2000, -300])), "dampk": float(rng.choice([5, 20]))},
                       **({"x": round(float(rng.uniform(20, 90)), 1)} if rng.random() < 0.3 else {})))
           for i, j in springs[M:]]
    spec = {"points": pts, "muscles": mus, "skeletons": sks}
    check_class(spec, mass_class)
    return spec


def check_class(spec, mass_class):
    """The body has the mass class it names (the generator's own guarantees)."""
    masses = [m for m, _, _ in spec["points"]]
    fixed = [f for _, _, f in spec["points"]]
    springs = [(i, j) for i, j, _ in spec["muscles"] + spec["skeletons"]]
    want = {"unit": 0, "classes": 3, "general": 2, "ding": 2}[mass_class]
    assert mass_mode(masses, fixed) == want, (mass_class, masses, fixed)
    if mass_class == "classes":
        assert 1.0 in masses
        assert any(masses[i] == masses[j] != 1.0 for i, j in springs), "no spring between equal non-unit masses"
        assert any(1.0 in (masses[i], masses[j]) for i, j in springs), "no spring with a unit endpoint"
    if mass_class == "ding":
        assert sum(fixed) == 1 and mass_mode(masses, [False] * len(masses)) == 3, "MM 2 only because of the DingPoint"


def expected_instance(mass_class):
    """(Topo struct, MM) the compiled kernel of this mass class must have."""
    return {"unit": ("TopoJit", 0), "classes": ("TopoJitP", 3), "general": ("TopoJit", 2), "ding": ("TopoJit", 2)}[mass_class]


def creature(spec):
    from walker_gym_b200 import Creature, DingPoint, Muscle, Point, Skeleton
    Point.clear()
    pts = [DingPoint(m, list(p)) if f else Point(m, list(p), [0, 0, 0]) for m, p, f in spec["points"]]
    return Creature(pts, [Muscle(pts[i], pts[j], **kw) for i, j, kw in spec["muscles"]],
                    [Skeleton(pts[i], pts[j], **kw) for i, j, kw in spec["skeletons"]])


def obs_dim(spec, in3d):
    return 3 * (3 if in3d else 2) * len(spec["points"]) + len(spec["muscles"])


# ---- cases ---------------------------------------------------------------------------------------------------------
# (N, S, M, mass class, graph feature)
PACKED_BODIES = [
    (8, 16, 16, "classes", ""), (8, 16, 0, "unit", ""), (2, 1, 1, "unit", ""), (8, 16, 8, "ding", "hub"),
    (8, 14, 4, "general", "isolated"), (7, 12, 2, "classes", "hub"), (7, 9, 9, "unit", "isolated"), (6, 11, 5, "ding", ""),
    (6, 9, 3, "classes", "isolated"), (6, 15, 8, "general", "hub"), (5, 8, 4, "unit", ""), (5, 6, 6, "classes", ""),
    (5, 4, 1, "general", "isolated"), (4, 6, 2, "ding", ""), (4, 5, 0, "classes", ""), (4, 3, 3, "unit", "isolated"),
    (3, 3, 2, "general", ""), (3, 2, 1, "unit", ""), (2, 1, 0, "general", ""), (8, 10, 7, "classes", "isolated"),
    (7, 16, 16, "general", ""), (6, 7, 4, "unit", "hub"), (3, 2, 2, "ding", ""), (8, 12, 3, "ding", "isolated"),
]
# 9..16 masses; the last two: <= 8 masses on state_layout="soa"
SOA_BODIES = [
    (16, 32, 32, "classes", "hub"), (16, 24, 8, "unit", "isolated"), (16, 20, 0, "general", ""), (15, 30, 4, "ding", "hub"),
    (14, 18, 2, "classes", "isolated"), (13, 25, 13, "unit", ""), (12, 32, 8, "general", "hub"), (12, 16, 5, "classes", ""),
    (11, 14, 14, "classes", "isolated"), (11, 22, 2, "unit", "hub"), (10, 12, 4, "general", ""), (10, 27, 7, "classes", "hub"),
    (9, 9, 9, "unit", ""), (9, 11, 3, "ding", ""), (10, 13, 6, "unit", "isolated"), (14, 21, 11, "general", "isolated"),
    (6, 10, 4, "classes", "hub"), (3, 3, 2, "general", ""),
]
ENV_CHOICES = dict(g=[100, 9.8, 0, 250.5], dampk=[0, 0, 0.5, 3], ground_high=[0, -20, 35.5], ground_k=[1000, 0, 321],
                   ground_damp=[100, 0, 12.5], friction=[100, 0, 7], rand_sigma=[0.1, 1.0], time_step=[0.01, 0.003])


def _case(kind, k, body):
    """Everything one lockstep case needs, derived from its index."""
    N, S, M, mass_class, feature = body
    seed = (1000 if kind == "packed" else 2000) + k
    spec = random_spec(seed, N, S, M, mass_class, feature)
    rng = np.random.default_rng(seed)
    in3d = k % 3 != 2
    layout = "row" if k % 2 == 0 else "feature"
    if kind == "soa" and k == 0:
        in3d, layout = True, "row"               # (16, 32, 32): D = 176, a 90 KB observation tile
    env_kw = {name: float(rng.choice(v)) for name, v in ENV_CHOICES.items()}
    return dict(kind=kind, id=f"{kind}{k}-{N}-{S}-{M}-{mass_class}{'-' + feature if feature else ''}-{'3d' if in3d else '2d'}-{layout}",
                spec=spec, mass_class=mass_class, in3d=in3d, layout=layout, env_kw=env_kw,
                auto="template" if k % 4 in (0, 3) else "jitter", integrator="run2" if k % 5 == 1 else "run1",
                k_sub=1 if N >= 16 else 1 + k % 4, E=JIT_MIN_ENVS + int(rng.integers(1, 2 * PACKED_BLOCK)),
                state_layout="soa" if kind == "soa" and N <= 8 else "auto", seed=seed)


def _named_soa_cases():
    """Box-v0's graph with a DingPoint and the hat graph with a 2.5 mass, in the SoA layout: MM 2 on in-tree graphs."""
    box = spec_of("box_v0")
    box["points"] = [(m, p, n == 1) for n, (m, p, _) in enumerate(box["points"])]
    hat = spec_of("hat")
    hat["points"] = [(2.5 if n == 3 else m, p, f) for n, (m, p, f) in enumerate(hat["points"])]
    out = []
    for k, (name, spec, in3d, layout) in enumerate((("box_v0-ding", box, True, "feature"), ("hat-2.5", hat, False, "row"))):
        out.append(dict(kind="soa", id=f"soa-{name}", spec=spec, mass_class="general", in3d=in3d, layout=layout, env_kw={},
                        auto="template", integrator="run1", k_sub=2, E=JIT_MIN_ENVS + 5 + k, state_layout="soa",
                        seed=77 + k))
    return out


PACKED_CASES = [_case("packed", k, b) for k, b in enumerate(PACKED_BODIES)]
SOA_CASES = [_case("soa", k, b) for k, b in enumerate(SOA_BODIES)] + _named_soa_cases()
# T steps per launch: packed bodies of every mass class with tensor actions; the first three also with in-kernel sources
MULTI_CASES = [PACKED_CASES[k] for k in (0, 1, 4, 3, 11, 13, 20, 2)]
GEN_CASES = [PACKED_CASES[k] for k in (0, 2, 4)]


def make_env(case, E=None, **over):
    from walker_gym_b200 import BatchedPhysicsEnv
    kw = dict(in3d=case["in3d"], auto_reset=case["auto"], max_steps=5, k_sub=case["k_sub"], seed=case["seed"],
              obs_layout=case["layout"], integrator=case["integrator"], keep_old_a=True, track_info=True,
              track_contacts=True, initial_reset=False, state_layout=case["state_layout"], **case["env_kw"])
    kw.update(over)
    return BatchedPhysicsEnv(creature(case["spec"]), case["E"] if E is None else E, DEV, **kw)


def oracle_for(case, E, **over):
    kw = dict(in3d=case["in3d"], auto_reset={"jitter": 1, "template": 2}[case["auto"]], max_steps=5, k_sub=case["k_sub"],
              seed=case["seed"], integrator=1 if case["integrator"] == "run2" else 0, **case["env_kw"])
    kw.update(over)
    body = wo.make_body(case["spec"])
    return body, wo.make_params(**kw), wo.init_state(body, E)


# ---- which instance ran ----------------------------------------------------------------------------------------------
# template parameters of the three families (wg_kernels_packed.cuh, wg_kernels.cuh, wg_kernels_multi.cuh)
FAMILY_PARAMS = {"step_static_packed_kernel": ("topo", "in3d", "obs", "mm"),
                 "step_static_kernel": ("topo", "in3d", "obs", "ept", "mm"),
                 "step_multi_packed_kernel": ("topo", "in3d", "mm", "args", "gen")}


def _mangled_args(s, i):
    """Template arguments of an Itanium-mangled name from s[i] (just after 'I') to the matching 'E'."""
    args = []
    while s[i] != "E":
        if s[i] == "L":                                            # literal: L<type><value>E
            m = re.compile(r"L[a-z]+(n?\d+)E").match(s, i)
            args.append(int(m.group(1).replace("n", "-")))
            i = m.end()
        elif s[i] == "N" or s[i].isdigit():                        # (nested) name, possibly with template arguments
            nested, name = s[i] == "N", None
            i += nested
            while True:
                if s.startswith("S_", i):
                    i += 2
                elif s[i].isdigit():
                    m = re.compile(r"\d+").match(s, i)
                    name = s[m.end():m.end() + int(m.group())]
                    i = m.end() + int(m.group())
                elif s[i] == "I":
                    _, i = _mangled_args(s, i + 1)
                else:
                    break
                if not nested:
                    break
            i += nested                                            # the 'E' that closes N...E
            args.append(name)
        else:
            raise ValueError(f"cannot read the mangled name {s!r} at {i}")
    return args, i + 1


def _demangled_args(s, i):
    """Top-level template arguments of a demangled name from s[i] (just after '<')."""
    args, depth, cur = [], 0, ""
    while True:
        c = s[i]
        i += 1
        if c == "<":
            depth += 1
        elif c == ">" and depth == 0:
            args.append(cur)
            break
        elif c == ">":
            depth -= 1
        elif c == "," and depth == 0:
            args.append(cur)
            cur = ""
            continue
        cur += c
    out = []
    for a in args:
        a = re.sub(r"^\((?:int|bool|unsigned int)\)", "", a.strip())
        a = {"true": "1", "false": "0"}.get(a, a)
        out.append(int(a) if re.fullmatch(r"-?\d+", a) else a.split("::")[-1].split("<")[0])
    return out


def instance(name):
    """{"family": ..., "topo": ..., "in3d": 0/1, "mm": ..., ...} of a step kernel name as torch.profiler reports it."""
    for fam, params in FAMILY_PARAMS.items():
        m = re.search(fam + r"(<|I)", name)
        if m:
            args = _demangled_args(name, m.end()) if m.group(1) == "<" else _mangled_args(name, m.end())[0]
            return dict(zip(params, args), family=fam)
    return {"family": None, "name": name}


def check_instance(label, family, mass_class=None, *, topo=None, mm=None, in3d=None, gen=None, obs_rm=None):
    """The probe `label` launched `family` with the Topo struct and MM of `mass_class`.  Returns False when
    torch.profiler reports no kernel names (the caller skips after its oracle comparison)."""
    names = kernel_names()
    if names is None:
        return False
    name = names[label]
    got = instance(name)
    if mass_class is not None:
        topo, mm = expected_instance(mass_class)
    want = {"family": family, "topo": topo, "mm": mm, "in3d": None if in3d is None else int(in3d),
            "gen": None if gen is None else int(gen), "obs": obs_rm}
    for k, v in want.items():
        if v is not None:
            assert got.get(k) == v, f"{label}: {k} = {got.get(k)!r}, want {v!r} ({name})"
    return True


def _skip_unnamed():
    pytest.skip("torch.profiler reports no kernel names: the compiled instance was not identified")


# ---- probes: one launch per case, built before the shared profiler session -----------------------------------------
def _zero_actions(env):
    import torch
    return torch.zeros(env.num_envs, env.M, device=DEV)


def _step_probe(label, env, warm=True):
    """(label, run) of one env.step; a first step before the session compiles a SoA instance (wg_step compiles it on
    its first launch)."""
    a = _zero_actions(env)
    if warm:
        env.step(a)
    return (label, lambda: env.step(a))


class jit_include:
    """WG_JIT_INCLUDE set to `path` (None: unset) for the duration; include_dir() reads it at every compile."""

    def __init__(self, path):
        self.path = path

    def __enter__(self):
        self.old = os.environ.get("WG_JIT_INCLUDE")
        if self.path is None:
            os.environ.pop("WG_JIT_INCLUDE", None)
        else:
            os.environ["WG_JIT_INCLUDE"] = self.path
        return self

    def __exit__(self, *exc):
        if self.old is None:
            os.environ.pop("WG_JIT_INCLUDE", None)
        else:
            os.environ["WG_JIT_INCLUDE"] = self.old
        return False


@register_probes
def _jit_probes():
    import torch
    from walker_gym_b200 import CPGActions
    out = []
    for c in PACKED_CASES + SOA_CASES:
        out.append(_step_probe(c["id"], make_env(c)))
    for c in MULTI_CASES:
        env = make_env(c, obs_layout="row", state_layout="packed", keep_old_a=False, track_info=False, track_contacts=False)
        acts = torch.zeros(1, env.num_envs, env.M, device=DEV)
        out.append((f"multi {c['id']}", lambda env=env, acts=acts: env.step_many(acts)))
    for c in GEN_CASES:
        env = make_env(c, obs_layout="row", state_layout="packed", keep_old_a=False, track_info=False, track_contacts=False)
        src = CPGActions(amp=[1.0] * env.M, freq=[2.0] * env.M)
        out.append((f"gen {c['id']}", lambda env=env, src=src: env.step_many(src, n_steps=1)))
    for c in BOUNDARY_CASES:
        for E in (JIT_MIN_ENVS - 1, JIT_MIN_ENVS):
            out.append(_step_probe(f"boundary {c['id']} {E}", make_env(c, E=E, state_layout="auto")))
    for label, case in cache_cases():
        out.append(_step_probe(f"cache {label}", make_env(case)))
    with tempfile.TemporaryDirectory() as empty, jit_include(empty):
        for label, case in failure_cases():
            out.append(_step_probe(f"failure {label}", make_env(case)))
    c = GRID_CASE
    out.append(_step_probe("grid", make_env(c, E=grid_envs(), keep_old_a=False, track_info=False, track_contacts=False),
                           warm=False))
    return out


# ---- 1. the body set covers the edges the kernels specialise on -------------------------------------------------------
def test_body_set_covers_the_specialisation_edges():
    """Isolated masses, a mass of degree >= 5, M = 0 and M = S, M in {2, 4, 8} (the SoA kernel's vector action load) and
    other M, row-major observation widths on both sides of gcd(D, 32) <= 2 (bulk store / padded tile), every mass
    class, and each MM by 2-D / 3-D by both observation layouts -- in each of the packed and the SoA sets."""
    for cases in (PACKED_CASES, SOA_CASES):
        feats = set()
        for c in cases:
            sp = c["spec"]
            N, M = len(sp["points"]), len(sp["muscles"])
            S = M + len(sp["skeletons"])
            deg = np.bincount([n for i, j, _ in sp["muscles"] + sp["skeletons"] for n in (i, j)], minlength=N)
            feats.add(("instance", expected_instance(c["mass_class"])[1], c["in3d"], c["layout"]))
            feats |= {("isolated", bool((deg == 0).any())), ("hub", bool(deg.max() >= 5)), ("M0", M == 0), ("MS", M == S),
                      ("vec", M in (2, 4, 8)), ("novec", M not in (0, 2, 4, 8)), ("class", c["mass_class"]),
                      ("in3d", c["in3d"]), ("layout", c["layout"])}
            if c["layout"] == "row":
                feats.add(("bulk", bool(np.gcd(obs_dim(sp, c["in3d"]), 32) <= 2)))
        for want in (("isolated", True), ("hub", True), ("M0", True), ("MS", True), ("vec", True), ("novec", True),
                     ("bulk", True), ("bulk", False), ("in3d", True), ("in3d", False), ("layout", "row"),
                     ("layout", "feature"), ("class", "unit"), ("class", "classes"), ("class", "general"), ("class", "ding")):
            assert want in feats, (cases[0]["kind"], want)
        for mm in (0, 3, 2):
            for in3d in (True, False):
                for layout in ("row", "feature"):
                    assert ("instance", mm, in3d, layout) in feats, (cases[0]["kind"], mm, in3d, layout)
    big = SOA_CASES[0]
    assert big["in3d"] and big["layout"] == "row" and obs_dim(big["spec"], True) == 176
    assert 4 * PACKED_BLOCK * (176 | 1) > 48 * 1024           # the tile needs the opt-in shared memory attribute


# ---- 2. / 3. lockstep on the packed and the SoA instances --------------------------------------------------------------
def _lockstep_case(c):
    env = make_env(c)
    want_layout = "packed" if c["kind"] == "packed" else "soa"
    assert env.state_layout == want_layout and env.kernel_variant == 0, (env.state_layout, env.kernel_variant)
    body, prm, st = oracle_for(c, env.num_envs)
    run_lockstep(env, body, prm, st, 12, np.random.default_rng(c["seed"]), noise_reset=True)
    family = "step_static_packed_kernel" if c["kind"] == "packed" else "step_static_kernel"
    if not check_instance(c["id"], family, c["mass_class"], in3d=c["in3d"], obs_rm=int(c["layout"] == "row")):
        _skip_unnamed()


@pytest.mark.parametrize("case", PACKED_CASES, ids=[c["id"] for c in PACKED_CASES])
def test_packed_instances_match_oracle(case):
    """step_static_packed_kernel<TopoJit[P], ...> at 4096 + a ragged remainder envs (state_layout="auto"), random
    environment parameters, run1 / run2, 1..4 substeps, template and jitter auto-reset: 12 steps bit for bit."""
    _lockstep_case(case)


@pytest.mark.parametrize("case", SOA_CASES, ids=[c["id"] for c in SOA_CASES])
def test_soa_instances_match_oracle(case):
    """step_static_kernel<TopoJit[P], IN3D, OBS, 1, MM> at >= 4096 envs: MM 0 / 3 / 2 by both observation layouts in 2-D
    and 3-D, the (16, 32, 32) body whose row-major tile needs the opt-in shared memory, two <= 8-mass bodies on
    state_layout="soa", and Box-v0 / hat graphs with a DingPoint / a 2.5 mass."""
    _lockstep_case(case)


# ---- 4. T steps per launch ---------------------------------------------------------------------------------------------
def _multi_env(c):
    env = make_env(c, obs_layout="row", state_layout="packed", keep_old_a=False, track_info=False, track_contacts=False,
                   track_stats=True)
    body, prm, st = oracle_for(c, env.num_envs)
    rng = np.random.default_rng(c["seed"] + 1)
    import torch
    nz = (rng.standard_normal((3 * env.N, env.num_envs)) * 0.1).astype(np.float32)
    env.reset(noise=torch.from_numpy(nz).to(DEV), mode="jitter")
    wo.reset(body, prm, st, mode=1, noise=nz)
    return env, body, prm, st, rng


def _check_block(env, st, out, obs, what):
    assert gu.same(obs.cpu().numpy(), out["obs"]), f"obs after {what}"
    for k in ("pos", "vel", "mx", "steps"):
        assert gu.same(getattr(env, k).cpu().numpy(), st[k]), f"{k} after {what}"


@pytest.mark.parametrize("case", MULTI_CASES, ids=[c["id"] for c in MULTI_CASES])
def test_step_many_instances_match_oracle(case):
    """step_multi_packed_kernel<TopoJit[P], IN3D, MM, ..., GEN = false>: blocks of 1, 9 and 16 steps of tensor actions,
    every step's reward and done, the last observation and the state after each block."""
    import torch
    env, body, prm, st, rng = _multi_env(case)
    ep = (np.zeros(env.num_envs, np.float32), np.zeros((4, env.num_envs), np.float32))
    for T in (1, 9, 16):
        acts = rng.uniform(-1, 1, (T, env.num_envs, env.M)).astype(np.float32)
        first = env.step_count
        obs, rew, done = env.step_many(torch.from_numpy(acts).to(DEV))
        for t in range(T):
            prm.step_index = first + t
            out = wo.step(body, prm, st, acts[t], ep_ret=ep[0], fin_stats=ep[1])
            assert gu.same(rew[t].cpu().numpy(), out["reward"]), f"reward @ block {T} step {t}"
            assert gu.same(done[t].cpu().numpy(), out["done"].astype(bool)), f"done @ block {T} step {t}"
        _check_block(env, st, out, obs, f"block {T}")
    assert gu.same(env.fin_stats.cpu().numpy(), ep[1]) and ep[1][3].sum() > 0
    if not check_instance(f"multi {case['id']}", "step_multi_packed_kernel", case["mass_class"], in3d=case["in3d"], gen=False):
        _skip_unnamed()


@pytest.mark.parametrize("case", GEN_CASES, ids=[c["id"] for c in GEN_CASES])
def test_step_many_in_kernel_action_sources_match_oracle(case):
    """step_multi_packed_kernel<..., GEN = true>: ScriptedActions and CPGActions evaluated in the kernel from each env's
    own (desynchronised) step counter, blocks of 1, 9 and 16 steps, against the oracle fed the same generated actions."""
    from walker_gym_b200 import CPGActions, ScriptedActions
    import torch
    env, body, prm, st, rng = _multi_env(case)
    M = env.M
    steps0 = rng.integers(0, 6, env.num_envs).astype(np.int32)
    env.set_state(steps=torch.from_numpy(steps0))
    st["steps"][:] = steps0
    table = rng.uniform(-1, 1, (3, M)).round(2).tolist()
    cpg = CPGActions(amp=rng.uniform(0.2, 3.0, M).tolist(), freq=rng.uniform(0.3, 9.0, M).tolist(),
                     phase=rng.uniform(-3, 3, M).tolist())
    sources = [(ScriptedActions(table, hold=2), ScriptedActions(table, hold=2).describe()),
               (cpg, cpg.describe(float(env.params.dt)))]
    for k, T in enumerate((1, 9, 16, 16, 9, 1)):
        src, desc = sources[k % 2]
        first = env.step_count
        obs, rew, done = env.step_many(src, n_steps=T)
        for t in range(T):
            prm.step_index = first + t
            out = wo.step(body, prm, st, wo.gen_actions(desc, st["steps"], M))
            assert gu.same(rew[t].cpu().numpy(), out["reward"]), f"reward @ block {k} step {t}"
            assert gu.same(done[t].cpu().numpy(), out["done"].astype(bool)), f"done @ block {k} step {t}"
        _check_block(env, st, out, obs, f"block {k} ({T} steps)")
    if not check_instance(f"gen {case['id']}", "step_multi_packed_kernel", case["mass_class"], in3d=case["in3d"], gen=True):
        _skip_unnamed()


# ---- 6. dispatch boundary ----------------------------------------------------------------------------------------------
BOUNDARY_CASES = [dict(PACKED_CASES[7], id="boundary-packed", auto="jitter", layout="row"),
                  dict(SOA_CASES[3], id="boundary-soa", auto="jitter", layout="row")]


@pytest.mark.parametrize("case", BOUNDARY_CASES, ids=[c["id"] for c in BOUNDARY_CASES])
def test_dispatch_boundary_4095_vs_4096(case):
    """The same body at 4095 envs (run-time-topology kernel) and 4096 envs (the compiled kernel) with jitter resets
    (Philox keyed by the global env id): the first 4095 envs are bit-identical for 12 steps, and the two sizes ran
    different kernels."""
    import torch
    envs = [make_env(case, E=E, state_layout="auto", max_steps=4) for E in (JIT_MIN_ENVS - 1, JIT_MIN_ENVS)]
    n = JIT_MIN_ENVS - 1
    rng = np.random.default_rng(case["seed"])
    for e in envs:
        e.reset(mode="jitter")
    ended = 0
    for t in range(12):
        act = torch.from_numpy(rng.uniform(-1, 1, (JIT_MIN_ENVS, envs[0].M)).astype(np.float32)).to(DEV)
        outs = [e.step(act[:e.num_envs].contiguous())[:3] for e in envs]
        for k, (a, b) in enumerate(zip(*outs)):
            assert gu.same(a[:n].cpu().numpy(), b[:n].cpu().numpy()), ("obs", "reward", "done")[k] + f" @ step {t}"
        ended += int(outs[1][2][:n].sum())
        for k in ("pos", "vel", "mx", "steps", "old_a"):
            assert gu.same(getattr(envs[0], k)[..., :n].cpu().numpy(), getattr(envs[1], k)[..., :n].cpu().numpy()), (k, t)
    assert ended > 0, "no episode ended: the jitter resets were not exercised"
    names = kernel_names()
    if names is None:
        _skip_unnamed()
    small = instance(names[f"boundary {case['id']} {n}"])
    assert small["family"] is None and "step_generic_kernel" in small["name"], small
    fam = "step_static_packed_kernel" if case is BOUNDARY_CASES[0] else "step_static_kernel"
    check_instance(f"boundary {case['id']} {JIT_MIN_ENVS}", fam, case["mass_class"])


# ---- 7. the compiled-kernel cache ----------------------------------------------------------------------------------
# one 4-mass graph (no in-tree body has it): muscles (0, 2), (3, 1); bones (0, 1), (1, 2), (2, 3), (3, 0)
CACHE_GRAPH = [(0, 2), (3, 1), (0, 1), (1, 2), (2, 3), (3, 0)]


def cache_spec(masses, ding=None, variant=0):
    """The cache graph with these masses; variant 1 changes every value that is a kernel argument (spring constants,
    damping, rest lengths, muscle limits, template positions)."""
    pos = [(-40, 60, 5), (45, 70, -8), (0, 10, 0), (10, 110, 3)]
    if variant:
        pos = [(x * 1.25 + 3, y * 0.8 + 6, z - 2) for x, y, z in pos]
    kw_m = [{"k": 800, "dampk": 15, "minl": 0.3, "maxl": 1.2}, {"k": -300, "dampk": 25}]
    kw_s = [{"k": 500}, {"k": 2000, "dampk": 5}, {"x": 61.5}, {}]
    if variant:
        kw_m = [{"k": 1300, "dampk": 7, "minl": 0.2, "maxl": 1.4}, {"k": 650, "dampk": 12, "minl": 0.5}]
        kw_s = [{"k": 900, "dampk": 30}, {"k": -150}, {"x": 40.25}, {"k": 3000, "x": 75.0}]
    return {"points": [(float(m), p, n == ding) for n, (m, p) in enumerate(zip(masses, pos))],
            "muscles": [(i, j, kw) for (i, j), kw in zip(CACHE_GRAPH[:2], kw_m)],
            "skeletons": [(i, j, kw) for (i, j), kw in zip(CACHE_GRAPH[2:], kw_s)]}


def _cache_case(label, spec, mass_class, in3d=True, layout="row", seed=5):
    check_class(spec, mass_class)
    return dict(kind="packed", id=f"cache-{label}", spec=spec, mass_class=mass_class, in3d=in3d, layout=layout, env_kw={},
                auto="template", integrator="run1", k_sub=2, E=JIT_MIN_ENVS + 3, state_layout="auto", seed=seed)


def cache_cases():
    """[(label, case)] in compile order: (2, 2, 1, 3) before (2, 3, 1, 3) and (3, 2, 1, 3), 3-D before 2-D."""
    return [
        ("a-2213", _cache_case("a-2213", cache_spec((2, 2, 1, 3)), "classes")),
        ("a-5517", _cache_case("a-5517", cache_spec((5, 5, 1, 7), variant=1), "classes", seed=6)),
        ("b-2313", _cache_case("b-2313", cache_spec((2, 3, 1, 3)), "classes")),
        ("b-3213", _cache_case("b-3213", cache_spec((3, 2, 1, 3)), "classes")),
        ("c-ding0", _cache_case("c-ding0", cache_spec((3, 5, 1, 3), ding=0), "ding")),
        ("c-ding3", _cache_case("c-ding3", cache_spec((3, 5, 1, 3), ding=3), "ding")),
        ("d-3d-row", _cache_case("d-3d-row", cache_spec((1, 1, 1, 1)), "unit")),
        ("d-3d-feature", _cache_case("d-3d-feature", cache_spec((1, 1, 1, 1)), "unit", layout="feature")),
        ("d-2d-row", _cache_case("d-2d-row", cache_spec((1, 1, 1, 1)), "unit", in3d=False)),
        ("d-2d-feature", _cache_case("d-2d-feature", cache_spec((1, 1, 1, 1)), "unit", in3d=False, layout="feature")),
    ]


@pytest.mark.parametrize("group", ["a", "b", "c", "d"])
def test_compiled_kernel_cache(group):
    """(a) same graph and class pattern, different values: one kernel, values as arguments; (b) class patterns
    (2, 2, 1, 3), (2, 3, 1, 3), (3, 2, 1, 3): three kernels; (c) a DingPoint at different indices: one MM 2 kernel;
    (d) the graph in 3-D and 2-D, row- and feature-major.  The envs of a group are stepped interleaved, each against its
    own oracle, after all of them were built (so each took its kernel from the cache as it stood)."""
    import torch
    cases = [(label, c) for label, c in cache_cases() if label.startswith(group)]
    runs = []
    for label, c in cases:
        env = make_env(c)
        assert env.state_layout == "packed"
        body, prm, st = oracle_for(c, env.num_envs)
        runs.append((label, c, env, body, prm, st, np.random.default_rng(c["seed"] + len(runs))))
    for t in range(10):
        for label, c, env, body, prm, st, rng in runs:
            act = rng.uniform(-1, 1, (env.num_envs, env.M)).astype(np.float32)
            prm.step_index = env.step_count
            obs, rew, done, _ = env.step(torch.from_numpy(act).to(DEV))
            out = wo.step(body, prm, st, act)
            o = obs.cpu().numpy()
            assert gu.same(o if c["layout"] == "row" else o.T, out["obs"]), f"{label}: obs @ step {t}"
            assert gu.same(rew.cpu().numpy(), out["reward"]), f"{label}: reward @ step {t}"
            assert gu.same(done.cpu().numpy(), out["done"].astype(bool)), f"{label}: done @ step {t}"
            for k in ("pos", "vel", "mx", "steps"):
                assert gu.same(getattr(env, k).cpu().numpy(), st[k]), f"{label}: {k} @ step {t}"
    if group == "c":         # the DingPoint stays where it is
        for label, c, env, body, prm, st, rng in runs:
            n = next(k for k, (_, _, f) in enumerate(c["spec"]["points"]) if f)
            tmpl = np.array(c["spec"]["points"][n][1], np.float32)
            assert (env.pos[3 * n:3 * n + 3].cpu().numpy() == tmpl[:, None]).all(), label
    for label, c, *_ in runs:
        if not check_instance(f"cache {label}", "step_static_packed_kernel", c["mass_class"], in3d=c["in3d"],
                              obs_rm=int(c["layout"] == "row")):
            _skip_unnamed()


# ---- 8. compile failure --------------------------------------------------------------------------------------------
def failure_cases():
    """Graphs no other test compiles (a failed compilation is cached per key): a packed-eligible body and a 12-mass one."""
    small = random_spec(9101, 5, 7, 3, "classes", "")
    big = random_spec(9102, 12, 17, 4, "unit", "isolated")
    return [("packed-eligible", dict(kind="packed", id="failure-packed", spec=small, mass_class="classes", in3d=True,
                                     layout="row", env_kw={}, auto="template", integrator="run1", k_sub=1,
                                     E=JIT_MIN_ENVS + 11, state_layout="auto", seed=9101)),
            ("soa", dict(kind="soa", id="failure-soa", spec=big, mass_class="unit", in3d=False, layout="feature", env_kw={},
                         auto="jitter", integrator="run1", k_sub=2, E=JIT_MIN_ENVS + 7, state_layout="auto", seed=9102))]


def test_compile_failure_falls_back_or_raises():
    """With WG_JIT_INCLUDE pointing at an empty directory the compiler cannot find the kernel headers:
    state_layout="auto" keeps a packed-eligible body on the SoA layout and the run-time-topology kernel,
    state_layout="packed" raises with the compiler's message, and a 12-mass body at >= 4096 envs runs the
    run-time-topology kernel -- each with the oracle's bits."""
    (_, small), (_, big) = failure_cases()
    with tempfile.TemporaryDirectory() as empty, jit_include(empty):
        for c in (small, big):          # wg_step tries (and fails) to compile the SoA kernel at the first step
            env = make_env(c)
            env.step(_zero_actions(env))
        with pytest.raises(Exception, match=r"(?s)run-time specialisation failed: nvrtc: .*wg_kernels_packed\.cuh"):
            make_env(small, state_layout="packed")
    for c in (small, big):              # the failures stay cached per key after the include directory is back
        env = make_env(c)
        assert env.state_layout == "soa", c["id"]
        body, prm, st = oracle_for(c, env.num_envs)
        run_lockstep(env, body, prm, st, 10, np.random.default_rng(c["seed"]), noise_reset=True)
    names = kernel_names()
    if names is None:
        _skip_unnamed()
    for label, _ in failure_cases():
        name = names[f"failure {label}"]
        assert "step_generic_kernel" in name and instance(name)["family"] is None, (label, name)


# ---- 9. one CTA past the first full wave ---------------------------------------------------------------------------
GRID_CASE = dict(PACKED_CASES[0], id="grid", layout="row", in3d=True, auto="template", k_sub=1, env_kw={})


def grid_envs():
    return 3 * n_sms() * PACKED_BLOCK + 1


def test_eight_mass_body_one_cta_past_the_first_wave():
    """The (8, 16, 16) packed body (3 CTAs of 128 envs per SM for its register count) at 3 * SMs * 128 + 1 envs:
    the head, a slice in the middle of the first wave, and the tail (the end of the first wave and the one CTA past
    it) against the oracle for 20 steps with template auto-resets."""
    import torch
    c = GRID_CASE
    E = grid_envs()
    env = make_env(c, E=E, keep_old_a=False, track_info=False, track_contacts=False, initial_reset=True, max_steps=7,
                   track_stats=True)
    assert env.state_layout == "packed"
    n = 4096
    slices = [(0, n), (E // 2 - n // 2, E // 2 + n // 2), (E - n, E)]
    lock = SliceLockstep(env, slices, max_steps=7, seed=c["seed"], spec=c["spec"], k_sub=1, in3d=True,
                         rand_sigma=0.1, block=PACKED_BLOCK)
    g = torch.Generator(device=DEV).manual_seed(3)
    for t in range(20):
        act = torch.rand(E, env.M, device=DEV, generator=g) * 2 - 1
        obs, rew, done, _ = env.step(act)
        lock.record(act, obs, rew, done)
    lock.flush()
    lock.check_state()
    assert lock.done_count > 0
    if not check_instance("grid", "step_static_packed_kernel", c["mass_class"], in3d=True, obs_rm=1):
        _skip_unnamed()
