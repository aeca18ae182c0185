/*
 * walker_gym_b200.h -- C ABI of libwalkergym_b200.so
 *
 * The drop-in boundary for walker-gym's physics step on B200 (sm_100a).
 * The reference has no FFI: its boundary is the Python class surface of
 * gym/optimized_env.py (PhysicsEnv.reset/step, make_env), which the host
 * package walker_gym_b200 keeps; these entry points are what that surface
 * binds underneath (ctypes, see INTEGRATION.md).  Plain pointers and sizes,
 * no torch types, nothing owned by the library: every buffer is caller-owned
 * device memory, every call is asynchronous on the caller's stream, the
 * library keeps no global state except a thread-local error string.
 *
 * Data layout (device memory, float32 unless noted), E = n_env:
 *   pos, vel, old_a : SoA  [(n*3 + c) * E + e]      n = mass, c = x/y/z
 *   mx              : SoA  [m * E + e]              m = muscle (current length Muscle.x)
 *   steps           : int32 [E]
 *   action          : row-major [E][act_dim] (act_layout 0) or feature-major [act_dim][E] (act_layout 1)
 *   obs             : row-major [E][D] (obs_layout 0) or feature-major [D][E] (obs_layout 1)
 *   reward [E], done uint8 [E], contact_* uint32 bitmask [E] (bit n = mass n)
 *   energy [E], centroid [3][E], ep_ret [E], fin_stats [4][E], nf_stats [2][E]
 *   noise           : SoA like pos; already scaled by sigma
 * D = 3 * (in3d ? 3 : 2) * n_mass + n_muscle   (Creature.getstat, gym/optimized_walker.py:129-162)
 *
 * Every function returns 0 on success or a negative wg_status; it never
 * throws and never synchronises the device.
 */
#ifndef WALKER_GYM_B200_H
#define WALKER_GYM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WG_ABI_VERSION 4
#define WG_MAX_MASS 32
#define WG_MAX_SPRING 96

typedef enum wg_status {
    WG_OK = 0,
    WG_ERR_BAD_ARG = -1,      /* null/ill-sized argument, N or S over the limits */
    WG_ERR_UNSUPPORTED = -2,  /* e.g. no CUDA device / wrong architecture */
    WG_ERR_CUDA = -3          /* a CUDA runtime call failed; see wg_last_error_string */
} wg_status;

/*
 * One morphology shared by all envs.  Replaces the object graph
 * Creature(phys, muscles, skeletons) of gym/optimized_walker.py:108-115 with
 * Point (gym/optimized_engine.py:42-68), Muscle (:7-21) and Skeleton (:69-82).
 * Springs [0, n_muscle) are the muscles in list order, [n_muscle, n_spring)
 * the skeletons: the order Creature.run applies them (:117-127).
 * Scalars are stored as the value NumPy would use at the point of use
 * (float32 for "weak" python scalars multiplied into float32 arrays).
 */
typedef struct wg_topology {
    int32_t n_mass, n_spring, n_muscle, reserved;
    double  mass[WG_MAX_MASS];          /* Point.m */
    uint8_t fixed[WG_MAX_MASS];         /* 1 = DingPoint: forced() ignored (gym/optimized_engine.py:414-416) */
    float   tmpl_pos[WG_MAX_MASS * 3];  /* creation-time positions, [n*3+c] */
    int32_t si[WG_MAX_SPRING], sj[WG_MAX_SPRING];   /* p1, p2 */
    float   sk[WG_MAX_SPRING];          /* k      */
    float   sdamp[WG_MAX_SPRING];       /* dampk  */
    float   srest[WG_MAX_SPRING];       /* Skeleton.x / Muscle.originx */
    float   mlo[WG_MAX_SPRING];         /* originx * minl   (Muscle.regulation, :27-30) */
    float   mhi[WG_MAX_SPRING];         /* originx * maxl */
    uint8_t sstring[WG_MAX_SPRING];     /* 1 = rope-type spring: no elastic force while shorter than its rest length
                                           (`if dx < 0 and string: f_size = 0`, Point.resilience,
                                           gym/optimized_engine.py:134-138, applied to Muscle.run / Skeleton.run; the
                                           damping term is unchanged).  The rule holds for float32 and float64
                                           (wg_step_x64) actions alike; with float64 actions a muscle's dx is the
                                           double one.  Bodies with such springs step through the run-time-topology
                                           kernels. */
} wg_topology;

/*
 * Environment constants.  Replaces the constructor arguments and attributes
 * of PhysicsEnv (gym/optimized_env.py:15-44).
 */
typedef struct wg_params {
    double   g;             /* gravity, applied as a force: a_y += (-g)/m in float64 (:148) */
    float    dampk;         /* global velocity damping (:151,180-182) */
    float    ground;        /* ground_high */
    float    fall_thresh;   /* float32(ground_high - 50): done when mean(y) < this (:218) */
    float    ground_k, ground_damp, friction;   /* contact spring, damper, friction (:162-172) */
    float    dt;            /* time_step (:42) */
    float    dt2;           /* float32(time_step ** 2): only used by integrator 1 */
    float    sigma;         /* rand_sigma of the in-kernel reset jitter (:59-62) */
    int32_t  in3d;
    int32_t  max_steps;     /* :44 */
    int32_t  k_sub;         /* physics substeps per env step (>= 1) */
    int32_t  auto_reset;    /* 0 none; 1 jitter-only = PhysicsEnv.reset (:53-68); 2 template = make_env again */
    int32_t  integrator;    /* 0 = Point.run1, semi-implicit Euler (gym/optimized_engine.py:258-272, what PhysicsEnv uses);
                               1 = Point.run2 (:274-288): pos += v*t + 0.5*a*t^2, then v += a*t */
    uint32_t seed_lo, seed_hi;   /* Philox key of the in-kernel jitter */
    uint32_t step_index;    /* global step number (Philox counter word), set by the caller each step */
    uint32_t env_offset;    /* global id of env 0 of this shard (multi-GPU invariance) */
    int32_t  end_nonfinite; /* 0 = the reference's done rule; 1 = also done on a step whose reward is not finite
                               (!(|reward| <= FLT_MAX)): an env whose state overflowed to inf / NaN ends its episode and,
                               with auto_reset 2, restarts from the template.  Needs auto_reset 0 or 2 (a jitter reset
                               keeps the overflowed positions) */
    int32_t  reserved1;
} wg_params;

/*
 * In-kernel action source for wg_step_multi: the action of every step of the launch is computed on chip from the
 * env's own step counter (Point-in-episode time), so an n_steps launch reads no action memory at all.
 *   mode 1, table: the scripted phase-table gait sketched at gym/walker.py:356-366 (`tt = (t // 50) % 3;
 *           c.act([...row tt...])`): action = table[((steps / hold) % n_rows)][muscle], steps = the env's step
 *           counter BEFORE the step (0 for the first step of an episode; an auto-reset restarts the gait);
 *   mode 2, cpg:   the sinusoidal pattern generator of the package lineage's Muscle.act
 *           (gym/optimized_walker/walker.py:56-90: `t += dt; sin(2 pi freq t + phase)`) as an action source:
 *           action = amp[m] * sin(2 pi * ((phase0[m] + (steps + 1) * dphase[m]) mod 2^24) / 2^24), the phase kept
 *           as a 24-bit fraction of a turn (dphase = round(freq * time_step * 2^24)) and the sine evaluated by the
 *           library's deterministic polynomial (IEEE +, *, fma only), so the oracle reproduces its bits.
 * Creature.act applies the generated value exactly like an action read from memory (add, then regulation()).
 */
#define WG_GEN_MAX_ROWS 32
#define WG_GEN_MAX_MUSCLE 16
typedef struct wg_action_gen {
    int32_t  mode;          /* 0 = off (buf->action is used), 1 = table, 2 = cpg */
    int32_t  n_rows;        /* table: 1..WG_GEN_MAX_ROWS */
    int32_t  hold;          /* table: env-steps each row is held (>= 1) */
    int32_t  reserved;
    float    table[WG_GEN_MAX_ROWS * WG_GEN_MAX_MUSCLE];   /* [row * WG_GEN_MAX_MUSCLE + muscle] */
    float    amp[WG_GEN_MAX_MUSCLE];
    uint32_t phase0[WG_GEN_MAX_MUSCLE];   /* 24-bit fractions of a turn */
    uint32_t dphase[WG_GEN_MAX_MUSCLE];
} wg_action_gen;

/* Caller-owned device buffers of one shard.  Optional ones may be NULL. */
typedef struct wg_buffers {
    float*       pos;           /* in/out */
    float*       vel;           /* in/out */
    float*       old_a;         /* out, optional: Point.old_a of the last substep */
    float*       mx;            /* in/out */
    int32_t*     steps;         /* in/out */
    const float* action;        /* in */
    int32_t      act_dim;       /* columns of action; only min(act_dim, n_muscle) are used (Creature.act :164-167) */
    int32_t      obs_layout;    /* 0 = [E][D] row-major, 1 = [D][E] */
    int32_t      act_layout;    /* 0 = [E][act_dim] row-major, 1 = [act_dim][E] (what a feature-major policy emits) */
    int32_t      reserved0;
    float*       obs;           /* out, optional */
    float*       reward;        /* out, optional */
    uint8_t*     done;          /* out, optional */
    uint32_t*    contact_pre;   /* out, optional: force-phase contact of the last substep (:154) */
    uint32_t*    contact_post;  /* out, optional: reward-phase contact (:200) */
    float*       energy;        /* out, optional: _calculate_energy (:240-248) */
    float*       centroid;      /* out, optional: info['centroid_position'] (:235) */
    float*       ep_ret;        /* in/out, optional: running episode return */
    float*       fin_stats;     /* in/out, optional: per-env sums over finished episodes:
                                   [0] return, [1] return^2, [2] length, [3] count */
    const float* noise;         /* in, optional: jitter used by auto-reset / wg_reset instead of Philox */
    const uint32_t* step_counter; /* in, optional: device scalar added to prm->step_index; lets a CUDA graph
                                   that replays wg_step advance the Philox counter without new parameters */
    float*       state_packed;  /* in/out, optional: the packed state layout (see below).  When set, pos / vel /
                                   mx / steps / ep_ret are ignored (they live inside it) */
    /* x64 mode only (wg_step_x64): */
    double*      mx64;          /* in/out: muscle lengths as doubles, [m * E + e] */
    uint8_t*     mx_weak;       /* in/out: 1 = the length is float32-typed (a fresh or just-clamped muscle), [m * E + e] */
    const double* action64;     /* in: float64 actions, laid out like action */
    /* wg_step_multi only: HOST pointer to an in-kernel action source (copied into the kernel parameters at launch);
     * when set with mode != 0, action must be NULL and n_action_steps is ignored */
    const wg_action_gen* action_gen;
    float*       nf_stats;      /* in/out, optional: per-env sums over finished episodes whose return is not finite:
                                   [0] count, [1] length.  Such an episode then goes here instead of into fin_stats.
                                   Needs fin_stats and the running return (ep_ret, or state_packed) */
} wg_buffers;

/*
 * x64 mode: PhysicsEnv.step driven with float64 ndarray actions, which is what the reference's own demo loop does
 * (gym/performance_demo.py:241-262: np.random.uniform).  `self.x += a` (gym/optimized_walker.py:33) then turns
 * Muscle.x into an np.float64 and NumPy evaluates the muscle's spring term in double (dx, f_size, force, force / m
 * added to the float32 accumulator in double); a muscle that regulation() clamped (:27-30) holds the limit object
 * and is float32-typed until the next action.  These are the double-typed objects of that path, per spring:
 */
typedef struct wg_x64 {
    double sk_d[WG_MAX_SPRING];     /* float(k) */
    double x0_d[WG_MAX_SPRING];     /* originx: np.float32 distance, or the python float the user passed */
    double mlo_d[WG_MAX_SPRING];    /* originx * minl as regulation() forms it (np.float32 or python float) */
    double mhi_d[WG_MAX_SPRING];    /* originx * maxl */
} wg_x64;

/*
 * Run-time specialisation.  A body with at most 8 masses and 16 springs that has no ahead-of-time kernel gets the
 * packed-state step kernel compiled for ITS spring graph and masses class with NVRTC (about one second, once per
 * process and (body, in3d, obs_layout) combination), so user-built creatures run the same register-resident code as
 * the in-tree bodies.  wg_step compiles on first use; wg_jit_prepare does it eagerly and reports a compiler or
 * loader failure (then use the SoA layout: the run-time-topology kernel needs no compiler).  With the SoA layout,
 * bodies of up to 16 masses and 32 springs stepped in batches of >= 4096 envs get the one-thread SoA kernel compiled
 * the same way (2-14 s once), and
 * fall back to the run-time-topology kernel silently if the compiler is missing.  Results are identical.
 */
int wg_jit_prepare(const wg_topology* topo, int in3d, int obs_layout);

/* 1 if this body has an ahead-of-time packed-state kernel (Balance / Box topologies and the smaller walker.py bodies: box, test,
 * intrian, hat, humanb, box4, leg2, leg -- unit / power-of-two / small-integer masses, no DingPoints), 2 if it can get
 * one at run time (WG_TUNE_JIT on, NVRTC present, <= 8 masses, <= 16 springs), else 0. */
int wg_packed_available(const wg_topology* topo);

/*
 * Packed state layout (only for bodies with wg_packed_available() == 1).
 * The R = 6*n_mass + n_muscle + 2 per-env scalars k -- pos rows 0..3N-1 (n*3+c), vel rows 3N..6N-1, muscle
 * lengths 6N..6N+M-1, steps (int32 bits) 6N+M, ep_ret 6N+M+1 -- are stored as [tile][k/4][128 envs][4]:
 *     index(e, k) = ((e >> 7) * R4 + (k >> 2)) * 512 + (e & 127) * 4 + (k & 3),   R4 = ceil(R / 4)
 * so a thread moves four scalars of its env with one 16-byte access, a warp moves 512 contiguous bytes, and a
 * tile of 128 envs is one contiguous R4 * 2 KiB block.  The buffer holds ceil(E / 128) * R4 * 512 floats.
 */
int64_t wg_packed_state_floats(const wg_topology* topo, int64_t n_env);

int         wg_abi_version(void);
const char* wg_last_error_string(void);

/* Observation length for this morphology (len(PhysicsEnv._get_observation()), :184-187). */
int wg_obs_dim(const wg_topology* topo, int in3d);

/* Which kernel wg_step will launch: 0 = generic (runtime topology), >0 = id of a
 * register-resident specialisation.  For tests and logs; not needed to call wg_step. */
int wg_kernel_variant(const wg_topology* topo);
/* Force the generic kernel (1) or restore automatic dispatch (0); returns the old value. */
int wg_force_generic(int on);
/* Kernel-selection knobs for experiments and tests; results never depend on them.
 *   WG_TUNE_TMA (0): 1 = use the persistent TMA-pipelined variant of the specialised SoA kernels when the
 *                    buffers allow it (E % 4 == 0, 16-byte aligned); default 0 (measured slower).
 *   WG_TUNE_PART (1): lanes per env of the mass-partitioned kernels:
 *                    -1 = automatic (default: wg_step uses 4 lanes for bodies of >= 16 masses stepped with >= 2
 *                    substeps, wg_pkg_update_physics 2 / 4 lanes from 12 / 18 points), 0 = never, 2 / 4 / 8 = forced.
 *   WG_TUNE_L2_PREFETCH (2): distance, in thread blocks, of the L2 prefetch issued by the packed-state and
 *                    mass-partitioned kernels (0 = off; default 256).
 * Returns the previous value, or WG_ERR_BAD_ARG. */
#define WG_TUNE_TMA 0
#define WG_TUNE_PART 1
#define WG_TUNE_L2_PREFETCH 2
#define WG_TUNE_JIT 3             /* 1 (default) = bodies without an ahead-of-time kernel get one compiled at run time */
#define WG_TUNE_POLICY_TC 4       /* wg_policy_act: 2 (default) = the warp-specialised tcgen05 / tensor-memory pipeline, 1 = the monolithic
                                   tcgen05 kernel, 0 = the mma.sync kernel (env WG_POLICY_TC) */
#define WG_TUNE_PDL 5             /* 1 (default) = the packed-state step kernel is launched with programmatic stream serialisation
                                   (cudaLaunchAttributeProgrammaticStreamSerialization): its CTAs may be scheduled while the
                                   previous kernel of the stream drains and wait (griddepcontrol.wait) before their first global
                                   access, so back-to-back steps lose no launch gap; 0 = plain launches (env WG_PDL) */
int wg_set_tuning(int key, int value);

/*
 * PhysicsEnv.step for n_env environments (gym/optimized_env.py:70-92):
 * Creature.act -> k_sub x _run_physics -> steps += 1 -> reward, done, info ->
 * optional auto-reset of done envs -> observation.  One kernel launch.
 */
int wg_step(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
            int64_t n_env, void* cuda_stream);

/*
 * n_steps consecutive PhysicsEnv.step calls (gym/optimized_env.py:70-92) in ONE launch, for callers that know
 * the next n_steps actions up front (scripted gaits / open-loop controllers like the phase table sketched at gym/walker.py:356-366,
 * action repeat, replay of a recorded action sequence).  The state stays in registers between the steps, so an
 * env-step costs its arithmetic plus 4 * n_muscle + 5 bytes of HBM traffic instead of the whole state.
 * Bit-identical to n_steps wg_step calls with prm->step_index advanced by one per call (an auto-reset at step t
 * of the block draws its jitter with Philox index step_index + t).
 *   buf->state_packed  required (packed layout); every body with an ahead-of-time packed kernel (the Balance / Box
 *                      graphs and walker.py's box, test, intrian, hat, humanb, box4, leg2, leg) and every body whose
 *                      packed kernel is compiled at run time (wg_packed_available() != 0), i.e. whatever wg_step
 *                      accepts on the packed layout
 *   buf->action        [n_action_steps][n_env][n_muscle] float32 (act_layout 0, act_dim == n_muscle), or null;
 *                      n_action_steps == n_steps: one action block per step; n_action_steps == 1: the same block is
 *                      applied at every step (action repeat / frame skip: Creature.act runs n_steps times with it)
 *   buf->action_gen    optional in-kernel action source (scripted table / CPG, see wg_action_gen) instead of buf->action:
 *                      the launch then reads no action memory at all
 *   buf->reward        [n_steps][n_env] float32, optional;  buf->done  [n_steps][n_env] uint8, optional
 *   buf->obs           [n_env][obs_dim] row-major observation after the LAST step (obs_layout 0), optional
 *   buf->old_a / contact_pre / contact_post / energy / centroid must be null.
 */
int wg_step_multi(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
                  int64_t n_env, int32_t n_steps, int32_t n_action_steps, void* cuda_stream);

/*
 * wg_step in x64 mode:buf->mx64 / mx_weak / action64 must be set (action is ignored; mx still receives the float32
 * view of the lengths, which is what the float32 observation carries).  Bit-identical to the reference driven
 * with float64 actions.  Runs the run-time-topology kernel (a compatibility path, not the throughput path).
 * wg_reset does not touch mx64 / mx_weak: after a template reset the caller sets them to x0_d / 1.
 * Returns WG_ERR_UNSUPPORTED for a body whose per-block tile (11 * n_mass + n_muscle + 3 rows of 129 floats) exceeds
 * the device's shared memory per block (on a B200 with 32 masses: 93 or more muscles with row-major observations,
 * 96 with feature-major ones); the check also runs when n_env == 0, so a call with no envs tells whether the body
 * can step.
 */
int wg_step_x64(const wg_topology* topo, const wg_x64* x64, const wg_params* prm, const wg_buffers* buf,
                int64_t n_env, void* cuda_stream);

/*
 * Creature.getstat (gym/optimized_walker.py:129-162) with its options, for every env: per point
 * [(pos - mid)[:d] * pk (midform) or pos[:d] * pk, v[:d] * vk, old_a[:d] * ak], then the centroid `mid` (3 values,
 * zeros without midform) if conmid, then Muscle.x * mk.  d = in3d ? 3 : 2; out has 3*d*n_mass + n_muscle (+3) entries
 * per env, row-major [E][D'] (out_layout 0) or [D'][E] (1).  The state is read from buf (SoA or packed); Point.old_a
 * from buf->old_a or, when that is null, from the acceleration entries of obs_default -- the observation the step
 * kernel wrote (layout buf->obs_layout, dimensionality env_in3d).  The python scalars pk / vk / ak / mk multiply
 * float32 arrays, i.e. they act as float32 (NEP 50).
 */
int wg_getstat(const wg_topology* topo, const wg_buffers* buf, const float* obs_default, int32_t env_in3d,
               int32_t in3d, float pk, float vk, float ak, float mk, int32_t midform, int32_t conmid,
               float* out, int32_t out_layout, int64_t n_env, void* cuda_stream);

/*
 * PhysicsEnv.reset (gym/optimized_env.py:53-68) for the envs whose mask byte is
 * non-zero (mask NULL = all).  mode 1 = jitter only (the reference's reset),
 * mode 2 = restore the template first (what make_env does, :273-294).
 * Writes obs if buf->obs is set.
 */
int wg_reset(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
             int64_t n_env, int mode, const uint8_t* mask, void* cuda_stream);

/*
 * Sum the per-env finished-episode accumulators into out8 (device, 8 doubles):
 * [sum return, sum return^2, sum length, count, non-finite count, non-finite length, 0, 0].
 * nf_stats may be NULL (then out8[4..5] = 0).  One kernel launch.  The caller
 * all-reduces out8 across ranks (NCCL) -- the only collective on this path.
 * wg_stats_reduce(f, n, o, s) is wg_stats_reduce_split(f, NULL, n, o, s).
 */
int wg_stats_reduce_split(const float* fin_stats, const float* nf_stats, int64_t n_env, double* out8, void* cuda_stream);
int wg_stats_reduce(const float* fin_stats, int64_t n_env, double* out8, void* cuda_stream);

/*
 * Host-buffer convenience used for end-to-end timing: copies `action` from
 * (pinned) host memory into buf->action, runs wg_step, and copies obs, reward
 * and done back to the host pointers (any may be NULL), all on cuda_stream.
 */
int wg_step_host(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
                 int64_t n_env, const float* h_action, float* h_obs, float* h_reward,
                 uint8_t* h_done, void* cuda_stream);

/*
 * The same for wg_step_multi: copies n_action_steps * n_env * n_muscle actions from (pinned) host memory into
 * buf->action, runs the n_steps-step launch, and copies the last observation [n_env][obs_dim], the per-step rewards
 * [n_steps][n_env] and dones back to the host pointers (any may be NULL), all on cuda_stream.  Per env-step the
 * PCIe traffic is 4 * n_muscle bytes up and 5 + 4 * obs_dim / n_steps bytes down.
 */
int wg_step_multi_host(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env,
                       int32_t n_steps, int32_t n_action_steps, const float* h_action, float* h_obs,
                       float* h_reward, uint8_t* h_done, void* cuda_stream);

/* =====================================================================================
 * The reference's *package* lineage (gym/optimized_walker/{core,env}.py): a second
 * physics model behind the same boundary.  Environment.update_physics (env.py:135-184)
 * has no action / observation / reward: it advances a point-and-spring system, so the
 * call takes a step count and keeps the state on chip for all n_steps substeps
 * (one HBM read and one HBM write of the state per launch).
 * ===================================================================================== */

/*
 * One point-and-spring system shared by all envs.  Replaces Environment.points /
 * ding_points / springs (gym/optimized_walker/env.py:39-41) as filled by add_point
 * (:56-72), add_ding_point (:74-90) and add_spring (:92-111).  Springs are applied in
 * list order (:149-150), which fixes the float32 accumulation order of every point.
 */
typedef struct wg_pkg_system {
    int32_t n_point, n_spring;
    double  mass[WG_MAX_MASS];          /* Point.m */
    uint8_t fixed[WG_MAX_MASS];         /* 1 = DingPoint (core.py:259-275): forced() ignored, not damped, no ground */
    int32_t si[WG_MAX_SPRING], sj[WG_MAX_SPRING];   /* point1, point2 */
    float   srest[WG_MAX_SPRING];       /* x: rest length (float32, as add_spring stores it) */
    float   sk[WG_MAX_SPRING];          /* k */
    uint8_t sstring[WG_MAX_SPRING];     /* string=True: no force while shorter than x (core.py:115-118) */
} wg_pkg_system;

/* Environment constructor arguments (gym/optimized_walker/env.py:10-37), as float32 at the point of use. */
typedef struct wg_pkg_params {
    float   gravity[3];     /* to_data(gravity) */
    float   damping;        /* v *= damping  (:153-154) */
    float   drag_c;         /* float32(-0.5 * air_resistance): drag = drag_c * |v| * v  (:157-161) */
    float   ground_level, restitution, friction;   /* (:167-181) */
    float   dt;             /* time_step */
    float   min_dist;       /* float32(Config.r): lower clamp of the spring length in anti_forced (core.py:89) */
    int32_t ground;         /* 0 = no ground */
} wg_pkg_params;

/*
 * n_steps x Environment.update_physics for n_env independent copies of the system.
 * pos, vel: in/out, SoA [(n*3 + c) * n_env + e]; old_a: optional out (Point.old_a of
 * the last step, same layout).  One kernel launch; asynchronous on cuda_stream.
 */
/* Which kernel wg_pkg_update_physics will launch: 0 = run-time topology (shared-memory state), > 0 = a
 * register-resident specialisation for one of the reference's small bodies (leg2, balance1-3, test).
 * wg_force_generic(1) forces 0.  Results never depend on it. */
int wg_pkg_kernel_variant(const wg_pkg_system* sys);

int wg_pkg_update_physics(const wg_pkg_system* sys, const wg_pkg_params* prm,
                          float* pos, float* vel, float* old_a,
                          int64_t n_env, int32_t n_steps, void* cuda_stream);

/* =====================================================================================
 * The caller of the hot path (BASELINE config 5): PPO rollout collection around wg_step.
 * The reference has no policy code; these entry points replace the per-step torch glue of
 * a rollout loop (gym/performance_demo.py:241-262 is the reference's random-action loop)
 * so that one env step costs two launches: wg_policy_act + wg_step.
 * ===================================================================================== */

/*
 * A gaussian MLP policy with two tanh hidden layers of 64 units and a value head, weights in
 * torch.nn.Linear layout (weight [out][in] row-major), all device pointers, float32.
 */
typedef struct wg_mlp_policy {
    const float* w1; const float* b1;        /* [64][obs_dim], [64] */
    const float* w2; const float* b2;        /* [64][64], [64] */
    const float* w_mu; const float* b_mu;    /* [act_dim][64], [act_dim] */
    const float* w_v; const float* b_v;      /* [1][64], [1] */
    const float* log_std;                    /* [act_dim] */
    int32_t obs_dim;                         /* 1..64 */
    int32_t act_dim;                         /* 1..7 */
    float   obs_scale, obs_clip;             /* x = clamp(nan_to_num(obs * obs_scale), +-obs_clip) */
    int32_t precision;                       /* 0 = float32-grade (3xTF32 error-compensated MMA), 1 = plain TF32 */
    int32_t reserved;
} wg_mlp_policy;

/*
 * One policy evaluation for n_env envs, one kernel launch:
 *   obs [n_env][obs_dim] (obs_layout 0) or [obs_dim][n_env] (obs_layout 1), as wg_step writes it
 *   -> mean, value = MLP(obs); action = mean + exp(log_std) * eps, eps ~ N(0,1) from Philox keyed by
 *      (seed, env_offset + env, step_index [+ *step_counter], action index); logp = log N(action; mean, std).
 * action [act_dim][n_env] (act_layout 1) or [n_env][act_dim] (0); logp, value [n_env]; mean [act_dim][n_env].
 * Any output may be NULL.  sample = 0 returns action = mean.
 */
int wg_policy_act(const wg_mlp_policy* pol, const float* obs, int32_t obs_layout, float* action, int32_t act_layout, float* logp,
                  float* value, float* mean, int64_t n_env, int32_t sample, uint32_t seed_lo, uint32_t seed_hi,
                  uint32_t step_index, const uint32_t* step_counter, uint32_t env_offset, void* cuda_stream);

/*
 * wg_policy_act immediately followed by wg_step with that action -- one env step of a PPO rollout (the caller of the hot
 * path, gym/performance_demo.py:241-262 with a policy instead of random actions) -- in ONE launch: the output warps of
 * the policy pipeline run PhysicsEnv.step of the env whose action they have just sampled, with the device functions of
 * the packed step kernel (the results are the bits of the two separate calls).  obs [n_env][38] row-major is this step's
 * observation; action [n_env][2] (row-major), logp, value, mean as in wg_policy_act (any may be NULL); buf as in wg_step:
 * buf->obs receives the NEXT observation, buf->reward / done / state_packed / fin_stats ... the step's results; buf->action is
 * ignored; the policy's Philox counter is step_index + *buf->step_counter, the env's prm->step_index + *buf->step_counter.
 * Exists for BASELINE config 5's environment -- Balance-v0's spring graph with the mass pattern [k, k, 1, j] (unit /
 * power-of-two / odd-integer masses), 3-D, packed state, row-major observations, WG_TUNE_POLICY_TC == 2; anything else
 * returns WG_ERR_UNSUPPORTED and the caller makes the two calls.
 */
int wg_policy_step(const wg_mlp_policy* pol, const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
                   const float* obs, float* action, float* logp, float* value, float* mean, int64_t n_env, int32_t sample,
                   uint32_t seed_lo, uint32_t seed_hi, uint32_t step_index, uint32_t env_offset, void* cuda_stream);

/* 1 if a tcgen05 policy kernel ever gave up waiting for its tensor-core work (a diagnostic: synchronises the device;
 * never set by a correct build), 0 otherwise, -1 on a CUDA error. */
int wg_policy_tc_status(void);

/*
 * GAE(lambda) over a trajectory: rewards [T][n_env], values [T+1][n_env], dones uint8 [T][n_env] ->
 * advantages, returns [T][n_env].  Rewards are sanitised first (NaN -> 0, clamp to +-reward_clip).
 */
int wg_gae(const float* rewards, const float* values, const uint8_t* dones, float* advantages, float* returns,
           int32_t horizon, int64_t n_env, float gamma, float lam, float reward_clip, void* cuda_stream);

/*
 * Measurement aid (bench.py --probe-stream): n_threads threads each read vec_reads and write vec_writes 16-byte
 * vectors from / to coalesced planes src[k][n_threads], dst[k][n_threads] and do nothing else.  Gives the HBM rate
 * that a kernel with the step kernel's read : write mix can reach on this GPU.
 */
int wg_stream_probe(const float* src, float* dst, int64_t n_threads, int32_t vec_reads, int32_t vec_writes, void* cuda_stream);

/*
 * Pinned (page-locked, portable, device-mapped) host memory for the host-buffer calls above.  The reference keeps
 * its arrays in pageable NumPy memory (gym/optimized_engine.py:84-89); a caller that feeds wg_step_host from such
 * arrays copies them into these buffers.  The pages are allocated and first-touched by the CALLING thread, so bind
 * the thread to the GPU's NUMA node first (walker_gym_b200.host.bind_to_device).  write_combined = 1 suits buffers
 * the host only writes (actions).  Because the memory is mapped, buf->obs / reward / done may point into it: the
 * step kernel then writes its results straight over PCIe ("zero-copy"), without a device staging buffer.
 */
int wg_host_alloc(void** out, uint64_t bytes, int write_combined);
int wg_host_free(void* p);

/*
 * Self-tests of the exact-arithmetic primitives the kernels are built from (csrc/wg_math.cuh), each against the
 * IEEE operation it replaces; every call ADDS the number of mismatching inputs to *d_mismatches (a device counter
 * the caller zeroes).  Asynchronous on cuda_stream.
 *   (The kernels evaluate the x / y halves of their 3-vectors with the packed twins of these primitives -- FMUL2 / FFMA2 /
 *   FADD2 -- and wg_selftest_div_smallint / wg_selftest_div3 check those twins on the same inputs, in both halves.)
 *   wg_selftest_div_smallint: x / m through the 3-FMA exact quotient (Point.forced's `f / self.m`,
 *       gym/optimized_engine.py:104-106, for integer masses and for the division by the number of masses) vs
 *       IEEE division, for every float32 bit pattern x in [x_begin, x_begin + x_count), x_begin + x_count <= 2^32;
 *       m = 1, a power of two <= 2048 or an odd integer in [3, 2047] (the divisors that ever take this path).
 *   wg_selftest_forced_list: float32(float64(a) + float64(f) / m) (a python-list force, gym/optimized_env.py:148-172)
 *       on n_pairs Philox-random (a, f) bit patterns.
 *   wg_selftest_sqrt: the inline sqrt of np.linalg.norm vs IEEE sqrt for every non-negative float32 and every NaN.
 *   wg_selftest_div3: `direction / current_dist` with one shared reciprocal (gym/optimized_walker.py:52-54) vs three
 *       IEEE divisions on n Philox-random inputs; mode 0 = independent bit patterns, 1 = L = norm(d), 2 = exponents
 *       at the guard boundaries (L near 2^-2 / 2^120 / subnormal / huge, quotients near 2^-100); general = 1 tests
 *       the variant the package-lineage kernel uses (arbitrary numerators; general = 0 assumes |d| <~ L, a direction,
 *       so mode 0 applies to general = 1 only).  Inputs are numbered first .. first + n - 1.  d_mismatches is
 *       uint64[2]: [0] += mismatches, [1] = 1 + the number of one failing input (if it was 0); d_dump (optional,
 *       float[10]) receives that input's d0 d1 d2 L, the three results and the three IEEE quotients.
 */
int wg_selftest_div_smallint(float m, uint64_t x_begin, uint64_t x_count, uint64_t* d_mismatches, void* cuda_stream);
int wg_selftest_forced_list(double m, uint32_t seed, uint64_t n_pairs, uint64_t* d_mismatches, void* cuda_stream);
int wg_selftest_sqrt(uint64_t* d_mismatches, void* cuda_stream);
int wg_selftest_div3(int mode, int general, uint32_t seed, uint64_t first, uint64_t n, uint64_t* d_mismatches, float* d_dump,
                     void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* WALKER_GYM_B200_H */
