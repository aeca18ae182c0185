/*
 * walker_oracle.c -- TEST INFRASTRUCTURE ONLY (the parity checker; never the
 * product, never shipped, never on the measured GPU path).
 *
 * A scalar CPU restatement, in plain C, of the physics step of walker-gym's
 * L1 "optimized flat" environment -- PhysicsEnv.step and everything below it.
 * Every function cites the reference file:line it restates (paths relative to
 * the reference checkout).  It reproduces the reference's float32/float64
 * mixed arithmetic *bit for bit* (NumPy 2.x NEP-50 promotion, OpenBLAS sdot
 * tail, NumPy pairwise summation), so parity tests can use exact equality.
 *
 * Pinning: the reference ships no tests or golden vectors (SURVEY.md 8c), so
 * this oracle is pinned against outputs of the reference itself, executed by
 * oracle/ref_harness.py in the authoring container and committed as fixtures
 * under tests/golden/ (generator: tests/golden/make_golden.py).  The
 * `-m "not gpu"` tests require bit equality between this file and those
 * fixtures.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off; no fast-math -- any
 * contraction or reassociation would break the bit-exactness argument).
 *
 * Memory layout (shared with the device library so the same arrays can be fed
 * to both): state is SoA, env fastest:  pos[(n*3+c)*E + e], vel likewise,
 * mx[m*E + e]; actions are row-major [E][M]; observations row-major [E][D].
 */
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <stdlib.h>

#define WGO_MAX_MASS 32
#define WGO_MAX_SPRING 96

typedef struct {
    int32_t n_mass, n_spring, n_muscle;      /* springs [0,M) are muscles, [M,S) skeletons: Creature.run order */
    double mass[WGO_MAX_MASS];               /* Point.m as the Python number it was given */
    uint8_t fixed[WGO_MAX_MASS];             /* DingPoint: forced() is a no-op (optimized_engine.py:414-416) */
    float tmpl_pos[WGO_MAX_MASS * 3];        /* morphology template (create_*_creature) */
    int32_t si[WGO_MAX_SPRING], sj[WGO_MAX_SPRING];
    float sk[WGO_MAX_SPRING];                /* float32(k)      -- NEP-50 weak python scalar */
    float sdamp[WGO_MAX_SPRING];             /* float32(dampk)  */
    float srest[WGO_MAX_SPRING];             /* skeleton.x / muscle.originx as float32 */
    float mlo[WGO_MAX_SPRING], mhi[WGO_MAX_SPRING]; /* float32(originx*minl), float32(originx*maxl) */
    uint8_t sstring[WGO_MAX_SPRING];         /* rope-type spring: no elastic force while shorter than its rest length --
                                                `if dx < 0 and string: f_size = 0` of Point.resilience
                                                (optimized_engine.py:134-138) applied to Muscle.run / Skeleton.run;
                                                the damping term is unchanged */
} wgo_body;

typedef struct {
    double g;                /* PhysicsEnv.g (python number) */
    float dampk;             /* float32(dampk) */
    float ground;            /* float32(ground_high) */
    float fall_thresh;       /* float32(ground_high - 50)  (optimized_env.py:218) */
    float ground_k, ground_damp, friction;
    float dt;                /* float32(time_step) */
    float dt2;               /* float32(time_step ** 2), integrator 1 only */
    float sigma;             /* rand_sigma for in-kernel reset noise */
    int32_t in3d, max_steps, k_sub;
    int32_t auto_reset;      /* 0 = none, 1 = jitter-only (reference reset()), 2 = template (make_env again) */
    int32_t integrator;      /* 0 = Point.run1, 1 = Point.run2 (optimized_engine.py:274-288) */
    uint32_t seed_lo, seed_hi;
    uint32_t step_index;     /* global step counter, part of the Philox counter */
    uint32_t env_offset;     /* global id of env 0 of this shard */
} wgo_params;

/* ---- NumPy / OpenBLAS arithmetic primitives --------------------------------- */

/* np.dot / np.linalg.norm on float32[3] go through OpenBLAS sdot, whose scalar
 * tail (n < 32) multiplies in float and accumulates in a double, rounding once
 * at the end (probed against NumPy 2.3.5 + OpenBLAS 0.3.30, 20k vectors). */
static inline float np_dot3(const float a[3], const float b[3]) {
    double acc = 0.0;
    float p0 = a[0] * b[0], p1 = a[1] * b[1], p2 = a[2] * b[2];
    acc += (double)p0; acc += (double)p1; acc += (double)p2;
    return (float)acc;
}
static inline float np_norm3(const float a[3]) { return sqrtf(np_dot3(a, a)); }

/* NumPy float32 pairwise summation (np.mean / np.sum over a 1-D array):
 * n < 8 sequential from -0.0; 8 <= n <= 128 eight interleaved accumulators. */
static float np_pairwise_sum(const float *a, int n) {
    if (n < 8) {
        float r = -0.0f;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    }
    float r[8];
    for (int j = 0; j < 8; j++) r[j] = a[j];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; j++) r[j] += a[i + j];
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}

/* Point.forced (optimized_engine.py:104-106) with a float32 ndarray force:
 * a += f / m, all float32 (m is a weak python scalar). */
static inline void forced_f32(float a[3], const float f[3], float mf, int fixed) {
    if (fixed) return;
    for (int c = 0; c < 3; c++) a[c] = a[c] + f[c] / mf;
}
/* Point.forced with a python *list* force (optimized_env.py:148-172 via the
 * harness shim): the list becomes a float64 ndarray, f/m is a float64 divide
 * and the in-place add runs in float64 before rounding into float32 a. */
static inline void forced_list(float a[3], const double f[3], double m, int fixed) {
    if (fixed) return;
    for (int c = 0; c < 3; c++) a[c] = (float)((double)a[c] + f[c] / m);
}

/* ---- deterministic N(0,1) for auto-reset (new functionality, no reference) --- */
/* Philox4x32-10 + Box-Muller whose log / sin / cos are built only from IEEE
 * + - * / sqrt and fmaf, so the device library reproduces them bit for bit.  */
static inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

/* natural log for x in (0, 1], |rel err| ~ 1e-7 */
static float det_logf(float x) {
    uint32_t ix = f2u(x);
    int32_t e = (int32_t)(ix - 0x3f3504f3u) >> 23;        /* m in [sqrt(1/2), sqrt(2)) */
    float m = u2f(ix - ((uint32_t)e << 23));
    float f = m - 1.0f;
    float s = f / (2.0f + f);
    float z = s * s;
    float w = z * z;
    float t1 = w * fmaf(w, 0.24279078841f, 0.40000972152f);
    float t2 = z * fmaf(w, 0.28498786688f, 0.66666662693f);
    float R = t2 + t1;
    float hfsq = 0.5f * f * f;
    float dk = (float)e;
    return fmaf(dk, 6.9313812256e-01f, f - (hfsq - fmaf(s, hfsq + R, dk * 9.0580006145e-06f)));
}
/* sin and cos of 2*pi*j/2^24 for a 24-bit integer j */
static void det_sincos2pi(uint32_t j, float *sn, float *cs) {
    uint32_t q = j >> 22;
    int32_t r = (int32_t)(j & 0x3fffffu);
    if (r >= (1 << 21)) { r -= (1 << 22); q += 1; }
    float th = (float)r * (1.5707963267948966f / 4194304.0f);   /* |th| <= pi/4 */
    float t2 = th * th;
    float sp = fmaf(t2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(t2, sp, -1.6666654611e-1f);
    float s = fmaf(th * t2, sp, th);
    float cp = fmaf(t2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(t2, cp, 4.166664568298827e-2f);
    float c = fmaf(t2 * t2, cp, fmaf(t2, -0.5f, 1.0f));
    switch (q & 3u) {
        case 0: *sn = s;  *cs = c;  break;
        case 1: *sn = c;  *cs = -s; break;
        case 2: *sn = -s; *cs = -c; break;
        default: *sn = -c; *cs = s; break;
    }
}
/* In-kernel action sources of wg_step_multi, restated: the scripted phase table sketched at gym/walker.py:356-366
 * (`tt = (t // 50) % 3; c.act([... row tt ...])`) and a sinusoidal pattern generator after the package lineage's
 * Muscle.act (gym/optimized_walker/walker.py:56-90: `t += dt; sin(2 pi freq t + phase)`) with the phase kept as a
 * 24-bit fraction of a turn.  steps[e] is env e's step counter BEFORE the step; out is [E][M] row-major.
 * mode 1: out = table[((steps / hold) % n_rows) * 16 + m];  mode 2: out = amp[m] * sin(2 pi ((phase0 + (steps+1) dphase) mod 2^24) / 2^24) */
void wgo_gen_actions(int mode, int n_rows, int hold, const float *table, const float *amp, const uint32_t *phase0,
                     const uint32_t *dphase, const int32_t *steps, int64_t E, int M, float *out) {
    for (int64_t e = 0; e < E; e++)
        for (int m = 0; m < M; m++) {
            if (mode == 1) out[e * M + m] = table[((steps[e] / hold) % n_rows) * 16 + m];
            else {
                float sn, cs;
                det_sincos2pi((phase0[m] + (uint32_t)(steps[e] + 1) * dphase[m]) & 0xffffffu, &sn, &cs);
                out[e * M + m] = amp[m] * sn;
            }
        }
}

/* three standard normals for (global env id, global step index, mass) */
void wgo_normal3(uint32_t seed_lo, uint32_t seed_hi, uint32_t env, uint32_t step, uint32_t mass, float out[3]) {
    uint32_t c[4] = { env, step, mass, 0x57474231u };
    philox4x32_10(c, seed_lo, seed_hi);
    float u1 = (float)((c[0] >> 8) + 1u) * (1.0f / 16777216.0f);
    float u3 = (float)((c[2] >> 8) + 1u) * (1.0f / 16777216.0f);
    float r1 = sqrtf(-2.0f * det_logf(u1));
    float r2 = sqrtf(-2.0f * det_logf(u3));
    float s1, c1, s2, c2;
    det_sincos2pi(c[1] >> 8, &s1, &c1);
    det_sincos2pi(c[3] >> 8, &s2, &c2);
    out[0] = r1 * c1; out[1] = r1 * s1; out[2] = r2 * c2;
    (void)s2;
}

/* ---- the step ----------------------------------------------------------------- */

/* "x64" mode: the reference driven with float64 ndarray actions (its own demo loop,
 * gym/performance_demo.py:241-262).  `self.x += a` (optimized_walker.py:33) then makes Muscle.x an np.float64, and
 * NumPy's promotion rules evaluate the muscle's spring term in double: dx = float64(L) - x, f_size = -dx * k,
 * force = f_size * direction (a float64 array), and Point.forced adds force / m to the float32 accumulator in
 * double, rounding once (:48-59 + optimized_engine.py:104-106).  A muscle that regulation() clamped (:27-30) holds
 * the limit object instead -- an np.float32 (or the python float the user passed) -- and is back on the float32
 * path until the next action.  So every muscle carries its length as a double plus a "weak" bit. */
typedef struct {
    double sk_d[WGO_MAX_SPRING];                          /* float(k) */
    double x0_d[WGO_MAX_SPRING];                          /* originx as the object the constructor kept */
    double mlo_d[WGO_MAX_SPRING], mhi_d[WGO_MAX_SPRING];  /* originx * minl, originx * maxl as the objects max()/min() compare */
} wgo_x64;

typedef struct {
    float pos[WGO_MAX_MASS][3], vel[WGO_MAX_MASS][3], acc[WGO_MAX_MASS][3], old_a[WGO_MAX_MASS][3];
    float mx[WGO_MAX_SPRING];
    double mx64[WGO_MAX_SPRING];      /* x64 mode only */
    uint8_t mxw[WGO_MAX_SPRING];      /* x64 mode: 1 = float32-typed ("weak") length: float32 arithmetic */
    const wgo_x64 *xb;                /* NULL = float32 mode */
} env_state;

/* Muscle.run / Skeleton.run (optimized_walker.py:45-67, 84-106): identical bodies. */
static void spring_run(const wgo_body *b, const wgo_params *p, env_state *s, int sp, float x) {
    (void)p;
    int i = b->si[sp], j = b->sj[sp];
    float mi = (float)b->mass[i], mj = (float)b->mass[j];
    float d12[3], dir[3], F[3], nF[3], dv[3], D[3], nD[3];
    for (int c = 0; c < 3; c++) d12[c] = s->pos[i][c] - s->pos[j][c];
    float L = np_norm3(d12);                                   /* :47 distant() */
    float dx = L - x;                                          /* :48 */
    float fs = (-dx) * b->sk[sp];                              /* :49  -dx*k: inverted Hooke as written
                                                                  (SURVEY 0.4); physical sign == negative k */
    if (b->sstring[sp] && dx < 0) fs = 0.0f;                   /* rope-type: f_size = 0 (optimized_engine.py:134-136) */
    for (int c = 0; c < 3; c++) dir[c] = s->pos[j][c] - s->pos[i][c];   /* :52 */
    if (L > 0) for (int c = 0; c < 3; c++) dir[c] = dir[c] / L;         /* :53-54 */
    if (s->xb && sp < b->n_muscle && !s->mxw[sp]) {
        /* np.float64 length: dx, f_size and force in double; forced() adds force / m in double */
        double dx64 = (double)L - s->mx64[sp];
        double fs64 = (-dx64) * s->xb->sk_d[sp];
        if (b->sstring[sp] && dx64 < 0) fs64 = 0.0;            /* rope-type, tested on the double dx */
        double F64[3], nF64[3];
        for (int c = 0; c < 3; c++) { F64[c] = fs64 * (double)dir[c]; nF64[c] = -F64[c]; }
        forced_list(s->acc[i], F64, b->mass[i], b->fixed[i]);
        forced_list(s->acc[j], nF64, b->mass[j], b->fixed[j]);
    } else {
    for (int c = 0; c < 3; c++) { F[c] = fs * dir[c]; nF[c] = -F[c]; }  /* :57 */
    forced_f32(s->acc[i], F, mi, b->fixed[i]);                          /* :58 */
    forced_f32(s->acc[j], nF, mj, b->fixed[j]);                         /* :59 */
    }
    for (int c = 0; c < 3; c++) dv[c] = s->vel[i][c] - s->vel[j][c];    /* :62 */
    float dk = np_dot3(dv, dir);                                        /* :63 */
    float cdk = dk * b->sdamp[sp];                                      /* :64 (dk*dampk)*direction */
    for (int c = 0; c < 3; c++) { D[c] = cdk * dir[c]; nD[c] = -D[c]; }
    forced_f32(s->acc[i], nD, mi, b->fixed[i]);                         /* :65 */
    forced_f32(s->acc[j], D, mj, b->fixed[j]);                          /* :66 */
}

/* PhysicsEnv._run_physics (optimized_env.py:140-178) + Point.run1
 * (optimized_engine.py:258-272).  Returns the force-phase contact bitmask. */
static uint32_t run_physics(const wgo_body *b, const wgo_params *p, env_state *s) {
    int N = b->n_mass, S = b->n_spring;
    uint32_t contact = 0;
    /* Creature.run (optimized_walker.py:117-127): zero, muscles, then skeletons */
    for (int n = 0; n < N; n++) for (int c = 0; c < 3; c++) s->acc[n][c] = 0.0f;
    for (int sp = 0; sp < S; sp++)
        spring_run(b, p, s, sp, sp < b->n_muscle ? s->mx[sp] : b->srest[sp]);
    for (int n = 0; n < N; n++) {
        double m = b->mass[n];
        float mf = (float)m;
        int fx = b->fixed[n];
        double fg[3] = { 0.0, -p->g, 0.0 };                        /* :148 gravity as a *force* */
        forced_list(s->acc[n], fg, m, fx);
        float fd[3];                                               /* :151,180-182 _damp: -k * p.v */
        float nk = -p->dampk;
        for (int c = 0; c < 3; c++) fd[c] = nk * s->vel[n][c];
        forced_f32(s->acc[n], fd, mf, fx);
        float deep = s->pos[n][1] - p->ground;                     /* :154,159 */
        if (deep < 0) {
            contact |= 1u << n;
            double f1[3] = { 0.0, (double)((-p->ground_k) * deep), 0.0 };       /* :162 */
            forced_list(s->acc[n], f1, m, fx);
            double f2[3] = { 0.0, (double)((-p->ground_damp) * s->vel[n][1]), 0.0 }; /* :165 */
            forced_list(s->acc[n], f2, m, fx);
            float ff = fabsf(deep) * p->friction;                  /* :168 */
            double f3[3] = { (double)((-s->vel[n][0]) * ff), 0.0,
                             p->in3d ? (double)((-s->vel[n][2]) * ff) : 0.0 };  /* :169-172 */
            forced_list(s->acc[n], f3, m, fx);
        }
    }
    /* Point.run1: v += a*t; pos += v*t; old_a = a  (two roundings each, no FMA) */
    for (int n = 0; n < N; n++)
        for (int c = 0; c < 3; c++) {
            if (p->integrator == 0) {
                float at = s->acc[n][c] * p->dt;
                s->vel[n][c] = s->vel[n][c] + at;
                float vt = s->vel[n][c] * p->dt;
                s->pos[n][c] = s->pos[n][c] + vt;
            } else {   /* Point.run2: p.pos += p.v*t + 0.5*p.a*t**2; p.v += p.a*t */
                float vt = s->vel[n][c] * p->dt;
                float ha = (0.5f * s->acc[n][c]) * p->dt2;
                s->pos[n][c] = s->pos[n][c] + (vt + ha);
                float at = s->acc[n][c] * p->dt;
                s->vel[n][c] = s->vel[n][c] + at;
            }
            s->old_a[n][c] = s->acc[n][c];
        }
    return contact;
}

/* Creature.getstat (optimized_walker.py:129-162) with the defaults PhysicsEnv uses. */
static void get_obs(const wgo_body *b, const wgo_params *p, const env_state *s, float *obs) {
    int N = b->n_mass, d = p->in3d ? 3 : 2, k = 0;
    float mid[3] = { 0.0f, 0.0f, 0.0f };
    for (int n = 0; n < N; n++) for (int c = 0; c < 3; c++) mid[c] = mid[c] + s->pos[n][c];
    for (int c = 0; c < 3; c++) mid[c] = mid[c] / (float)N;
    for (int n = 0; n < N; n++) {
        for (int c = 0; c < d; c++) obs[k++] = s->pos[n][c] - mid[c];
        for (int c = 0; c < d; c++) obs[k++] = s->vel[n][c];
        for (int c = 0; c < d; c++) obs[k++] = s->old_a[n][c];
    }
    for (int m = 0; m < b->n_muscle; m++) obs[k++] = s->mx[m];
}

int wgo_obs_dim(const wgo_body *b, int in3d) { return 3 * (in3d ? 3 : 2) * b->n_mass + b->n_muscle; }

static void load_env(const wgo_body *b, env_state *s, int64_t E, int64_t e, const float *pos, const float *vel,
                     const float *old_a, const float *mx) {
    for (int n = 0; n < b->n_mass; n++)
        for (int c = 0; c < 3; c++) {
            s->pos[n][c] = pos[(int64_t)(n * 3 + c) * E + e];
            s->vel[n][c] = vel[(int64_t)(n * 3 + c) * E + e];
            s->old_a[n][c] = old_a ? old_a[(int64_t)(n * 3 + c) * E + e] : 0.0f;
        }
    for (int m = 0; m < b->n_muscle; m++) s->mx[m] = mx[(int64_t)m * E + e];
}
static void store_env(const wgo_body *b, const env_state *s, int64_t E, int64_t e, float *pos, float *vel,
                      float *old_a, float *mx) {
    for (int n = 0; n < b->n_mass; n++)
        for (int c = 0; c < 3; c++) {
            pos[(int64_t)(n * 3 + c) * E + e] = s->pos[n][c];
            vel[(int64_t)(n * 3 + c) * E + e] = s->vel[n][c];
            if (old_a) old_a[(int64_t)(n * 3 + c) * E + e] = s->old_a[n][c];
        }
    for (int m = 0; m < b->n_muscle; m++) mx[(int64_t)m * E + e] = s->mx[m];
}

/* PhysicsEnv.reset (optimized_env.py:53-68) = "jitter": v[:d] += noise, steps = 0.
 * "template" = what make_env does again: fresh creature, then the same jitter. */
static void apply_reset(const wgo_body *b, const wgo_params *p, env_state *s, int mode,
                        const float *noise, int64_t E, int64_t e, uint32_t step_index) {
    int d = p->in3d ? 3 : 2;
    if (mode == 2) {
        for (int n = 0; n < b->n_mass; n++)
            for (int c = 0; c < 3; c++) {
                s->pos[n][c] = b->tmpl_pos[n * 3 + c]; s->vel[n][c] = 0.0f; s->old_a[n][c] = 0.0f;
            }
        for (int m = 0; m < b->n_muscle; m++) {
            s->mx[m] = b->srest[m];
            if (s->xb) { s->mx64[m] = s->xb->x0_d[m]; s->mxw[m] = 1; }      /* a fresh Muscle: x = originx */
        }
    }
    for (int n = 0; n < b->n_mass; n++) {
        float z[3];
        if (noise) {
            for (int c = 0; c < 3; c++) z[c] = noise[(int64_t)(n * 3 + c) * E + e];
        } else {
            wgo_normal3(p->seed_lo, p->seed_hi, p->env_offset + (uint32_t)e, step_index, (uint32_t)n, z);
            for (int c = 0; c < 3; c++) z[c] = p->sigma * z[c];
        }
        for (int c = 0; c < d; c++) s->vel[n][c] = s->vel[n][c] + z[c];
    }
}

/*
 * One env-step for E envs: PhysicsEnv.step (optimized_env.py:70-92).
 *   act (Creature.act, optimized_walker.py:164-167; Muscle.act/regulation :27-35)
 *   k_sub x _run_physics
 *   steps += 1; reward (:189-205); done (:207-230); info (:232-248)
 *   optional auto-reset of done envs, then observation (:184-187).
 * Optional outputs may be NULL.  noise (if given) is the already-scaled jitter
 * [N*3][E] used by auto-reset instead of the Philox stream.
 */
static int step_impl(const wgo_body *b, const wgo_params *p, int64_t E,
             float *pos, float *vel, float *old_a, float *mx, int32_t *steps,
             const float *action, int32_t act_dim,
             float *obs, float *reward, uint8_t *done,
             uint32_t *contact_pre, uint32_t *contact_post,
             float *energy, float *centroid,
             float *ep_ret, float *fin_stats,
             const float *noise,
             const wgo_x64 *xb, double *mx64, uint8_t *mx_weak, const double *action64) {
    int N = b->n_mass, M = b->n_muscle;
    int D = wgo_obs_dim(b, p->in3d);
    if (N > WGO_MAX_MASS || b->n_spring > WGO_MAX_SPRING) return -1;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < E; e++) {
        env_state s;
        load_env(b, &s, E, e, pos, vel, old_a, mx);
        s.xb = xb;
        /* Creature.act: for i < min(M, len(a)): x += a; x = max(x, lo); x = min(x, hi) */
        int na = act_dim < M ? act_dim : M;
        if (xb) {
            for (int m = 0; m < M; m++) { s.mx64[m] = mx64[(int64_t)m * E + e]; s.mxw[m] = mx_weak[(int64_t)m * E + e]; }
            for (int m = 0; m < na; m++) {
                double x = s.mx64[m] + action64[e * act_dim + m];    /* anything + np.float64 -> np.float64 */
                uint8_t weak = 0;
                if (xb->mlo_d[m] > x) { x = xb->mlo_d[m]; weak = 1; }  /* max() returns the limit OBJECT: float32-typed */
                if (xb->mhi_d[m] < x) { x = xb->mhi_d[m]; weak = 1; }
                s.mx64[m] = x; s.mxw[m] = weak;
            }
            for (int m = 0; m < M; m++) s.mx[m] = (float)s.mx64[m];  /* float32 view: weak muscles, observation */
        } else
        for (int m = 0; m < na; m++) {
            float x = s.mx[m] + action[e * act_dim + m];
            if (b->mlo[m] > x) x = b->mlo[m];       /* python max(x, lo): lo wins only if lo > x */
            if (b->mhi[m] < x) x = b->mhi[m];       /* python min(x, hi) */
            s.mx[m] = x;
        }
        uint32_t cpre = 0;
        for (int k = 0; k < p->k_sub; k++) cpre = run_physics(b, p, &s);
        int32_t st = steps[e] + 1;
        /* _get_reward */
        float ys[WGO_MAX_MASS], sp[WGO_MAX_MASS];
        uint32_t cpost = 0; int ncon = 0;
        for (int n = 0; n < N; n++) {
            ys[n] = s.pos[n][1];
            sp[n] = np_norm3(s.vel[n]);
            if (s.pos[n][1] - p->ground < 0) { cpost |= 1u << n; ncon++; }
        }
        float cy = np_pairwise_sum(ys, N) / (float)N;
        float avgv = np_pairwise_sum(sp, N) / (float)N;
        float vpen = (-avgv) * 0.1f;
        float cpen = (float)(-(double)ncon * 0.5);
        float rew = (cy + vpen) + cpen;
        /* _is_done */
        int dn = 0;
        if (st >= p->max_steps) dn = 1;
        else if (cy < p->fall_thresh) dn = 1;
        else {
            int all_stopped = 1;
            for (int n = 0; n < N; n++) if (!(sp[n] < 0.1f)) all_stopped = 0;
            if (all_stopped && st > 100) dn = 1;
        }
        if (reward) reward[e] = rew;
        if (done) done[e] = (uint8_t)dn;
        if (contact_pre) contact_pre[e] = cpre;
        if (contact_post) contact_post[e] = cpost;
        if (energy) {   /* _calculate_energy :240-248 */
            float ke[WGO_MAX_MASS], pe[WGO_MAX_MASS];
            for (int n = 0; n < N; n++) {
                ke[n] = (float)b->mass[n] * (sp[n] * sp[n]);
                pe[n] = (float)(b->mass[n] * p->g) * (s.pos[n][1] - p->ground);
            }
            energy[e] = 0.5f * np_pairwise_sum(ke, N) + np_pairwise_sum(pe, N);
        }
        if (centroid) { /* np.mean(axis=0): sequential over points, then / N */
            for (int c = 0; c < 3; c++) {
                float acc = s.pos[0][c];
                for (int n = 1; n < N; n++) acc = acc + s.pos[n][c];
                centroid[c * E + e] = acc / (float)N;
            }
        }
        if (ep_ret) {
            float r = ep_ret[e] + rew;
            if (dn && fin_stats) {       /* per-env finished-episode accumulators */
                fin_stats[0 * E + e] += r;
                fin_stats[1 * E + e] += r * r;
                fin_stats[2 * E + e] += (float)st;
                fin_stats[3 * E + e] += 1.0f;
            }
            ep_ret[e] = (dn && p->auto_reset) ? 0.0f : r;
        }
        if (dn && p->auto_reset) {
            apply_reset(b, p, &s, p->auto_reset, noise, E, e, p->step_index);
            st = 0;
        }
        steps[e] = st;
        if (obs) get_obs(b, p, &s, obs + e * D);
        store_env(b, &s, E, e, pos, vel, old_a, mx);
        if (xb) for (int m = 0; m < M; m++) { mx64[(int64_t)m * E + e] = s.mx64[m]; mx_weak[(int64_t)m * E + e] = s.mxw[m]; }
    }
    return 0;
}

int wgo_step(const wgo_body *b, const wgo_params *p, int64_t E,
             float *pos, float *vel, float *old_a, float *mx, int32_t *steps,
             const float *action, int32_t act_dim,
             float *obs, float *reward, uint8_t *done,
             uint32_t *contact_pre, uint32_t *contact_post,
             float *energy, float *centroid,
             float *ep_ret, float *fin_stats,
             const float *noise) {
    return step_impl(b, p, E, pos, vel, old_a, mx, steps, action, act_dim, obs, reward, done, contact_pre, contact_post,
                     energy, centroid, ep_ret, fin_stats, noise, NULL, NULL, NULL, NULL);
}

/* PhysicsEnv.step driven with float64 ndarray actions (x64 mode, see wgo_x64): mx64 [M][E] double and mx_weak [M][E]
 * are the muscle lengths and their type bits (in/out); mx receives the float32 view. */
int wgo_step_x64(const wgo_body *b, const wgo_x64 *xb, const wgo_params *p, int64_t E,
                 float *pos, float *vel, float *old_a, float *mx, double *mx64, uint8_t *mx_weak, int32_t *steps,
                 const double *action64, int32_t act_dim,
                 float *obs, float *reward, uint8_t *done,
                 uint32_t *contact_pre, uint32_t *contact_post,
                 float *energy, float *centroid,
                 float *ep_ret, float *fin_stats,
                 const float *noise) {
    if (!xb || !mx64 || !mx_weak || (act_dim > 0 && !action64)) return -1;
    return step_impl(b, p, E, pos, vel, old_a, mx, steps, NULL, act_dim, obs, reward, done, contact_pre, contact_post,
                     energy, centroid, ep_ret, fin_stats, noise, xb, mx64, mx_weak, action64);
}
int wgo_sizeof_x64(void) { return (int)sizeof(wgo_x64); }

/* Explicit reset of the envs whose mask byte is non-zero (mask NULL = all). */
int wgo_reset(const wgo_body *b, const wgo_params *p, int64_t E, int mode,
              float *pos, float *vel, float *old_a, float *mx, int32_t *steps,
              float *obs, const uint8_t *mask, const float *noise) {
    int D = wgo_obs_dim(b, p->in3d);
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < E; e++) {
        if (mask && !mask[e]) continue;
        env_state s;
        load_env(b, &s, E, e, pos, vel, old_a, mx);
        s.xb = NULL;
        apply_reset(b, p, &s, mode, noise, E, e, p->step_index);
        steps[e] = 0;
        if (obs) get_obs(b, p, &s, obs + e * D);
        store_env(b, &s, E, e, pos, vel, old_a, mx);
    }
    return 0;
}

/* =============================================================================================
 * L2: the reference's *package* lineage -- Environment.update_physics of
 * gym/optimized_walker/env.py:135-184 on top of gym/optimized_walker/core.py (Point.forced :81-83,
 * anti_forced :85-91, resilience :93-121, run1 :184-200, DingPoint :259-275).  A different physics
 * model from the gym-style env above: physically signed springs with optional one-sided ("string")
 * behaviour, gravity as an acceleration (g*m/m), multiplicative velocity damping, quadratic drag,
 * and a ground that clamps the position and reflects the velocity.  No observation/reward/done.
 * ============================================================================================= */
typedef struct {
    int32_t n_point, n_spring;
    double mass[WGO_MAX_MASS];
    uint8_t ding[WGO_MAX_MASS];
    int32_t si[WGO_MAX_SPRING], sj[WGO_MAX_SPRING];
    float sx[WGO_MAX_SPRING];        /* rest length as float32 */
    float sk[WGO_MAX_SPRING];        /* float32(k) */
    uint8_t sstring[WGO_MAX_SPRING]; /* rope: no force while shorter than the rest length */
} wgo_l2_system;

typedef struct {
    float gravity[3];      /* to_data(gravity): float32 */
    float damping;         /* float32(damping) */
    float drag_c;          /* float32(-0.5 * air_resistance)  (python product, then weak cast) */
    float ground_level, restitution, friction, dt;
    float min_dist;        /* float32(Config.r) = float32(16e-36) */
    int32_t ground;
} wgo_l2_params;

static void l2_anti_forced(float a[3], const float self_pos[3], const float other_pos[3], float nfs,
                           float m, int ding, float min_dist) {
    float dir[3];                                                 /* core.py:87 */
    for (int c = 0; c < 3; c++) dir[c] = other_pos[c] - self_pos[c];
    float dist = np_norm3(dir);                                   /* :89 max(norm, Config.r) */
    if (min_dist > dist) dist = min_dist;
    if (ding) return;                                             /* DingPoint.forced: pass */
    for (int c = 0; c < 3; c++) {
        float f = (nfs * dir[c]) / dist;                          /* :90 -f_size * direction / distance */
        a[c] = a[c] + f / m;                                      /* :83 */
    }
}

int wgo_l2_step(const wgo_l2_system *sys, const wgo_l2_params *p, int64_t E, int32_t n_steps,
                float *pos, float *vel, float *old_a) {
    const int P = sys->n_point, S = sys->n_spring;
    if (P > WGO_MAX_MASS || S > WGO_MAX_SPRING) return -1;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < E; e++) {
        float ps[WGO_MAX_MASS][3], vs[WGO_MAX_MASS][3], as[WGO_MAX_MASS][3];
        for (int n = 0; n < P; n++)
            for (int c = 0; c < 3; c++) { ps[n][c] = pos[(int64_t)(n * 3 + c) * E + e]; vs[n][c] = vel[(int64_t)(n * 3 + c) * E + e]; }
        for (int t = 0; t < n_steps; t++) {
            for (int n = 0; n < P; n++) for (int c = 0; c < 3; c++) as[n][c] = 0.0f;          /* env.py:141-142 */
            for (int n = 0; n < P; n++) {                                                    /* :145-146 gravity*m */
                if (sys->ding[n]) continue;
                float mf = (float)sys->mass[n];
                for (int c = 0; c < 3; c++) as[n][c] = as[n][c] + (p->gravity[c] * mf) / mf;
            }
            for (int s = 0; s < S; s++) {                                                    /* :149-150 resilience */
                int i = sys->si[s], j = sys->sj[s];
                float d[3];
                for (int c = 0; c < 3; c++) d[c] = ps[i][c] - ps[j][c];
                float cur = np_norm3(d);                                                     /* core.py:102 */
                float dx = cur - sys->sx[s];
                float nfs = (dx < 0 && sys->sstring[s]) ? 0.0f : -((-dx) * sys->sk[s]);      /* :115-118, then -f_size */
                l2_anti_forced(as[i], ps[i], ps[j], nfs, (float)sys->mass[i], sys->ding[i], p->min_dist);
                l2_anti_forced(as[j], ps[j], ps[i], nfs, (float)sys->mass[j], sys->ding[j], p->min_dist);
            }
            for (int n = 0; n < P; n++) {
                if (sys->ding[n]) continue;
                for (int c = 0; c < 3; c++) vs[n][c] = vs[n][c] * p->damping;                  /* env.py:153-154 */
            }
            for (int n = 0; n < P; n++) {                                                    /* :157-161 drag */
                if (sys->ding[n]) continue;
                float speed = np_norm3(vs[n]);
                float cs = p->drag_c * speed;
                float mf = (float)sys->mass[n];
                for (int c = 0; c < 3; c++) as[n][c] = as[n][c] + (cs * vs[n][c]) / mf;
            }
            for (int n = 0; n < P; n++)                                                      /* Point.run1 */
                for (int c = 0; c < 3; c++) {
                    float at = as[n][c] * p->dt;
                    vs[n][c] = vs[n][c] + at;
                    float vt = vs[n][c] * p->dt;
                    ps[n][c] = ps[n][c] + vt;
                }
            if (p->ground)                                                                   /* :167-181 */
                for (int n = 0; n < P; n++) {
                    if (sys->ding[n]) continue;
                    if (ps[n][1] <= p->ground_level) {
                        ps[n][1] = p->ground_level;
                        if (vs[n][1] < 0) {
                            vs[n][1] = (-vs[n][1]) * p->restitution;
                            vs[n][0] = vs[n][0] * p->friction;
                            vs[n][2] = vs[n][2] * p->friction;
                        }
                    }
                }
        }
        for (int n = 0; n < P; n++)
            for (int c = 0; c < 3; c++) {
                pos[(int64_t)(n * 3 + c) * E + e] = ps[n][c];
                vel[(int64_t)(n * 3 + c) * E + e] = vs[n][c];
                if (old_a) old_a[(int64_t)(n * 3 + c) * E + e] = as[n][c];
            }
    }
    return 0;
}
int wgo_sizeof_l2_system(void) { return (int)sizeof(wgo_l2_system); }
int wgo_sizeof_l2_params(void) { return (int)sizeof(wgo_l2_params); }

#ifdef _OPENMP
#include <omp.h>
void wgo_set_num_threads(int n) { if (n > 0) omp_set_num_threads(n); }
int wgo_get_max_threads(void) { return omp_get_max_threads(); }
#else
void wgo_set_num_threads(int n) { (void)n; }
int wgo_get_max_threads(void) { return 1; }
#endif

int wgo_sizeof_body(void) { return (int)sizeof(wgo_body); }
int wgo_sizeof_params(void) { return (int)sizeof(wgo_params); }
