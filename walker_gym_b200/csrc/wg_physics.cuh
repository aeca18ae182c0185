// wg_physics.cuh -- the per-env physics of walker-gym's PhysicsEnv.step, written
// once as templates over
//   Topo  : the spring/muscle topology (compile-time tables for the register-
//           resident specialisations, run-time tables for the generic kernel),
//   Store : where the per-env state lives (registers or a shared-memory tile).
// One thread owns one env; springs are applied strictly in the reference's list
// order with its four separate accumulations per endpoint, so the float32
// result is bit-identical to the reference (gym/optimized_walker.py:45-127,
// gym/optimized_env.py:140-230, gym/optimized_engine.py:104-106,258-272).
#pragma once
#include "wg_math.cuh"

namespace wg {

constexpr int kMaxMass = 32;
constexpr int kMaxSpring = 96;

// Per-morphology scalars, passed by value in the kernel parameters (constant bank).
template <int MAXN, int MAXS>
struct BodyVals {
    double gm[MAXN];        // (-g) / m  in float64: gravity "force" per unit mass (optimized_env.py:148)
    double mass_d[MAXN];    // Point.m
    float mass_f[MAXN];     // float32(m): divisor of float32 forces
    float mass_r[MAXN];     // RN(1 / float32(m))
    double mass_rd[MAXN];   // RN(1 / m) in float64
    int32_t mass_kind[MAXN];// div_const kind of each mass (0 unit, 1 pow2, 2 small integer, 3 general)
    ConstDiv ndiv;          // division by the number of masses (centroid / means)
    float mg_f[MAXN];       // float32(m * g): potential-energy weight (:245)
    float tmpl[MAXN * 3];   // creation-time positions
    float sk[MAXS], sdamp[MAXS], srest[MAXS];
    float mlo[MAXS], mhi[MAXS];
    uint32_t fixed_mask;    // DingPoint bits
    uint32_t unit_mask;     // bit n: m == 1 (x / 1 is exact, float64 division skipped)
    int32_t si[MAXS], sj[MAXS];   // only read by the run-time topology
    int32_t n_mass, n_spring, n_muscle;
    uint32_t string_mask[(MAXS + 31) / 32];   // rope-type springs (run-time topology only: f_size = 0 while dx < 0)
};

struct EnvConst {
    float ndampk;           // -dampk
    float ground, fall_thresh;
    float nground_k, nground_damp, friction;
    float dt, dt2, sigma;
    int32_t max_steps, k_sub, auto_reset, integrator;
    uint32_t seed_lo, seed_hi, step_index, env_offset;
    int32_t dampk_is_zero;
    int32_t end_nonfinite;  // 1 = a step whose reward is not finite ends the episode (epilogue_reduce)
};

// ---- state stores -------------------------------------------------------------
template <int N, int M>
struct RegStore {
    float p_[N][3], v_[N][3], a_[N][3];
    float mx_[M > 0 ? M : 1];
    __device__ __forceinline__ float& pos(int n, int c) { return p_[n][c]; }
    __device__ __forceinline__ float& vel(int n, int c) { return v_[n][c]; }
    __device__ __forceinline__ float& acc(int n, int c) { return a_[n][c]; }
    __device__ __forceinline__ float& mx(int m) { return mx_[m]; }
};
// shared-memory tile: element (row, thread) at base[row * stride + tid], conflict-free per warp
struct SmemStore {
    float* base; int stride; int N;
    __device__ __forceinline__ float& pos(int n, int c) { return base[(n * 3 + c) * stride]; }
    __device__ __forceinline__ float& vel(int n, int c) { return base[(3 * N + n * 3 + c) * stride]; }
    __device__ __forceinline__ float& acc(int n, int c) { return base[(6 * N + n * 3 + c) * stride]; }
    __device__ __forceinline__ float& mx(int m) { return base[(9 * N + m) * stride]; }
    // scratch rows after the muscles: 2*N floats (ys / speeds)
    __device__ __forceinline__ float& scratch(int M, int i) { return base[(9 * N + M + i) * stride]; }
};

// ---- topologies ---------------------------------------------------------------
struct RuntimeTopo {
    static constexpr bool kStatic = false;
    static constexpr int kId = 0;
    int N_, S_, M_;
    const int32_t* si_; const int32_t* sj_;
    __device__ __forceinline__ int n() const { return N_; }
    __device__ __forceinline__ int s() const { return S_; }
    __device__ __forceinline__ int m() const { return M_; }
    __device__ __forceinline__ int si(int k) const { return si_[k]; }
    __device__ __forceinline__ int sj(int k) const { return sj_[k]; }
};

#define WG_STATIC_TOPO(NAME, ID, NN, SS, MM, ...)                                               \
    struct NAME {                                                                               \
        static constexpr bool kStatic = true;                                                   \
        static constexpr int kId = ID, N = NN, S = SS, M = MM;                                  \
        __host__ __device__ static constexpr int n() { return NN; }                             \
        __host__ __device__ static constexpr int s() { return SS; }                             \
        __host__ __device__ static constexpr int m() { return MM; }                             \
        __host__ __device__ static constexpr int ep(int k) {                                    \
            constexpr int t[2 * SS] = { __VA_ARGS__ };                                          \
            return t[k];                                                                        \
        }                                                                                       \
        __host__ __device__ static constexpr int si(int k) { return ep(2 * k); }                \
        __host__ __device__ static constexpr int sj(int k) { return ep(2 * k + 1); }            \
    };

// ---- physics ------------------------------------------------------------------

// Two successive Point.forced calls on mass n with float32 ndarray forces:
//   a += f / m;  a += g / m        (gym/optimized_engine.py:104-106)
// MM is the body-wide mass mode chosen at launch: 0 = every mass is 1 (x / 1 == x, no division at
// all), 1 = every mass is 1, a power of two or a small integer (exact 3-instruction division),
// 2 = arbitrary masses.  The per-mass choice is a warp-uniform branch on a kernel parameter.
template <int MM, class BV>
__device__ __forceinline__ void forced2(V3& a, const V3& f, const V3& g, const BV& bv, int n) {
    if (MM == 0) {
        a = v3_add_prod(v3_add_prod(a, f), g);            // f and g are packed products: scalar additions
        return;
    }
    int kind = 2;
    if (MM == 2) kind = bv.mass_kind[n];
    if (kind == 0) {
        a = v3_add_prod(v3_add_prod(a, f), g);
    } else if (kind <= 2) {
        // one straight-line path for every mass of the body (MM 1: with m == 1 (r == 1) the sequence degenerates to
        // q0 = x, rem = 0, q = x, so unit masses need no branch).  Three packed quotients: (f.x, f.y), (g.x, g.y) and the
        // two z components together -- they share the divisor
        const float m = bv.mass_f[n], r = bv.mass_r[n];
        const float2 qf = div_smallint2(f.xy, m, r), qg = div_smallint2(g.xy, m, r), qz = div_smallint2(make_float2(f.z, g.z), m, r);
        a.xy = __fadd2_rn(__fadd2_rn(a.xy, qf), qg);
        a.z = (a.z + qz.x) + qz.y;
    } else {
        const float m = bv.mass_f[n];
        a.xy = make_float2((a.xy.x + div_rn(f.xy.x, m)) + div_rn(g.xy.x, m), (a.xy.y + div_rn(f.xy.y, m)) + div_rn(g.xy.y, m));
        a.z = (a.z + div_rn(f.z, m)) + div_rn(g.z, m);
    }
}

// Muscle.run / Skeleton.run (optimized_walker.py:45-67 == :84-106)
template <class Store>
__device__ __forceinline__ V3 load_acc(Store& st, int n) { return v3(st.acc(n, 0), st.acc(n, 1), st.acc(n, 2)); }
template <class Store>
__device__ __forceinline__ void store_acc(Store& st, int n, const V3& a) { st.acc(n, 0) = a.xy.x; st.acc(n, 1) = a.xy.y; st.acc(n, 2) = a.z; }

template <int MM, bool USE_SKIP = (MM == 2), class Topo, class BV, class Store>
__device__ __forceinline__ void spring_run(const Topo& topo, const BV& bv, Store& st, int sp, float x, uint32_t skip_mask) {
    const int i = topo.si(sp), j = topo.sj(sp);
    const V3 pi = v3(st.pos(i, 0), st.pos(i, 1), st.pos(i, 2)), pj = v3(st.pos(j, 0), st.pos(j, 1), st.pos(j, 2));
    V3 d = v3_sub(pj, pi);                                                  // direction = p2 - p1
    // distant(p1, p2) = norm(p1 - p2): p1 - p2 == -(p2 - p1) exactly and only its squares are used, so the norm is
    // taken of the direction's components (three subtractions less per spring)
    const float L = unit_dir(d);                                            // L = |d|, then d /= L (one rare-path region)
    const float dx = L - x;
    float fs = (-dx) * bv.sk[sp];                                         // -dx * k (sign as written)
    // rope-type springs (`if dx < 0 and string: f_size = 0`, gym/optimized_engine.py:134-136): a per-spring flag of
    // the run-time topology only -- bodies with such springs never reach the compile-time specialisations.  The rule
    // holds for both action dtypes: spring_run_x64 applies it to the float64 length of a strong muscle
    if constexpr (!Topo::kStatic) { if (((bv.string_mask[sp >> 5] >> (sp & 31)) & 1u) && dx < 0.0f) fs = 0.0f; }
    const V3 F = v3_scale(d, fs);
    const V3 vd = v3_sub(v3(st.vel(i, 0), st.vel(i, 1), st.vel(i, 2)), v3(st.vel(j, 0), st.vel(j, 1), st.vel(j, 2)));
    const float dk = np_dot3(vd, d);
    const float cd = dk * bv.sdamp[sp];
    const V3 D = v3_scale(d, cd);
    const V3 nF = v3_neg(F), nD = v3_neg(D);
    // skip_mask: masses whose accumulator this thread must not touch -- DingPoints (forced() is a no-op)
    // and, in the mass-partitioned kernel, masses owned by another lane.  Compiled out (USE_SKIP false)
    // in the one-thread-per-env kernels for bodies without DingPoints.
    if constexpr (MM == 3) {
        // mass pattern known at compile time (Topo::unit / Topo::same, constant-folded after unrolling): a unit mass
        // needs no division, and two endpoints of equal mass share the quotients -- (-F)/m == -(F/m) and
        // D/m == -((-D)/m) exactly, so p2's increments are the negated increments of p1.  Per endpoint three packed
        // quotients: (F.x, F.y), (-D.x, -D.y) and the two z components together.
        const bool ui = Topo::unit(i), uj = Topo::unit(j);
        float2 qF = F.xy, qD = nD.xy, qz = make_float2(F.z, nD.z);          // F / m_i, (-D) / m_i
        if (!ui) {
            qF = div_smallint2(qF, bv.mass_f[i], bv.mass_r[i]);
            qD = div_smallint2(qD, bv.mass_f[i], bv.mass_r[i]);
            qz = div_smallint2(qz, bv.mass_f[i], bv.mass_r[i]);
        }
        V3 ai = load_acc(st, i);
        // unit mass: qF / qD are the packed PRODUCTS themselves and must be added with scalar additions (wg_math.cuh CAUTION)
        ai.xy = ui ? add2_prod(add2_prod(ai.xy, qF), qD) : __fadd2_rn(__fadd2_rn(ai.xy, qF), qD);
        ai.z = (ai.z + qz.x) + qz.y;
        store_acc(st, i, ai);
        float2 pF, pD, pz;                                                  // (-F) / m_j, D / m_j
        if (Topo::same(i, j)) { pF = neg2(qF); pD = neg2(qD); pz = neg2(qz); }
        else if (uj) { pF = nF.xy; pD = D.xy; pz = make_float2(nF.z, D.z); }
        else {
            pF = div_smallint2(nF.xy, bv.mass_f[j], bv.mass_r[j]);
            pD = div_smallint2(D.xy, bv.mass_f[j], bv.mass_r[j]);
            pz = div_smallint2(make_float2(nF.z, D.z), bv.mass_f[j], bv.mass_r[j]);
        }
        V3 aj = load_acc(st, j);
        const bool j_raw = Topo::same(i, j) ? ui : uj;                      // p2's increments are (negated) raw products
        aj.xy = j_raw ? add2_prod(add2_prod(aj.xy, pF), pD) : __fadd2_rn(__fadd2_rn(aj.xy, pF), pD);
        aj.z = (aj.z + pz.x) + pz.y;
        store_acc(st, j, aj);
        return;
    }
    if (!USE_SKIP || !((skip_mask >> i) & 1u)) {                            // p1.forced(force); p1.forced(-damp)
        V3 a = load_acc(st, i);
        forced2<MM>(a, F, nD, bv, i);
        store_acc(st, i, a);
    }
    if (!USE_SKIP || !((skip_mask >> j) & 1u)) {                            // p2.forced(-force); p2.forced(damp)
        V3 a = load_acc(st, j);
        forced2<MM>(a, nF, D, bv, j);
        store_acc(st, j, a);
    }
}

// ---- x64 mode -----------------------------------------------------------------------------------------------------
// The reference driven with float64 ndarray actions (its own demo loop, gym/performance_demo.py:241-262):
// `self.x += a` (optimized_walker.py:33) makes Muscle.x an np.float64 and NumPy then evaluates the muscle's spring
// term in double -- dx = float64(L) - x, f_size = -dx * k, force = f_size * direction (a float64 array), and
// Point.forced adds force / m to the float32 accumulator in double, rounding once (:48-59, optimized_engine.py:104-106).
// A muscle that regulation() clamped (:27-30) holds the limit object (np.float32 / python float) and is on the float32
// path until the next action.  Direction and damping stay float32 either way.
struct X64Vals {
    double sk_d[kMaxSpring];                          // float(k)
    double x0_d[kMaxSpring];                          // originx, the object a fresh Muscle holds
    double mlo_d[kMaxSpring], mhi_d[kMaxSpring];      // originx * minl, originx * maxl as max() / min() compare them
};

template <class Topo, class BV, class Store>
__device__ __forceinline__ void spring_run_x64(const Topo& topo, const BV& bv, Store& st, int sp, double x, double k_d,
                                               uint32_t skip_mask) {
    const int i = topo.si(sp), j = topo.sj(sp);
    const float pix = st.pos(i, 0), piy = st.pos(i, 1), piz = st.pos(i, 2);
    const float pjx = st.pos(j, 0), pjy = st.pos(j, 1), pjz = st.pos(j, 2);
    float d0 = pjx - pix, d1 = pjy - piy, d2 = pjz - piz;
    const float L = np_norm3(d0, d1, d2);
    div3_len(d0, d1, d2, L);
    const double dx = (double)L - x;
    double fs = (-dx) * k_d;
    if (((bv.string_mask[sp >> 5] >> (sp & 31)) & 1u) && dx < 0.0) fs = 0.0;   // rope-type, tested on the double dx
    const double F[3] = { fs * (double)d0, fs * (double)d1, fs * (double)d2 };
    const float dk = np_dot3(st.vel(i, 0) - st.vel(j, 0), st.vel(i, 1) - st.vel(j, 1),
                             st.vel(i, 2) - st.vel(j, 2), d0, d1, d2);
    const float cd = dk * bv.sdamp[sp];
    const float D[3] = { cd * d0, cd * d1, cd * d2 };
    if (!((skip_mask >> i) & 1u)) {                                        // p1.forced(force); p1.forced(-damp)
        const double m = bv.mass_d[i];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const float a = (float)((double)st.acc(i, c) + F[c] / m);
            st.acc(i, c) = a + div_const(-D[c], bv.mass_f[i], bv.mass_r[i], bv.mass_kind[i]);
        }
    }
    if (!((skip_mask >> j) & 1u)) {                                        // p2.forced(-force); p2.forced(damp)
        const double m = bv.mass_d[j];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const float a = (float)((double)st.acc(j, c) + (-F[c]) / m);
            st.acc(j, c) = a + div_const(D[c], bv.mass_f[j], bv.mass_r[j], bv.mass_kind[j]);
        }
    }
}

// Rarely used variants, kept out of line so that they do not dilute the hot instruction stream.
static __device__ __noinline__ float3 damp_cold(float3 a, float3 v, float ndampk, float m, float r, int kind) {
    a.x = a.x + div_const(ndampk * v.x, m, r, kind);
    a.y = a.y + div_const(ndampk * v.y, m, r, kind);
    a.z = a.z + div_const(ndampk * v.z, m, r, kind);
    return a;
}
static __device__ __noinline__ void run2_cold(float3& p, float3& v, float3 a, float dt, float dt2) {
    p.x = p.x + (v.x * dt + (0.5f * a.x) * dt2);
    p.y = p.y + (v.y * dt + (0.5f * a.y) * dt2);
    p.z = p.z + (v.z * dt + (0.5f * a.z) * dt2);
    v.x = v.x + a.x * dt; v.y = v.y + a.y * dt; v.z = v.z + a.z * dt;
}

// Environment forces on mass n (gravity, damping, ground contact: gym/optimized_env.py:146-175) followed by
// the integrator (Point.run1 / run2).  Returns the force-phase contact flag.
// UNIT: 1 = this mass is known at compile time to be 1 (mass mode 0, or mode 3's unit-mass point), 0 = known not to
// need the run-time kind (modes 1 and 3: the exact-remainder quotient, which is also right for m == 1), -1 = run time.
template <bool IN3D, int MM, int UNIT = -1, class BV, class Store>
__device__ __forceinline__ bool point_step(const BV& bv, const EnvConst& ec, Store& st, int n) {
    const bool fixed = (MM == 2) && ((bv.fixed_mask >> n) & 1u);
    float ax = st.acc(n, 0), ay = st.acc(n, 1), az = st.acc(n, 2);
    const float vx = st.vel(n, 0), vy = st.vel(n, 1), vz = st.vel(n, 2);
    const float deep = st.pos(n, 1) - ec.ground;
    const bool hit = deep < 0.0f;
    if (!fixed) {
        ay = (float)((double)ay + bv.gm[n]);                 // forced([0, -g, 0])
        if (ec.dampk_is_zero) {                               // forced(-0 * v): +-0, or NaN for non-finite v
            // one FMA per component: the product is an exact zero (or NaN), so fma(-0, v, a) == a + (-0 * v) bit for bit,
            // signs of zero included
            const float2 axy = __ffma2_rn(bc2(ec.ndampk), make_float2(vx, vy), make_float2(ax, ay));
            ax = axy.x; ay = axy.y; az = __fmaf_rn(ec.ndampk, vz, az);
        } else {                                              // forced(-k * v): float32 force / m  (cold: dampk defaults to 0)
            const float3 r = damp_cold(make_float3(ax, ay, az), make_float3(vx, vy, vz), ec.ndampk,
                                       bv.mass_f[n], bv.mass_r[n], bv.mass_kind[n]);
            ax = r.x; ay = r.y; az = r.z;
        }
        if (hit) {
            const double m = bv.mass_d[n], rd = bv.mass_rd[n];
            const float ff = fabsf(deep) * ec.friction;             // friction
            if constexpr (MM == 0 || UNIT == 1) {                    // unit mass: float32 additions (see forced_list_k)
                ay = forced_list_k<0>(ay, ec.nground_k * deep, m, rd);       // ground spring
                ay = forced_list_k<0>(ay, ec.nground_damp * vy, m, rd);      // ground damper
                ax = forced_list_k<0>(ax, (-vx) * ff, m, rd);
                if (IN3D) az = forced_list_k<0>(az, (-vz) * ff, m, rd);
            } else if constexpr (MM == 1 || MM == 3) {               // unit / power-of-two / odd-integer masses: no dispatch
                ay = forced_list_k<2>(ay, ec.nground_k * deep, m, rd);
                ay = forced_list_k<2>(ay, ec.nground_damp * vy, m, rd);
                ax = forced_list_k<2>(ax, (-vx) * ff, m, rd);
                if (IN3D) az = forced_list_k<2>(az, (-vz) * ff, m, rd);
            } else {
                const int kd = bv.mass_kind[n];
                ay = forced_list(ay, ec.nground_k * deep, m, rd, kd);
                ay = forced_list(ay, ec.nground_damp * vy, m, rd, kd);
                ax = forced_list(ax, (-vx) * ff, m, rd, kd);
                if (IN3D) az = forced_list(az, (-vz) * ff, m, rd, kd);
            }
        }
    }
    if (ec.integrator == 0) {
        // Point.run1: v += a*t; pos += v*t   (old_a = a stays in acc)
        // products packed, additions scalar (a packed addition of a packed product would be contracted: wg_math.cuh CAUTION)
        const float2 dt2v = bc2(ec.dt);
        const float2 nvxy = add2_prod(make_float2(vx, vy), __fmul2_rn(make_float2(ax, ay), dt2v));        // v + a * t
        const float nvz = vz + az * ec.dt;
        st.vel(n, 0) = nvxy.x; st.vel(n, 1) = nvxy.y; st.vel(n, 2) = nvz;
        const float2 npxy = add2_prod(make_float2(st.pos(n, 0), st.pos(n, 1)), __fmul2_rn(nvxy, dt2v));   // pos + v * t
        st.pos(n, 0) = npxy.x; st.pos(n, 1) = npxy.y;
        st.pos(n, 2) = st.pos(n, 2) + nvz * ec.dt;
    } else {
        // Point.run2 (gym/optimized_engine.py:274-288): pos += v*t + (0.5*a)*t**2; then v += a*t  (cold path)
        float3 p = make_float3(st.pos(n, 0), st.pos(n, 1), st.pos(n, 2)), v = make_float3(vx, vy, vz);
        run2_cold(p, v, make_float3(ax, ay, az), ec.dt, ec.dt2);
        st.pos(n, 0) = p.x; st.pos(n, 1) = p.y; st.pos(n, 2) = p.z;
        st.vel(n, 0) = v.x; st.vel(n, 1) = v.y; st.vel(n, 2) = v.z;
    }
    st.acc(n, 0) = ax; st.acc(n, 1) = ay; st.acc(n, 2) = az;
    return hit;
}

// point_step for every mass; returns the force-phase contact mask.  Mass mode 3 (compile-time mass pattern) walks the
// masses by template recursion so that the unit-mass points get their float32 contact forces.
template <bool IN3D, int MM, class Topo, int N0, class BV, class Store>
__device__ __forceinline__ uint32_t point_steps_static(const BV& bv, const EnvConst& ec, Store& st) {
    if constexpr (N0 >= Topo::N) return 0u;
    else {
        const uint32_t c = point_step<IN3D, MM, (Topo::unit(N0) ? 1 : 0)>(bv, ec, st, N0) ? (1u << N0) : 0u;
        return c | point_steps_static<IN3D, MM, Topo, N0 + 1>(bv, ec, st);
    }
}
template <bool IN3D, int MM, class Topo, class BV, class Store>
__device__ __forceinline__ uint32_t all_point_steps(const Topo& topo, const BV& bv, const EnvConst& ec, Store& st) {
    if constexpr (MM == 3) return point_steps_static<IN3D, MM, Topo, 0>(bv, ec, st);
    else {
        uint32_t contact = 0;
        const int N = topo.n();
#pragma unroll
        for (int n = 0; n < N; n++)
            if (point_step<IN3D, MM>(bv, ec, st, n)) contact |= 1u << n;
        return contact;
    }
}

// PhysicsEnv._run_physics + Point.run1: one substep.  Returns the force-phase contact mask.
template <bool IN3D, int MM, class Topo, class BV, class Store>
__device__ __forceinline__ uint32_t run_physics(const Topo& topo, const BV& bv, const EnvConst& ec, Store& st) {
    const int N = topo.n(), S = topo.s(), M = topo.m();
    // Creature.run: zero, muscles, skeletons
#pragma unroll
    for (int n = 0; n < N; n++) { st.acc(n, 0) = 0.0f; st.acc(n, 1) = 0.0f; st.acc(n, 2) = 0.0f; }
#pragma unroll
    for (int sp = 0; sp < M; sp++) spring_run<MM>(topo, bv, st, sp, st.mx(sp), bv.fixed_mask);
#pragma unroll
    for (int sp = M; sp < S; sp++) spring_run<MM>(topo, bv, st, sp, bv.srest[sp], bv.fixed_mask);
    uint32_t contact = 0;
    contact = all_point_steps<IN3D, MM>(topo, bv, ec, st);
    return contact;
}

// NumPy float32 pairwise sum over n values produced by get(i)
template <class Get>
__device__ __forceinline__ float np_pairwise_sum(int n, Get get) {
    if (n < 8) {
        float r = -0.0f;
#pragma unroll
        for (int i = 0; i < n; i++) r = r + get(i);
        return r;
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = get(j);
    int i = 8;
    const int lim = n - (n % 8);
#pragma unroll
    for (; i < lim; i += 8) {
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = r[j] + get(i + j);
    }
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (; i < n; i++) res = res + get(i);
    return res;
}

// Reset of one mass: optional template restore, then the velocity jitter of PhysicsEnv.reset.
template <bool IN3D, class BV, class Store>
__device__ __forceinline__ void reset_mass(const BV& bv, const EnvConst& ec, Store& st, int n, int mode,
                                           const float* __restrict__ noise, int64_t E, int64_t e, uint32_t step_index) {
    if (mode == 2) {
#pragma unroll
        for (int c = 0; c < 3; c++) { st.pos(n, c) = bv.tmpl[n * 3 + c]; st.vel(n, c) = 0.0f; st.acc(n, c) = 0.0f; }
    }
    float z[3];
    if (noise) {
#pragma unroll
        for (int c = 0; c < 3; c++) z[c] = noise[(int64_t)(n * 3 + c) * E + e];
    } else {
        normal3(ec.seed_lo, ec.seed_hi, ec.env_offset + (uint32_t)e, step_index, (uint32_t)n, z);
#pragma unroll
        for (int c = 0; c < 3; c++) z[c] = ec.sigma * z[c];
    }
    st.vel(n, 0) = st.vel(n, 0) + z[0];
    st.vel(n, 1) = st.vel(n, 1) + z[1];
    if (IN3D) st.vel(n, 2) = st.vel(n, 2) + z[2];
}

// Template reset + jitter (PhysicsEnv.reset, optimized_env.py:53-68; make_env :273-294)
template <bool IN3D, class Topo, class BV, class Store>
__device__ __forceinline__ void apply_reset(const Topo& topo, const BV& bv, const EnvConst& ec, Store& st,
                                            int mode, const float* __restrict__ noise, int64_t E, int64_t e,
                                            uint32_t step_index) {
    const int N = topo.n(), M = topo.m();
    if (mode == 2) {
#pragma unroll
        for (int m = 0; m < M; m++) st.mx(m) = bv.srest[m];
    }
#pragma unroll
    for (int n = 0; n < N; n++) reset_mass<IN3D>(bv, ec, st, n, mode, noise, E, e, step_index);
}

// Creature.getstat with PhysicsEnv's defaults; emit(k, value) receives the D entries in order.
template <bool IN3D, class Topo, class Store, class Emit>
__device__ __forceinline__ void get_obs(const Topo& topo, const ConstDiv& nd, Store& st, Emit emit) {
    const int N = topo.n(), M = topo.m();
    constexpr int d = IN3D ? 3 : 2;
    float mid[3] = { 0.0f, 0.0f, 0.0f };
    float2 mxy = make_float2(0.0f, 0.0f);                    // np.mean(axis=0): sequential sums, x / y packed
#pragma unroll
    for (int n = 0; n < N; n++) { mxy = __fadd2_rn(mxy, make_float2(st.pos(n, 0), st.pos(n, 1))); mid[2] = mid[2] + st.pos(n, 2); }
    mid[0] = div_const(mxy.x, nd.m, nd.r, nd.kind);
    mid[1] = div_const(mxy.y, nd.m, nd.r, nd.kind);
    mid[2] = div_const(mid[2], nd.m, nd.r, nd.kind);
    const float2 nmid = make_float2(-mid[0], -mid[1]);
    int k = 0;
#pragma unroll
    for (int n = 0; n < N; n++) {
        const float2 rel = __fadd2_rn(make_float2(st.pos(n, 0), st.pos(n, 1)), nmid);        // pos - mid
        emit(k++, rel.x); emit(k++, rel.y);
#pragma unroll
        for (int c = 2; c < d; c++) emit(k++, st.pos(n, c) - mid[c]);
#pragma unroll
        for (int c = 0; c < d; c++) emit(k++, st.vel(n, c));
#pragma unroll
        for (int c = 0; c < d; c++) emit(k++, st.acc(n, c));
    }
#pragma unroll
    for (int m = 0; m < M; m++) emit(k++, st.mx(m));
}

}  // namespace wg
