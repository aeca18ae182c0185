// wg_kernels_part.cuh -- K1 for larger bodies: P adjacent lanes share one env ("mass partition").
//
// A body with N >= 8 masses costs ~750 bytes of per-env state and tens of thousands of instructions
// per env-step; with one thread per env a B200 SM holds too few envs to hide latency, and the fully
// unrolled specialisation does not fit the instruction caches.  Here the masses of a body are split
// into P parts (host side: breadth-first order of the spring graph cut into P chunks, so connected
// pieces stay together) and lane `part` of an env
//   * evaluates, in the reference's list order, every spring that touches one of its masses and
//     accumulates only into ITS masses' accelerations (a spring that crosses two parts is evaluated by
//     both owners -- same inputs, same operations, same bits);
//   * applies the environment forces and integrates its own masses.
// Per-mass accumulation order is therefore exactly the reference's, so the result is bit-identical to
// the one-thread-per-env kernels, while an env exposes P-fold parallelism.  The state of the block's
// envs lives in a shared-memory tile [row][env] (odd pitch) for the whole step: one coalesced read and
// one coalesced write of HBM per env-step, rolled loops (small code), two __syncwarp per substep.
#pragma once
#include "wg_kernels.cuh"

namespace wg {

constexpr int kMaxPart = 8;

struct PartTables {
    uint8_t spring[kMaxPart][kMaxSpring];   // springs touching part p, ascending (= list order)
    uint8_t mass[kMaxPart][kMaxMass];       // masses owned by part p
    uint8_t n_spring[kMaxPart], n_mass[kMaxPart];
    uint32_t own_mask[kMaxPart];
};

struct PartArgs {
    StepArgs<kMaxMass, kMaxSpring> A;
    PartTables pt;
};

template <bool IN3D, int P, bool ROWMAJOR, int MM>
__global__ void __launch_bounds__(kBlock)
step_part_kernel(const __grid_constant__ PartArgs PA) {
    const auto& A = PA.A;
    extern __shared__ float smem[];
    // lanes of one warp work on different springs and masses: per-spring / per-mass constants would be
    // divergent constant-bank reads (serialised per distinct address), so the tables are staged once per
    // block in shared memory
    __shared__ BodyVals<kMaxMass, kMaxSpring> bv;
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&A.bv);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&bv);
        for (int i = threadIdx.x; i < (int)(sizeof(bv) / 4); i += kBlock) dst[i] = src[i];
    }
    constexpr int EB = kBlock / P;                 // envs per block
    constexpr int PITCH = EB + 1;
    constexpr int d = IN3D ? 3 : 2;
    const int N = A.bv.n_mass, S = A.bv.n_spring, M = A.bv.n_muscle;
    const int D = 3 * d * N + M;
    __shared__ uint16_t obs_src[3 * 3 * kMaxMass + kMaxSpring], obs_cen[3 * 3 * kMaxMass + kMaxSpring];
    for (int k = threadIdx.x; k < D; k += blockDim.x) {                // Creature.getstat's entry order
        int src, cen = 0;
        if (k < 3 * d * N) {
            const int n = k / (3 * d), rr = k - n * 3 * d, sec = rr / d, c = rr - sec * d;
            src = sec * 3 * N + n * 3 + c;
            if (sec == 0) cen = 9 * N + M + 2 * N + c;
        } else {
            src = 9 * N + (k - 3 * d * N);
        }
        obs_src[k] = (uint16_t)src; obs_cen[k] = (uint16_t)cen;
    }
    const int ROWS = 11 * N + M + 3;               // pos, vel, acc, mx, ys, speeds, centroid
    RuntimeTopo topo{ N, S, M, bv.si, bv.sj };
    const int tid = threadIdx.x, lane = tid & 31;
    const int el = tid / P, part = tid % P;        // env within the block, lane's part
    const int64_t E = A.E;
    const int64_t e0 = (int64_t)blockIdx.x * EB;
    const int64_t e = e0 + el;
    const bool valid = e < E;
    const int64_t rem = E - e0;
    const int nvalid = rem < EB ? (int)rem : EB;
    SmemStore st{ smem + el, PITCH, N };
    // per-part tables in shared memory (lanes of a warp read different parts)
    uint8_t* tab = reinterpret_cast<uint8_t*>(smem + ROWS * PITCH);
    uint8_t* my_springs = tab + part * kMaxSpring;
    uint8_t* my_masses = tab + P * kMaxSpring + part * kMaxMass;
    for (int i = tid; i < P * kMaxSpring; i += kBlock) tab[i] = PA.pt.spring[i / kMaxSpring][i % kMaxSpring];
    for (int i = tid; i < P * kMaxMass; i += kBlock) tab[P * kMaxSpring + i] = PA.pt.mass[i / kMaxMass][i % kMaxMass];
    const int n_my_springs = PA.pt.n_spring[part], n_my_masses = PA.pt.n_mass[part];
    const uint32_t skip = A.bv.fixed_mask | ~PA.pt.own_mask[part];
    __syncthreads();                               // staged tables visible

    // L2 prefetch for a block dispatched `pf_dist` blocks later: every row segment of that block is one
    // 128-byte-class span, so each thread asks for one line (pos/vel rows, then muscle rows)
    if (A.pf_dist > 0) {
        const int64_t pe0 = ((int64_t)blockIdx.x + A.pf_dist) * EB;
        if (pe0 + EB <= E) {
            for (int r = tid; r < 6 * N + M; r += kBlock) {
                const float* ptr = r < 3 * N ? A.pos + (int64_t)r * E + pe0
                                 : r < 6 * N ? A.vel + (int64_t)(r - 3 * N) * E + pe0 : A.mx + (int64_t)(r - 6 * N) * E + pe0;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
            }
        }
    }
    // ---- single HBM read: the block's EB envs of every state row, coalesced ----
    // cp.async (global -> shared without a register round trip): every thread has all of its elements in flight at
    // once; the plain load-then-store loop serialised on DRAM latency (35 % of the kernel's stall samples at k_sub 1)
    for (int idx = tid; idx < 6 * N * EB; idx += kBlock) {
        const int r = idx / EB, c = idx - r * EB;
        if (c < nvalid) {
            const float* src = r < 3 * N ? A.pos + (int64_t)r * E + e0 + c : A.vel + (int64_t)(r - 3 * N) * E + e0 + c;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem + r * PITCH + c)), "l"(src) : "memory");
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    {   // Creature.act while loading the muscle lengths
        const int na = A.act_dim < M ? A.act_dim : M;
        for (int idx = tid; idx < M * EB; idx += kBlock) {
            const int m = idx / EB, c = idx - m * EB;
            if (c < nvalid) {
                float x = A.mx[(int64_t)m * E + e0 + c];
                if (m < na) {
                    x = x + (A.act_layout ? A.action[(int64_t)m * E + e0 + c] : A.action[(e0 + c) * A.act_dim + m]);
                    if (bv.mlo[m] > x) x = bv.mlo[m];
                    if (bv.mhi[m] < x) x = bv.mhi[m];
                }
                smem[(9 * N + m) * PITCH + c] = x;
            }
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    uint32_t cpre = 0;
    for (int k = 0; k < A.ec.k_sub; k++) {
        if (valid) {
            for (int q = 0; q < n_my_masses; q++) { const int n = my_masses[q]; st.acc(n, 0) = 0.0f; st.acc(n, 1) = 0.0f; st.acc(n, 2) = 0.0f; }
            for (int q = 0; q < n_my_springs; q++) {
                const int sp = my_springs[q];
                spring_run<MM, true>(topo, bv, st, sp, sp < M ? st.mx(sp) : bv.srest[sp], skip);
            }
        }
        __syncwarp();                              // everyone has read the old positions / velocities
        cpre = 0;
        if (valid)
            for (int q = 0; q < n_my_masses; q++) { const int n = my_masses[q]; if (point_step<IN3D, MM>(bv, A.ec, st, n)) cpre |= 1u << n; }
        __syncwarp();                              // new positions / velocities visible to the env's other lanes
    }
    // ---- reward / done / info: speeds in parallel, the reduction on the env's first lane ----
    if (valid)
        for (int q = 0; q < n_my_masses; q++) {
            const int n = my_masses[q];
            st.scratch(M, n) = st.pos(n, 1);
            st.scratch(M, N + n) = np_norm3(st.vel(n, 0), st.vel(n, 1), st.vel(n, 2));
        }
#pragma unroll
    for (int off = 1; off < P; off <<= 1) cpre |= __shfl_xor_sync(0xffffffffu, cpre, off);
    __syncwarp();
    int do_reset = 0;
    if (valid && part == 0) {
        const int32_t sn = A.steps[e] + 1;
        EpiOut o;
        epilogue_reduce(N, bv, A.ec, st, sn, A.energy != nullptr, A.centroid != nullptr, A.truncated != nullptr,
                        [&](int i) -> float& { return st.scratch(M, i); },
                        [&](int i) -> float& { return st.scratch(M, N + i); }, o);
        if (A.reward) A.reward[e] = o.reward;
        if (A.done) A.done[e] = (uint8_t)o.done;
        if (A.truncated) A.truncated[e] = (uint8_t)o.trunc;
        if (A.contact_pre) A.contact_pre[e] = cpre;
        if (A.contact_post) A.contact_post[e] = o.cpost;
        if (A.energy) A.energy[e] = o.energy;
        if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
        if (A.ep_ret) {
            const float r = A.ep_ret[e] + o.reward;
            if (o.done) account_episode(A, E, e, r, sn);
            A.ep_ret[e] = (o.done && A.ec.auto_reset) ? 0.0f : r;
        }
        if (o.done && A.final_obs) store_final_obs<IN3D>(topo, A, st, E, e, ROWMAJOR);   // the env's whole state is in st
        do_reset = (o.done && A.ec.auto_reset) ? 1 : 0;
        A.steps[e] = do_reset ? 0 : sn;
        if (do_reset && A.ec.auto_reset == 2)
            for (int m = 0; m < M; m++) st.mx(m) = bv.srest[m];
    }
    do_reset = __shfl_sync(0xffffffffu, do_reset, lane - part);
    if (valid && do_reset) {                       // each lane resets its own masses (Philox keyed per mass)
        const uint32_t si = step_index_of(A);
        for (int q = 0; q < n_my_masses; q++) reset_mass<IN3D>(bv, A.ec, st, my_masses[q], A.ec.auto_reset, A.noise, E, e, si);
    }
    __syncwarp();
    if (valid && part == 0 && A.obs && ROWMAJOR) {  // getstat centroid: sequential sum over the masses, then / N
        float mid[3] = { 0.0f, 0.0f, 0.0f };
        for (int n = 0; n < N; n++) { mid[0] = mid[0] + st.pos(n, 0); mid[1] = mid[1] + st.pos(n, 1); mid[2] = mid[2] + st.pos(n, 2); }
        const ConstDiv nd = bv.ndiv;
        st.scratch(M, 2 * N + 0) = div_const(mid[0], nd.m, nd.r, nd.kind);
        st.scratch(M, 2 * N + 1) = div_const(mid[1], nd.m, nd.r, nd.kind);
        st.scratch(M, 2 * N + 2) = div_const(mid[2], nd.m, nd.r, nd.kind);
    }
    if (valid && part == 0 && A.obs && !ROWMAJOR)
        get_obs<IN3D>(topo, bv.ndiv, st, [&](int k, float v) { A.obs[(int64_t)k * E + e] = v; });
    __syncthreads();
    // ---- single HBM write of the state, coalesced ----
    for (int idx = tid; idx < 3 * N * EB; idx += kBlock) {
        const int r = idx / EB, c = idx - r * EB;
        if (c < nvalid) {
            A.pos[(int64_t)r * E + e0 + c] = smem[r * PITCH + c];
            A.vel[(int64_t)r * E + e0 + c] = smem[(3 * N + r) * PITCH + c];
            if (A.old_a) A.old_a[(int64_t)r * E + e0 + c] = smem[(6 * N + r) * PITCH + c];
        }
    }
    for (int idx = tid; idx < M * EB; idx += kBlock) {
        const int m = idx / EB, c = idx - m * EB;
        if (c < nvalid) A.mx[(int64_t)m * E + e0 + c] = smem[(9 * N + m) * PITCH + c];
    }
    if (ROWMAJOR && A.obs) {                        // whole warps stream observation rows out of the tile
        const int warp = tid >> 5;
        // entry k of an observation row = tile row obs_src[k] (minus the centroid row obs_cen[k] for positions)
        for (int r = warp; r < nvalid; r += kBlock / 32) {
            const float* col = smem + r;
            float* out = A.obs + (e0 + r) * D;
            for (int k = lane; k < D; k += 32) {
                float v = col[obs_src[k] * PITCH];
                const int cr = obs_cen[k];
                if (cr) v = v - col[cr * PITCH];
                out[k] = v;
            }
        }
    }
}

// =====================================================================================================================
// Bodies made of P identical, disconnected units (BASELINE config 4's enlarged morphology is 4 Balance units; the
// compat Environment steps a *list* of creatures the same way): lane u of an env owns unit u and runs the unit's
// register-resident physics -- the code of the one-unit specialisation, UnitTopo's compile-time spring table, the
// unit's constants in the constant bank -- for all k_sub substeps without touching memory; only the env-level tail
// (reward / done over all masses in NumPy's summation order, auto-reset, observation) goes through the shared tile.
// Global mass U::N*u + n is unit u's mass n; global spring U::M*u + s (s < U::M, the muscles) or
// M + (U::S-U::M)*u + (s-U::M) (the bones) is its spring s: the order in which a mass accumulates its springs is the
// reference's (all muscles, then all bones, each in list order), so the bits are those of every other kernel.
// =====================================================================================================================
template <class U, int UMM>
struct UnitsArgs {
    PartArgs P;                        // env-level tables (pt unused)
    BodyVals<U::N, U::S> ubv;          // the unit's constants (identical for every unit: checked on the host)
    float link_k, link_damp, link_rest;   // LINKED units: the bone joining unit u's mass LA to unit u+1's mass LB
};

// One endpoint's share of Skeleton.run (gym/optimized_walker.py:84-106) for a bone whose other endpoint lives in a
// neighbouring lane: p1 = (pi, vi), p2 = (pj, vj) exactly as spring_run reads them; SIDE 0 accumulates p1's two
// increments (F / m, (-D) / m), SIDE 1 p2's ((-F) / m, D / m) into acc (the mass with local index n of this unit).
// Both owners evaluate the same operations on the same inputs, so each gets the bits the one-thread kernel computes.
template <int MM, int SIDE, class U, class BV>
__device__ __forceinline__ void link_half(const BV& bv, int n, const float (&pi)[3], const float (&vi)[3],
                                          const float (&pj)[3], const float (&vj)[3], float k, float damp, float rest,
                                          float (&acc)[3]) {
    // the same operations as spring_run, x / y halves packed (wg_math.cuh)
    V3 d = v3_sub(v3(pj[0], pj[1], pj[2]), v3(pi[0], pi[1], pi[2]));
    const float L = unit_dir(d);
    const float dx = L - rest;
    const float fs = (-dx) * k;
    const V3 F = v3_scale(d, fs);
    const float dk = np_dot3(v3_sub(v3(vi[0], vi[1], vi[2]), v3(vj[0], vj[1], vj[2])), d);
    const float cd = dk * damp;
    const V3 D = v3_scale(d, cd);
    bool unit = (MM == 0);
    if constexpr (MM == 3) unit = U::unit(n);
    const V3 f1 = SIDE == 0 ? F : v3_neg(F), f2 = SIDE == 0 ? v3_neg(D) : D;
    float2 axy = make_float2(acc[0], acc[1]);
    if (unit) {                                         // raw packed products: scalar additions (wg_math.cuh CAUTION)
        axy = add2_prod(add2_prod(axy, f1.xy), f2.xy);
        acc[2] = (acc[2] + f1.z) + f2.z;
    } else {
        const float m = bv.mass_f[n], r = bv.mass_r[n];
        const float2 q1 = div_smallint2(f1.xy, m, r), q2 = div_smallint2(f2.xy, m, r), qz = div_smallint2(make_float2(f1.z, f2.z), m, r);
        axy = __fadd2_rn(__fadd2_rn(axy, q1), q2);
        acc[2] = (acc[2] + qz.x) + qz.y;
    }
    acc[0] = axy.x; acc[1] = axy.y;
}

// positions of every mass of an env in the per-env scratch (the env-level tail reads them in NumPy's order)
struct ScratchPos {
    float* p;                                         // [3N] for this env
    __device__ __forceinline__ float& pos(int n, int c) { return p[n * 3 + c]; }
};
// a unit's registers addressed by GLOBAL mass / muscle index (reset_mass and friends take global indices)
template <class U>
struct UnitView {
    RegStore<U::N, U::M>& rs; int m0, g0;
    __device__ __forceinline__ float& pos(int n, int c) { return rs.p_[n - m0][c]; }
    __device__ __forceinline__ float& vel(int n, int c) { return rs.v_[n - m0][c]; }
    __device__ __forceinline__ float& acc(int n, int c) { return rs.a_[n - m0][c]; }
    __device__ __forceinline__ float& mx(int m) { return rs.mx_[m - g0]; }
};

// KB threads per CTA = KB / P envs.  Nothing of the state goes through shared memory: lane u loads unit u's rows
// straight into registers (a warp request = P rows x 32/P consecutive envs: whole 32-byte sectors), steps it, and
// stores it back; shared memory only carries the env-level scratch (heights, speeds, positions, centroid) and the
// row-major observation tile, which leaves with one TMA bulk store per warp.
#ifndef WG_UNITS_THREADS_PER_SM
#define WG_UNITS_THREADS_PER_SM 768
#endif
// LA >= 0: LINKED units -- one connected body.  After every unit's own bones the skeleton list holds P-1 link bones,
// link u joining unit u's mass LA (its p1) to unit u+1's mass LB (its p2), all with the same constants.  Each substep,
// after the unit's springs and before the integration, a lane fetches its neighbours' link endpoints with warp
// shuffles and evaluates its side of the left link (it owns p2 = its LB) and of the right link (it owns p1 = its LA):
// per-mass accumulation order is the list's (unit springs, then link u-1, then link u).
template <class U, bool IN3D, int P, bool ROWMAJOR, int MM, int KB, int LA = -1, int LB = -1>
__global__ void __launch_bounds__(KB, WG_UNITS_THREADS_PER_SM / KB)
step_units_kernel(const __grid_constant__ UnitsArgs<U, MM> UA) {
    const auto& A = UA.P.A;
    constexpr int N = P * U::N, M = P * U::M, d = IN3D ? 3 : 2, D = 3 * d * N + M;
    constexpr int EB = KB / P, EW = 32 / P;           // envs per block / per warp
    constexpr int SCR = 5 * N + 4;                    // per env: ys[N], speeds[N], pos[3N], centroid[3], pad
    constexpr bool OBS_BULK = ROWMAJOR && ((EW * D * 4) % 16 == 0);
    extern __shared__ __align__(128) float smem[];
    float* const otile = smem + ((EB * SCR + 31) / 32) * 32;          // [EB][D], 128-byte aligned
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int el = tid / P, u = tid % P;
    const int m0 = U::N * u, g0 = U::M * u;
    const int64_t E = A.E;
    const int64_t e0 = (int64_t)blockIdx.x * EB;
    const int64_t e = e0 + el;
    const bool valid = e < E;
    const uint32_t vmask = __ballot_sync(0xffffffffu, valid);     // the warp's valid lanes (whole envs): shuffle mask of the links
    float* const scr = smem + el * SCR;
    RegStore<U::N, U::M> rs;
    uint32_t cpre = 0;
    if (valid) {
        // ---- single HBM read: this lane's unit, coalesced per (row, 32/P envs) ----
#pragma unroll
        for (int n = 0; n < U::N; n++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                rs.p_[n][c] = A.pos[(int64_t)((m0 + n) * 3 + c) * E + e];
                rs.v_[n][c] = A.vel[(int64_t)((m0 + n) * 3 + c) * E + e];
                rs.a_[n][c] = 0.0f;
            }
        const int na = A.act_dim < M ? A.act_dim : M;
#pragma unroll
        for (int m = 0; m < U::M; m++) {                // Creature.act on this unit's muscles
            float x = A.mx[(int64_t)(g0 + m) * E + e];
            if (g0 + m < na) {
                x = x + (A.act_layout ? A.action[(int64_t)(g0 + m) * E + e] : A.action[e * A.act_dim + g0 + m]);
                if (UA.ubv.mlo[m] > x) x = UA.ubv.mlo[m];
                if (UA.ubv.mhi[m] < x) x = UA.ubv.mhi[m];
            }
            rs.mx(m) = x;
        }
        const U utopo;
        uint32_t cu = 0;
        if constexpr (LA < 0) {
            for (int k = 0; k < A.ec.k_sub; k++) cu = run_physics<IN3D, MM>(utopo, UA.ubv, A.ec, rs);
        } else {
            for (int k = 0; k < A.ec.k_sub; k++) {
                // Creature.run: zero, muscles, this unit's bones (run_physics up to the integration)
#pragma unroll
                for (int n = 0; n < U::N; n++) { rs.a_[n][0] = 0.0f; rs.a_[n][1] = 0.0f; rs.a_[n][2] = 0.0f; }
#pragma unroll
                for (int sp = 0; sp < U::M; sp++) spring_run<MM>(utopo, UA.ubv, rs, sp, rs.mx(sp), 0u);
#pragma unroll
                for (int sp = U::M; sp < U::S; sp++) spring_run<MM>(utopo, UA.ubv, rs, sp, UA.ubv.srest[sp], 0u);
                // the link bones: neighbours' endpoints over shuffles (pre-integration state of this substep)
                float lp[3], lv[3], rp[3], rv[3];
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    lp[c] = __shfl_up_sync(vmask, rs.p_[LA][c], 1);          // unit u-1's mass LA
                    lv[c] = __shfl_up_sync(vmask, rs.v_[LA][c], 1);
                    rp[c] = __shfl_down_sync(vmask, rs.p_[LB][c], 1);        // unit u+1's mass LB
                    rv[c] = __shfl_down_sync(vmask, rs.v_[LB][c], 1);
                }
                if (u > 0) link_half<MM, 1, U>(UA.ubv, LB, lp, lv, rs.p_[LB], rs.v_[LB], UA.link_k, UA.link_damp, UA.link_rest, rs.a_[LB]);
                if (u + 1 < P) link_half<MM, 0, U>(UA.ubv, LA, rs.p_[LA], rs.v_[LA], rp, rv, UA.link_k, UA.link_damp, UA.link_rest, rs.a_[LA]);
                cu = all_point_steps<IN3D, MM>(utopo, UA.ubv, A.ec, rs);
            }
        }
        cpre = cu << m0;
        // ---- env-level scratch: heights, speeds, positions ----
#pragma unroll
        for (int n = 0; n < U::N; n++) {
            scr[m0 + n] = rs.p_[n][1];
            scr[N + m0 + n] = np_norm3(rs.v_[n][0], rs.v_[n][1], rs.v_[n][2]);
#pragma unroll
            for (int c = 0; c < 3; c++) scr[2 * N + (m0 + n) * 3 + c] = rs.p_[n][c];
        }
    }
#pragma unroll
    for (int off = 1; off < P; off <<= 1) cpre |= __shfl_xor_sync(0xffffffffu, cpre, off);
    __syncwarp();
    int do_reset = 0;
    if (valid && u == 0) {                              // reward / done / info on the env's first lane
        const int32_t sn = A.steps[e] + 1;
        EpiOut o;
        ScratchPos sp{ scr + 2 * N };
        epilogue_reduce(N, A.bv, A.ec, sp, sn, A.energy != nullptr, A.centroid != nullptr, A.truncated != nullptr,
                        [&](int i) -> float& { return scr[i]; }, [&](int i) -> float& { return scr[N + i]; }, o);
        if (A.reward) A.reward[e] = o.reward;
        if (A.done) A.done[e] = (uint8_t)o.done;
        if (A.truncated) A.truncated[e] = (uint8_t)o.trunc;
        if (A.contact_pre) A.contact_pre[e] = cpre;
        if (A.contact_post) A.contact_post[e] = o.cpost;
        if (A.energy) A.energy[e] = o.energy;
        if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
        if (A.ep_ret) {
            const float r = A.ep_ret[e] + o.reward;
            if (o.done) account_episode(A, E, e, r, sn);
            A.ep_ret[e] = (o.done && A.ec.auto_reset) ? 0.0f : r;
        }
        do_reset = (o.done ? 2 : 0) | ((o.done && A.ec.auto_reset) ? 1 : 0);
        A.steps[e] = (do_reset & 1) ? 0 : sn;
    }
    (void)vmask;
    do_reset = __shfl_sync(0xffffffffu, do_reset, lane - u);
    const bool ended = (do_reset & 2) != 0;
    do_reset &= 1;
    // this lane's entries of an observation row: masses m0 .. m0+U::N-1 and muscles g0 .. g0+U::M-1 (mid: the centroid)
    auto emit_unit = [&](const float (&mid)[3], auto put) {
#pragma unroll
        for (int n = 0; n < U::N; n++) {
            const int k0 = (m0 + n) * 3 * d;
#pragma unroll
            for (int c = 0; c < d; c++) {
                put(k0 + c, rs.p_[n][c] - mid[c]);
                put(k0 + d + c, rs.v_[n][c]);
                put(k0 + 2 * d + c, rs.a_[n][c]);
            }
        }
#pragma unroll
        for (int m = 0; m < U::M; m++) put(3 * d * N + g0 + m, rs.mx(m));
    };
    auto centroid = [&]() {                             // getstat centroid: sequential sum over all masses, then / N
        float mid[3] = { 0.0f, 0.0f, 0.0f };
#pragma unroll
        for (int n = 0; n < N; n++) { mid[0] = mid[0] + scr[2 * N + n * 3]; mid[1] = mid[1] + scr[2 * N + n * 3 + 1]; mid[2] = mid[2] + scr[2 * N + n * 3 + 2]; }
        const ConstDiv nd = A.bv.ndiv;
        scr[5 * N + 0] = div_const(mid[0], nd.m, nd.r, nd.kind);
        scr[5 * N + 1] = div_const(mid[1], nd.m, nd.r, nd.kind);
        scr[5 * N + 2] = div_const(mid[2], nd.m, nd.r, nd.kind);
    };
    if (A.final_obs) {                                  // the final row from the pre-reset state: each lane its own part
        if (valid && ended && u == 0) centroid();
        __syncwarp();
        if (valid && ended) {
            const float mid[3] = { scr[5 * N + 0], scr[5 * N + 1], scr[5 * N + 2] };
            float* const fo = A.final_obs;
            emit_unit(mid, [&](int k, float v) { if (ROWMAJOR) fo[e * D + k] = v; else fo[(int64_t)k * E + e] = v; });
        }
        __syncwarp();                                   // the centroid is read before the reset below moves the positions
    }
    if (valid && do_reset) {                            // each lane resets its own unit (Philox keyed per global mass)
        const uint32_t si = step_index_of(A);
        UnitView<U> view{ rs, m0, g0 };
        if (A.ec.auto_reset == 2) {
#pragma unroll
            for (int m = 0; m < U::M; m++) rs.mx(m) = UA.ubv.srest[m];
        }
#pragma unroll
        for (int n = 0; n < U::N; n++) reset_mass<IN3D>(A.bv, A.ec, view, m0 + n, A.ec.auto_reset, A.noise, E, e, si);
#pragma unroll
        for (int n = 0; n < U::N; n++)
#pragma unroll
            for (int c = 0; c < 3; c++) scr[2 * N + (m0 + n) * 3 + c] = rs.p_[n][c];
    }
    __syncwarp();
    if (valid && A.obs && u == 0) centroid();
    __syncwarp();
    if (valid && A.obs) {
        const float mid[3] = { scr[5 * N + 0], scr[5 * N + 1], scr[5 * N + 2] };
        emit_unit(mid, [&](int k, float v) {
            if (ROWMAJOR) { if (OBS_BULK) otile[el * D + k] = v; else A.obs[e * D + k] = v; }
            else A.obs[(int64_t)k * E + e] = v;
        });
    }
    if (valid) {
        // ---- single HBM write of the state ----
#pragma unroll
        for (int n = 0; n < U::N; n++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                A.pos[(int64_t)((m0 + n) * 3 + c) * E + e] = rs.p_[n][c];
                A.vel[(int64_t)((m0 + n) * 3 + c) * E + e] = rs.v_[n][c];
                if (A.old_a) A.old_a[(int64_t)((m0 + n) * 3 + c) * E + e] = rs.a_[n][c];
            }
#pragma unroll
        for (int m = 0; m < U::M; m++) A.mx[(int64_t)(g0 + m) * E + e] = rs.mx(m);
    }
    if (OBS_BULK && A.obs) {
        // the warp's EW observation rows are one contiguous span of global memory: one TMA bulk store
        __syncwarp();
        const int64_t ew = e0 + (int64_t)warp * EW;
        const int64_t remw = E - ew;
        if (remw > 0) {
            float* wt = otile + warp * EW * D;
            if (remw >= EW && ((reinterpret_cast<uintptr_t>(A.obs) & 15u) == 0) && ((ew * D * 4) % 16 == 0)) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { bulk_s2g(A.obs + ew * D, wt, (uint32_t)(EW * D * 4)); bulk_commit(); bulk_wait_read0(); }
            } else {
                const int nvw = remw < EW ? (int)remw : EW;
                for (int idx = lane; idx < nvw * D; idx += 32) A.obs[ew * D + idx] = wt[idx];
            }
        }
    }
}

}  // namespace wg
