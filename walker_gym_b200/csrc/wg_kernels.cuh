// wg_kernels.cuh -- the fused step kernel (K1), the reset kernel (K2) and the
// episode-statistics reduction (K3).
//
// K1 performs, in ONE launch and with ONE read and ONE write of the state per
// env step: Creature.act, k_sub x (_run_physics + Point.run1), steps += 1,
// reward, done, info, episode statistics, auto-reset and the observation.
// HBM-bound by design (sparse per-env stencil, no tensor cores): all global
// accesses are coalesced SoA vectors of EPT consecutive envs per thread; the
// row-major [E][D] observation is transposed through a padded shared-memory
// tile and written back as fully coalesced rows.
#pragma once
#include "wg_physics.cuh"

namespace wg {

#ifndef WG_BLOCK
#define WG_BLOCK 128
#endif
#ifndef WG_MIN_BLOCKS
#define WG_MIN_BLOCKS 6
#endif
constexpr int kBlock = WG_BLOCK;

template <int MAXN, int MAXS>
struct StepArgs {
    BodyVals<MAXN, MAXS> bv;
    EnvConst ec;
    float* pos; float* vel; float* old_a; float* mx; int32_t* steps;
    const float* action; float* obs; float* reward; uint8_t* done;
    uint32_t* contact_pre; uint32_t* contact_post; float* energy; float* centroid;
    float* ep_ret; float* fin_stats; const float* noise;
    const uint32_t* step_counter;
    float* state_packed;
    int64_t E;
    int32_t pf_dist;          // packed kernel: L2 prefetch distance in tiles (0 = off)
    int32_t act_dim, act_layout;
    float* nf_stats;          // optional [2][E]: count and length sum of finished episodes whose return is not finite
};

// NF (template flag of the kernel families whose keep-mode code must stay exactly what it was, see
// step_static_packed_kernel): false compiles the non-finite handling out -- the instance then ignores
// ec.end_nonfinite and nf_stats, and the host launches it only when both are off.

// ---- TMA 1-D bulk store helpers (shared memory -> global), used for the observation rows ----------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__host__ __device__ constexpr int gcd_c(int a, int b) { return b == 0 ? a : gcd_c(b, a % b); }

// packed state layout [tile][k/4][128][4] (include/walker_gym_b200.h)
__host__ __device__ __forceinline__ int64_t packed_index(int64_t e, int k, int r4) {
    return (((e >> 7) * r4 + (k >> 2)) << 9) + ((e & 127) << 2) + (k & 3);
}

// Philox counter word of this launch: the by-value step index plus the optional device-side counter
template <class Args>
__device__ __forceinline__ uint32_t step_index_of(const Args& A) {
    return A.ec.step_index + (A.step_counter ? __ldg(A.step_counter) : 0u);
}

// ---- vector access of EPT consecutive envs --------------------------------------
template <int EPT> struct Vec;
template <> struct Vec<1> { using F = float;  using I = int32_t; using U = uint32_t; using B = uint8_t; };
template <> struct Vec<2> { using F = float2; using I = int2;    using U = uint2;    using B = uchar2; };
template <> struct Vec<4> { using F = float4; using I = int4;    using U = uint4;    using B = uchar4; };

template <int EPT, class T, class V>
__device__ __forceinline__ void ld_vec(const T* p, T (&out)[EPT]) {
    V v = *reinterpret_cast<const V*>(p);
    const T* s = reinterpret_cast<const T*>(&v);
#pragma unroll
    for (int j = 0; j < EPT; j++) out[j] = s[j];
}
template <int EPT, class T, class V>
__device__ __forceinline__ void st_vec(T* p, const T (&in)[EPT]) {
    V v;
    T* s = reinterpret_cast<T*>(&v);
#pragma unroll
    for (int j = 0; j < EPT; j++) s[j] = in[j];
    *reinterpret_cast<V*>(p) = v;
}
#define WG_LDF(ptr, arr) ld_vec<EPT, float, typename Vec<EPT>::F>(ptr, arr)
#define WG_STF(ptr, arr) st_vec<EPT, float, typename Vec<EPT>::F>(ptr, arr)

// ---- per-env epilogue: reward, done, info, stats, auto-reset (shared by both kernels) ----
struct EpiOut { float reward; uint32_t cpost; int done; float energy; float cen[3]; };

// reward, done and info from the per-mass heights ys(i) and speeds sp(i) (already filled in)
template <bool NF = true, class BV, class Store, class YS, class SP>
__device__ __forceinline__ void epilogue_reduce(int N, const BV& bv, const EnvConst& ec, Store& st, int32_t steps_now,
                                                bool want_energy, bool want_centroid, YS ys, SP sp, EpiOut& o) {
    uint32_t cpost = 0; int ncon = 0;
#pragma unroll
    for (int n = 0; n < N; n++)
        if (ys(n) - ec.ground < 0.0f) { cpost |= 1u << n; ncon++; }
    const ConstDiv nd = bv.ndiv;
    const float cy = div_const(np_pairwise_sum(N, [&](int i) { return ys(i); }), nd.m, nd.r, nd.kind);
    const float avgv = div_const(np_pairwise_sum(N, [&](int i) { return sp(i); }), nd.m, nd.r, nd.kind);
    const float vpen = (-avgv) * 0.1f;
    const float cpen = -0.5f * (float)ncon;
    o.reward = (cy + vpen) + cpen;
    o.cpost = cpost;
    int dn = 0;                                                  // _is_done (:207-230)
    if (steps_now >= ec.max_steps) dn = 1;
    else if (cy < ec.fall_thresh) dn = 1;
    else {
        bool all_stopped = true;
#pragma unroll
        for (int n = 0; n < N; n++) all_stopped = all_stopped && (sp(n) < 0.1f);
        if (all_stopped && steps_now > 100) dn = 1;
    }
    // opt-in (wg_params.end_nonfinite): an env whose state overflowed ends its episode.  The reward sums every mass
    // height and speed, so an inf / NaN anywhere in the state reaches it in the same step.
    if (NF && ec.end_nonfinite && !is_finite(o.reward)) dn = 1;
    o.done = dn;
    if (want_energy) {                                           // _calculate_energy (:240-248)
        const float ke = np_pairwise_sum(N, [&](int i) { return bv.mass_f[i] * (sp(i) * sp(i)); });
        const float pe = np_pairwise_sum(N, [&](int i) { return bv.mg_f[i] * (ys(i) - ec.ground); });
        o.energy = 0.5f * ke + pe;
    }
    if (want_centroid) {                                         // np.mean(axis=0): sequential
#pragma unroll
        for (int c = 0; c < 3; c++) {
            float acc = st.pos(0, c);
#pragma unroll
            for (int n = 1; n < N; n++) acc = acc + st.pos(n, c);
            o.cen[c] = div_const(acc, nd.m, nd.r, nd.kind);
        }
    }
}

// episode statistics of env i whose episode just ended with return r after len steps: fin_stats [4][E] sums return,
// return^2, length and count.  With nf_stats [2][E] bound, an episode whose return is not finite is counted there
// instead (count, length sum), so one overflowed episode cannot make the mean return of the whole batch NaN.
// Every step kernel accounts a finished episode through this function.
template <bool NF = true, class Args>
__device__ __forceinline__ void account_episode(const Args& A, int64_t E, int64_t i, float r, int32_t len) {
    if (!A.fin_stats) return;
    if (NF && A.nf_stats && !is_finite(r)) {
        A.nf_stats[0 * E + i] += 1.0f;
        A.nf_stats[1 * E + i] += (float)len;
        return;
    }
    A.fin_stats[0 * E + i] += r;
    A.fin_stats[1 * E + i] += r * r;
    A.fin_stats[2 * E + i] += (float)len;
    A.fin_stats[3 * E + i] += 1.0f;
}

template <bool IN3D, bool NF = true, class Topo, class BV, class Store, class YS, class SP>
__device__ __forceinline__ void epilogue(const Topo& topo, const BV& bv, const EnvConst& ec, Store& st,
                                         int32_t steps_now, bool want_energy, bool want_centroid,
                                         YS ys, SP sp, EpiOut& o) {
    const int N = topo.n();
#pragma unroll
    for (int n = 0; n < N; n++) {                               // _get_reward (optimized_env.py:189-205)
        ys(n) = st.pos(n, 1);
        sp(n) = np_norm3(v3(st.vel(n, 0), st.vel(n, 1), st.vel(n, 2)));
    }
    epilogue_reduce<NF>(N, bv, ec, st, steps_now, want_energy, want_centroid, ys, sp, o);
}

// =================================================================================
// K1, register-resident specialisation: Topo is compile-time, EPT envs per thread.
// =================================================================================
// OBS: 0 = feature-major [D][E] (stores coalesced straight from registers),
//      1 = row-major [E][D] staged through a padded shared-memory tile, each warp streaming its
//          own 32*EPT rows (one contiguous span of global memory) with only a __syncwarp,
// Args: StepArgs<Topo::N, Topo::S> for the ahead-of-time specialisations; the run-time compiled ones (wg_jit.cu) take
// the full-size StepArgs<kMaxMass, kMaxSpring>.
template <class Topo, bool IN3D, int OBS, int EPT, int MM, class Args = StepArgs<Topo::N, Topo::S>>
__global__ void __launch_bounds__(kBlock, (Topo::N <= 4 && EPT == 1) ? WG_MIN_BLOCKS : 1)
step_static_kernel(const __grid_constant__ Args A) {
    constexpr bool ROWMAJOR = (OBS == 1);
    constexpr int N = Topo::N, M = Topo::M;
    constexpr int D = 3 * (IN3D ? 3 : 2) * N + M;
    // Row-major observations leave through a per-warp shared-memory tile.  When gcd(D, 32) <= 2 the rows
    // are stored unpadded (owner-thread writes then conflict at most 2-way) so that the warp's 32 rows
    // are byte-for-byte the contiguous 32*D*4-byte span of global memory they go to, and ONE TMA bulk
    // store (cp.async.bulk, SASS UBLKCP) per warp replaces 3*D per-thread instructions; otherwise the
    // tile has an odd pitch (conflict-free) and lanes copy it out.
    constexpr bool OBS_BULK = (OBS == 1) && (EPT == 1) && gcd_c(D, 32) <= 2;
    constexpr int STRIDE = OBS_BULK ? D : (D | 1);
    constexpr int TILE_ENVS = kBlock * EPT;
    extern __shared__ __align__(128) float tile[];
    const Topo topo;
    const int tid = threadIdx.x;
    const int64_t E = A.E;
    const int64_t e0 = (int64_t)blockIdx.x * TILE_ENVS;
    const int64_t e = e0 + (int64_t)tid * EPT;    // first env of this thread (E % EPT == 0 is guaranteed)
    const bool valid = e < E;

    if (valid) {
        RegStore<N, M> st[EPT];
        int32_t stp[EPT];
        // ---- single HBM read of the state: coalesced vectors of EPT envs ----
        // (32-bit row offsets -- one IMAD.WIDE per access -- measured 6 % slower than 64-bit add chains)
        const int64_t Eu = E;
        const float* const ppos = A.pos + e;
        const float* const pvel = A.vel + e;
        const float* const pmx = A.mx + e;
#pragma unroll
        for (int n = 0; n < N; n++) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                float t[EPT];
                WG_LDF(ppos + (decltype(Eu))(n * 3 + c) * Eu, t);
#pragma unroll
                for (int j = 0; j < EPT; j++) st[j].pos(n, c) = t[j];
                WG_LDF(pvel + (decltype(Eu))(n * 3 + c) * Eu, t);
#pragma unroll
                for (int j = 0; j < EPT; j++) st[j].vel(n, c) = t[j];
            }
        }
#pragma unroll
        for (int m = 0; m < M; m++) {
            float t[EPT];
            WG_LDF(pmx + (decltype(Eu))m * Eu, t);
#pragma unroll
            for (int j = 0; j < EPT; j++) st[j].mx(m) = t[j];
        }
        ld_vec<EPT, int32_t, typename Vec<EPT>::I>(A.steps + e, stp);
        float epr[EPT];
        if (A.ep_ret) WG_LDF(A.ep_ret + e, epr);

        // actions: when the row has exactly M columns the EPT rows of this thread are one aligned vector
        constexpr int AV = EPT * M;
        constexpr bool kVecOk = (M > 0) && (AV == 2 || AV == 4 || AV == 8);
        float actv[kVecOk ? AV : 1];
        const bool act_vec = kVecOk && A.act_layout == 0 && A.act_dim == M && ((reinterpret_cast<uintptr_t>(A.action) & 15u) == 0);
        if (act_vec) {
            const float* ap = A.action + e * M;
            if (AV == 2) { const float2 v = *reinterpret_cast<const float2*>(ap); actv[0] = v.x; actv[AV > 1 ? 1 : 0] = v.y; }
            else {
#pragma unroll
                for (int q = 0; q < AV / 4; q++) {
                    const float4 v = *reinterpret_cast<const float4*>(ap + 4 * q);
                    actv[(4 * q + 0) % AV] = v.x; actv[(4 * q + 1) % AV] = v.y;
                    actv[(4 * q + 2) % AV] = v.z; actv[(4 * q + 3) % AV] = v.w;
                }
            }
        }
        float rew[EPT]; uint8_t dnb[EPT]; uint32_t cpre[EPT], cpost[EPT];
        float eng[EPT], cen[3][EPT];
#pragma unroll
        for (int j = 0; j < EPT; j++) {
            // ---- Creature.act (optimized_walker.py:164-167; Muscle.act/regulation :27-35) ----
            const int na = A.act_dim < M ? A.act_dim : M;
#pragma unroll
            for (int m = 0; m < M; m++) {
                if (m < na) {
                    float x = st[j].mx(m) + (act_vec ? actv[j * M + m]
                                             : A.act_layout ? A.action[(int64_t)m * E + e + j] : A.action[(e + j) * A.act_dim + m]);
                    if (A.bv.mlo[m] > x) x = A.bv.mlo[m];       // python max(x, lo)
                    if (A.bv.mhi[m] < x) x = A.bv.mhi[m];       // python min(x, hi)
                    st[j].mx(m) = x;
                }
            }
            // ---- k_sub x (_run_physics + run1) ----
            uint32_t cp = 0;
            for (int k = 0; k < A.ec.k_sub; k++) cp = run_physics<IN3D, MM>(topo, A.bv, A.ec, st[j]);
            cpre[j] = cp;
            // ---- reward / done / info ----
            const int32_t sn = stp[j] + 1;
            float ysr[N], spr[N];
            EpiOut o;
            epilogue<IN3D>(topo, A.bv, A.ec, st[j], sn, A.energy != nullptr, A.centroid != nullptr,
                           [&](int i) -> float& { return ysr[i]; }, [&](int i) -> float& { return spr[i]; }, o);
            rew[j] = o.reward; dnb[j] = (uint8_t)o.done; cpost[j] = o.cpost;
            eng[j] = o.energy; cen[0][j] = o.cen[0]; cen[1][j] = o.cen[1]; cen[2][j] = o.cen[2];
            stp[j] = sn;
            if (A.ep_ret) {
                const float r = epr[j] + o.reward;
                if (o.done) account_episode(A, E, e + j, r, sn);
                epr[j] = (o.done && A.ec.auto_reset) ? 0.0f : r;
            }
            if (o.done && A.ec.auto_reset) {
                apply_reset<IN3D>(topo, A.bv, A.ec, st[j], A.ec.auto_reset, A.noise, E, e + j, step_index_of(A));
                stp[j] = 0;
            }
            // ---- observation of the (possibly reset) state ----
            if (A.obs) {
                if (OBS == 1) {
                    float* row = tile + (tid * EPT + j) * STRIDE;
                    get_obs<IN3D>(topo, A.bv.ndiv, st[j], [&](int k, float v) { row[k] = v; });
                } else {
                    get_obs<IN3D>(topo, A.bv.ndiv, st[j], [&](int k, float v) { A.obs[(int64_t)k * E + e + j] = v; });
                }
            }
        }
        // ---- single HBM write of the state ----
#pragma unroll
        for (int n = 0; n < N; n++) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                float t[EPT];
#pragma unroll
                for (int j = 0; j < EPT; j++) t[j] = st[j].pos(n, c);
                WG_STF(A.pos + e + (decltype(Eu))(n * 3 + c) * Eu, t);
#pragma unroll
                for (int j = 0; j < EPT; j++) t[j] = st[j].vel(n, c);
                WG_STF(A.vel + e + (decltype(Eu))(n * 3 + c) * Eu, t);
                if (A.old_a) {
#pragma unroll
                    for (int j = 0; j < EPT; j++) t[j] = st[j].acc(n, c);
                    WG_STF(A.old_a + e + (decltype(Eu))(n * 3 + c) * Eu, t);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < M; m++) {
            float t[EPT];
#pragma unroll
            for (int j = 0; j < EPT; j++) t[j] = st[j].mx(m);
            WG_STF(A.mx + e + (decltype(Eu))m * Eu, t);
        }
        st_vec<EPT, int32_t, typename Vec<EPT>::I>(A.steps + e, stp);
        if (A.ep_ret) WG_STF(A.ep_ret + e, epr);
        if (A.reward) WG_STF(A.reward + e, rew);
        if (A.done) st_vec<EPT, uint8_t, typename Vec<EPT>::B>(A.done + e, dnb);
        if (A.contact_pre) st_vec<EPT, uint32_t, typename Vec<EPT>::U>(A.contact_pre + e, cpre);
        if (A.contact_post) st_vec<EPT, uint32_t, typename Vec<EPT>::U>(A.contact_post + e, cpost);
        if (A.energy) WG_STF(A.energy + e, eng);
        if (A.centroid) {
#pragma unroll
            for (int c = 0; c < 3; c++) WG_STF(A.centroid + (int64_t)c * E + e, cen[c]);
        }
    }
    // ---- row-major observation: each warp owns 32*EPT consecutive rows = one contiguous span ----
    if (ROWMAJOR && A.obs) {
        static_assert(D >= 16, "copy-out assumes at most two row wraps per 32 lanes");
        __syncwarp();
        constexpr int RW = 32 * EPT;                       // rows per warp
        constexpr int PAD = STRIDE - D;
        const int warp = tid >> 5, lane = tid & 31;
        const int64_t ew = e0 + (int64_t)warp * RW;         // first env of this warp
        const int64_t rem = E - ew;
        if (rem > 0) {
            const float* src = tile + warp * RW * STRIDE + lane;
            float* out = A.obs + ew * D + lane;
            if (OBS_BULK && rem >= RW && ((reinterpret_cast<uintptr_t>(A.obs) & 15u) == 0)) {
                fence_proxy_async();                  // the lanes' tile writes -> visible to the copy engine
                __syncwarp();
                if (lane == 0) {
                    bulk_s2g(A.obs + ew * D, tile + warp * RW * STRIDE, (uint32_t)(RW * D * 4));
                    bulk_commit();
                    bulk_wait_read0();                // shared memory must outlive the copy's reads
                }
            } else if (rem >= RW) {
#pragma unroll
                for (int i = 0; i < EPT * D; i++) {         // idx = 32*i + lane -> row el, column idx - el*D
                    constexpr int dummy = 0; (void)dummy;
                    const int base = (32 * i) / D, r0 = (32 * i) % D;
                    const int t = lane + r0;
                    const int el = base + (t >= D ? 1 : 0) + (t >= 2 * D ? 1 : 0);
                    out[32 * i] = src[32 * i + el * PAD];
                }
            } else {
                const int total = (int)rem * D;
                for (int idx = lane; idx < total; idx += 32) {
                    const int el = idx / D;
                    out[idx - lane] = src[idx - lane + el * PAD];
                }
            }
        }
    }
}

// =================================================================================
// K1, generic: run-time topology, per-env state in a shared-memory tile that stays
// resident across the k_sub substeps; one thread per env.
// =================================================================================
// x64 mode (see wg_physics.cuh): the muscle lengths live as doubles plus a type bit; XArgs = X64Args adds their buffers,
// the float64 actions and the double-typed tables, XArgs = NoX64 is the plain float32 kernel.
struct NoX64 { static constexpr bool kOn = false; };
struct X64Args {
    static constexpr bool kOn = true;
    X64Vals v;
    double* mx64; uint8_t* mx_weak; const double* action64;
};

template <bool IN3D, bool ROWMAJOR, class XArgs = NoX64>
__global__ void __launch_bounds__(kBlock)
step_generic_kernel(const __grid_constant__ StepArgs<kMaxMass, kMaxSpring> A, const __grid_constant__ XArgs XA) {
    constexpr bool X64 = XArgs::kOn;
    extern __shared__ float smem[];
    const int N = A.bv.n_mass, S = A.bv.n_spring, M = A.bv.n_muscle;
    constexpr int d = IN3D ? 3 : 2;
    const int D = 3 * d * N + M;
    constexpr int PITCH = kBlock + 1;             // odd pitch: row-wise and column-wise access conflict-free
    RuntimeTopo topo{ N, S, M, A.bv.si, A.bv.sj };
    const int tid = threadIdx.x;
    __shared__ uint16_t obs_src[3 * 3 * kMaxMass + kMaxSpring], obs_cen[3 * 3 * kMaxMass + kMaxSpring];
    if (ROWMAJOR) {
        for (int k = tid; k < D; k += kBlock) {                     // Creature.getstat's entry order
            int src, cen = 0;
            if (k < 3 * d * N) {
                const int n = k / (3 * d), r = k - n * 3 * d, part = r / d, c = r - part * d;
                src = part * 3 * N + n * 3 + c;
                if (part == 0) cen = 9 * N + M + 2 * N + c;
            } else {
                src = 9 * N + (k - 3 * d * N);
            }
            obs_src[k] = (uint16_t)src; obs_cen[k] = (uint16_t)cen;
        }
    }
    const int64_t E = A.E;
    const int64_t e0 = (int64_t)blockIdx.x * kBlock;
    const int64_t e = e0 + tid;
    const bool valid = e < E;
    SmemStore st{ smem + tid, PITCH, N };
    // scratch rows: [0,N) ys, [N,2N) speeds, [2N,2N+3) centroid used by the obs copy-out
    if (valid) {
        for (int r = 0; r < 3 * N; r++) {
            st.base[r * PITCH] = A.pos[(int64_t)r * E + e];
            st.base[(3 * N + r) * PITCH] = A.vel[(int64_t)r * E + e];
        }
        const int na = A.act_dim < M ? A.act_dim : M;
        uint32_t cp = 0;
        if constexpr (X64) {
            // the post-action double lengths and type bits go back to their coalesced [M][E] arrays, which the substeps
            // read: staged in shared memory they would cost 3M more rows and keep large bodies from launching
            for (int m = 0; m < M; m++) {
                double x = XA.mx64[(int64_t)m * E + e];
                if (m < na) {                                               // anything + np.float64 -> np.float64
                    x = x + (A.act_layout ? XA.action64[(int64_t)m * E + e] : XA.action64[e * A.act_dim + m]);
                    uint8_t weak = 0;
                    if (XA.v.mlo_d[m] > x) { x = XA.v.mlo_d[m]; weak = 1; }   // max() returns the limit object
                    if (XA.v.mhi_d[m] < x) { x = XA.v.mhi_d[m]; weak = 1; }
                    XA.mx64[(int64_t)m * E + e] = x;
                    XA.mx_weak[(int64_t)m * E + e] = weak;
                }
                st.mx(m) = (float)x;                                        // float32 view: weak muscles, observation
            }
            for (int k = 0; k < A.ec.k_sub; k++) {
                for (int n = 0; n < N; n++) { st.acc(n, 0) = 0.0f; st.acc(n, 1) = 0.0f; st.acc(n, 2) = 0.0f; }
                for (int sp = 0; sp < M; sp++) {
                    if (XA.mx_weak[(int64_t)sp * E + e])
                        spring_run<2>(topo, A.bv, st, sp, st.mx(sp), A.bv.fixed_mask);
                    else
                        spring_run_x64(topo, A.bv, st, sp, XA.mx64[(int64_t)sp * E + e], XA.v.sk_d[sp], A.bv.fixed_mask);
                }
                for (int sp = M; sp < S; sp++) spring_run<2>(topo, A.bv, st, sp, A.bv.srest[sp], A.bv.fixed_mask);
                cp = 0;
                for (int n = 0; n < N; n++)
                    if (point_step<IN3D, 2>(A.bv, A.ec, st, n)) cp |= 1u << n;
            }
        } else {
        for (int m = 0; m < M; m++) st.mx(m) = A.mx[(int64_t)m * E + e];
        for (int m = 0; m < na; m++) {
            float x = st.mx(m) + (A.act_layout ? A.action[(int64_t)m * E + e] : A.action[e * A.act_dim + m]);
            if (A.bv.mlo[m] > x) x = A.bv.mlo[m];
            if (A.bv.mhi[m] < x) x = A.bv.mhi[m];
            st.mx(m) = x;
        }
        for (int k = 0; k < A.ec.k_sub; k++) cp = run_physics<IN3D, 2>(topo, A.bv, A.ec, st);
        }
        int32_t sn = A.steps[e] + 1;
        EpiOut o;
        epilogue<IN3D>(topo, A.bv, A.ec, st, sn, A.energy != nullptr, A.centroid != nullptr,
                       [&](int i) -> float& { return st.scratch(M, i); },
                       [&](int i) -> float& { return st.scratch(M, N + i); }, o);
        if (A.reward) A.reward[e] = o.reward;
        if (A.done) A.done[e] = (uint8_t)o.done;
        if (A.contact_pre) A.contact_pre[e] = cp;
        if (A.contact_post) A.contact_post[e] = o.cpost;
        if (A.energy) A.energy[e] = o.energy;
        if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
        if (A.ep_ret) {
            const float r = A.ep_ret[e] + o.reward;
            if (o.done) account_episode(A, E, e, r, sn);
            A.ep_ret[e] = (o.done && A.ec.auto_reset) ? 0.0f : r;
        }
        if (o.done && A.ec.auto_reset) {
            apply_reset<IN3D>(topo, A.bv, A.ec, st, A.ec.auto_reset, A.noise, E, e, step_index_of(A));
            sn = 0;
            if constexpr (X64) {
                if (A.ec.auto_reset == 2)                                   // a fresh Muscle: x = originx
                    for (int m = 0; m < M; m++) {
                        XA.mx64[(int64_t)m * E + e] = XA.v.x0_d[m];
                        XA.mx_weak[(int64_t)m * E + e] = 1;
                    }
            }
        }
        A.steps[e] = sn;
        for (int r = 0; r < 3 * N; r++) {
            A.pos[(int64_t)r * E + e] = st.base[r * PITCH];
            A.vel[(int64_t)r * E + e] = st.base[(3 * N + r) * PITCH];
            if (A.old_a) A.old_a[(int64_t)r * E + e] = st.base[(6 * N + r) * PITCH];
        }
        for (int m = 0; m < M; m++) A.mx[(int64_t)m * E + e] = st.mx(m);
        if (A.obs) {
            if (ROWMAJOR) {
                // centroid of getstat (sequential sum, then / N) for the cooperative copy-out below
                float mid[3] = { 0.0f, 0.0f, 0.0f };
                for (int n = 0; n < N; n++) { mid[0] = mid[0] + st.pos(n, 0); mid[1] = mid[1] + st.pos(n, 1); mid[2] = mid[2] + st.pos(n, 2); }
                const ConstDiv nd = A.bv.ndiv;
                st.scratch(M, 2 * N + 0) = div_const(mid[0], nd.m, nd.r, nd.kind);
                st.scratch(M, 2 * N + 1) = div_const(mid[1], nd.m, nd.r, nd.kind);
                st.scratch(M, 2 * N + 2) = div_const(mid[2], nd.m, nd.r, nd.kind);
            } else {
                get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float v) { A.obs[(int64_t)k * E + e] = v; });
            }
        }
    }
    if (ROWMAJOR && A.obs) {
        // Each warp streams whole observation rows straight out of the state tile:
        // lanes run over the D entries of one env, so global stores are coalesced
        // and the (row, env) shared-memory reads hit distinct banks (odd pitch).
        __syncthreads();
        const int64_t rem = E - e0;
        const int nvalid = rem < kBlock ? (int)rem : kBlock;
        const int warp = tid >> 5, lane = tid & 31;
        // entry k of an observation row = tile row obs_src[k] (minus the centroid row obs_cen[k] for positions):
        // a per-block lookup table instead of index arithmetic per element
        for (int el = warp; el < nvalid; el += kBlock / 32) {
            const float* col = smem + el;
            float* out = A.obs + (e0 + el) * D;
            for (int k = lane; k < D; k += 32) {
                float v = col[obs_src[k] * PITCH];
                const int cr = obs_cen[k];
                if (cr) v = v - col[cr * PITCH];
                out[k] = v;
            }
        }
    }
}

// =================================================================================
// K2: PhysicsEnv.reset for masked envs.  Not on the hot path: generic, local-memory state.
// =================================================================================
struct LocalStore {
    float p_[kMaxMass][3], v_[kMaxMass][3], a_[kMaxMass][3], mx_[kMaxSpring];
    __device__ __forceinline__ float& pos(int n, int c) { return p_[n][c]; }
    __device__ __forceinline__ float& vel(int n, int c) { return v_[n][c]; }
    __device__ __forceinline__ float& acc(int n, int c) { return a_[n][c]; }
    __device__ __forceinline__ float& mx(int m) { return mx_[m]; }
};

template <bool IN3D>
__global__ void __launch_bounds__(kBlock)
reset_kernel(const __grid_constant__ StepArgs<kMaxMass, kMaxSpring> A, int mode, const uint8_t* mask, int obs_layout) {
    const int N = A.bv.n_mass, S = A.bv.n_spring, M = A.bv.n_muscle;
    constexpr int d = IN3D ? 3 : 2;
    const int D = 3 * d * N + M;
    const int64_t E = A.E;
    const int64_t e = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (e >= E) return;
    if (mask && !mask[e]) return;
    RuntimeTopo topo{ N, S, M, A.bv.si, A.bv.sj };
    LocalStore st;
    const int r4 = (6 * N + M + 2 + 3) / 4;
    float* const sp = A.state_packed;
    for (int r = 0; r < 3 * N; r++) {
        st.p_[r / 3][r % 3] = sp ? sp[packed_index(e, r, r4)] : A.pos[(int64_t)r * E + e];
        st.v_[r / 3][r % 3] = sp ? sp[packed_index(e, 3 * N + r, r4)] : A.vel[(int64_t)r * E + e];
        st.a_[r / 3][r % 3] = A.old_a ? A.old_a[(int64_t)r * E + e] : 0.0f;
    }
    for (int m = 0; m < M; m++) st.mx_[m] = sp ? sp[packed_index(e, 6 * N + m, r4)] : A.mx[(int64_t)m * E + e];
    apply_reset<IN3D>(topo, A.bv, A.ec, st, mode, A.noise, E, e, step_index_of(A));
    if (sp) {
        sp[packed_index(e, 6 * N + M, r4)] = __int_as_float(0);
        sp[packed_index(e, 6 * N + M + 1, r4)] = 0.0f;
    } else {
        A.steps[e] = 0;
        if (A.ep_ret) A.ep_ret[e] = 0.0f;
    }
    for (int r = 0; r < 3 * N; r++) {
        if (sp) { sp[packed_index(e, r, r4)] = st.p_[r / 3][r % 3]; sp[packed_index(e, 3 * N + r, r4)] = st.v_[r / 3][r % 3]; }
        else { A.pos[(int64_t)r * E + e] = st.p_[r / 3][r % 3]; A.vel[(int64_t)r * E + e] = st.v_[r / 3][r % 3]; }
        if (A.old_a) A.old_a[(int64_t)r * E + e] = st.a_[r / 3][r % 3];
    }
    for (int m = 0; m < M; m++) {
        if (sp) sp[packed_index(e, 6 * N + m, r4)] = st.mx_[m]; else A.mx[(int64_t)m * E + e] = st.mx_[m];
    }
    if (A.obs) {
        // jitter-only reset without an old_a buffer: the acceleration slots of the
        // observation still hold Point.old_a of the last step -- leave them alone.
        const bool keep_acc = (mode == 1) && (A.old_a == nullptr);
        get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float v) {
            if (keep_acc && k < 3 * d * N && (k % (3 * d)) >= 2 * d) return;
            if (obs_layout == 0) A.obs[e * D + k] = v; else A.obs[(int64_t)k * E + e] = v;
        });
    }
}

// =================================================================================
// K3: deterministic single-block reduction of the finished-episode accumulators:
// out8 = [fin_stats rows 0..3, nf_stats rows 0..1 (0 when nf is null), 0, 0].
// =================================================================================
template <int THREADS>
__global__ void __launch_bounds__(THREADS) stats_reduce_kernel(const float* __restrict__ fin, const float* __restrict__ nf,
                                                               int64_t E, double* out8) {
    constexpr int Q = 6;
    __shared__ double part[Q][32];
    double acc[Q] = { 0.0, 0.0, 0.0, 0.0, 0.0, 0.0 };
    for (int64_t i = threadIdx.x; i < E; i += blockDim.x) {
#pragma unroll
        for (int q = 0; q < 4; q++) acc[q] += (double)fin[(int64_t)q * E + i];
        if (nf) {
            acc[4] += (double)nf[i];
            acc[5] += (double)nf[E + i];
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < Q; q++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc[q] += __shfl_down_sync(0xffffffffu, acc[q], off);
        if (lane == 0) part[q][warp] = acc[q];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int q = 0; q < Q; q++) {
            double v = lane < (int)(blockDim.x >> 5) ? part[q][lane] : 0.0;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if (lane == 0) out8[q] = v;
        }
        if (lane == 0) { out8[6] = 0.0; out8[7] = 0.0; }
    }
}

}  // namespace wg
