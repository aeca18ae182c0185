// wg_kernels_packed.cuh -- K1 on the packed state layout: vectorised float4 HBM access.
//
// State layout [tile][k/4][128 envs][4] (include/walker_gym_b200.h): the R = 6N + M + 2 scalars of an env
// (positions, velocities, muscle lengths, step counter, running return) are grouped four at a time, so
// thread t of a tile moves its env's whole state with R4 = ceil(R/4) 16-byte loads and R4 16-byte stores
// (7 + 7 for Balance-v0 instead of 28 + 28 scalar accesses), every access is `tile base + immediate`, a warp
// access is 512 contiguous bytes and a tile is one contiguous R4 * 2 KiB block of HBM.  Everything between
// the loads and the stores is the same register-resident code as step_static_kernel.
#pragma once
#include "wg_kernels.cuh"

namespace wg {

#ifndef WG_PACKED_BLOCK
#define WG_PACKED_BLOCK 128
#endif
#ifndef WG_PACKED_MIN_BLOCKS
#define WG_PACKED_MIN_BLOCKS (768 / WG_PACKED_BLOCK)
#endif
// threads per CTA of the packed kernel: a multiple of the 128-env tile (a CTA covers PB / 128 consecutive tiles)
constexpr int kPackedBlock = WG_PACKED_BLOCK;
static_assert(kPackedBlock % 128 == 0, "the packed layout is tiled by 128 envs");

// Args: StepArgs<Topo::N, Topo::S> for the ahead-of-time specialisations; the run-time compiled ones (wg_jit.cu) take
// the full-size StepArgs<kMaxMass, kMaxSpring> the host can fill for any body.
// NF: the non-finite handling (wg_params.end_nonfinite, buf->nf_stats), the truncation flag (buf->truncated) and the
// final observation (buf->final_obs) are compiled in; the launcher takes the NF = false instance when all four are off, so the reference's semantics run exactly the code they ran before the option existed.
// MINB: resident CTAs per SM the compiler must allow (0 = the default for the body size).  The 7-CTA instance (72
// registers) exists for grids that fit ONE wave at 7 CTAs per SM but not at 6 -- BASELINE config 3 as written, 2^20 envs
// over 8 GPUs = 1024 CTAs per GPU against 148 x 6 = 888 slots: a second, 14 %-full wave would double the step time.
__host__ __device__ constexpr int packed_min_blocks(int n_mass, int minb) {
    return minb > 0 ? minb : (n_mass <= 4 ? WG_PACKED_MIN_BLOCKS : (n_mass <= 6 ? 512 : 384) / WG_PACKED_BLOCK);
}
template <class Topo, bool IN3D, int OBS, int MM, class Args = StepArgs<Topo::N, Topo::S>, bool NF = true, int MINB = 0>
__global__ void __launch_bounds__(kPackedBlock, packed_min_blocks(Topo::N, MINB))
step_static_packed_kernel(const __grid_constant__ Args A) {
    constexpr int N = Topo::N, M = Topo::M;
    constexpr int D = 3 * (IN3D ? 3 : 2) * N + M;
    constexpr int R = 6 * N + M + 2, R4 = (R + 3) / 4;
    constexpr int K_MX = 6 * N, K_STEPS = 6 * N + M, K_EPRET = K_STEPS + 1;
    constexpr bool OBS_BULK = (OBS == 1) && gcd_c(D, 32) <= 2;
    constexpr int STRIDE = OBS_BULK ? D : (D | 1);
    extern __shared__ __align__(128) float tile[];
    const Topo topo;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t E = A.E;
    constexpr int kBlock = 128;                       // envs per state tile (shadows the CTA size of the SoA kernels)
    const int64_t e0 = (int64_t)blockIdx.x * kPackedBlock;
    const int64_t e = e0 + tid;
    const bool valid = e < E;
    const int64_t tile_idx = (int64_t)blockIdx.x * (kPackedBlock / kBlock) + (tid >> 7);
    float4* const base = reinterpret_cast<float4*>(A.state_packed) + tile_idx * (R4 * kBlock) + (tid & 127);

    // Programmatic dependent launch: let the NEXT kernel of the stream be scheduled as soon as every CTA of this grid has
    // started (its CTAs then sit in freed slots, past their prologue), and wait here for the PREVIOUS kernel's memory
    // before the first global access -- back-to-back steps lose no launch gap.  Both are no-ops without the launch attribute.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // L2 prefetch: a tile is one contiguous block, so one thread can ask the copy engine to pull the tile that a
    // CTA launched `pf_dist` blocks later will read (CTAs are dispatched in index order) from HBM into L2 with a
    // single cp.async.bulk.prefetch; that CTA's loads then pay L2 instead of DRAM latency.
    if ((tid & 127) == 0 && A.pf_dist > 0) {
        const int64_t pt = tile_idx + A.pf_dist;
        if (pt * kBlock + kBlock <= E) {
            const float* ps = A.state_packed + pt * (R4 * kBlock * 4);
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ps), "r"((uint32_t)(R4 * kBlock * 16)) : "memory");
            if (M > 0 && A.action && A.act_layout == 0 && A.act_dim == M && ((reinterpret_cast<uintptr_t>(A.action) & 15u) == 0))
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(A.action + pt * kBlock * M),
                             "r"((uint32_t)(kBlock * M * 4)) : "memory");
        }
    }

    if (valid) {
        // ---- single HBM read of the state: R4 coalesced 16-byte loads at immediate offsets ----
        float v[R4 * 4];
#pragma unroll
        for (int g = 0; g < R4; g++) {
            const float4 q = base[g * kBlock];
            v[4 * g + 0] = q.x; v[4 * g + 1] = q.y; v[4 * g + 2] = q.z; v[4 * g + 3] = q.w;
        }
        RegStore<N, M> st;
#pragma unroll
        for (int k = 0; k < 3 * N; k++) { st.p_[k / 3][k % 3] = v[k]; st.v_[k / 3][k % 3] = v[3 * N + k]; }
#pragma unroll
        for (int m = 0; m < M; m++) st.mx(m) = v[K_MX + m];
        int32_t stp = __float_as_int(v[K_STEPS]);
        float epr = v[K_EPRET];

        // ---- Creature.act: the env's M actions are one aligned vector when the row has exactly M columns ----
        float act[M > 0 ? M : 1];
        const int na = A.act_dim < M ? A.act_dim : M;
        const bool act_vec = (M == 2 || M == 4) && A.act_layout == 0 && A.act_dim == M &&
                             ((reinterpret_cast<uintptr_t>(A.action) & 15u) == 0);
        if (act_vec) {
            if (M == 2) { const float2 a = *reinterpret_cast<const float2*>(A.action + e * 2); act[0] = a.x; act[M > 1 ? 1 : 0] = a.y; }
            else { const float4 a = *reinterpret_cast<const float4*>(A.action + e * 4);
                   act[0] = a.x; act[M > 1 ? 1 : 0] = a.y; act[M > 2 ? 2 : 0] = a.z; act[M > 3 ? 3 : 0] = a.w; }
        }
#pragma unroll
        for (int m = 0; m < M; m++) {
            if (m < na) {
                float x = st.mx(m) + (act_vec ? act[m] : A.act_layout ? A.action[(int64_t)m * E + e] : A.action[e * A.act_dim + m]);
                if (A.bv.mlo[m] > x) x = A.bv.mlo[m];       // python max(x, lo)
                if (A.bv.mhi[m] < x) x = A.bv.mhi[m];       // python min(x, hi)
                st.mx(m) = x;
            }
        }
        // ---- k_sub x (_run_physics + run1), reward / done / info ----
        uint32_t cp = 0;
        for (int k = 0; k < A.ec.k_sub; k++) cp = run_physics<IN3D, MM>(topo, A.bv, A.ec, st);
        const int32_t sn = stp + 1;
        float ysr[N], spr[N];
        EpiOut o;
        epilogue<IN3D, NF>(topo, A.bv, A.ec, st, sn, A.energy != nullptr, A.centroid != nullptr, NF && A.truncated != nullptr,
                       [&](int i) -> float& { return ysr[i]; }, [&](int i) -> float& { return spr[i]; }, o);
        stp = sn;
        {   // episode statistics: the running return lives in the packed state
            const float r = epr + o.reward;
            if (o.done) account_episode<NF>(A, E, e, r, sn);
            epr = (o.done && A.ec.auto_reset) ? 0.0f : r;
        }
        if (NF && o.done && A.final_obs) store_final_obs<IN3D>(topo, A, st, E, e, OBS == 1);
        if (o.done && A.ec.auto_reset) {
            apply_reset<IN3D>(topo, A.bv, A.ec, st, A.ec.auto_reset, A.noise, E, e, step_index_of(A));
            stp = 0;
        }
        if (A.obs) {
            if (OBS == 1) {
                float* row = tile + tid * STRIDE;
                get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float val) { row[k] = val; });
            } else {
                get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float val) { A.obs[(int64_t)k * E + e] = val; });
            }
        }
        // ---- single HBM write of the state: R4 coalesced 16-byte stores ----
#pragma unroll
        for (int k = 0; k < 3 * N; k++) { v[k] = st.p_[k / 3][k % 3]; v[3 * N + k] = st.v_[k / 3][k % 3]; }
#pragma unroll
        for (int m = 0; m < M; m++) v[K_MX + m] = st.mx(m);
        v[K_STEPS] = __int_as_float(stp);
        v[K_EPRET] = epr;
#pragma unroll
        for (int g = 0; g < R4; g++) base[g * kBlock] = make_float4(v[4 * g + 0], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
        if (A.old_a) {
#pragma unroll
            for (int k = 0; k < 3 * N; k++) A.old_a[(int64_t)k * E + e] = st.a_[k / 3][k % 3];
        }
        if (A.reward) A.reward[e] = o.reward;
        if (A.done) A.done[e] = (uint8_t)o.done;
        if (NF && A.truncated) A.truncated[e] = (uint8_t)o.trunc;
        if (A.contact_pre) A.contact_pre[e] = cp;
        if (A.contact_post) A.contact_post[e] = o.cpost;
        if (A.energy) A.energy[e] = o.energy;
        if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
    }
    // ---- row-major observation: one TMA bulk store per warp (or the padded-tile copy-out) ----
    if (OBS == 1 && A.obs) {
        __syncwarp();
        const int64_t ew = e0 + (int64_t)warp * 32;
        const int64_t remw = E - ew;
        if (remw > 0) {
            float* wt = tile + warp * 32 * STRIDE;
            if (OBS_BULK && remw >= 32 && ((reinterpret_cast<uintptr_t>(A.obs) & 15u) == 0)) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { bulk_s2g(A.obs + ew * D, wt, (uint32_t)(32 * D * 4)); bulk_commit(); bulk_wait_read0(); }
            } else {
                const int nvw = remw < 32 ? (int)remw : 32;
                const int total = nvw * D;
                float* out = A.obs + ew * D;
                for (int idx = lane; idx < total; idx += 32) {
                    const int el = idx / D;
                    out[idx] = wt[idx + el * (STRIDE - D)];
                }
            }
        }
    }
}

}  // namespace wg
