// wg_kernels_tma.cuh -- K1 as a persistent, TMA-pipelined kernel (the default for the
// register-resident specialisations whenever the buffers are 16-byte aligned and E % 4 == 0).
//
// One CTA (128 threads, one env per thread) walks tiles of 128 envs with stride gridDim.x;
// the grid is a multiple of the SM count.  A tile's inputs are consumed into registers at the
// very start of its compute phase, so ONE shared-memory stage suffices: as soon as every thread
// holds its inputs, the state rows of tile i+1 -- (6N + M + 2) rows of 512 contiguous bytes plus
// the action block -- are put in flight: lanes of warp 0 issue one cp.async.bulk (TMA 1-D bulk
// copy, SASS UBLKCP) per row and an mbarrier counts the bytes.  The whole compute of tile i
// overlaps the HBM reads of tile i+1: latency is hidden by the copy engine, not by occupancy.  Outputs: the state goes straight
// from registers to coalesced global stores; the row-major observation of each warp's 32 envs
// is one contiguous 32*D*4-byte span, staged in shared memory and written back with a single
// bulk store per warp (or the padded-tile copy-out when D would bank-conflict).
#pragma once
#include "wg_kernels.cuh"

namespace wg {

#ifndef WG_TMA_MIN_BLOCKS
#define WG_TMA_MIN_BLOCKS 6
#endif

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WG_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra WG_DONE;\n\t"
        "bra WG_WAIT;\n\t"
        "WG_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}


template <class Topo, bool IN3D>
struct TmaLayout {
    static constexpr int N = Topo::N, M = Topo::M;
    static constexpr int D = 3 * (IN3D ? 3 : 2) * N + M;
    static constexpr int ROW_STEPS = 6 * N + M, ROW_EPRET = ROW_STEPS + 1, ROWS = ROW_STEPS + 2;
    static constexpr int STAGE_FLOATS = ROWS * kBlock + kBlock * (M > 0 ? M : 1);
    // unpadded rows allow a single bulk store per warp; the owner-thread writes then conflict gcd(D,32)-way
    static constexpr bool OBS_BULK = gcd_c(D, 32) <= 2;
    static constexpr int DP = OBS_BULK ? D : (D | 1);
    static constexpr size_t smem_bytes(bool obs_tile) {
        return sizeof(float) * (STAGE_FLOATS + (obs_tile ? kBlock * DP : 0)) + 2 * sizeof(uint64_t) + 16;
    }
};

// One env, inputs already in registers: Creature.act -> k_sub x physics -> reward/done/info -> episode
// statistics -> auto-reset -> observation (into the warp's shared-memory tile or feature-major global)
// -> the single coalesced HBM write of the state.  Shared by the pipelined kernels below.
template <class Topo, bool IN3D, int OBS, int MM, int DP, class Args>
__device__ __forceinline__ void env_compute_store(const Args& A, RegStore<Topo::N, Topo::M>& st, int32_t stp, float epr,
                                                  const float* act, bool act_staged, int64_t e, int lane, float* wtile) {
    constexpr int N = Topo::N, M = Topo::M;
    const Topo topo;
    const int64_t E = A.E;
    {
            // ---- Creature.act ----
            const int na = A.act_dim < M ? A.act_dim : M;
#pragma unroll
            for (int m = 0; m < M; m++) {
                if (m < na) {
                    float x = st.mx(m) + (act_staged ? act[m] : A.act_layout ? A.action[(int64_t)m * E + e] : A.action[e * A.act_dim + m]);
                    if (A.bv.mlo[m] > x) x = A.bv.mlo[m];
                    if (A.bv.mhi[m] < x) x = A.bv.mhi[m];
                    st.mx(m) = x;
                }
            }
            uint32_t cp = 0;
            for (int k = 0; k < A.ec.k_sub; k++) cp = run_physics<IN3D, MM>(topo, A.bv, A.ec, st);
            const int32_t sn = stp + 1;
            float ysr[N], spr[N];
            EpiOut o;
            epilogue<IN3D>(topo, A.bv, A.ec, st, sn, A.energy != nullptr, A.centroid != nullptr, A.truncated != nullptr,
                           [&](int i) -> float& { return ysr[i]; }, [&](int i) -> float& { return spr[i]; }, o);
            stp = sn;
            if (A.ep_ret) {
                const float r = epr + o.reward;
                if (o.done) account_episode(A, E, e, r, sn);
                A.ep_ret[e] = (o.done && A.ec.auto_reset) ? 0.0f : r;
            }
            if (o.done && A.final_obs) store_final_obs<IN3D>(topo, A, st, E, e, OBS == 1);
            if (o.done && A.ec.auto_reset) {
                apply_reset<IN3D>(topo, A.bv, A.ec, st, A.ec.auto_reset, A.noise, E, e, step_index_of(A));
                stp = 0;
            }
            if (A.obs) {
                if (OBS == 1) {
                    float* row = wtile + lane * DP;
                    get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float v) { row[k] = v; });
                } else {
                    get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float v) { A.obs[(int64_t)k * E + e] = v; });
                }
            }
            // ---- single HBM write of the state: coalesced stores straight from registers ----
#pragma unroll
            for (int r = 0; r < 3 * N; r++) {
                A.pos[(int64_t)r * E + e] = st.p_[r / 3][r % 3];
                A.vel[(int64_t)r * E + e] = st.v_[r / 3][r % 3];
                if (A.old_a) A.old_a[(int64_t)r * E + e] = st.a_[r / 3][r % 3];
            }
#pragma unroll
            for (int m = 0; m < M; m++) A.mx[(int64_t)m * E + e] = st.mx(m);
            A.steps[e] = stp;
            if (A.reward) A.reward[e] = o.reward;
            if (A.done) A.done[e] = (uint8_t)o.done;
            if (A.truncated) A.truncated[e] = (uint8_t)o.trunc;
            if (A.contact_pre) A.contact_pre[e] = cp;
            if (A.contact_post) A.contact_post[e] = o.cpost;
            if (A.energy) A.energy[e] = o.energy;
            if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
        }
}

template <class Topo, bool IN3D, int OBS, int MM>
__global__ void __launch_bounds__(kBlock, WG_TMA_MIN_BLOCKS)
step_static_tma_kernel(const __grid_constant__ StepArgs<Topo::N, Topo::S> A) {
    using LY = TmaLayout<Topo, IN3D>;
    constexpr int N = Topo::N, M = Topo::M, D = LY::D, DP = LY::DP;
    extern __shared__ __align__(128) float smem_f[];
    float* const stage_buf = smem_f;
    float* const obs_tile = smem_f + LY::STAGE_FLOATS;
    uint64_t* const full = reinterpret_cast<uint64_t*>(
        smem_f + LY::STAGE_FLOATS + ((OBS == 1 && A.obs) ? kBlock * DP : 0) + 2);       // 8-byte aligned: all counts even
    const Topo topo;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t E = A.E;
    const int64_t n_tiles = (E + kBlock - 1) / kBlock;
    const bool act_bulk = (M > 0) && A.action && A.act_dim == M && A.act_layout == 0;

    if (tid == 0) {
        mbar_init(&full[0], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // warp 0: one bulk copy per state row of `tile`
    auto issue = [&](int64_t tile) {
        const int64_t e0 = tile * kBlock;
        const int64_t rem = E - e0;
        const uint32_t nv = rem < kBlock ? (uint32_t)rem : (uint32_t)kBlock;
        const uint32_t row_bytes = nv * 4u;
        const uint32_t n_rows = (uint32_t)LY::ROW_STEPS + 1u + (A.ep_ret ? 1u : 0u);
        if (lane == 0) mbar_expect_tx(&full[0], n_rows * row_bytes + (act_bulk ? nv * (uint32_t)M * 4u : 0u));
        __syncwarp();
        float* dst = stage_buf;
        for (int r = lane; r <= LY::ROWS; r += 32) {
            const void* src = nullptr;
            uint32_t bytes = row_bytes;
            if (r < 3 * N) src = A.pos + (int64_t)r * E + e0;
            else if (r < 6 * N) src = A.vel + (int64_t)(r - 3 * N) * E + e0;
            else if (r < LY::ROW_STEPS) src = A.mx + (int64_t)(r - 6 * N) * E + e0;
            else if (r == LY::ROW_STEPS) src = A.steps + e0;
            else if (r == LY::ROW_EPRET) { if (A.ep_ret) src = A.ep_ret + e0; }
            else if (act_bulk) { src = A.action + e0 * M; bytes = nv * (uint32_t)M * 4u; }
            if (src) bulk_g2s(dst + r * kBlock, src, bytes, &full[0]);
        }
    };

    int64_t tile = blockIdx.x;
    if (warp == 0 && tile < n_tiles) issue(tile);

    for (int it = 0; tile < n_tiles; tile += gridDim.x, ++it) {
        const int64_t next = tile + gridDim.x;
        mbar_wait(&full[0], (uint32_t)it & 1u);

        const int64_t e0 = tile * kBlock;
        const int64_t e = e0 + tid;
        const bool valid = e < E;
        const float* in = stage_buf + tid;
        RegStore<N, M> st;
        int32_t stp = 0;
        float epr = 0.0f;
        float act[M > 0 ? M : 1];
        if (valid) {
#pragma unroll
            for (int r = 0; r < 3 * N; r++) { st.p_[r / 3][r % 3] = in[r * kBlock]; st.v_[r / 3][r % 3] = in[(3 * N + r) * kBlock]; }
#pragma unroll
            for (int m = 0; m < M; m++) st.mx(m) = in[(6 * N + m) * kBlock];
            stp = __float_as_int(in[LY::ROW_STEPS * kBlock]);
            if (A.ep_ret) epr = in[LY::ROW_EPRET * kBlock];
            if (act_bulk) {
                const float* ap = stage_buf + LY::ROWS * kBlock + tid * M;
#pragma unroll
                for (int m = 0; m < M; m++) act[m] = ap[m];
            }
        }
        __syncthreads();          // every thread holds its inputs in registers: the stage is free again
        if (warp == 0 && next < n_tiles) issue(next);                  // in flight during the whole compute below

        float* wtile = obs_tile + warp * 32 * DP;
        if (OBS == 1 && A.obs) {  // the previous bulk store of this warp must have finished reading its tile
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
        }
        if (valid) env_compute_store<Topo, IN3D, OBS, MM, DP>(A, st, stp, epr, act, act_bulk, e, lane, wtile);
        if (OBS == 1 && A.obs) {
            const int64_t ew = e0 + (int64_t)warp * 32;
            const int64_t remw = E - ew;
            if (remw > 0) {
                const int nvw = remw < 32 ? (int)remw : 32;
                if (LY::OBS_BULK) {
                    fence_proxy_async();             // generic-proxy tile writes -> visible to the bulk copy engine
                    __syncwarp();
                    if (lane == 0) { bulk_s2g(A.obs + ew * D, wtile, (uint32_t)(nvw * D * 4)); bulk_commit(); }
                } else {
                    __syncwarp();
                    const int total = nvw * D;
                    float* out = A.obs + ew * D;
                    for (int idx = lane; idx < total; idx += 32) {
                        const int el = idx / D;
                        out[idx] = wtile[idx + el * (DP - D)];
                    }
                    __syncwarp();
                }
            }
        }
    }
    if (OBS == 1 && A.obs && LY::OBS_BULK && lane == 0) bulk_wait_read0();   // smem must outlive the last bulk store
}

}  // namespace wg
