// wg_kernels_multi.cuh -- T consecutive PhysicsEnv.step calls in ONE launch on the packed state layout.
//
// wg_step is HBM-bound: an env-step moves its whole state in and out of HBM (381 B for Balance-v0 with the
// observation row).  When the caller already knows the next T actions (scripted gaits, CPG / open-loop controllers,
// action repeat / frame skip, evaluation of a recorded action sequence) the state can stay in registers for all T
// steps: one state read, T x (Creature.act -> k_sub x _run_physics -> reward / done -> auto-reset), one state
// write, one observation row (that of the last step).  Per step only the action (4M bytes) is read and reward +
// done (5 bytes) are written, so the kernel leaves the HBM roofline of the single-step kernel behind and runs at
// the instruction rate of the bit-exact arithmetic.  Every step is the same device code as
// step_static_packed_kernel (gym/optimized_env.py:70-92), so results equal T wg_step calls bit for bit, including
// the Philox index of an auto-reset in the middle of the block (step index + t).
#pragma once
#include "wg_kernels_packed.cuh"

namespace wg {

// resident CTAs per SM the compiler must allow (small bodies): the kernel is instruction bound, so this trades
// registers per thread against warps per scheduler
#ifndef WG_MULTI_MIN_BLOCKS
#define WG_MULTI_MIN_BLOCKS WG_PACKED_MIN_BLOCKS
#endif

// threads per CTA (a multiple of the 128-env tile) and, optionally, a per-scheduler named barrier at the top of every
// step that keeps the warps sharing an instruction cache in phase (experiment knobs; see DESIGN.md K1-multi)
#ifndef WG_MULTI_BLOCK
#define WG_MULTI_BLOCK 128
#endif
#ifndef WG_MULTI_SYNC
#define WG_MULTI_SYNC 0
#endif
constexpr int kMultiBlock = WG_MULTI_BLOCK;
static_assert(kMultiBlock % 128 == 0, "the packed layout is tiled by 128 envs");
__host__ __device__ constexpr int multi_min_blocks(int n_mass) {
    const int threads = n_mass <= 4 ? WG_MULTI_MIN_BLOCKS * 128 : (n_mass <= 6 ? 512 : 384);
    return threads / kMultiBlock > 0 ? threads / kMultiBlock : 1;
}

// In-kernel action source (mirror of wg_action_gen, include/walker_gym_b200.h): a scripted phase table indexed by the
// env's step counter (gym/walker.py:356-366) or a sinusoidal pattern generator (gym/optimized_walker/walker.py:56-90)
constexpr int kGenRows = 32, kGenMuscle = 16;
struct ActionGen {
    int32_t mode, n_rows, hold, reserved;
    float table[kGenRows * kGenMuscle];
    float amp[kGenMuscle];
    uint32_t phase0[kGenMuscle], dphase[kGenMuscle];
};
// the action of muscle m for an env whose step counter (before the step) is `stp`
__device__ __forceinline__ float gen_action(const ActionGen& G, int m, int32_t stp) {
    if (G.mode == 1) return G.table[((stp / G.hold) % G.n_rows) * kGenMuscle + m];
    float sn, cs;
    det_sincos2pi((G.phase0[m] + (uint32_t)(stp + 1) * G.dphase[m]) & 0xffffffu, sn, cs);
    return G.amp[m] * sn;
}

// action: [T][E][M] row-major (act_stride = E * M), or one [E][M] block applied at every step (act_stride = 0:
// action repeat), or generated on chip (G.mode != 0); reward: [T][E]; done: [T][E]; obs: [E][D] row-major, after the
// last step.
// GEN: compile-time switch for the in-kernel action sources -- the tensor-action instance (GEN = false) stays exactly
// the code it was (the loop is instruction-cache sensitive: a run-time branch around the generator cost it 6 %).
// NF: as for step_static_packed_kernel (the non-finite handling and the truncation flag compiled in; launched with all of
// them off only as NF = false).
template <class Topo, bool IN3D, int MM, class Args = StepArgs<Topo::N, Topo::S>, bool GEN = false, bool NF = true>
__global__ void __launch_bounds__(kMultiBlock, multi_min_blocks(Topo::N))
step_multi_packed_kernel(const __grid_constant__ Args A, const int n_steps, const int64_t act_stride,
                         const __grid_constant__ ActionGen G) {
    constexpr int N = Topo::N, M = Topo::M;
    constexpr int D = 3 * (IN3D ? 3 : 2) * N + M;
    constexpr int R = 6 * N + M + 2, R4 = (R + 3) / 4;
    constexpr int K_MX = 6 * N, K_STEPS = 6 * N + M, K_EPRET = K_STEPS + 1;
    constexpr bool OBS_BULK = gcd_c(D, 32) <= 2;
    constexpr int STRIDE = OBS_BULK ? D : (D | 1);
    extern __shared__ __align__(128) float tile[];
    const Topo topo;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t E = A.E;
    constexpr int kBlock = 128;
    const int64_t e0 = (int64_t)blockIdx.x * kMultiBlock;
    const int64_t e = e0 + tid;
    const bool valid = e < E;
    const int64_t tile_idx = (int64_t)blockIdx.x * (kMultiBlock / kBlock) + (tid >> 7);
    float4* const base = reinterpret_cast<float4*>(A.state_packed) + tile_idx * (R4 * kBlock) + (tid & 127);

    if (valid) {
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
        const uint32_t si0 = step_index_of(A);
        const float* ap = A.action ? A.action + e * M : nullptr;

        // the first step's actions; inside the loop step t + 1's are requested before step t's physics
        float act[M > 0 ? M : 1];
#pragma unroll
        for (int m = 0; m < M; m++) act[m] = ap ? __ldg(ap + m) : 0.0f;

#pragma unroll 1
        for (int t = 0; t < n_steps; t++) {
#if WG_MULTI_SYNC
            if (e0 + kMultiBlock <= E)      // whole CTA valid: the warps of one scheduler start every step together
                asm volatile("bar.sync %0, %1;" ::"r"(1 + (warp & 3)), "r"(kMultiBlock / 4) : "memory");
#endif
            // ---- Creature.act ----
            if constexpr (GEN) {                // generated on chip from the env's own step counter: no action memory
#pragma unroll
                for (int m = 0; m < M; m++) {
                    float x = st.mx(m) + gen_action(G, m, stp);
                    if (A.bv.mlo[m] > x) x = A.bv.mlo[m];
                    if (A.bv.mhi[m] < x) x = A.bv.mhi[m];
                    st.mx(m) = x;
                }
            } else if (ap) {
#pragma unroll
                for (int m = 0; m < M; m++) {
                    float x = st.mx(m) + act[m];
                    if (A.bv.mlo[m] > x) x = A.bv.mlo[m];       // python max(x, lo)
                    if (A.bv.mhi[m] < x) x = A.bv.mhi[m];       // python min(x, hi)
                    st.mx(m) = x;
                }
                if (t + 1 < n_steps) {
                    ap += act_stride;
#pragma unroll
                    for (int m = 0; m < M; m++) act[m] = __ldg(ap + m);
                }
            }
            // ---- k_sub x (_run_physics + run1), reward / done ----
            for (int k = 0; k < A.ec.k_sub; k++) (void)run_physics<IN3D, MM>(topo, A.bv, A.ec, st);
            const int32_t sn = stp + 1;
            float ysr[N], spr[N];
            EpiOut o;
            epilogue<IN3D, NF>(topo, A.bv, A.ec, st, sn, false, false, NF && A.truncated != nullptr,
                           [&](int i) -> float& { return ysr[i]; }, [&](int i) -> float& { return spr[i]; }, o);
            stp = sn;
            {
                const float r = epr + o.reward;
                if (o.done) account_episode<NF>(A, E, e, r, sn);
                epr = (o.done && A.ec.auto_reset) ? 0.0f : r;
            }
            if (o.done && A.ec.auto_reset) {
                apply_reset<IN3D>(topo, A.bv, A.ec, st, A.ec.auto_reset, A.noise, E, e, si0 + (uint32_t)t);
                stp = 0;
            }
            if (A.reward) A.reward[(int64_t)t * E + e] = o.reward;
            if (A.done) A.done[(int64_t)t * E + e] = (uint8_t)o.done;
            if (NF && A.truncated) A.truncated[(int64_t)t * E + e] = (uint8_t)o.trunc;
        }

        if (A.obs) {
            float* row = tile + tid * STRIDE;
            get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float val) { row[k] = val; });
        }
#pragma unroll
        for (int k = 0; k < 3 * N; k++) { v[k] = st.p_[k / 3][k % 3]; v[3 * N + k] = st.v_[k / 3][k % 3]; }
#pragma unroll
        for (int m = 0; m < M; m++) v[K_MX + m] = st.mx(m);
        v[K_STEPS] = __int_as_float(stp);
        v[K_EPRET] = epr;
#pragma unroll
        for (int g = 0; g < R4; g++) base[g * kBlock] = make_float4(v[4 * g + 0], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
    }
    // ---- row-major observation of the last step: one TMA bulk store per warp (or the padded-tile copy-out) ----
    if (A.obs) {
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

#ifndef __CUDACC_RTC__          // host-side launch helpers (not part of a run-time compiled translation unit)
static_assert(sizeof(ActionGen) == sizeof(wg_action_gen) && kGenRows == WG_GEN_MAX_ROWS && kGenMuscle == WG_GEN_MAX_MUSCLE,
              "ActionGen mirrors wg_action_gen");
inline void fill_gen(ActionGen& G, const wg_buffers* b) {
    if (b->action_gen && b->action_gen->mode != 0) memcpy(&G, b->action_gen, sizeof(G));
    else { G.mode = 0; G.n_rows = 1; G.hold = 1; }
}

template <class Topo, bool IN3D, int MM>
inline int launch_multi_packed(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, int n_steps,
                               int64_t act_stride, cudaStream_t s) {
    StepArgs<Topo::N, Topo::S> A;
    fill_args(A, t, p, b, E);
    constexpr int D = 3 * (IN3D ? 3 : 2) * Topo::N + Topo::M;
    constexpr bool bulk = gcd_c(D, 32) <= 2;
    const size_t smem = b->obs ? sizeof(float) * kMultiBlock * (bulk ? D : (D | 1)) : 0;
    static thread_local ActionGen G;
    fill_gen(G, b);
    using SA = StepArgs<Topo::N, Topo::S>;
    const bool nf = p->end_nonfinite || b->nf_stats || b->truncated;
    auto kern = G.mode ? (nf ? step_multi_packed_kernel<Topo, IN3D, MM, SA, true, true> : step_multi_packed_kernel<Topo, IN3D, MM, SA, true, false>)
                       : (nf ? step_multi_packed_kernel<Topo, IN3D, MM, SA, false, true> : step_multi_packed_kernel<Topo, IN3D, MM, SA, false, false>);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(unsigned)((E + kMultiBlock - 1) / kMultiBlock), kMultiBlock, smem, s>>>(A, n_steps, act_stride, G);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "step kernel (multi) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// unit masses (mode 0) or unit / power-of-two / small-integer masses (mode 1); 2-D and 3-D
template <class Topo>
inline int launch_multi_flags(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, int n_steps,
                              int64_t act_stride, cudaStream_t s) {
    if (mass_mode(t) == 0)
        return p->in3d ? launch_multi_packed<Topo, true, 0>(t, p, b, E, n_steps, act_stride, s)
                       : launch_multi_packed<Topo, false, 0>(t, p, b, E, n_steps, act_stride, s);
    return p->in3d ? launch_multi_packed<Topo, true, 1>(t, p, b, E, n_steps, act_stride, s)
                   : launch_multi_packed<Topo, false, 1>(t, p, b, E, n_steps, act_stride, s);
}
#endif

}  // namespace wg
