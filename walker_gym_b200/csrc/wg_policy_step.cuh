// wg_policy_step.cuh -- the env step of BASELINE config 5 fused INTO the policy pipeline (wg_policy_ws.cuh): the output
// warps that have just sampled an env's action also run that env's PhysicsEnv.step -- the same device functions as the
// packed step kernel (wg_kernels_packed.cuh: Creature.act, k_sub x _run_physics, reward / done / info, episode statistics,
// auto-reset, observation), on the same packed state layout, bit for bit -- instead of a second kernel that has to wait
// for the whole policy grid.  The step's ~1400 instructions per env fill issue slots the pipeline leaves idle (it is
// bound by the XU pipe and by stage latencies at ~60 % issue utilisation), the action never leaves registers, and one
// launch per env step remains.
#pragma once
#include "wg_kernels_packed.cuh"

namespace wg {

struct NoStep {                                   // wg_policy_act: the policy alone
    static constexpr bool kFused = false;
    static constexpr int kObsFloats = 0, kStateRegs = 1;
};

template <class Topo, bool IN3D, int MM>
struct FusedStep {
    static constexpr bool kFused = true;
    static constexpr int N = Topo::N, M = Topo::M, D = 3 * (IN3D ? 3 : 2) * N + M;
    static constexpr int R = 6 * N + M + 2, R4 = (R + 3) / 4, kStateRegs = 4 * R4;
    static constexpr int K_MX = 6 * N, K_STEPS = 6 * N + M, K_EPRET = K_STEPS + 1;
    static constexpr int kObsFloats = kTcTile * D;               // the tile's next observations, staged for TMA bulk stores
    StepArgs<N, Topo::S> A;

    __device__ __forceinline__ float4* base(int64_t tile, int row) const {
        return reinterpret_cast<float4*>(A.state_packed) + tile * (R4 * 128) + row;
    }
    // the env's packed state: R4 coalesced 16-byte loads, issued before the output warp waits for the heads
    __device__ __forceinline__ void load(float (&v)[kStateRegs], int64_t tile, int row) const {
        const float4* b = base(tile, row);
#pragma unroll
        for (int g = 0; g < R4; g++) {
            const float4 q = b[g * 128];
            v[4 * g + 0] = q.x; v[4 * g + 1] = q.y; v[4 * g + 2] = q.z; v[4 * g + 3] = q.w;
        }
    }
    // PhysicsEnv.step of env e with the action in registers; the observation row goes to obs_row (shared memory)
    __device__ __forceinline__ void step(float (&v)[kStateRegs], const float (&act)[M > 0 ? M : 1], int64_t tile, int row,
                                         int64_t e, float* obs_row) const {
        const Topo topo;
        const int64_t E = A.E;
        RegStore<N, M> st;
#pragma unroll
        for (int k = 0; k < 3 * N; k++) { st.p_[k / 3][k % 3] = v[k]; st.v_[k / 3][k % 3] = v[3 * N + k]; }
#pragma unroll
        for (int m = 0; m < M; m++) st.mx(m) = v[K_MX + m];
        int32_t stp = __float_as_int(v[K_STEPS]);
        float epr = v[K_EPRET];
#pragma unroll
        for (int m = 0; m < M; m++) {                            // Creature.act: add, then regulation()
            float x = st.mx(m) + act[m];
            if (A.bv.mlo[m] > x) x = A.bv.mlo[m];                // python max(x, lo)
            if (A.bv.mhi[m] < x) x = A.bv.mhi[m];                // python min(x, hi)
            st.mx(m) = x;
        }
        uint32_t cp = 0;
        for (int k = 0; k < A.ec.k_sub; k++) cp = run_physics<IN3D, MM>(topo, A.bv, A.ec, st);
        const int32_t sn = stp + 1;
        float ysr[N], spr[N];
        EpiOut o;
        epilogue<IN3D>(topo, A.bv, A.ec, st, sn, A.energy != nullptr, A.centroid != nullptr, false,
                       [&](int i) -> float& { return ysr[i]; }, [&](int i) -> float& { return spr[i]; }, o);
        stp = sn;
        {   // episode statistics: the running return lives in the packed state
            const float r = epr + o.reward;
            if (o.done) account_episode(A, E, e, r, sn);
            epr = (o.done && A.ec.auto_reset) ? 0.0f : r;
        }
        if (o.done && A.ec.auto_reset) {
            apply_reset<IN3D>(topo, A.bv, A.ec, st, A.ec.auto_reset, A.noise, E, e, step_index_of(A));
            stp = 0;
        }
        get_obs<IN3D>(topo, A.bv.ndiv, st, [&](int k, float val) { obs_row[k] = val; });
#pragma unroll
        for (int k = 0; k < 3 * N; k++) { v[k] = st.p_[k / 3][k % 3]; v[3 * N + k] = st.v_[k / 3][k % 3]; }
#pragma unroll
        for (int m = 0; m < M; m++) v[K_MX + m] = st.mx(m);
        v[K_STEPS] = __int_as_float(stp);
        v[K_EPRET] = epr;
        float4* b = base(tile, row);
#pragma unroll
        for (int g = 0; g < R4; g++) b[g * 128] = make_float4(v[4 * g + 0], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
        if (A.old_a) {
#pragma unroll
            for (int k = 0; k < 3 * N; k++) A.old_a[(int64_t)k * E + e] = st.a_[k / 3][k % 3];
        }
        if (A.reward) A.reward[e] = o.reward;
        if (A.done) A.done[e] = (uint8_t)o.done;
        if (A.contact_pre) A.contact_pre[e] = cp;
        if (A.contact_post) A.contact_post[e] = o.cpost;
        if (A.energy) A.energy[e] = o.energy;
        if (A.centroid) { A.centroid[e] = o.cen[0]; A.centroid[E + e] = o.cen[1]; A.centroid[2 * E + e] = o.cen[2]; }
    }
};

}  // namespace wg
