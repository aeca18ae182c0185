// wg_launch.cuh -- host-side launch helpers shared by the per-morphology translation units.
#pragma once
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "../../include/walker_gym_b200.h"
#include "wg_kernels.cuh"
#include "wg_kernels_tma.cuh"
#include "wg_kernels_part.cuh"
#include "wg_kernels_packed.cuh"

namespace wg {

int fail(int code, const char* fmt, const char* a = "");
int tuning(int key);      // current value of a WG_TUNE_* knob (wg_abi.cu)

// ---- register-resident specialisations --------------------------------------------
// endpoints listed as (p1, p2) pairs, muscles first then skeletons (Creature.run order)
// Balance-v0: gym/optimized_walker.py:176-199 (also walker.py balance/balance2/balance3)
WG_STATIC_TOPO(TopoBalance, 1, 4, 5, 2, 0,2, 1,2, 0,1, 0,3, 1,3)
// Balance-v0 with the mass pattern of create_balance_creature ([k, k, 1, j]: point 2 has unit mass, points 0 and 1
// share one): mass mode 3 skips the unit-mass divisions and shares the quotients of the (0,1) bone at compile time
struct TopoBalanceV0 : TopoBalance {
    __host__ __device__ static constexpr bool unit(int n) { return n == 2; }
    __host__ __device__ static constexpr bool same(int i, int j) { return (i == 0 && j == 1) || (i == 1 && j == 0); }
};
// Box-v0: gym/optimized_walker.py:201-224 (== walker.py box2)
WG_STATIC_TOPO(TopoBox, 2, 4, 5, 4, 0,1, 0,2, 3,1, 3,2, 1,2)
// 4x Balance in one env (N=16, S=20, M=8): the enlarged morphology of BASELINE config 4.
// muscles of unit u: (4u+0,4u+2),(4u+1,4u+2); skeletons: (4u+0,4u+1),(4u+0,4u+3),(4u+1,4u+3)
WG_STATIC_TOPO(TopoQuad, 3, 16, 20, 8,
               0,2, 1,2, 4,6, 5,6, 8,10, 9,10, 12,14, 13,14,
               0,1, 0,3, 1,3, 4,5, 4,7, 5,7, 8,9, 8,11, 9,11, 12,13, 12,15, 13,15)
// walker.py insect (:255-293): N=13, 8 muscles, 15 skeletons
WG_STATIC_TOPO(TopoInsect, 4, 13, 23, 8,
               9,4, 9,5, 10,5, 10,6, 11,6, 11,7, 12,7, 12,8,
               0,1, 0,4, 0,5, 1,2, 1,5, 1,6, 2,3, 2,6, 2,7, 3,7, 3,8, 4,5, 5,6, 6,7, 7,8)

// Smaller walker.py bodies (gym/walker.py:112-353; spring order = muscles then skeletons as the builders list them):
// packed-state kernels only.
WG_STATIC_TOPO(TopoLegacyBox, 5, 4, 5, 2, 0,2, 1,3, 0,1, 1,2, 2,3)                       // box (:160-171)
WG_STATIC_TOPO(TopoTest, 6, 4, 6, 1, 1,2, 0,1, 0,3, 2,3, 0,2, 1,3)                       // test (:112-136)
WG_STATIC_TOPO(TopoIntrian, 7, 3, 3, 3, 0,2, 1,2, 0,1)                                   // intrian (:225-234)
WG_STATIC_TOPO(TopoHat, 8, 5, 7, 4, 1,3, 1,4, 2,3, 2,4, 0,1, 0,2, 1,2)                   // hat (:339-353)
WG_STATIC_TOPO(TopoHumanb, 9, 6, 9, 4, 2,4, 2,5, 3,4, 3,5, 0,1, 0,2, 1,2, 1,3, 2,3)      // humanb (:236-253)
WG_STATIC_TOPO(TopoBox4, 10, 6, 9, 8, 0,2, 0,3, 0,4, 0,5, 1,2, 1,3, 1,4, 1,5, 0,1)       // box4 (:295-312)
WG_STATIC_TOPO(TopoLeg2, 11, 7, 11, 4, 1,3, 4,6, 0,2, 0,5, 0,1, 0,4, 1,4, 1,2, 2,3, 4,5, 5,6)              // leg2 (:138-158)
WG_STATIC_TOPO(TopoLeg, 12, 8, 13, 3, 1,3, 2,4, 5,7, 0,1, 0,2, 1,2, 2,3, 3,4, 3,5, 4,5, 4,6, 5,6, 6,7)     // leg (:314-337)
int launch_leg2_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_leg_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_legacy_box_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_test_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_intrian_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_hat_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_humanb_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_box4_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);

// one entry point per translation unit (ept = envs per thread the caller verified as legal)
int launch_balance(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int ept, cudaStream_t);
int launch_balance_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_box_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_box(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int ept, cudaStream_t);
int launch_quad(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int ept, cudaStream_t);
int launch_insect(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int ept, cudaStream_t);
int launch_generic_step(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_part_step(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int parts, cudaStream_t);
int launch_reset(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int mode, const uint8_t* mask, cudaStream_t);
int launch_stats(const float* fin_stats, const float* nf_stats, int64_t E, double* out8, cudaStream_t);

// classify a host-known divisor for div_const (see wg_math.cuh)
inline ConstDiv make_const_div(float m) {
    ConstDiv c; c.m = m; c.r = 1.0f / m; c.kind = 3;
    int ex = 0;
    const float fr = frexpf(m, &ex);
    if (m == 1.0f) c.kind = 0;
    else if (fr == 0.5f && ex > -100 && ex < 100) c.kind = 1;              // power of two: reciprocal exact
    // odd integers only: for an even m that is not a power of two, x / m can fall exactly halfway between two
    // SUBNORMAL float32 values (x = (2k+1) * (m/2) * 2^-149), and the 3-FMA quotient, which works with the inexact
    // RN(1/m), breaks such ties the wrong way (found by wg_selftest_div_smallint: 2 796 202 of the 2^32 x for m = 6);
    // with an odd m no quotient is ever a tie.  Even non-powers of two take the IEEE division.
    else if (m >= 3.0f && m <= 2047.0f && m == floorf(m) && fmodf(m, 2.0f) == 1.0f) c.kind = 2;
    return c;
}

template <int MAXN, int MAXS>
inline void fill_args(StepArgs<MAXN, MAXS>& A, const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E) {
    memset(&A, 0, sizeof(A));
    auto& bv = A.bv;
    bv.n_mass = t->n_mass; bv.n_spring = t->n_spring; bv.n_muscle = t->n_muscle;
    for (int n = 0; n < t->n_mass; n++) {
        bv.mass_d[n] = t->mass[n];
        bv.mass_f[n] = (float)t->mass[n];
        const ConstDiv cd = make_const_div(bv.mass_f[n]);
        bv.mass_r[n] = cd.r; bv.mass_kind[n] = cd.kind;
        bv.mass_rd[n] = 1.0 / t->mass[n];
        bv.gm[n] = (-p->g) / t->mass[n];                  // np.asarray([0,-g,0]) / m  (float64)
        bv.mg_f[n] = (float)(t->mass[n] * p->g);          // python m*g, then float32 at the multiply
        if (t->fixed[n]) bv.fixed_mask |= 1u << n;
        if (t->mass[n] == 1.0) bv.unit_mask |= 1u << n;
        for (int c = 0; c < 3; c++) bv.tmpl[n * 3 + c] = t->tmpl_pos[n * 3 + c];
    }
    for (int s = 0; s < t->n_spring; s++) {
        bv.si[s] = t->si[s]; bv.sj[s] = t->sj[s];
        bv.sk[s] = t->sk[s]; bv.sdamp[s] = t->sdamp[s]; bv.srest[s] = t->srest[s];
        bv.mlo[s] = t->mlo[s]; bv.mhi[s] = t->mhi[s];
        if (t->sstring[s]) bv.string_mask[s >> 5] |= 1u << (s & 31);
    }
    bv.ndiv = make_const_div((float)t->n_mass);
    auto& ec = A.ec;
    ec.ndampk = -p->dampk;
    ec.dampk_is_zero = (p->dampk == 0.0f);
    ec.ground = p->ground; ec.fall_thresh = p->fall_thresh;
    ec.nground_k = -p->ground_k; ec.nground_damp = -p->ground_damp; ec.friction = p->friction;
    ec.dt = p->dt; ec.dt2 = p->dt2; ec.sigma = p->sigma; ec.integrator = p->integrator;
    ec.max_steps = p->max_steps; ec.k_sub = p->k_sub; ec.auto_reset = p->auto_reset;
    ec.seed_lo = p->seed_lo; ec.seed_hi = p->seed_hi; ec.step_index = p->step_index; ec.env_offset = p->env_offset;
    ec.end_nonfinite = p->end_nonfinite;
    A.nf_stats = b->nf_stats; A.truncated = b->truncated; A.final_obs = b->final_obs;
    A.pos = b->pos; A.vel = b->vel; A.old_a = b->old_a; A.mx = b->mx; A.steps = b->steps;
    A.action = b->action; A.obs = b->obs; A.reward = b->reward; A.done = b->done;
    A.contact_pre = b->contact_pre; A.contact_post = b->contact_post; A.energy = b->energy; A.centroid = b->centroid;
    A.ep_ret = b->ep_ret; A.fin_stats = b->fin_stats; A.noise = b->noise;
    A.step_counter = b->step_counter; A.state_packed = b->state_packed;
    A.pf_dist = tuning(WG_TUNE_L2_PREFETCH);
    A.E = E; A.act_dim = b->action ? b->act_dim : 0; A.act_layout = b->act_layout;
}

// body-wide mass mode (see forced2): 0 all unit, 1 unit / power of two / small integer, 2 general
inline int mass_mode(const wg_topology* t) {
    int mode = 0;
    for (int n = 0; n < t->n_mass; n++) {
        const int k = make_const_div((float)t->mass[n]).kind;
        if (k == 3) return 2;
        if (k != 0) mode = 1;
    }
    return mode;
}

template <class Topo, bool IN3D, int OBS, int EPT, int MM>
inline int launch_static(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    StepArgs<Topo::N, Topo::S> A;
    fill_args(A, t, p, b, E);
    constexpr int D = 3 * (IN3D ? 3 : 2) * Topo::N + Topo::M;
    constexpr bool bulk = (OBS == 1) && (EPT == 1) && gcd_c(D, 32) <= 2;      // must mirror the kernel's OBS_BULK
    const size_t smem = (OBS == 1 && b->obs) ? sizeof(float) * kBlock * EPT * (bulk ? D : (D | 1)) : 0;
    auto kern = step_static_kernel<Topo, IN3D, OBS, EPT, MM>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    const int64_t tile = (int64_t)kBlock * EPT;
    const unsigned grid = (unsigned)((E + tile - 1) / tile);
    kern<<<grid, kBlock, smem, s>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "step kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// ---- persistent TMA-pipelined variant ----------------------------------------------------------
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// every bulk copy needs 16-byte aligned addresses and sizes: E % 4 == 0 and aligned base pointers
inline bool tma_ok(const wg_buffers* b, int64_t E) {
    if (!tuning(WG_TUNE_TMA) || (E % 4) != 0) return false;
    return aligned16(b->pos) && aligned16(b->vel) && aligned16(b->mx) && aligned16(b->steps) &&
           aligned16(b->ep_ret) && aligned16(b->action) && aligned16(b->obs);
}

template <class Topo, bool IN3D, int OBS, int MM>
inline int launch_static_tma(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    using LY = TmaLayout<Topo, IN3D>;
    StepArgs<Topo::N, Topo::S> A;
    fill_args(A, t, p, b, E);
    const size_t smem = LY::smem_bytes(OBS == 1 && b->obs);
    auto kern = step_static_tma_kernel<Topo, IN3D, OBS, MM>;
    static thread_local int cached_dev = -1, ctas_per_sm = 0, n_sm = 0;
    static thread_local size_t cached_smem = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev || smem != cached_smem) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, kBlock, smem);
        if (e != cudaSuccess || ctas_per_sm < 1) return fail(WG_ERR_CUDA, "occupancy query: %s", cudaGetErrorString(e));
        cached_dev = dev; cached_smem = smem;
    }
    const int64_t n_tiles = (E + kBlock - 1) / kBlock;
    const int64_t resident = (int64_t)n_sm * ctas_per_sm;        // persistent grid: a multiple of the SM count
    const unsigned grid = (unsigned)(n_tiles < resident ? n_tiles : resident);
    kern<<<grid, kBlock, smem, s>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "step kernel (tma) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// SMs of the current device (cached per thread and device)
inline int sm_count() {
    static thread_local int dev_cached = -1, sms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev != dev_cached) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) sms = v;
        dev_cached = dev;
    }
    return sms;
}

// ---- packed state layout: float4 state access --------------------------------------------------------
template <class Topo, bool IN3D, int OBS, int MM>
inline int launch_static_packed(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    StepArgs<Topo::N, Topo::S> A;
    fill_args(A, t, p, b, E);
    constexpr int D = 3 * (IN3D ? 3 : 2) * Topo::N + Topo::M;
    constexpr bool bulk = (OBS == 1) && gcd_c(D, 32) <= 2;
    const size_t smem = (OBS == 1 && b->obs) ? sizeof(float) * kPackedBlock * (bulk ? D : (D | 1)) : 0;
    using SA = StepArgs<Topo::N, Topo::S>;
    const bool nf = p->end_nonfinite || b->nf_stats || b->truncated || b->final_obs;   // compiled into NF = true only
    auto kern = nf ? step_static_packed_kernel<Topo, IN3D, OBS, MM, SA, true> : step_static_packed_kernel<Topo, IN3D, OBS, MM, SA, false>;
    const int64_t n_blocks = (E + kPackedBlock - 1) / kPackedBlock;
    if constexpr (Topo::N <= 4 && IN3D && OBS == 1 && (MM == 0 || MM == 3) && WG_PACKED_MIN_BLOCKS == 6 && WG_PACKED_BLOCK == 128) {
        // a grid of (6, 7] CTAs per SM: one wave with the 7-CTA instance instead of one full wave plus a sliver
        const int64_t sms = sm_count();
        if (n_blocks > 6 * sms && n_blocks <= 7 * sms)
            kern = nf ? step_static_packed_kernel<Topo, IN3D, OBS, MM, SA, true, 7> : step_static_packed_kernel<Topo, IN3D, OBS, MM, SA, false, 7>;
    }
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    cudaError_t e;
    if (tuning(WG_TUNE_PDL)) {            // programmatic dependent launch: see the top of step_static_packed_kernel
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)n_blocks); cfg.blockDim = dim3(kPackedBlock); cfg.dynamicSmemBytes = smem; cfg.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, kern, A);
    } else {
        kern<<<(unsigned)n_blocks, kPackedBlock, smem, s>>>(A);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "step kernel (packed) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// GENERAL = true also instantiates mass mode 2 (arbitrary masses, DingPoints) for this topology
template <class Topo, bool GENERAL = false>
inline int launch_packed_flags(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    int mm = mass_mode(t);
    for (int n = 0; n < t->n_mass; n++) if (t->fixed[n]) mm = 2;
    const bool rm = b->obs_layout == 0;
    if (mm == 2) {
        if constexpr (GENERAL) {
#define WG_PK2(I3, OB) launch_static_packed<Topo, I3, OB, 2>(t, p, b, E, s)
            if (p->in3d) return rm ? WG_PK2(true, 1) : WG_PK2(true, 0);
            return rm ? WG_PK2(false, 1) : WG_PK2(false, 0);
#undef WG_PK2
        } else {
            return fail(WG_ERR_BAD_ARG, "this body's packed kernel needs unit / power-of-two / small-integer masses and no DingPoints%s");
        }
    }
    if constexpr (GENERAL) {          // the Balance spring graph: is it also Balance-v0's mass pattern?
        if (mm == 1 && t->mass[2] == 1.0 && t->mass[0] == t->mass[1] && t->mass[0] != 1.0 && t->mass[3] != 1.0) {
#define WG_PK3(I3, OB) launch_static_packed<TopoBalanceV0, I3, OB, 3>(t, p, b, E, s)
            if (p->in3d) return rm ? WG_PK3(true, 1) : WG_PK3(true, 0);
            return rm ? WG_PK3(false, 1) : WG_PK3(false, 0);
#undef WG_PK3
        }
    }
#define WG_PK(I3, OB) (mm == 0 ? launch_static_packed<Topo, I3, OB, 0>(t, p, b, E, s) : launch_static_packed<Topo, I3, OB, 1>(t, p, b, E, s))
    if (p->in3d) return rm ? WG_PK(true, 1) : WG_PK(true, 0);
    return rm ? WG_PK(false, 1) : WG_PK(false, 0);
#undef WG_PK
}

template <class Topo, bool IN3D, int EPT, int MM>
inline int launch_static_obs(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    const int om = b->obs_layout == 1 ? 0 : 1;       // OBS template value: 0 feature-major, 1 row-major
    if constexpr (EPT == 1 && Topo::N <= 4) {
        if (tma_ok(b, E))
            return om == 0 ? launch_static_tma<Topo, IN3D, 0, MM>(t, p, b, E, s) : launch_static_tma<Topo, IN3D, 1, MM>(t, p, b, E, s);
    }
    return om == 0 ? launch_static<Topo, IN3D, 0, EPT, MM>(t, p, b, E, s) : launch_static<Topo, IN3D, 1, EPT, MM>(t, p, b, E, s);
}

// static kernels exist for mass modes 0 and 1; bodies with arbitrary masses use the generic kernel
template <class Topo, int EPT>
inline int launch_static_flags(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    const int mm = mass_mode(t);
    if (p->in3d) return mm == 0 ? launch_static_obs<Topo, true, EPT, 0>(t, p, b, E, s) : launch_static_obs<Topo, true, EPT, 1>(t, p, b, E, s);
    return mm == 0 ? launch_static_obs<Topo, false, EPT, 0>(t, p, b, E, s) : launch_static_obs<Topo, false, EPT, 1>(t, p, b, E, s);
}

}  // namespace wg
