// wg_policy.cuh -- the caller of the hot path (SURVEY 8 f1, BASELINE config 5): PPO rollout collection.
//
//   policy_act_kernel : obs [D][E] -> gaussian MLP policy (D -> 64 -> 64 -> {M means, 1 value}, tanh) ->
//                       sampled action [M][E], log-prob [E], value [E]; ONE launch per env step, reading the
//                       observation exactly as the step kernel wrote it (feature-major) and writing the action in
//                       the layout the step kernel reads.  The three small GEMMs run on the tensor cores
//                       (mma.sync m16n8k8 TF32; with SPLIT every product is the 3-term error-compensated
//                       a_hi*b_hi + a_lo*b_hi + a_hi*b_lo, i.e. float32-grade accuracy); activations never leave
//                       registers between layers: the k-slots of each MMA are permuted so that the accumulator
//                       fragment of one layer IS the A fragment of the next (no shuffles, no shared memory).
//   gae_kernel        : GAE(lambda) advantages / returns over a [T][E] trajectory, one thread per env.
//   gae_trunc_kernel  : the same with time-limit truncations bootstrapped from a value of the final state.
//
// This is floating-point ML glue, not the bit-exact physics: it is checked against a plain PyTorch float32
// reference with a stated tolerance (tests/test_cuda_policy.py).
#pragma once
#include "wg_math.cuh"

namespace wg {

constexpr int kPolH = 64;          // hidden width (both layers)
constexpr int kPolBlock = 128;     // 4 warps x 32 envs per tile

struct PolicyArgs {
    const float* w1; const float* b1;        // torch.nn.Linear layout: weight [64][D] row-major, bias [64]
    const float* w2; const float* b2;        // [64][64], [64]
    const float* w_mu; const float* b_mu;    // [M][64], [M]
    const float* w_v; const float* b_v;      // [1][64], [1]
    const float* log_std;                    // [M]
    const float* obs;                        // [D][E] feature-major (obs_layout 1) or [E][D] row-major (obs_layout 0)
    float* action;                           // [M][E] (act_layout 1) or [E][M] (act_layout 0); optional
    float* logp;                             // [E], optional
    float* value;                            // [E], optional
    float* mean;                             // [M][E], optional (the distribution mean, for the PPO update / tests)
    const uint32_t* step_counter;            // optional device scalar added to step_index (CUDA-graph replays)
    int64_t E;
    int32_t D, M, act_layout, sample;        // sample 0: action = mean
    int32_t obs_layout;
    float obs_scale, obs_clip;
    uint32_t seed_lo, seed_hi, step_index, env_offset;
};

__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// D(16x8) += A(16x8, row) * B(8x8, col); fragments per PTX ISA "mma.m16n8k8 .tf32"
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// Activation -> TF32 operand(s) WITHOUT the conversion unit: cvt.rna.tf32 issues on the XU pipe (16 lanes / clock / SM),
// which it shares with the tanh's MUFU operations and which ncu showed to be the busiest pipe of both policy kernels
// (45 %).  SPLIT: hi = the float32 rounded to 11 significant bits by integer arithmetic (add half an ulp of TF32 to the
// magnitude, clear the 13 low bits: round-to-nearest, ties away from zero == cvt.rna for every finite value whose
// rounding does not overflow -- activations are clipped observations and tanh outputs), lo = x - hi exactly (left as
// float32: the MMA reads only its TF32 bits, residual ~2^-22 |x|); a NaN activation stays NaN through lo.  Plain TF32:
// Veltkamp's split (three float32 operations on the FMA pipe; NaN-preserving, no integer wrap-around of a NaN).
template <bool SPLIT>
__device__ __forceinline__ void act_split(float x, uint32_t& hi, uint32_t& lo) {
    if (SPLIT) {
        hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
        lo = __float_as_uint(__fsub_rn(x, __uint_as_float(hi)));
    } else {
        const float c = __fmul_rn(x, 8193.0f);                 // 2^13 + 1: keeps 24 - 13 = 11 significant bits
        hi = __float_as_uint(__fadd_rn(c, __fsub_rn(x, c)));
        lo = 0u;
    }
}
template <bool SPLIT>
__device__ __forceinline__ void split4(const float (&x)[4], uint32_t (&hi)[4], uint32_t (&lo)[4]) {
#pragma unroll
    for (int i = 0; i < 4; i++) act_split<SPLIT>(x[i], hi[i], lo[i]);
}
// c += A * B with A given as float32 values (split on the fly) and B as pre-split hi / lo planes
template <bool SPLIT>
__device__ __forceinline__ void mma3(float (&c)[4], const uint32_t (&ahi)[4], const uint32_t (&alo)[4],
                                     uint2 bhi, uint2 blo) {
    if (SPLIT) {
        mma_tf32(c, alo, bhi.x, bhi.y);
        mma_tf32(c, ahi, blo.x, blo.y);
    }
    mma_tf32(c, ahi, bhi.x, bhi.y);
}
// tanh: SPLIT (float32-grade) 1 - 2 / (exp(2x) + 1) from ex2.approx / rcp.approx (abs error ~2e-7);
// otherwise the hardware tanh.approx (2^-11), matching the TF32 products it is used with
template <bool SPLIT>
__device__ __forceinline__ float pol_tanh(float x) {
    if (!SPLIT) {
        float y;
        asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    }
    float e;                              // no clamp needed: exp -> inf gives 1 - 2/inf = 1, exp -> 0 gives 1 - 2 = -1
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));      // exp(2x)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return __fmaf_rn(-2.0f, r, 1.0f);
}

// shared-memory planes of one weight matrix [n_rows][KP] (tf32 bit patterns), hi then lo
// PERM_KT > 0: the layer-1 input permutation -- physical column 8*kk + 2*t + j holds feature (2*PERM_KT)*t + 2*kk + j,
// so that the features one thread feeds into its A fragments over all k-tiles are contiguous in an observation row.
template <bool SPLIT, int PERM_KT = 0>
__device__ __forceinline__ void fill_plane(uint32_t* dst, int n_rows, int KP, int n_valid_rows, int k_valid,
                                           const float* __restrict__ w, int ld, const float* __restrict__ w_last) {
    // rows < n_valid_rows come from w (leading dimension ld); row n_valid_rows (if w_last) from w_last; rest 0
    for (int idx = threadIdx.x; idx < n_rows * KP; idx += blockDim.x) {
        const int n = idx / KP;
        int k = idx - n * KP;
        if (PERM_KT > 0) k = k < 8 * PERM_KT ? (2 * PERM_KT) * ((k & 7) >> 1) + 2 * (k >> 3) + (k & 1) : k_valid;
        float v = 0.0f;
        if (k < k_valid) {
            if (n < n_valid_rows) v = w[n * ld + k];
            else if (n == n_valid_rows && w_last) v = w_last[k];
        }
        const uint32_t hi = to_tf32(v);
        if (SPLIT) {
            // hi and lo of a column pair share one 16-byte vector {hi(k), hi(k+1), lo(k), lo(k+1)}: one LDS.128 per
            // B fragment instead of two LDS.64 (row pitch 2*KP words == 16 mod 32: conflict-free quarter-warps)
            const int kc = idx - n * KP;
            uint32_t* q = dst + ((size_t)n * KP + (kc & ~1)) * 2 + (kc & 1);
            q[0] = hi;
            q[2] = to_tf32(v - __uint_as_float(hi));
        } else {
            dst[idx] = hi;
        }
    }
}
// B fragment (b0, b1) of columns k, k+1 of row n: hi and lo planes
template <bool SPLIT>
__device__ __forceinline__ void load_b(const uint32_t* W, int n, int KP, int k, uint2& bhi, uint2& blo) {
    if (SPLIT) {
        const uint4 b = *reinterpret_cast<const uint4*>(W + ((size_t)n * KP + k) * 2);
        bhi = make_uint2(b.x, b.y); blo = make_uint2(b.z, b.w);
    } else {
        bhi = *reinterpret_cast<const uint2*>(W + (size_t)n * KP + k);
        blo = make_uint2(0u, 0u);
    }
}

template <int KT1>
struct PolicySmem {
    static constexpr int KP1 = KT1 <= 5 ? 40 : 72;     // row pitch == 8 (mod 32) words: conflict-free 64-bit fragment loads
    static constexpr int KP2 = 72;
    static constexpr int words(bool split) {
        return (split ? 2 : 1) * (kPolH * KP1 + kPolH * KP2 + 8 * KP2) + kPolH + kPolH + 8 + 8;
    }
};

// two standard normals for (env, step, action pair): Philox4x32-10 + Box-Muller (fast intrinsics: sampling noise
// is not part of any parity contract; it only has to be reproducible and independent of the sharding)
__device__ __forceinline__ float2 pol_normal2(uint32_t seed_lo, uint32_t seed_hi, uint32_t env, uint32_t step, uint32_t pair) {
    uint32_t c[4] = { env, step, pair, 0x504f4c31u };
    philox4x32_10(c, seed_lo, seed_hi);
    const float u1 = (float)((c[0] >> 8) + 1u) * (1.0f / 16777216.0f);
    const float u2 = (float)(c[1] >> 8) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, co;
    __sincosf(6.283185307179586f * u2, &s, &co);
    return make_float2(r * co, r * s);
}

// MT = m-tiles (16 envs each) per warp.  A CTA always covers a tile of 128 envs: 128 / (16 * MT) warps.  MT = 1
// (8 warps per CTA, ~120 registers, 16 warps per SM) overlaps tensor and ALU work better than MT = 2 (half the
// fragment loads per MMA, but only 8 warps per SM): measured 1.6x faster.
template <int KT1, bool SPLIT, int MT>
__global__ void __launch_bounds__(32 * (kPolBlock / (16 * MT)), 2)
policy_act_kernel(const __grid_constant__ PolicyArgs A) {
    using L = PolicySmem<KT1>;
    constexpr int KP1 = L::KP1, KP2 = L::KP2, NPL = SPLIT ? 2 : 1;
    extern __shared__ __align__(16) uint32_t psm[];
    uint32_t* const W1 = psm;                                  // [NPL][64][KP1]
    uint32_t* const W2 = W1 + NPL * kPolH * KP1;               // [NPL][64][KP2]
    uint32_t* const WH = W2 + NPL * kPolH * KP2;               // [NPL][8][KP2]: rows 0..M-1 means, row M value
    float* const B1 = reinterpret_cast<float*>(WH + NPL * 8 * KP2);
    float* const B2 = B1 + kPolH;
    float* const BH = B2 + kPolH;
    float* const LS = BH + 8;
    const int D = A.D, M = A.M;
    fill_plane<SPLIT, KT1>(W1, kPolH, KP1, kPolH, D, A.w1, D, nullptr);
    fill_plane<SPLIT>(W2, kPolH, KP2, kPolH, kPolH, A.w2, kPolH, nullptr);
    fill_plane<SPLIT>(WH, 8, KP2, M, kPolH, A.w_mu, kPolH, A.w_v);
    for (int i = threadIdx.x; i < kPolH; i += blockDim.x) { B1[i] = A.b1[i]; B2[i] = A.b2[i]; }
    if (threadIdx.x < 8) {
        const int n = threadIdx.x;
        BH[n] = n < M ? A.b_mu[n] : (n == M ? A.b_v[0] : 0.0f);
        LS[n] = n < M ? A.log_std[n] : 0.0f;
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int64_t E = A.E;
    const int64_t n_tiles = (E + kPolBlock - 1) / kPolBlock;
    const uint32_t step = A.step_index + (A.step_counter ? __ldg(A.step_counter) : 0u);
    const bool row_vec = (D % 2 == 0) && ((reinterpret_cast<uintptr_t>(A.obs) & 7u) == 0);

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t e0 = tile * kPolBlock + warp * (16 * MT);    // this warp: envs e0 .. e0 + 16*MT - 1
        if (e0 >= E) continue;
        // env rows of this thread's fragments: (mt, h) -> e0 + 16*mt + 8*h + g
        int64_t er[MT][2];
        bool ev[MT][2];
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
#pragma unroll
            for (int h = 0; h < 2; h++) { er[mt][h] = e0 + 16 * mt + 8 * h + g; ev[mt][h] = er[mt][h] < E; }

        // ---- layer 1: h1 = tanh(W1 x + b1); A fragments straight from the feature-major observation ----
        float acc[MT][8][4];
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
#pragma unroll
            for (int nt = 0; nt < 8; nt++)
#pragma unroll
                for (int i = 0; i < 4; i++) acc[mt][nt][i] = 0.0f;
#pragma unroll
        for (int kk = 0; kk < KT1; kk++) {
            // k-slot t <-> feature f0, slot t+4 <-> f1; over the k-tiles thread t covers features [2*KT1*t, 2*KT1*(t+1)):
            // contiguous bytes of a row-major observation row, so every 32-byte sector a warp touches is fully used
            const int f0 = 2 * KT1 * t + 2 * kk, f1 = f0 + 1;
            uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
            for (int mt = 0; mt < MT; mt++) {
                float x[4];                                              // a0 (g, f0), a1 (g+8, f0), a2 (g, f1), a3 (g+8, f1)
                if (A.obs_layout == 0 && row_vec) {
                    // row-major observation rows: features f0, f0+1 of one env are one aligned 8-byte load
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const float2 v = (f0 < D && ev[mt][h]) ? __ldg(reinterpret_cast<const float2*>(A.obs + er[mt][h] * D + f0))
                                                               : make_float2(0.0f, 0.0f);
                        x[h] = v.x; x[2 + h] = v.y;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int f = (i & 2) ? f1 : f0, h = i & 1;
                        x[i] = (f < D && ev[mt][h]) ? __ldg(A.obs + (A.obs_layout ? (int64_t)f * E + er[mt][h] : er[mt][h] * D + f)) : 0.0f;
                    }
                }
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    float v = x[i] * A.obs_scale;                        // nan_to_num + clamp of the torch reference
                    x[i] = (v != v) ? 0.0f : fminf(fmaxf(v, -A.obs_clip), A.obs_clip);
                }
                split4<SPLIT>(x, ahi[mt], alo[mt]);
            }
#pragma unroll
            for (int nt = 0; nt < 8; nt++) {
                uint2 bhi, blo;
                load_b<SPLIT>(W1, 8 * nt + g, KP1, 8 * kk + 2 * t, bhi, blo);
#pragma unroll
                for (int mt = 0; mt < MT; mt++) mma3<SPLIT>(acc[mt][nt], ahi[mt], alo[mt], bhi, blo);
            }
        }
        // bias + tanh, then split once into the A fragments of layer 2: accumulator (g,2t) (g,2t+1) (g+8,2t) (g+8,2t+1)
        // -> a0 a2 a1 a3 under the k-slot permutation
        uint32_t h1hi[MT][8][4], h1lo[MT][8][4];
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
#pragma unroll
            for (int nt = 0; nt < 8; nt++) {
                const float bA = B1[8 * nt + 2 * t], bB = B1[8 * nt + 2 * t + 1];
                const float x[4] = { pol_tanh<SPLIT>(acc[mt][nt][0] + bA), pol_tanh<SPLIT>(acc[mt][nt][2] + bA),
                                     pol_tanh<SPLIT>(acc[mt][nt][1] + bB), pol_tanh<SPLIT>(acc[mt][nt][3] + bB) };
                split4<SPLIT>(x, h1hi[mt][nt], h1lo[mt][nt]);
            }

        // ---- layer 2 + heads: n-tile nt2 of h2 is k-tile nt2 of the heads, so h2 is consumed group by group.
        // Four n-tiles x MT m-tiles are accumulated together: independent MMA chains keep the tensor pipe busy
        // (one chain per accumulator would serialise on the MMA latency).
        float hd[MT][4];
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
#pragma unroll
            for (int i = 0; i < 4; i++) hd[mt][i] = 0.0f;
#pragma unroll
        for (int grp = 0; grp < 2; grp++) {
            float a2[4][MT][4];
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int mt = 0; mt < MT; mt++)
#pragma unroll
                    for (int i = 0; i < 4; i++) a2[q][mt][i] = 0.0f;
#pragma unroll
            for (int kk = 0; kk < 8; kk++) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint2 bhi, blo;
                    load_b<SPLIT>(W2, 8 * (4 * grp + q) + g, KP2, 8 * kk + 2 * t, bhi, blo);
#pragma unroll
                    for (int mt = 0; mt < MT; mt++) mma3<SPLIT>(a2[q][mt], h1hi[mt][kk], h1lo[mt][kk], bhi, blo);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int nt2 = 4 * grp + q;
                const float bA = B2[8 * nt2 + 2 * t], bB = B2[8 * nt2 + 2 * t + 1];
                uint2 bhi, blo;
                load_b<SPLIT>(WH, g, KP2, 8 * nt2 + 2 * t, bhi, blo);
#pragma unroll
                for (int mt = 0; mt < MT; mt++) {
                    const float x[4] = { pol_tanh<SPLIT>(a2[q][mt][0] + bA), pol_tanh<SPLIT>(a2[q][mt][2] + bA),
                                         pol_tanh<SPLIT>(a2[q][mt][1] + bB), pol_tanh<SPLIT>(a2[q][mt][3] + bB) };
                    uint32_t ahi[4], alo[4];
                    split4<SPLIT>(x, ahi, alo);
                    mma3<SPLIT>(hd[mt], ahi, alo, bhi, blo);
                }
            }
        }

        // ---- gaussian noise: the tile needs one Philox + Box-Muller evaluation per (env row, action pair); spread them
        // over all lanes (evaluation q = pair * 16*MT + row on lane q % 32) instead of leaving them to the few lanes that
        // own an action pair, then hand each owner its pair with two shuffles ----
        constexpr int ROWS = 16 * MT, JMAX = (ROWS * 4 + 31) / 32;
        const int n_eval = A.sample ? ROWS * ((M + 1) / 2) : 0;
        float2 zq[JMAX];
#pragma unroll
        for (int j = 0; j < JMAX; j++) {
            zq[j] = make_float2(0.0f, 0.0f);
            if (32 * j < n_eval) {                                            // warp-uniform
                const int q = 32 * j + lane;
                const int64_t eq = e0 + q % ROWS;
                if (q < n_eval && eq < E)
                    zq[j] = pol_normal2(A.seed_lo, A.seed_hi, A.env_offset + (uint32_t)eq, step, (uint32_t)(q / ROWS));
            }
        }
        // ---- heads: this thread holds outputs n = 2t, 2t+1 of env rows (mt, h); n < M mean, n == M value ----
#pragma unroll
        for (int mt = 0; mt < MT; mt++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int64_t e = er[mt][h];
                float lp = 0.0f;
                float out[2] = { hd[mt][2 * h + 0] + BH[2 * t], hd[mt][2 * h + 1] + BH[2 * t + 1] };
                float2 z = make_float2(0.0f, 0.0f);
                const int qo = ROWS * t + 16 * mt + 8 * h + g;                // this thread's evaluation (pair t, its env row)
#pragma unroll
                for (int j = 0; j < JMAX; j++) {
                    if (32 * j < n_eval) {                                    // warp-uniform
                        const float zx = __shfl_sync(0xffffffffu, zq[j].x, qo & 31);
                        const float zy = __shfl_sync(0xffffffffu, zq[j].y, qo & 31);
                        if ((qo >> 5) == j) z = make_float2(zx, zy);
                    }
                }
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int n = 2 * t + j;
                    if (n < M) {
                        const float ls = LS[n], eps = j ? z.y : z.x;
                        const float act = A.sample ? __fmaf_rn(__expf(ls), eps, out[j]) : out[j];
                        lp += -0.5f * eps * eps - ls - 0.9189385332046727f;
                        if (ev[mt][h]) {
                            if (A.mean) A.mean[(int64_t)n * E + e] = out[j];
                            if (A.action) A.action[A.act_layout ? (int64_t)n * E + e : e * M + n] = act;
                        }
                    } else if (n == M && ev[mt][h] && A.value) {
                        A.value[e] = out[j];
                    }
                }
                lp += __shfl_xor_sync(0xffffffffu, lp, 1);
                lp += __shfl_xor_sync(0xffffffffu, lp, 2);
                if (t == 0 && ev[mt][h] && A.logp) A.logp[e] = lp;
            }
    }
}

// GAE(lambda): adv_t = delta_t + gamma*lam*nonterminal_t*adv_{t+1}, delta_t = r_t + gamma*V_{t+1}*nonterminal_t - V_t;
// returns = adv + V.  Rewards are sanitised the way the torch collector did (nan -> 0, clamp to +-clip).
static __global__ void __launch_bounds__(256)
gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values, const uint8_t* __restrict__ dones,
           float* __restrict__ adv, float* __restrict__ ret, int T, int64_t E, float gamma, float lam, float clip) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    float a = 0.0f, vnext = values[(int64_t)T * E + e];
    for (int t = T - 1; t >= 0; t--) {
        float r = rewards[(int64_t)t * E + e];
        r = (r != r) ? 0.0f : fminf(fmaxf(r, -clip), clip);
        const float nt = dones[(int64_t)t * E + e] ? 0.0f : 1.0f;
        const float v = values[(int64_t)t * E + e];
        const float delta = r + gamma * vnext * nt - v;
        a = delta + gamma * lam * nt * a;
        adv[(int64_t)t * E + e] = a;
        ret[(int64_t)t * E + e] = a + v;
        vnext = v;
    }
}

// GAE(lambda) that bootstraps time-limit truncations: the value after step t is V_{t+1} when the episode goes on, 0 when it
// terminated, and final_values_t when it was truncated (a done step with truncated_t set); the advantage carry is cut on
// every done.  final_values is sanitised like the rewards.  Selects only: final_values rows of the other envs are never
// read into the arithmetic, so garbage there (NaN, inf) cannot leak.  With no truncated step and finite values
// the bits are gae_kernel's.
static __global__ void __launch_bounds__(256)
gae_trunc_kernel(const float* __restrict__ rewards, const float* __restrict__ values, const uint8_t* __restrict__ dones,
                 const uint8_t* __restrict__ truncated, const float* __restrict__ final_values, float* __restrict__ adv,
                 float* __restrict__ ret, int T, int64_t E, float gamma, float lam, float clip) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    float a = 0.0f, vnext = values[(int64_t)T * E + e];
    for (int t = T - 1; t >= 0; t--) {
        const int64_t i = (int64_t)t * E + e;
        float r = rewards[i];
        r = (r != r) ? 0.0f : fminf(fmaxf(r, -clip), clip);
        const bool d = dones[i] != 0;
        float boot = vnext;
        if (d) {
            boot = 0.0f;
            if (truncated[i]) {
                const float f = final_values[i];
                boot = (f != f) ? 0.0f : fminf(fmaxf(f, -clip), clip);
            }
        }
        const float v = values[i];
        const float delta = r + gamma * boot - v;
        a = d ? delta : delta + gamma * lam * a;
        adv[i] = a;
        ret[i] = a + v;
        vnext = v;
    }
}

}  // namespace wg
