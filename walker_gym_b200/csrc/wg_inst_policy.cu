// wg_inst_policy.cu -- rollout-side kernels: the fused MLP policy (wg_policy_act) and GAE (wg_gae).
#include "wg_launch.cuh"
#include "wg_policy.cuh"
#include "wg_policy_tc.cuh"
#include "wg_policy_ws.cuh"
namespace wg {

#ifndef WG_POLICY_MT
#define WG_POLICY_MT 1
#endif
template <int KT1, bool SPLIT>
static int launch_policy_t(const PolicyArgs& A, cudaStream_t s) {
    constexpr int MT = WG_POLICY_MT;
    auto kern = policy_act_kernel<KT1, SPLIT, MT>;
    const size_t smem = sizeof(uint32_t) * (size_t)PolicySmem<KT1>::words(SPLIT);
    static thread_local int cached_dev = -1, n_sm = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int64_t n_tiles = (A.E + kPolBlock - 1) / kPolBlock;
    const int64_t resident = (int64_t)n_sm * 2;                 // persistent: weights are staged once per CTA
    kern<<<(unsigned)(n_tiles < resident ? n_tiles : resident), 32 * (kPolBlock / (16 * MT)), smem, s>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "policy kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// ---- tcgen05 / TMEM variant (wg_policy_tc.cuh) ----
__device__ int g_policy_tc_error = 0;          // set by a CTA that gave up waiting for its MMAs (never in a correct build)

template <int K1, bool SPLIT>
static int launch_policy_tc_t(const PolicyArgs& A, cudaStream_t s) {
    auto kern = policy_act_tc_kernel<K1, SPLIT>;
    const size_t smem = TcSmem<K1>::bytes(A.D);
    static thread_local int cached_dev = -1, n_sm = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    int* flag = nullptr;
    cudaGetSymbolAddress((void**)&flag, g_policy_tc_error);
    const int64_t n_tiles = (A.E + kTcTile - 1) / kTcTile;
    const int64_t resident = (int64_t)n_sm * (smem * 2 <= 227 * 1024 ? 2 : 1);      // persistent: weights staged once per CTA
    kern<<<(unsigned)(n_tiles < resident ? n_tiles : resident), kTcThreads, smem, s>>>(A, flag);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "policy kernel (tcgen05) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

template <int K1, bool SPLIT, class SA = NoStep>
static int launch_policy_ws_t(const PolicyArgs& A, cudaStream_t s, const SA& S = SA{}) {
    auto kern = policy_act_ws_kernel<K1, SPLIT, SA>;
    const size_t smem = WsSmem<K1, SA::kObsFloats * WsCfg<SA>::kGroupsO>::bytes(A.D);
    static thread_local int cached_dev = -1, n_sm = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    int* flag = nullptr;
    cudaGetSymbolAddress((void**)&flag, g_policy_tc_error);
    const int64_t n_tiles = (A.E + kTcTile - 1) / kTcTile;
    const unsigned grid = (unsigned)(n_tiles < n_sm ? n_tiles : n_sm);                       // one persistent CTA per SM
    if (tuning(WG_TUNE_PDL)) {           // programmatic dependent launch: the kernel's prologue overlaps the previous kernel's tail
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(WsCfg<SA>::kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, kern, A, flag, S);
    } else {
        kern<<<grid, WsCfg<SA>::kThreads, smem, s>>>(A, flag, S);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "policy kernel (tcgen05, warp-specialised) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

// wg_policy_step: the policy pipeline with the env step fused into its output warps (Balance-v0's body and mass pattern,
// 3-D, packed state, row-major observations and actions -- BASELINE config 5's environment)
int launch_policy_step(const PolicyArgs& A, int precision, const wg_topology* t, const wg_params* p, const wg_buffers* b,
                       int64_t E, cudaStream_t s) {
    using SA = FusedStep<TopoBalanceV0, true, 3>;
    static_assert(SA::D == 38 && SA::M == 2, "Balance-v0 in 3-D");
    SA S;
    fill_args(S.A, t, p, b, E);
    return precision == 0 ? launch_policy_ws_t<40, true, SA>(A, s, S) : launch_policy_ws_t<40, false, SA>(A, s, S);
}

int policy_tc_error() {
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_policy_tc_error, sizeof(int)) != cudaSuccess) return -1;
    return v;
}

static int launch_policy_tc(const PolicyArgs& A, int precision, int variant, cudaStream_t s) {
    const int k1 = ((A.D + 1 + 7) / 8) * 8;          // obs_dim + the bias column, in k-steps of 8
#define WG_POLTC(K) (variant == 2 ? (precision == 0 ? launch_policy_ws_t<K, true>(A, s) : launch_policy_ws_t<K, false>(A, s)) \
                                  : (precision == 0 ? launch_policy_tc_t<K, true>(A, s) : launch_policy_tc_t<K, false>(A, s)))
    if (k1 <= 24) return WG_POLTC(24);
    if (k1 <= 32) return WG_POLTC(32);
    if (k1 <= 40) return WG_POLTC(40);
    if (k1 <= 48) return WG_POLTC(48);
    return WG_POLTC(72);
#undef WG_POLTC
}

int launch_policy(const PolicyArgs& A, int precision, cudaStream_t s) {
    if (tuning(WG_TUNE_POLICY_TC) > 0) return launch_policy_tc(A, precision, tuning(WG_TUNE_POLICY_TC), s);
    const int kt = (A.D + 7) / 8;
#define WG_POL(KT) (precision == 0 ? launch_policy_t<KT, true>(A, s) : launch_policy_t<KT, false>(A, s))
    if (kt <= 3) return WG_POL(3);
    if (kt <= 4) return WG_POL(4);
    if (kt <= 5) return WG_POL(5);
    return WG_POL(8);
#undef WG_POL
}

// Streaming probe: every thread reads R and writes W 16-byte vectors (coalesced planes), nothing else.  Measures the
// HBM rate a kernel with the step kernel's read : write mix can reach at all (bench.py --probe-stream).
__global__ void __launch_bounds__(128) stream_probe_kernel(const float4* __restrict__ src, float4* __restrict__ dst,
                                                           int64_t n, int R, int W) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < R; k++) { const float4 v = src[(int64_t)k * n + i]; acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
    for (int k = 0; k < W; k++) { acc.x += 1.0f; dst[(int64_t)k * n + i] = acc; }
}
int launch_stream_probe(const float* src, float* dst, int64_t n, int R, int W, cudaStream_t s) {
    stream_probe_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(reinterpret_cast<const float4*>(src),
                                                                    reinterpret_cast<float4*>(dst), n, R, W);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "stream probe launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

int launch_gae(const float* rewards, const float* values, const uint8_t* dones, float* adv, float* ret, int T, int64_t E,
               float gamma, float lam, float clip, cudaStream_t s) {
    gae_kernel<<<(unsigned)((E + 255) / 256), 256, 0, s>>>(rewards, values, dones, adv, ret, T, E, gamma, lam, clip);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "gae kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

int launch_gae_trunc(const float* rewards, const float* values, const uint8_t* dones, const uint8_t* truncated,
                     const float* final_values, float* adv, float* ret, int T, int64_t E, float gamma, float lam, float clip,
                     cudaStream_t s) {
    gae_trunc_kernel<<<(unsigned)((E + 255) / 256), 256, 0, s>>>(rewards, values, dones, truncated, final_values, adv, ret, T, E,
                                                                 gamma, lam, clip);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "gae (truncation) kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

}  // namespace wg
