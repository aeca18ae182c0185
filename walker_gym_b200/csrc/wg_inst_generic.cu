// wg_inst_generic.cu -- run-time-topology step kernel, reset kernel (K2), stats reduction (K3).
#include <atomic>

#include "wg_launch.cuh"
namespace wg {
// the per-env tile of the run-time-topology kernel: 11 * N + M + 3 rows of kBlock + 1 floats (x64 mode included)
static size_t generic_smem(const wg_topology* t) {
    return sizeof(float) * (size_t)(11 * t->n_mass + t->n_muscle + 3) * (kBlock + 1);
}

// Dynamic shared memory a block of `kern` can have on the current device: the device's opt-in limit per block (queried
// once per device) less the kernel's static shared memory.
static int smem_room(const void* kern, size_t* room) {
    constexpr int kMaxDevices = 64;
    static std::atomic<int> optin[kMaxDevices];                 // 0 = not queried yet
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
    int lim = dev < kMaxDevices ? optin[dev].load(std::memory_order_relaxed) : 0;
    if (lim == 0) {
        e = cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
        if (dev < kMaxDevices) optin[dev].store(lim, std::memory_order_relaxed);
    }
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncGetAttributes: %s", cudaGetErrorString(e));
    *room = (size_t)lim > fa.sharedSizeBytes ? (size_t)lim - fa.sharedSizeBytes : 0;
    return WG_OK;
}

// x64 mode has only the run-time-topology kernel: a body whose tile does not fit a block is refused
template <bool IN3D, bool ROWMAJOR>
static int check_generic_x64(const wg_topology* t) {
    const size_t smem = generic_smem(t);
    if (smem <= 48 * 1024) return WG_OK;
    size_t room = 0;
    const int rc = smem_room((const void*)step_generic_kernel<IN3D, ROWMAJOR, X64Args>, &room);
    if (rc != WG_OK || smem <= room) return rc;
    char msg[256];
    snprintf(msg, sizeof(msg), "x64 mode: a body of %d masses and %d muscles needs %zu bytes of shared memory per block "
             "(11 * n_mass + n_muscle + 3 rows of %d floats), this device allows %zu for the %s-observation kernel",
             t->n_mass, t->n_muscle, smem, kBlock + 1, room, ROWMAJOR ? "row-major" : "feature-major");
    return fail(WG_ERR_UNSUPPORTED, "%s", msg);
}

int check_generic_step_x64(const wg_topology* t, const wg_params* p, const wg_buffers* b) {
    const bool rm = b->obs_layout == 0;
    if (p->in3d) return rm ? check_generic_x64<true, true>(t) : check_generic_x64<true, false>(t);
    return rm ? check_generic_x64<false, true>(t) : check_generic_x64<false, false>(t);
}

template <bool IN3D, bool ROWMAJOR>
static int launch_generic_x64(const wg_topology* t, const wg_x64* x, const wg_params* p, const wg_buffers* b, int64_t E,
                              cudaStream_t s) {
    static thread_local StepArgs<kMaxMass, kMaxSpring> A;
    static thread_local X64Args XA;
    fill_args(A, t, p, b, E);
    for (int k = 0; k < t->n_spring; k++) {
        XA.v.sk_d[k] = x->sk_d[k]; XA.v.x0_d[k] = x->x0_d[k]; XA.v.mlo_d[k] = x->mlo_d[k]; XA.v.mhi_d[k] = x->mhi_d[k];
    }
    XA.mx64 = b->mx64; XA.mx_weak = b->mx_weak; XA.action64 = b->action64;
    A.act_dim = b->action64 ? b->act_dim : 0;
    const size_t smem = generic_smem(t);
    auto kern = step_generic_kernel<IN3D, ROWMAJOR, X64Args>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    kern<<<(unsigned)((E + kBlock - 1) / kBlock), kBlock, smem, s>>>(A, XA);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "generic step kernel (x64) launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

int launch_generic_step_x64(const wg_topology* t, const wg_x64* x, const wg_params* p, const wg_buffers* b, int64_t E,
                            cudaStream_t s) {
    const bool rm = b->obs_layout == 0;
    if (p->in3d) return rm ? launch_generic_x64<true, true>(t, x, p, b, E, s) : launch_generic_x64<true, false>(t, x, p, b, E, s);
    return rm ? launch_generic_x64<false, true>(t, x, p, b, E, s) : launch_generic_x64<false, false>(t, x, p, b, E, s);
}

template <bool IN3D, bool ROWMAJOR>
static int launch_generic(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    StepArgs<kMaxMass, kMaxSpring> A;
    const size_t smem = generic_smem(t);
    auto kern = step_generic_kernel<IN3D, ROWMAJOR, NoX64>;
    if (smem > 48 * 1024) {
        // a tile too large for one block: the mass-partitioned kernel with two lanes per env computes the same bits
        // with about half of it per block
        size_t room = 0;
        const int rc = smem_room((const void*)kern, &room);
        if (rc != WG_OK) return rc;
        if (smem > room) return launch_part_step(t, p, b, E, 2, s);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    fill_args(A, t, p, b, E);
    const unsigned grid = (unsigned)((E + kBlock - 1) / kBlock);
    kern<<<grid, kBlock, smem, s>>>(A, NoX64{});
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "generic step kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}


int launch_generic_step(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    const bool rm = b->obs_layout == 0;
    if (p->in3d) return rm ? launch_generic<true, true>(t, p, b, E, s) : launch_generic<true, false>(t, p, b, E, s);
    return rm ? launch_generic<false, true>(t, p, b, E, s) : launch_generic<false, false>(t, p, b, E, s);
}

// ---- mass-partitioned kernel --------------------------------------------------------------------
// Breadth-first order of the spring graph (components one after another), cut into `parts` chunks of
// near-equal size: connected pieces stay together, so few springs cross parts.
static void build_partition(const wg_topology* t, int parts, PartTables& pt) {
    const int N = t->n_mass, S = t->n_spring;
    int order[kMaxMass], n_order = 0;
    bool seen[kMaxMass] = {};
    for (int root = 0; root < N; root++) {
        if (seen[root]) continue;
        int head = n_order;
        order[n_order++] = root; seen[root] = true;
        while (head < n_order) {
            const int u = order[head++];
            for (int s = 0; s < S; s++) {
                int v = -1;
                if (t->si[s] == u) v = t->sj[s]; else if (t->sj[s] == u) v = t->si[s];
                if (v >= 0 && !seen[v]) { seen[v] = true; order[n_order++] = v; }
            }
        }
    }
    int owner[kMaxMass];
    memset(&pt, 0, sizeof(pt));
    for (int q = 0; q < N; q++) {
        const int p = (int)(((int64_t)q * parts) / N);
        owner[order[q]] = p;
    }
    for (int n = 0; n < N; n++) {                       // ascending mass order inside a part
        const int p = owner[n];
        pt.mass[p][pt.n_mass[p]++] = (uint8_t)n;
        pt.own_mask[p] |= 1u << n;
    }
    for (int s = 0; s < S; s++) {                       // ascending spring order = Creature.run order
        const int pi = owner[t->si[s]], pj = owner[t->sj[s]];
        pt.spring[pi][pt.n_spring[pi]++] = (uint8_t)s;
        if (pj != pi) pt.spring[pj][pt.n_spring[pj]++] = (uint8_t)s;
    }
}

template <bool IN3D, int P, bool ROWMAJOR, int MM>
static int launch_part(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    static thread_local PartArgs tl;
    PartArgs& args = tl;
    fill_args(args.A, t, p, b, E);
    build_partition(t, P, args.pt);
    constexpr int EB = kBlock / P;
    const size_t smem = sizeof(float) * (size_t)(11 * t->n_mass + t->n_muscle + 3) * (EB + 1) + (size_t)P * (kMaxSpring + kMaxMass);
    auto kern = step_part_kernel<IN3D, P, ROWMAJOR, MM>;
    if (smem > 32 * 1024) {          // the kernel also has ~4 KB of static shared memory (staged tables)
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    const unsigned grid = (unsigned)((E + EB - 1) / EB);
    kern<<<grid, kBlock, smem, s>>>(args);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "partitioned step kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

template <int P>
static int launch_part_p(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, cudaStream_t s) {
    const bool rm = b->obs_layout == 0;
    bool any_fixed = false;
    for (int n = 0; n < t->n_mass; n++) any_fixed = any_fixed || t->fixed[n];
    const int mm = any_fixed ? 2 : mass_mode(t);        // DingPoints need the general path
#define WG_PART_DISPATCH(MMV)                                                                                      \
    (p->in3d ? (rm ? launch_part<true, P, true, MMV>(t, p, b, E, s) : launch_part<true, P, false, MMV>(t, p, b, E, s)) \
             : (rm ? launch_part<false, P, true, MMV>(t, p, b, E, s) : launch_part<false, P, false, MMV>(t, p, b, E, s)))
    if (mm == 0) return WG_PART_DISPATCH(0);
    if (mm == 1) return WG_PART_DISPATCH(1);
    return WG_PART_DISPATCH(2);
#undef WG_PART_DISPATCH
}

int launch_part_step(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, int parts, cudaStream_t s) {
    switch (parts) {
        case 2: return launch_part_p<2>(t, p, b, E, s);
        case 4: return launch_part_p<4>(t, p, b, E, s);
        case 8: return launch_part_p<8>(t, p, b, E, s);
        default: return fail(WG_ERR_BAD_ARG, "parts must be 2, 4 or 8%s");
    }
}

int launch_reset(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E, int mode, const uint8_t* mask, cudaStream_t s) {
    StepArgs<kMaxMass, kMaxSpring> A;
    fill_args(A, t, p, b, E);
    const unsigned grid = (unsigned)((E + kBlock - 1) / kBlock);
    if (p->in3d) reset_kernel<true><<<grid, kBlock, 0, s>>>(A, mode, mask, b->obs_layout);
    else reset_kernel<false><<<grid, kBlock, 0, s>>>(A, mode, mask, b->obs_layout);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "reset kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}

int launch_stats(const float* fin_stats, const float* nf_stats, int64_t E, double* out8, cudaStream_t s) {
    stats_reduce_kernel<1024><<<1, 1024, 0, s>>>(fin_stats, nf_stats, E, out8);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "stats kernel launch: %s", cudaGetErrorString(e));
    return WG_OK;
}
}  // namespace wg
