// wg_abi.cu -- C ABI (include/walker_gym_b200.h): validation and kernel dispatch.
// Built by plain nvcc for sm_100a only; no torch headers, no globals besides a
// thread-local error string and the "force generic" test switch.
#include <atomic>
#include <cstdarg>
#include <cstdlib>

#include "wg_launch.cuh"
#include "wg_policy.cuh"

namespace wg {
int balance_units(const wg_topology*);
int launch_balance_units(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int R, cudaStream_t);
int balance_chain_units(const wg_topology*);
int launch_balance_chain(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int R, cudaStream_t);
bool jit_eligible(const wg_topology*);
bool jit_runtime_available();
bool jit_eligible_soa(const wg_topology*);
int jit_prepare(const wg_topology*, int in3d, int obs_layout, cudaKernel_t* kernel, int kind);      // kind: 0 SoA, 1 packed, 2 T-steps-per-launch
int launch_jit_multi(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int n_steps, int64_t act_stride, cudaStream_t);
int launch_jit_soa(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_jit_packed(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int launch_policy(const PolicyArgs& A, int precision, cudaStream_t s);
int policy_tc_error();
int launch_policy_step(const PolicyArgs& A, int precision, const wg_topology* t, const wg_params* p, const wg_buffers* b,
                       int64_t E, cudaStream_t s);
int launch_stream_probe(const float* src, float* dst, int64_t n, int R, int W, cudaStream_t s);
int launch_gae(const float* rewards, const float* values, const uint8_t* dones, float* adv, float* ret, int T, int64_t E,
               float gamma, float lam, float clip, cudaStream_t s);
int launch_gae_trunc(const float* rewards, const float* values, const uint8_t* dones, const uint8_t* truncated,
                     const float* final_values, float* adv, float* ret, int T, int64_t E, float gamma, float lam, float clip,
                     cudaStream_t s);

static thread_local char g_err[512] = "";
static std::atomic<int> g_force_generic{0};
static int env_int(const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; }
static std::atomic<int> g_tune[6] = { {env_int("WG_TMA", 0)}, {env_int("WG_PART", -1)}, {env_int("WG_L2_PREFETCH", 256)},
                                      {env_int("WG_JIT", 1)}, {env_int("WG_POLICY_TC", 2)}, {env_int("WG_PDL", 1)} };
int tuning(int key) { return g_tune[key].load(std::memory_order_relaxed); }

int fail(int code, const char* fmt, const char* a) {
    snprintf(g_err, sizeof(g_err), fmt, a);
    return code;
}

template <class Topo>
static bool topo_matches(const wg_topology* t) {
    if (t->n_mass != Topo::N || t->n_spring != Topo::S || t->n_muscle != Topo::M) return false;
    for (int s = 0; s < Topo::S; s++)
        if (t->si[s] != Topo::si(s) || t->sj[s] != Topo::sj(s)) return false;
    return true;
}

// topology id of the register-resident specialisation this body's spring graph matches (0 = none), whatever its masses
static int topo_id(const wg_topology* t) {
    if (topo_matches<TopoBalance>(t)) return TopoBalance::kId;
    if (topo_matches<TopoBox>(t)) return TopoBox::kId;
    if (topo_matches<TopoQuad>(t)) return TopoQuad::kId;
    if (topo_matches<TopoInsect>(t)) return TopoInsect::kId;
    if (topo_matches<TopoLegacyBox>(t)) return TopoLegacyBox::kId;
    if (topo_matches<TopoTest>(t)) return TopoTest::kId;
    if (topo_matches<TopoIntrian>(t)) return TopoIntrian::kId;
    if (topo_matches<TopoHat>(t)) return TopoHat::kId;
    if (topo_matches<TopoHumanb>(t)) return TopoHumanb::kId;
    if (topo_matches<TopoBox4>(t)) return TopoBox4::kId;
    if (topo_matches<TopoLeg2>(t)) return TopoLeg2::kId;
    if (topo_matches<TopoLeg>(t)) return TopoLeg::kId;
    return 0;
}
static bool has_strings(const wg_topology* t) {
    for (int s = 0; s < t->n_spring; s++) if (t->sstring[s]) return true;
    return false;
}
static bool general_masses(const wg_topology* t) {      // arbitrary masses or DingPoints: mass mode 2
    if (mass_mode(t) == 2) return true;
    for (int n = 0; n < t->n_mass; n++) if (t->fixed[n]) return true;
    return false;
}

static int pick_variant(const wg_topology* t) {
    if (g_force_generic.load() || has_strings(t)) return 0;      // rope-type springs: a flag of the run-time topology only
    // only the Balance topology's packed kernel carries the general path (full IEEE division, DingPoint masks)
    if (general_masses(t)) return 0;
    return topo_id(t);
}

// bodies with a packed-state kernel
static bool packed_variant(int v) { return v == TopoBalance::kId || v == TopoBox::kId || (v >= TopoLegacyBox::kId && v <= TopoLeg::kId); }
// the kernel a packed-state call launches: like pick_variant, plus the Balance topology with general masses
constexpr int kJitId = 99;     // a kernel compiled at run time for this body's spring graph (wg_jit.cu)
static int packed_pick(const wg_topology* t) {
    if (g_force_generic.load() || has_strings(t)) return 0;
    const int id = topo_id(t);
    if (general_masses(t)) { if (id == TopoBalance::kId) return id; }
    else if (packed_variant(id)) return id;
    return (tuning(WG_TUNE_JIT) && jit_eligible(t) && jit_runtime_available()) ? kJitId : 0;
}

static int validate(const wg_topology* t, const wg_params* p, const wg_buffers* b, int64_t E) {
    if (!t || !p || !b) return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (t->n_mass < 1 || t->n_mass > WG_MAX_MASS) return fail(WG_ERR_BAD_ARG, "n_mass out of range [1, 32]%s");
    if (t->n_spring < 0 || t->n_spring > WG_MAX_SPRING) return fail(WG_ERR_BAD_ARG, "n_spring out of range [0, 96]%s");
    if (t->n_muscle < 0 || t->n_muscle > t->n_spring) return fail(WG_ERR_BAD_ARG, "n_muscle out of range%s");
    for (int s = 0; s < t->n_spring; s++)
        if (t->si[s] < 0 || t->si[s] >= t->n_mass || t->sj[s] < 0 || t->sj[s] >= t->n_mass || t->si[s] == t->sj[s])
            return fail(WG_ERR_BAD_ARG, "spring endpoint out of range or degenerate%s");
    if (E < 0 || E > ((int64_t)1 << 31) - 1) return fail(WG_ERR_BAD_ARG, "n_env out of range%s");
    if (p->k_sub < 1) return fail(WG_ERR_BAD_ARG, "k_sub must be >= 1%s");
    if (p->auto_reset < 0 || p->auto_reset > 2) return fail(WG_ERR_BAD_ARG, "auto_reset must be 0, 1 or 2%s");
    if (p->integrator < 0 || p->integrator > 1) return fail(WG_ERR_BAD_ARG, "integrator must be 0 (run1) or 1 (run2)%s");
    if (p->end_nonfinite != 0 && p->end_nonfinite != 1) return fail(WG_ERR_BAD_ARG, "end_nonfinite must be 0 or 1%s");
    if (p->end_nonfinite && p->auto_reset == 1)
        return fail(WG_ERR_BAD_ARG, "end_nonfinite needs auto_reset 0 or 2: a jitter reset keeps the overflowed positions%s");
    if (b->nf_stats && (!b->fin_stats || (!b->ep_ret && !b->state_packed)))
        return fail(WG_ERR_BAD_ARG, "nf_stats needs fin_stats and the running return (ep_ret or state_packed)%s");
    if (b->state_packed) {
        if (!packed_pick(t))
            return fail(WG_ERR_BAD_ARG, "the packed state layout needs a body with wg_packed_available() == 1%s");
        if (reinterpret_cast<uintptr_t>(b->state_packed) & 15u) return fail(WG_ERR_BAD_ARG, "state_packed must be 16-byte aligned%s");
    } else if (!b->pos || !b->vel || !b->steps || (t->n_muscle > 0 && !b->mx))
        return fail(WG_ERR_BAD_ARG, "pos/vel/mx/steps must be set%s");
    if (b->obs_layout != 0 && b->obs_layout != 1) return fail(WG_ERR_BAD_ARG, "obs_layout must be 0 or 1%s");
    if (b->final_obs && !b->obs) return fail(WG_ERR_BAD_ARG, "final_obs needs obs%s");
    if (b->act_layout != 0 && b->act_layout != 1) return fail(WG_ERR_BAD_ARG, "act_layout must be 0 or 1%s");
    if (b->action && b->act_dim < 0) return fail(WG_ERR_BAD_ARG, "act_dim < 0%s");
    return WG_OK;
}

#define WG_MULTI_DECL(name) int launch_##name##_multi(const wg_topology*, const wg_params*, const wg_buffers*, int64_t E, int n_steps, int64_t act_stride, cudaStream_t)
WG_MULTI_DECL(balance); WG_MULTI_DECL(box); WG_MULTI_DECL(legacy_box); WG_MULTI_DECL(test); WG_MULTI_DECL(intrian);
WG_MULTI_DECL(hat); WG_MULTI_DECL(humanb); WG_MULTI_DECL(box4); WG_MULTI_DECL(leg2); WG_MULTI_DECL(leg);
#undef WG_MULTI_DECL
int launch_generic_step_x64(const wg_topology*, const wg_x64*, const wg_params*, const wg_buffers*, int64_t E, cudaStream_t);
int check_generic_step_x64(const wg_topology*, const wg_params*, const wg_buffers*);
int launch_pkg_update(const wg_pkg_system*, const wg_pkg_params*, float* pos, float* vel, float* old_a,
                      int64_t E, int32_t n_steps, bool force_generic, cudaStream_t);
int pkg_variant(const wg_pkg_system*);

}  // namespace wg

using namespace wg;

extern "C" {

int wg_abi_version(void) { return WG_ABI_VERSION; }
const char* wg_last_error_string(void) { return g_err; }

int wg_obs_dim(const wg_topology* topo, int in3d) {
    if (!topo) return fail(WG_ERR_BAD_ARG, "null topology%s");
    return 3 * (in3d ? 3 : 2) * topo->n_mass + topo->n_muscle;
}

int wg_kernel_variant(const wg_topology* topo) {
    if (!topo) return fail(WG_ERR_BAD_ARG, "null topology%s");
    return pick_variant(topo);
}

int wg_packed_available(const wg_topology* topo) {
    if (!topo) return fail(WG_ERR_BAD_ARG, "null topology%s");
    const int v = packed_pick(topo);
    return v == kJitId ? 2 : (v ? 1 : 0);
}

int wg_jit_prepare(const wg_topology* topo, int in3d, int obs_layout) {
    if (!topo) return fail(WG_ERR_BAD_ARG, "null topology%s");
    if (packed_pick(topo) != kJitId) return WG_OK;            // an ahead-of-time kernel (or none): nothing to compile
    return jit_prepare(topo, in3d, obs_layout, nullptr, 1);
}

int wg_force_generic(int on) { return g_force_generic.exchange(on ? 1 : 0); }

int64_t wg_packed_state_floats(const wg_topology* topo, int64_t n_env) {
    if (!topo || n_env < 0) return fail(WG_ERR_BAD_ARG, "bad argument to wg_packed_state_floats%s");
    const int64_t r4 = (6 * topo->n_mass + topo->n_muscle + 2 + 3) / 4;
    return ((n_env + 127) / 128) * r4 * 512;
}

int wg_set_tuning(int key, int value) {
    if (key < 0 || key > 5) return fail(WG_ERR_BAD_ARG, "unknown tuning key%s");
    if (key == WG_TUNE_PART && value != -1 && value != 0 && value != 2 && value != 4 && value != 8)
        return fail(WG_ERR_BAD_ARG, "PART must be -1, 0, 2, 4 or 8%s");
    if (key == WG_TUNE_L2_PREFETCH && (value < 0 || value > (1 << 20))) return fail(WG_ERR_BAD_ARG, "L2 prefetch distance out of range%s");
    return g_tune[key].exchange(value);
}

int wg_step(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env, void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (n_env == 0) return WG_OK;
    cudaStream_t s = (cudaStream_t)cuda_stream;
    // one env per thread: two envs per thread (128 registers, 16 warps/SM) measured 35 % slower
    if (buf->state_packed) {
        switch (packed_pick(topo)) {
            case TopoBalance::kId:   return launch_balance_packed(topo, prm, buf, n_env, s);
            case TopoBox::kId:       return launch_box_packed(topo, prm, buf, n_env, s);
            case TopoLegacyBox::kId: return launch_legacy_box_packed(topo, prm, buf, n_env, s);
            case TopoTest::kId:      return launch_test_packed(topo, prm, buf, n_env, s);
            case TopoIntrian::kId:   return launch_intrian_packed(topo, prm, buf, n_env, s);
            case TopoHat::kId:       return launch_hat_packed(topo, prm, buf, n_env, s);
            case TopoHumanb::kId:    return launch_humanb_packed(topo, prm, buf, n_env, s);
            case TopoLeg2::kId:      return launch_leg2_packed(topo, prm, buf, n_env, s);
            case TopoLeg::kId:       return launch_leg_packed(topo, prm, buf, n_env, s);
            case kJitId:             return launch_jit_packed(topo, prm, buf, n_env, s);
            default:                 return launch_box4_packed(topo, prm, buf, n_env, s);
        }
    }
    // bodies made of identical disconnected Balance units (config 4's enlarged morphology): one lane per unit, the
    // unit's physics register-resident for all substeps (WG_TUNE_PART -1 = automatic; 0 / 2 / 4 / 8 select the older paths)
    if (tuning(WG_TUNE_PART) < 0 && !g_force_generic.load() && !has_strings(topo)) {
        const int R = balance_units(topo);
        if (R) return launch_balance_units(topo, prm, buf, n_env, R, s);
        // the same units chained into ONE connected body by link bones: neighbour endpoints over warp shuffles
        const int Rc = balance_chain_units(topo);
        if (Rc) return launch_balance_chain(topo, prm, buf, n_env, Rc, s);
    }
    // larger bodies: several lanes per env (mass partition); automatic choice by body size
    int parts = tuning(WG_TUNE_PART);
    // measured (2^20 envs, us per env-step, lanes per env 1 / 2 / 4): quad (N = 16) k_sub 1: 986 / 1516 / 988, k_sub 2:
    // 1194 / 1752 / 1165, k_sub 8: 2493 / 3032 / 2284; insect (N = 13, static kernel) k_sub 1: 425 / 1237 / 1009,
    // k_sub 8: 1510 / 2828 / 3477; leg (N = 8) k_sub 1: 391 / 589 / 659; leg2 (N = 7): 319 / 525 / 630.
    // The partition only pays for the largest bodies once several substeps amortise its staging.
    if (parts < 0) parts = (topo->n_mass >= 16 && prm->k_sub >= 2) ? 4 : 0;
    if (parts > topo->n_mass) parts = 0;
    if (parts >= 2 && !g_force_generic.load()) return launch_part_step(topo, prm, buf, n_env, parts, s);
    switch (pick_variant(topo)) {      // SoA state: ids >= 5 have packed kernels only and take the generic kernel here
        case TopoBalance::kId: return launch_balance(topo, prm, buf, n_env, 1, s);
        case TopoBox::kId:     return launch_box(topo, prm, buf, n_env, 1, s);
        case TopoQuad::kId:    return launch_quad(topo, prm, buf, n_env, 1, s);
        case TopoInsect::kId:  return launch_insect(topo, prm, buf, n_env, 1, s);
        default:
            // no ahead-of-time kernel: a kernel compiled for this spring graph at run time (up to 16 masses); if the
            // run-time compiler is missing or fails, the run-time-topology kernel (same bits)
            // (only for batches that amortise the seconds of compilation)
            if (n_env >= 4096 && !g_force_generic.load() && !has_strings(topo) && tuning(WG_TUNE_JIT) && jit_eligible_soa(topo) && jit_runtime_available() &&
                launch_jit_soa(topo, prm, buf, n_env, s) == WG_OK)
                return WG_OK;
            return launch_generic_step(topo, prm, buf, n_env, s);
    }
}

int wg_step_multi(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env, int32_t n_steps,
                  int32_t n_action_steps, void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (n_steps < 1 || n_steps > 65536) return fail(WG_ERR_BAD_ARG, "n_steps out of range [1, 65536]%s");
    if (n_action_steps != n_steps && n_action_steps != 1) return fail(WG_ERR_BAD_ARG, "n_action_steps must be n_steps or 1 (action repeat)%s");
    if (!buf->state_packed) return fail(WG_ERR_BAD_ARG, "wg_step_multi needs the packed state layout%s");
    if (buf->final_obs) return fail(WG_ERR_BAD_ARG, "wg_step_multi returns only the last observation: final_obs must be null%s");
    if (buf->obs && buf->obs_layout != 0) return fail(WG_ERR_BAD_ARG, "wg_step_multi writes row-major observations%s");
    if (buf->action && (buf->act_layout != 0 || buf->act_dim != topo->n_muscle))
        return fail(WG_ERR_BAD_ARG, "wg_step_multi reads actions as [n_action_steps][n_env][n_muscle]%s");
    if (buf->action_gen && buf->action_gen->mode != 0) {
        const wg_action_gen* g = buf->action_gen;
        if (buf->action) return fail(WG_ERR_BAD_ARG, "wg_step_multi: action must be null when an in-kernel action source is set%s");
        if (g->mode != 1 && g->mode != 2) return fail(WG_ERR_BAD_ARG, "wg_action_gen.mode must be 0, 1 (table) or 2 (cpg)%s");
        if (topo->n_muscle > WG_GEN_MAX_MUSCLE) return fail(WG_ERR_BAD_ARG, "in-kernel action sources drive at most 16 muscles%s");
        if (g->mode == 1 && (g->n_rows < 1 || g->n_rows > WG_GEN_MAX_ROWS || g->hold < 1))
            return fail(WG_ERR_BAD_ARG, "wg_action_gen table: n_rows in [1, 32], hold >= 1%s");
    }
    if (buf->old_a || buf->contact_pre || buf->contact_post || buf->energy || buf->centroid)
        return fail(WG_ERR_BAD_ARG, "wg_step_multi has no per-step info outputs (old_a / contact / energy / centroid must be null)%s");
    if (n_env == 0) return WG_OK;
    cudaStream_t s = (cudaStream_t)cuda_stream;
    const int64_t as = n_action_steps == 1 ? 0 : n_env * (int64_t)topo->n_muscle;
    // the kernel family wg_step would pick for this body on the packed layout: an ahead-of-time instance (the Balance
    // graph also with arbitrary masses / DingPoints) or one compiled at run time for the body's spring graph
    const int pick = packed_pick(topo);
    if (pick == kJitId) return launch_jit_multi(topo, prm, buf, n_env, n_steps, as, s);
    switch (pick) {
#define WG_MULTI_CASE(T, name) case T::kId: return launch_##name##_multi(topo, prm, buf, n_env, n_steps, as, s)
        WG_MULTI_CASE(TopoBalance, balance); WG_MULTI_CASE(TopoBox, box); WG_MULTI_CASE(TopoLegacyBox, legacy_box);
        WG_MULTI_CASE(TopoTest, test); WG_MULTI_CASE(TopoIntrian, intrian); WG_MULTI_CASE(TopoHat, hat);
        WG_MULTI_CASE(TopoHumanb, humanb); WG_MULTI_CASE(TopoBox4, box4); WG_MULTI_CASE(TopoLeg2, leg2); WG_MULTI_CASE(TopoLeg, leg);
#undef WG_MULTI_CASE
        default: return fail(WG_ERR_UNSUPPORTED, "wg_step_multi: this body has no packed-state kernel%s");
    }
}

int wg_step_x64(const wg_topology* topo, const wg_x64* x64, const wg_params* prm, const wg_buffers* buf, int64_t n_env,
                void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (!x64) return fail(WG_ERR_BAD_ARG, "null wg_x64%s");
    if (buf->state_packed) return fail(WG_ERR_BAD_ARG, "x64 mode uses the SoA state layout%s");
    if (topo->n_muscle > 0 && (!buf->mx64 || !buf->mx_weak)) return fail(WG_ERR_BAD_ARG, "mx64 / mx_weak must be set%s");
    if (buf->act_dim > 0 && !buf->action64) return fail(WG_ERR_BAD_ARG, "action64 must be set when act_dim > 0%s");
    rc = check_generic_step_x64(topo, prm, buf);               // also for n_env == 0: lets callers check a body up front
    if (rc != WG_OK) return rc;
    if (n_env == 0) return WG_OK;
    return launch_generic_step_x64(topo, x64, prm, buf, n_env, (cudaStream_t)cuda_stream);
}

int wg_reset(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env, int mode,
             const uint8_t* mask, void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (mode != 1 && mode != 2) return fail(WG_ERR_BAD_ARG, "reset mode must be 1 (jitter) or 2 (template)%s");
    if (n_env == 0) return WG_OK;
    return launch_reset(topo, prm, buf, n_env, mode, mask, (cudaStream_t)cuda_stream);
}

int wg_stats_reduce_split(const float* fin_stats, const float* nf_stats, int64_t n_env, double* out8, void* cuda_stream) {
    if (!fin_stats || !out8 || n_env < 0) return fail(WG_ERR_BAD_ARG, "bad argument to wg_stats_reduce%s");
    return launch_stats(fin_stats, nf_stats, n_env, out8, (cudaStream_t)cuda_stream);
}

int wg_stats_reduce(const float* fin_stats, int64_t n_env, double* out8, void* cuda_stream) {
    return wg_stats_reduce_split(fin_stats, nullptr, n_env, out8, cuda_stream);
}

int wg_step_host(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env,
                 const float* h_action, float* h_obs, float* h_reward, uint8_t* h_done, void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (buf->truncated || buf->final_obs) return fail(WG_ERR_BAD_ARG, "wg_step_host does not take buf->truncated / final_obs%s");
    cudaStream_t s = (cudaStream_t)cuda_stream;
    cudaError_t e = cudaSuccess;
    if (h_action) {
        if (!buf->action) return fail(WG_ERR_BAD_ARG, "wg_step_host: device action buffer missing%s");
        e = cudaMemcpyAsync((void*)buf->action, h_action, sizeof(float) * n_env * buf->act_dim, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "H2D action: %s", cudaGetErrorString(e));
    }
    rc = wg_step(topo, prm, buf, n_env, cuda_stream);
    if (rc != WG_OK) return rc;
    const int D = wg_obs_dim(topo, prm->in3d);
    if (h_obs && buf->obs) e = cudaMemcpyAsync(h_obs, buf->obs, sizeof(float) * n_env * D, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && h_reward && buf->reward) e = cudaMemcpyAsync(h_reward, buf->reward, sizeof(float) * n_env, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && h_done && buf->done) e = cudaMemcpyAsync(h_done, buf->done, n_env, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "D2H results: %s", cudaGetErrorString(e));
    return WG_OK;
}

int wg_step_multi_host(const wg_topology* topo, const wg_params* prm, const wg_buffers* buf, int64_t n_env, int32_t n_steps,
                       int32_t n_action_steps, const float* h_action, float* h_obs, float* h_reward, uint8_t* h_done,
                       void* cuda_stream) {
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    if (n_steps < 1 || (n_action_steps != n_steps && n_action_steps != 1)) return fail(WG_ERR_BAD_ARG, "bad n_steps / n_action_steps%s");
    if (buf->truncated || buf->final_obs) return fail(WG_ERR_BAD_ARG, "wg_step_multi_host does not take buf->truncated / final_obs%s");
    cudaStream_t s = (cudaStream_t)cuda_stream;
    cudaError_t e = cudaSuccess;
    if (h_action) {
        if (!buf->action) return fail(WG_ERR_BAD_ARG, "wg_step_multi_host: device action buffer missing%s");
        e = cudaMemcpyAsync((void*)buf->action, h_action, sizeof(float) * n_action_steps * n_env * buf->act_dim, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return fail(WG_ERR_CUDA, "H2D actions: %s", cudaGetErrorString(e));
    }
    rc = wg_step_multi(topo, prm, buf, n_env, n_steps, n_action_steps, cuda_stream);
    if (rc != WG_OK) return rc;
    const int D = wg_obs_dim(topo, prm->in3d);
    if (h_obs && buf->obs) e = cudaMemcpyAsync(h_obs, buf->obs, sizeof(float) * n_env * D, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && h_reward && buf->reward)
        e = cudaMemcpyAsync(h_reward, buf->reward, sizeof(float) * n_steps * n_env, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && h_done && buf->done) e = cudaMemcpyAsync(h_done, buf->done, (size_t)n_steps * n_env, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) return fail(WG_ERR_CUDA, "D2H results: %s", cudaGetErrorString(e));
    return WG_OK;
}

int wg_pkg_kernel_variant(const wg_pkg_system* sys) {
    if (!sys) return fail(WG_ERR_BAD_ARG, "null system%s");
    return g_force_generic.load() ? 0 : pkg_variant(sys);
}

int wg_pkg_update_physics(const wg_pkg_system* sys, const wg_pkg_params* prm, float* pos, float* vel, float* old_a,
                          int64_t n_env, int32_t n_steps, void* cuda_stream) {
    if (!sys || !prm) return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (sys->n_point < 1 || sys->n_point > WG_MAX_MASS) return fail(WG_ERR_BAD_ARG, "n_point out of range [1, 32]%s");
    if (sys->n_spring < 0 || sys->n_spring > WG_MAX_SPRING) return fail(WG_ERR_BAD_ARG, "n_spring out of range [0, 96]%s");
    for (int s = 0; s < sys->n_spring; s++)
        if (sys->si[s] < 0 || sys->si[s] >= sys->n_point || sys->sj[s] < 0 || sys->sj[s] >= sys->n_point)
            return fail(WG_ERR_BAD_ARG, "spring endpoint out of range%s");
    if (n_env < 0 || n_env > ((int64_t)1 << 31) - 1) return fail(WG_ERR_BAD_ARG, "n_env out of range%s");
    if (n_steps < 0) return fail(WG_ERR_BAD_ARG, "n_steps < 0%s");
    if (n_env == 0 || n_steps == 0) return WG_OK;
    if (!pos || !vel) return fail(WG_ERR_BAD_ARG, "pos/vel must be set%s");
    return launch_pkg_update(sys, prm, pos, vel, old_a, n_env, n_steps, g_force_generic.load() != 0, (cudaStream_t)cuda_stream);
}

int wg_policy_act(const wg_mlp_policy* pol, const float* obs, int32_t obs_layout, float* action, int32_t act_layout, float* logp,
                  float* value, float* mean, int64_t n_env, int32_t sample, uint32_t seed_lo, uint32_t seed_hi,
                  uint32_t step_index, const uint32_t* step_counter, uint32_t env_offset, void* cuda_stream) {
    if (!pol || !obs) return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (!pol->w1 || !pol->b1 || !pol->w2 || !pol->b2 || !pol->w_mu || !pol->b_mu || !pol->w_v || !pol->b_v || !pol->log_std)
        return fail(WG_ERR_BAD_ARG, "wg_mlp_policy: every weight pointer must be set%s");
    if (pol->obs_dim < 1 || pol->obs_dim > 64) return fail(WG_ERR_BAD_ARG, "obs_dim out of range [1, 64]%s");
    if (pol->act_dim < 1 || pol->act_dim > 7) return fail(WG_ERR_BAD_ARG, "act_dim out of range [1, 7]%s");
    if (pol->precision != 0 && pol->precision != 1) return fail(WG_ERR_BAD_ARG, "precision must be 0 or 1%s");
    if (act_layout != 0 && act_layout != 1) return fail(WG_ERR_BAD_ARG, "act_layout must be 0 or 1%s");
    if (obs_layout != 0 && obs_layout != 1) return fail(WG_ERR_BAD_ARG, "obs_layout must be 0 or 1%s");
    if (n_env < 0 || n_env > ((int64_t)1 << 31) - 1) return fail(WG_ERR_BAD_ARG, "n_env out of range%s");
    if (n_env == 0) return WG_OK;
    PolicyArgs A;
    A.obs_layout = obs_layout;
    A.w1 = pol->w1; A.b1 = pol->b1; A.w2 = pol->w2; A.b2 = pol->b2; A.w_mu = pol->w_mu; A.b_mu = pol->b_mu;
    A.w_v = pol->w_v; A.b_v = pol->b_v; A.log_std = pol->log_std;
    A.obs = obs; A.action = action; A.logp = logp; A.value = value; A.mean = mean; A.step_counter = step_counter;
    A.E = n_env; A.D = pol->obs_dim; A.M = pol->act_dim; A.act_layout = act_layout; A.sample = sample ? 1 : 0;
    A.obs_scale = pol->obs_scale; A.obs_clip = pol->obs_clip;
    A.seed_lo = seed_lo; A.seed_hi = seed_hi; A.step_index = step_index; A.env_offset = env_offset;
    return launch_policy(A, pol->precision, (cudaStream_t)cuda_stream);
}

int wg_policy_step(const wg_mlp_policy* pol, const wg_topology* topo, const wg_params* prm, const wg_buffers* buf,
                   const float* obs, float* action, float* logp, float* value, float* mean, int64_t n_env, int32_t sample,
                   uint32_t seed_lo, uint32_t seed_hi, uint32_t step_index, uint32_t env_offset, void* cuda_stream) {
    if (!pol || !obs) return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (!pol->w1 || !pol->b1 || !pol->w2 || !pol->b2 || !pol->w_mu || !pol->b_mu || !pol->w_v || !pol->b_v || !pol->log_std)
        return fail(WG_ERR_BAD_ARG, "wg_mlp_policy: every weight pointer must be set%s");
    if (pol->precision != 0 && pol->precision != 1) return fail(WG_ERR_BAD_ARG, "precision must be 0 or 1%s");
    int rc = validate(topo, prm, buf, n_env);
    if (rc != WG_OK) return rc;
    // the fused kernel exists for BASELINE config 5's environment: Balance-v0's spring graph and mass pattern [k, k, 1, j]
    // (unit / power-of-two / odd-integer masses), 3-D, packed state, row-major observations, two muscles
    const bool body_ok = !g_force_generic.load() && !has_strings(topo) && !general_masses(topo) && topo_id(topo) == TopoBalance::kId &&
                         mass_mode(topo) == 1 && topo->mass[2] == 1.0 && topo->mass[0] == topo->mass[1] && topo->mass[0] != 1.0 &&
                         topo->mass[3] != 1.0;
    if (!body_ok || !prm->in3d || !buf->state_packed || buf->obs_layout != 0 || pol->obs_dim != 38 || pol->act_dim != 2 ||
        tuning(WG_TUNE_POLICY_TC) != 2)
        return fail(WG_ERR_UNSUPPORTED, "wg_policy_step: fused policy + step exists for Balance-v0 (3-D, packed state, row-major observations) with the tcgen05 pipeline%s");
    if (buf->truncated || buf->final_obs)
        return fail(WG_ERR_UNSUPPORTED, "wg_policy_step does not write buf->truncated / final_obs: make the two calls%s");
    if (n_env == 0) return WG_OK;
    PolicyArgs A;
    A.obs_layout = 0;
    A.w1 = pol->w1; A.b1 = pol->b1; A.w2 = pol->w2; A.b2 = pol->b2; A.w_mu = pol->w_mu; A.b_mu = pol->b_mu;
    A.w_v = pol->w_v; A.b_v = pol->b_v; A.log_std = pol->log_std;
    A.obs = obs; A.action = action; A.logp = logp; A.value = value; A.mean = mean; A.step_counter = buf->step_counter;
    A.E = n_env; A.D = 38; A.M = 2; A.act_layout = 0; A.sample = sample ? 1 : 0;
    A.obs_scale = pol->obs_scale; A.obs_clip = pol->obs_clip;
    A.seed_lo = seed_lo; A.seed_hi = seed_hi; A.step_index = step_index; A.env_offset = env_offset;
    return launch_policy_step(A, pol->precision, topo, prm, buf, n_env, (cudaStream_t)cuda_stream);
}

int wg_policy_tc_status(void) { return policy_tc_error(); }

int wg_stream_probe(const float* src, float* dst, int64_t n_threads, int32_t vec_reads, int32_t vec_writes, void* cuda_stream) {
    if (!src || !dst || n_threads < 0 || vec_reads < 0 || vec_writes < 0) return fail(WG_ERR_BAD_ARG, "bad argument to wg_stream_probe%s");
    if (n_threads == 0) return WG_OK;
    return launch_stream_probe(src, dst, n_threads, vec_reads, vec_writes, (cudaStream_t)cuda_stream);
}

int wg_gae(const float* rewards, const float* values, const uint8_t* dones, float* advantages, float* returns,
           int32_t horizon, int64_t n_env, float gamma, float lam, float reward_clip, void* cuda_stream) {
    if (!rewards || !values || !dones || !advantages || !returns) return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (horizon < 0 || n_env < 0) return fail(WG_ERR_BAD_ARG, "horizon / n_env < 0%s");
    if (horizon == 0 || n_env == 0) return WG_OK;
    return launch_gae(rewards, values, dones, advantages, returns, horizon, n_env, gamma, lam, reward_clip,
                      (cudaStream_t)cuda_stream);
}

int wg_gae_trunc(const float* rewards, const float* values, const uint8_t* dones, const uint8_t* truncated,
                 const float* final_values, float* advantages, float* returns, int32_t horizon, int64_t n_env, float gamma,
                 float lam, float reward_clip, void* cuda_stream) {
    if (!rewards || !values || !dones || !truncated || !final_values || !advantages || !returns)
        return fail(WG_ERR_BAD_ARG, "null argument%s");
    if (horizon < 0 || n_env < 0) return fail(WG_ERR_BAD_ARG, "horizon / n_env < 0%s");
    if (horizon == 0 || n_env == 0) return WG_OK;
    return launch_gae_trunc(rewards, values, dones, truncated, final_values, advantages, returns, horizon, n_env, gamma, lam,
                            reward_clip, (cudaStream_t)cuda_stream);
}

}  // extern "C"
