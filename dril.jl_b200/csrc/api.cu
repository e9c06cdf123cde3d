// libdril_b200.so — C ABI implementation (include/dril_b200.h): handles, launch logic,
// host<->device staging.  All compute is in the kernels of rollout.cuh / gae.cuh / update.cuh.
#include <dlfcn.h>
#include <math.h>
#include <cmath>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>
#include <utility>

#include "common.cuh"
#include "gae.cuh"
#include "rollout.cuh"
#include "update.cuh"
#include "update_tc.cuh"
#include "update_ft.cuh"
#include "update_ftg.cuh"
#include "rollout_tc.cuh"
#include "rollout_syn.cuh"
#include "rollout_gtc.cuh"

#define DRIL_SMEM_MAX 232448  // 227 KB opt-in per CTA on sm_100
#define DRIL_RESULT_SLOTS 4   // iterations that may be enqueued before their results are read
#define DRIL_GPLANES 8        // gradient partial planes per CTA (sample-range splits of the dW tiles)

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void dril_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char* dril_last_error(void) { return g_err; }
extern "C" int32_t dril_version(void) { return 200; }
#ifndef DRIL_SOURCE_HASH
#define DRIL_SOURCE_HASH "unknown"
#endif
/* SHA-256 prefix of the sources + flags this library was compiled from (dril.jl_b200/build.py decides staleness with it) */
static const char g_source_hash_marker[] = "DRIL_SOURCE_HASH=" DRIL_SOURCE_HASH;      // build.py finds the marker in the file (no dlopen)
extern "C" const char* dril_source_hash(void) { return g_source_hash_marker + 17; }
// ---------------------------------------------------------------------------------------
// options
// ---------------------------------------------------------------------------------------
static int g_opt_tc = getenv("DRIL_TC") ? atoi(getenv("DRIL_TC")) : 1;
// features-on-lanes tcgen05 loss/grad kernel (update_ft.cuh) instead of the samples-on-lanes one (update_tc.cuh)
static int g_opt_ft = getenv("DRIL_FT") ? atoi(getenv("DRIL_FT")) : 1;
// general rollout kernel: actor only in the step loop, values by one batched tcgen05 critic pass afterwards (shapes of update_ftg.cuh)
static int g_opt_defer_critic = getenv("DRIL_DEFER_CRITIC") ? atoi(getenv("DRIL_DEFER_CRITIC")) : 1;
static int g_opt_ftg = getenv("DRIL_FTG") ? atoi(getenv("DRIL_FTG")) : 1;   // general-shape features-on-lanes kernel (update_ftg.cuh); 2: also where update_ft.cuh applies
static int g_opt_tc_rollout = getenv("DRIL_TC_ROLLOUT") ? atoi(getenv("DRIL_TC_ROLLOUT")) : 1;   // tensor-core rollout (CartPole, [64,64])
static int g_opt_tc_actor = getenv("DRIL_TC_ACTOR") ? atoi(getenv("DRIL_TC_ACTOR")) : 1;   // general rollout: actor forward on tcgen05 (rollout_gtc.cuh)
static int g_opt_syn_rollout = getenv("DRIL_SYN_ROLLOUT") ? atoi(getenv("DRIL_SYN_ROLLOUT")) : 1;   // thread-per-env rollout (synthetic env, small policy)
static int g_opt_persistent = getenv("DRIL_PERSISTENT") ? atoi(getenv("DRIL_PERSISTENT")) : 1;   // [64,64] tcgen05 update: all minibatch steps of an update in one cooperative launch
static int g_opt_tail = getenv("DRIL_TAIL") ? atoi(getenv("DRIL_TAIL")) : 1;   // fused reduce/clip/Adam tail of the TC kernel
// fp32 loss/grad kernel, wide nets: one net per pass with shared activation rows (fixed per policy at creation)
static int g_opt_single_net = getenv("DRIL_SINGLE_NET") ? atoi(getenv("DRIL_SINGLE_NET")) : 1;
// fp32 loss/grad kernel: layers with padded dims multiple of 16 on mma.sync 3xTF32 tiles (fixed per policy at creation)
static int g_opt_mma = getenv("DRIL_MMA") ? atoi(getenv("DRIL_MMA")) : 1;
extern "C" int32_t dril_set_option(const char* key, int32_t value) {
    DRIL_REQUIRE(key, "key is NULL");
    if (!strcmp(key, "tc")) { g_opt_tc = value; return DRIL_OK; }
    if (!strcmp(key, "ft")) { g_opt_ft = value; return DRIL_OK; }
    if (!strcmp(key, "ftg")) { g_opt_ftg = value; return DRIL_OK; }
    if (!strcmp(key, "defer_critic")) { g_opt_defer_critic = value; return DRIL_OK; }
    if (!strcmp(key, "fused_tail")) { g_opt_tail = value; return DRIL_OK; }
    if (!strcmp(key, "tc_rollout")) { g_opt_tc_rollout = value; return DRIL_OK; }
    if (!strcmp(key, "syn_rollout")) { g_opt_syn_rollout = value; return DRIL_OK; }
    if (!strcmp(key, "tc_actor")) { g_opt_tc_actor = value; return DRIL_OK; }
    if (!strcmp(key, "persistent")) { g_opt_persistent = value; return DRIL_OK; }
    if (!strcmp(key, "single_net")) { g_opt_single_net = value; return DRIL_OK; }   // policies created afterwards
    if (!strcmp(key, "mma")) { g_opt_mma = value; return DRIL_OK; }                 // policies created afterwards
    dril_set_error("unknown option '%s'", key);
    return DRIL_ERR_INVALID;
}
// the tensor-core loss/grad kernel covers the reference's default layer: hidden_dims = [64, 64], obs_dim <= 4,
// Discrete(n <= 2)
// the general-shape features-on-lanes kernel (update_ftg.cuh): 2 or 3 hidden layers of width 64 / 128 (same in both nets),
// obs_dim <= 15, Discrete(n <= 4) or Box of dimension <= 2, and everything resident in shared memory
static bool ftg_eligible(const PolicyDesc& pd) {
    const int L = pd.n_layers - 1;
    if (L < 2 || L > 3 || pd.obs_dim > FTG_MAX_OBS || pd.act_n > (pd.act_kind == DRIL_ACT_DISCRETE ? 4 : 2)) return false;
    for (int l = 0; l < L; ++l) {
        if (pd.L[0][l].N != pd.L[1][l].N) return false;
        if (pd.L[0][l].N != 64 && pd.L[0][l].N != 128) return false;
    }
    return ftg_layout(pd).total <= DRIL_SMEM_MAX - 2048;
}
static bool tc_eligible(const PolicyDesc& pd) {
    if (pd.n_layers != 3 || pd.obs_dim > 4 || pd.act_kind != DRIL_ACT_DISCRETE || pd.act_n > 2) return false;
    for (int net = 0; net < 2; ++net) {
        if (pd.L[net][0].N != 64 || pd.L[net][1].K != 64 || pd.L[net][1].N != 64 || pd.L[net][2].K != 64) return false;
        if (pd.L[net][2].Np != 4) return false;
    }
    return true;
}

// the kind sets the rollout kernels are instantiated for (env.cuh): CartPole, Pendulum and the synthetic env run the ones built
// for those kinds alone, every other kind the ones built for all kinds, each plain, with per-env parameters (dril_env_set_params),
// observing its parameters (dril_env_set_observe_params) or with an observation history (dril_env_set_obs_history), and the
// last two with observation noise or action delay (dril_env_set_obs_noise, dril_env_set_action_delay)
static constexpr unsigned k_kind_sets[] = {
    ENV_KS_CLASSIC, env_param_kind_set(DRIL_ENV_CARTPOLE), env_obs_param_kind_set(DRIL_ENV_CARTPOLE), env_hist_kind_set(DRIL_ENV_CARTPOLE),
    ENV_KS_ALL, env_param_kind_set(DRIL_ENV_ACROBOT), env_obs_param_kind_set(DRIL_ENV_ACROBOT), env_hist_kind_set(DRIL_ENV_ACROBOT),
    env_perturb_kind_set(DRIL_ENV_CARTPOLE), env_hist_perturb_kind_set(DRIL_ENV_CARTPOLE),
    env_perturb_kind_set(DRIL_ENV_ACROBOT), env_hist_perturb_kind_set(DRIL_ENV_ACROBOT)};
// f(std::integral_constant<unsigned, KS>) for the entry KS == ks of k_kind_sets (nullptr for a kind set not in the list)
template <class F, size_t... I>
static void* ks_pick(unsigned ks, F f, std::index_sequence<I...>) {
    void* fn = nullptr;
    ((ks == k_kind_sets[I] ? (void)(fn = f(std::integral_constant<unsigned, k_kind_sets[I]>{})) : (void)0), ...);
    return fn;
}
template <class F>
static void* ks_pick(unsigned ks, F f) { return ks_pick(ks, f, std::make_index_sequence<sizeof(k_kind_sets) / sizeof(unsigned)>{}); }
static void* rollout_fn(bool ws, unsigned ks) {
    return ks_pick(ks, [ws](auto k) {
        constexpr unsigned KS = decltype(k)::value;
        return ws ? (void*)rollout_kernel<true, KS> : (void*)rollout_kernel<false, KS>;
    });
}
static void* rollout_fast_fn(bool ws, unsigned ks) {
    return ks_pick(ks, [ws](auto k) {
        constexpr unsigned KS = decltype(k)::value;
        return ws ? (void*)rollout_fast_kernel<true, KS> : (void*)rollout_fast_kernel<false, KS>;
    });
}
// tcgen05-actor rollout by hidden-layer count, kind set and action count (2 or 4 staged output columns, gtc_nout); the 4-column
// variant exists for the all-kinds sets only, which also serve the other kinds
static void* rollout_gtc_fn(int L, unsigned ks, int act_n) {
    if (act_n > 2) {
        ks |= env_has_params(ks) ? env_param_kind_set(DRIL_ENV_ACROBOT) : ENV_KS_ALL;
        return ks_pick(ks, [L](auto k) -> void* {
            constexpr unsigned KS = decltype(k)::value;
            if constexpr (env_in(KS, DRIL_ENV_ACROBOT)) return L == 2 ? (void*)rollout_gtc_kernel<2, KS, 4> : (void*)rollout_gtc_kernel<3, KS, 4>;
            else return nullptr;
        });
    }
    return ks_pick(ks, [L](auto k) {
        constexpr unsigned KS = decltype(k)::value;
        return L == 2 ? (void*)rollout_gtc_kernel<2, KS, 2> : (void*)rollout_gtc_kernel<3, KS, 2>;
    });
}

extern "C" int32_t dril_device_count(int32_t* count) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        dril_set_error("no usable CUDA device (%s); libdril_b200 has no CPU fallback", cudaGetErrorString(e));
        if (count) *count = 0;
        return DRIL_ERR_CUDA;
    }
    if (count) *count = n;
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// NCCL through dlopen (no link-time dependency: single-GPU use never touches it)
// ---------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm*, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int32_t nccl_load() {
    if (g_nccl.lib) return DRIL_OK;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) { dril_set_error("cannot dlopen libnccl.so.2: %s", dlerror()); return DRIL_ERR_NCCL; }
    g_nccl.GetUniqueId = (int (*)(nccl_uid*))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(nccl_comm*, int, nccl_uid, int))dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(nccl_comm))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce) {
        dril_set_error("libnccl is missing required symbols");
        return DRIL_ERR_NCCL;
    }
    return DRIL_OK;
}
#define DRIL_NCCL(expr)                                                                              \
    do {                                                                                             \
        int _r = (expr);                                                                             \
        if (_r != 0) {                                                                               \
            dril_set_error("NCCL error %d (%s) at %s:%d", _r,                                        \
                           g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "?", __FILE__, __LINE__); \
            return DRIL_ERR_NCCL;                                                                    \
        }                                                                                            \
    } while (0)
enum { NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8, NCCL_SUM = 0 };

// ---------------------------------------------------------------------------------------
// handles
// ---------------------------------------------------------------------------------------
struct ProfSpan { int kind; cudaEvent_t a, b; };

struct dril_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    uint64_t seed = 0;
    int sm_count = 0;
    int64_t launches = 0;
    bool profiling = false;
    double prof_ms[DRIL_K_COUNT] = {0};
    int64_t prof_n[DRIL_K_COUNT] = {0};
    std::vector<ProfSpan> spans;
    std::vector<cudaEvent_t> free_events;
    nccl_comm comm = nullptr;
    int rank = 0, nranks = 1;
    cudaEvent_t user_ev[16] = {nullptr};
    // peer-memory allreduce (CUDA IPC)
    void* p2p_region = nullptr;
    void* p2p_peer_base[DRIL_MAX_RANKS] = {nullptr};
    P2PDev p2p;
    bool p2p_enabled = false;
    void* l2_scratch = nullptr;
    size_t l2_bytes = 0;
    std::vector<struct dril_policy*> policies;   // live policies of this ctx (their env back-pointers are cleared by dril_env_destroy)
};

struct dril_buffer {
    dril_ctx* ctx;
    void* slab = nullptr;
    BufDev d;
    int act_elems;  // per-sample action elements
    TcRolloutScratch tcs = {nullptr, nullptr, nullptr, nullptr, 0};   // tensor-core rollout: inputs of the batched critic pass
    void* tcs_slab = nullptr;
    DeferredCritic dcs = {nullptr, nullptr, nullptr, nullptr, 0};      // general rollout with the critic deferred to a batched pass
    void* dcs_slab = nullptr;
    bool is_view = false;   // rows [t0, t0 + T) of another buffer (chunked collection): no tensor-core rollout scratch
};

struct dril_env {
    dril_ctx* ctx;
    EnvDev d;
    dril_buffer* compat = nullptr;   // 1-step buffer for the act!/observe compatibility path
    void* compat_actions = nullptr;  // device staging
    float* compat_obs = nullptr;     // device [n][D]
    MonitorRing ring;
    int max_blocks = 0;
    int64_t total_episodes = 0;
    PolicyDesc nopolicy;             // zeroed descriptor for policy-less launches
    // data-parallel runs: per-rollout normaliser moments, the statistics every rank started the rollout with, and the small
    // fp64 exchange buffer [explained-variance moments 4 | monitor sums 3 | normaliser moments 2 (D + 1) + 2]
    double* roll_moments = nullptr;
    double* xr = nullptr;
    float* norm_snap = nullptr;
    long long* norm_snap_cnt = nullptr;
    unsigned obs_ks = 0;             // ENV_KS_OBS_PARAMS (dril_env_set_observe_params), ENV_KS_HISTORY (dril_env_set_obs_history:
                                     // k > 1 or velocities masked) or 0: the observation layout, as a kind-set bit
    bool default_params = false;     // parameters held at lo = hi = the defaults only because obs_ks is set or the env is perturbed
    bool observed = false;           // an observation was made (observe, step, rollout, evaluate): the width is fixed
};
// observation noise or action delay on: the ENV_KS_PERTURB kernels
static bool env_perturbed(const dril_env* e) { return e->d.obs_noise || e->d.act_delay; }
// the kind set whose kernels run env e (one of k_kind_sets)
static unsigned env_ks(const dril_env* e) {
    const int kind = e->d.kind;
    if (env_perturbed(e)) return env_param_kind_set(kind) | e->obs_ks | ENV_KS_PERTURB;
    return e->obs_ks ? env_param_kind_set(kind) | e->obs_ks : e->d.has_params ? env_param_kind_set(kind) : env_kind_set(kind);
}

struct dril_policy {
    dril_ctx* ctx;
    PolicyDesc pd;
    float *flat = nullptr, *pack = nullptr, *m = nullptr, *v = nullptr, *g = nullptr, *gpart = nullptr;
    int *flat2pack = nullptr, *flat2packT = nullptr, *flat2g = nullptr;
    unsigned char* f2planes = nullptr;   // partial planes holding contributions to each parameter's gradient
    unsigned char* f2planes_one = nullptr;   // tensor-core path: one partial plane per CTA
    double* sq_part = nullptr;
    unsigned int* ticket = nullptr;
    int loss_M4 = 0, loss_splits = 1;
    bool loss_ws = true;
    long long* step = nullptr;
    double *iter_acc = nullptr, *ev_acc = nullptr, *mbstats = nullptr, *adv_partial = nullptr;
    int* stop_flag = nullptr;
    int gpart_ctas = 0;
    int plan_single = -1;      // single-net pass mode of the fp32 loss kernel, fixed when the policy is created
    int plan_mma = -1;         // mma.sync tiles for the wide layers of the fp32 loss kernel, fixed when the policy is created
    int mbstats_cap = 0;
    uint64_t seed = 0;
    uint32_t step_index = 0;
    // last iteration bookkeeping
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    // iterations in flight (dril_ppo_iteration_async -> dril_iteration_result, FIFO)
    struct Slot {
        cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // rollout start, update start, update end, record on host
        IterRecord* host = nullptr;                                    // pinned
        dril_env* env = nullptr;
        long long n_local = 0;
        float lr = 0.f;
    } slots[DRIL_RESULT_SLOTS];
    IterRecord* rec_dev = nullptr;       // [DRIL_RESULT_SLOTS]
    unsigned long long slot_head = 0, slot_tail = 0;
    dril_env* last_env = nullptr;
    dril_buffer* last_buf = nullptr;
    float last_lr = 0.f;
    int64_t last_steps = 0;
    // scratch for the host-pointer entry points
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    // update_ft.cuh / update_ftg.cuh: per-sample records of the buffer (packed once per update) and the current epoch's
    // samples as shuffled tile records
    float* ft_recs = nullptr;
    size_t ft_recs_floats = 0;
    int ft_rec_stride = 0;
    unsigned char* ft_tiles = nullptr;
    size_t ft_tiles_bytes = 0;
    int ft_tiles_per_mb = 0;
    long long ft_batch = 1;
    long long ft_epoch_tile0 = 0;      // first tile of the current epoch when all epochs of an update were staged at once
    // Adam betas of the most recent update (dril_ppo_hyper carries them per call); Optimisers.Adam defaults until then
    double beta1 = 0.9, beta2 = 0.999;
};

// ---------------------------------------------------------------------------------------
// launch bookkeeping / profiling
// ---------------------------------------------------------------------------------------
struct Span {
    dril_ctx* c;
    int kind;
    cudaEvent_t a = nullptr, b = nullptr;
    Span(dril_ctx* c_, int kind_) : c(c_), kind(kind_) {
        c->launches += 1;
        if (c->profiling) {
            a = take(); b = take();
            cudaEventRecord(a, c->stream);
        }
    }
    cudaEvent_t take() {
        if (!c->free_events.empty()) { cudaEvent_t e = c->free_events.back(); c->free_events.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    ~Span() {
        if (c->profiling) {
            cudaEventRecord(b, c->stream);
            c->spans.push_back({kind, a, b});
        }
    }
};
static void flush_spans(dril_ctx* c) {
    if (c->spans.empty()) return;
    cudaStreamSynchronize(c->stream);
    for (auto& s : c->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) { c->prof_ms[s.kind] += ms; c->prof_n[s.kind] += 1; }
        c->free_events.push_back(s.a); c->free_events.push_back(s.b);
    }
    c->spans.clear();
}

template <typename T>
static int32_t dmalloc(T** p, size_t n) {
    DRIL_CUDA(cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)));
    return DRIL_OK;
}
static int32_t ensure_scratch(dril_policy* p, size_t bytes) {
    if (p->scratch_bytes >= bytes) return DRIL_OK;
    if (p->scratch) cudaFree(p->scratch);
    p->scratch = nullptr; p->scratch_bytes = 0;
    DRIL_CUDA(cudaMalloc(&p->scratch, bytes));
    p->scratch_bytes = bytes;
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
extern "C" int32_t dril_ctx_create(int32_t device, uint64_t seed, dril_ctx** out) {
    DRIL_REQUIRE(out, "out is NULL");
    int32_t n = 0;
    DRIL_TRY(dril_device_count(&n));
    DRIL_REQUIRE(device >= 0 && device < n, "device %d out of range (%d devices)", device, n);
    DRIL_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    DRIL_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        dril_set_error("device %d is sm_%d%d; libdril_b200 is built for sm_100a only", device, prop.major, prop.minor);
        return DRIL_ERR_UNSUPPORTED;
    }
    dril_ctx* c = new dril_ctx();
    c->device = device;
    c->seed = seed;
    c->sm_count = prop.multiProcessorCount;
    DRIL_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (unsigned ks : k_kind_sets)
        for (int ws = 0; ws < 2; ++ws) {
            DRIL_CUDA(cudaFuncSetAttribute(rollout_fn(ws, ks), cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
            DRIL_CUDA(cudaFuncSetAttribute(rollout_fast_fn(ws, ks), cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
        }
    DRIL_CUDA(cudaFuncSetAttribute(policy_apply_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
    DRIL_CUDA(cudaFuncSetAttribute(policy_apply_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
    DRIL_CUDA(cudaFuncSetAttribute(ppo_loss_grad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
    DRIL_CUDA(cudaFuncSetAttribute(ppo_loss_grad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX));
    DRIL_CUDA(cudaFuncSetAttribute(ppo_loss_grad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
    DRIL_CUDA(cudaFuncSetAttribute(ppo_loss_grad_ft_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM_BYTES));
    DRIL_CUDA(cudaFuncSetAttribute(ppo_loss_grad_ft_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM_BYTES));
    {
        const void* fns[] = {(const void*)ppo_loss_grad_ftg_kernel<2, 0, 1>, (const void*)ppo_loss_grad_ftg_kernel<2, 0, 2>,
                             (const void*)ppo_loss_grad_ftg_kernel<2, 1, 1>, (const void*)ppo_loss_grad_ftg_kernel<2, 1, 2>,
                             (const void*)ppo_loss_grad_ftg_kernel<3, 0, 1>, (const void*)ppo_loss_grad_ftg_kernel<3, 0, 2>,
                             (const void*)ppo_loss_grad_ftg_kernel<3, 1, 1>, (const void*)ppo_loss_grad_ftg_kernel<3, 1, 2>,
                             (const void*)ppo_loss_grad_ftg_kernel<2, 0, 3>, (const void*)ppo_loss_grad_ftg_kernel<2, 0, 4>,
                             (const void*)ppo_loss_grad_ftg_kernel<3, 0, 3>, (const void*)ppo_loss_grad_ftg_kernel<3, 0, 4>};
        for (const void* fn : fns) DRIL_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX - 2048));   // 1 KB of static shared memory
        for (int L = 2; L <= 3; ++L)
            for (unsigned ks : k_kind_sets)
                for (int an = 2; an <= 4; an += 2)
                    DRIL_CUDA(cudaFuncSetAttribute(rollout_gtc_fn(L, ks, an), cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX - 2048));
        DRIL_CUDA(cudaFuncSetAttribute(critic_values_ftg_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX - 2048));
        DRIL_CUDA(cudaFuncSetAttribute(critic_values_ftg_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, DRIL_SMEM_MAX - 2048));
    }
    DRIL_CUDA(cudaFuncSetAttribute(rollout_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_SMEM_BYTES));
    DRIL_CUDA(cudaFuncSetAttribute(rollout_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_SMEM_BYTES));
    *out = c;
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_destroy(dril_ctx* c) {
    if (!c) return DRIL_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    flush_spans(c);
    for (auto e : c->free_events) cudaEventDestroy(e);
    for (auto e : c->user_ev) if (e) cudaEventDestroy(e);
    if (c->l2_scratch) cudaFree(c->l2_scratch);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    cudaStreamDestroy(c->stream);
    delete c;
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_synchronize(dril_ctx* c) {
    DRIL_REQUIRE(c, "ctx is NULL");
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_launch_count(dril_ctx* c, int64_t* launches) {
    DRIL_REQUIRE(c && launches, "NULL argument");
    *launches = c->launches;
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_set_profiling(dril_ctx* c, int32_t on) {
    DRIL_REQUIRE(c, "ctx is NULL");
    flush_spans(c);
    c->profiling = on != 0;
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_reset_profile(dril_ctx* c) {
    DRIL_REQUIRE(c, "ctx is NULL");
    flush_spans(c);
    for (int i = 0; i < DRIL_K_COUNT; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_get_profile(dril_ctx* c, int32_t kind, double* total_ms, int64_t* launches) {
    DRIL_REQUIRE(c && kind >= 0 && kind < DRIL_K_COUNT, "bad profile kind %d", kind);
    flush_spans(c);
    if (total_ms) *total_ms = c->prof_ms[kind];
    if (launches) *launches = c->prof_n[kind];
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_event_record(dril_ctx* c, int32_t slot) {
    DRIL_REQUIRE(c && slot >= 0 && slot < 16, "bad event slot");
    DRIL_CUDA(cudaSetDevice(c->device));
    if (!c->user_ev[slot]) DRIL_CUDA(cudaEventCreate(&c->user_ev[slot]));
    DRIL_CUDA(cudaEventRecord(c->user_ev[slot], c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_event_elapsed_ms(dril_ctx* c, int32_t a, int32_t b, float* ms) {
    DRIL_REQUIRE(c && ms && a >= 0 && a < 16 && b >= 0 && b < 16 && c->user_ev[a] && c->user_ev[b], "bad event slots");
    DRIL_CUDA(cudaEventSynchronize(c->user_ev[b]));
    DRIL_CUDA(cudaEventElapsedTime(ms, c->user_ev[a], c->user_ev[b]));
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_flush_l2(dril_ctx* c) {
    DRIL_REQUIRE(c, "ctx is NULL");
    DRIL_CUDA(cudaSetDevice(c->device));
    if (!c->l2_scratch) {
        c->l2_bytes = (size_t)256 << 20;   // > 126 MB L2
        DRIL_CUDA(cudaMalloc(&c->l2_scratch, c->l2_bytes));
    }
    DRIL_CUDA(cudaMemsetAsync(c->l2_scratch, 0, c->l2_bytes, c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_ctx_sm_count(dril_ctx* c, int32_t* sms) {
    DRIL_REQUIRE(c && sms, "NULL argument");
    *sms = c->sm_count;
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// comm
// ---------------------------------------------------------------------------------------
extern "C" int32_t dril_comm_unique_id(uint8_t id_out[128]) {
    DRIL_TRY(nccl_load());
    nccl_uid id;
    DRIL_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, 128);
    return DRIL_OK;
}
extern "C" int32_t dril_comm_init(dril_ctx* c, int32_t rank, int32_t nranks, const uint8_t id[128]) {
    DRIL_REQUIRE(c && id && nranks >= 1 && rank >= 0 && rank < nranks, "bad comm arguments");
    DRIL_TRY(nccl_load());
    DRIL_CUDA(cudaSetDevice(c->device));
    nccl_uid uid;
    memcpy(&uid, id, 128);
    DRIL_NCCL(g_nccl.CommInitRank(&c->comm, nranks, uid, rank));
    c->rank = rank; c->nranks = nranks;
    return DRIL_OK;
}
extern "C" int32_t dril_comm_destroy(dril_ctx* c) {
    DRIL_REQUIRE(c, "ctx is NULL");
    if (c->comm) { cudaStreamSynchronize(c->stream); g_nccl.CommDestroy(c->comm); c->comm = nullptr; }
    if (c->p2p_enabled) {
        for (int r = 0; r < c->nranks; ++r) if (r != c->rank && c->p2p_peer_base[r]) cudaIpcCloseMemHandle(c->p2p_peer_base[r]);
        c->p2p_enabled = false;
    }
    c->rank = 0; c->nranks = 1;
    return DRIL_OK;
}
#define P2P_HDR_BYTES 256   // [0] flag (u64), [8] seq (u64), [16] err (int)
#define P2P_MAX_CTA 256
extern "C" int32_t dril_comm_p2p_export(dril_ctx* c, int64_t n_slots, uint8_t handle_out[64]) {
    DRIL_REQUIRE(c && handle_out && n_slots >= 1, "bad p2p arguments");
    DRIL_REQUIRE(c->nranks >= 1 && c->nranks <= DRIL_MAX_RANKS, "p2p allreduce supports up to %d ranks", DRIL_MAX_RANKS);
    DRIL_CUDA(cudaSetDevice(c->device));
    if (c->p2p_region) { cudaFree(c->p2p_region); c->p2p_region = nullptr; c->p2p_enabled = false; }
    size_t slots = ((size_t)n_slots + 63) & ~(size_t)63;
    // [header | gbuf[2][slots] (pull exchange) | recv[2][nranks][slots] (push exchange) | cflag[nranks][P2P_MAX_CTA] |
    //  srecv[2][nranks][P2P_SMALL_MAX] doubles | sflag[DRIL_MAX_RANKS]]; header: [0] flag, [8] seq, [16] err, [24] small_seq
    size_t bytes = P2P_HDR_BYTES + 2 * slots * sizeof(float) + 2 * (size_t)c->nranks * slots * sizeof(float) +
                   (size_t)c->nranks * P2P_MAX_CTA * sizeof(unsigned long long) +
                   2 * (size_t)c->nranks * P2P_SMALL_MAX * sizeof(double) + DRIL_MAX_RANKS * sizeof(unsigned long long);
    DRIL_CUDA(cudaMalloc(&c->p2p_region, bytes));
    DRIL_CUDA(cudaMemset(c->p2p_region, 0, bytes));
    memset(&c->p2p, 0, sizeof(c->p2p));
    c->p2p.n_slots = (int)slots;
    cudaIpcMemHandle_t h;
    DRIL_CUDA(cudaIpcGetMemHandle(&h, c->p2p_region));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle_out, &h, 64);
    return DRIL_OK;
}
extern "C" int32_t dril_comm_p2p_import(dril_ctx* c, const uint8_t* handles) {
    DRIL_REQUIRE(c && handles && c->p2p_region, "dril_comm_p2p_export must be called first");
    DRIL_CUDA(cudaSetDevice(c->device));
    char* local = (char*)c->p2p_region;
    for (int r = 0; r < c->nranks; ++r) {
        void* base = nullptr;
        if (r == c->rank) base = c->p2p_region;
        else {
            cudaIpcMemHandle_t h;
            memcpy(&h, handles + 64 * r, 64);
            DRIL_CUDA(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
        }
        c->p2p_peer_base[r] = base;
        c->p2p.peer_flag[r] = (const volatile unsigned long long*)base;
        c->p2p.peer_gbuf[r] = (const float*)((char*)base + P2P_HDR_BYTES);
        char* recv = (char*)base + P2P_HDR_BYTES + 2 * (size_t)c->p2p.n_slots * sizeof(float);
        c->p2p.peer_recv[r] = (float*)recv;
        c->p2p.peer_cflag[r] = (unsigned long long*)(recv + 2 * (size_t)c->nranks * c->p2p.n_slots * sizeof(float));
        char* small = (char*)c->p2p.peer_cflag[r] + (size_t)c->nranks * P2P_MAX_CTA * sizeof(unsigned long long);
        c->p2p.peer_srecv[r] = (double*)small;
        c->p2p.peer_sflag[r] = (unsigned long long*)(small + 2 * (size_t)c->nranks * P2P_SMALL_MAX * sizeof(double));
    }
    c->p2p.local_srecv = c->p2p.peer_srecv[c->rank];
    c->p2p.local_sflag = c->p2p.peer_sflag[c->rank];
    c->p2p.small_seq = (unsigned long long*)(local + 24);
    c->p2p.local_recv = c->p2p.peer_recv[c->rank];
    c->p2p.local_cflag = c->p2p.peer_cflag[c->rank];
    c->p2p.max_cta = P2P_MAX_CTA;
    c->p2p.local_flag = (volatile unsigned long long*)local;
    c->p2p.local_seq = (unsigned long long*)(local + 8);
    c->p2p.err = (int*)(local + 16);
    c->p2p.local_gbuf = (float*)(local + P2P_HDR_BYTES);
    c->p2p.nranks = c->nranks; c->p2p.rank = c->rank;
    c->p2p_enabled = true;
    return DRIL_OK;
}
static int32_t allreduce_sum(dril_ctx* c, void* buf, size_t count, bool is_double) {
    if (!c->comm || c->nranks == 1) return DRIL_OK;
    Span sp(c, DRIL_K_ALLREDUCE);
    DRIL_NCCL(g_nccl.AllReduce(buf, buf, count, is_double ? NCCL_FLOAT64 : NCCL_FLOAT32, NCCL_SUM, c->comm, c->stream));
    return DRIL_OK;
}

// in-place sum over ranks of two small fp64 arrays (either may be empty): peer memory if available, else NCCL
static int32_t allreduce_small(dril_ctx* c, double* a, int na, double* b, int nb) {
    if (c->nranks == 1 || na + nb == 0) return DRIL_OK;
    if (c->p2p_enabled && na + nb <= P2P_SMALL_MAX) {
        Span sp(c, DRIL_K_ALLREDUCE);
        p2p_small_allreduce_kernel<<<1, P2P_SMALL_MAX, 0, c->stream>>>(c->p2p, a, na, b, nb);
        DRIL_CUDA(cudaGetLastError());
        return DRIL_OK;
    }
    if (na) DRIL_TRY(allreduce_sum(c, a, (size_t)na, true));
    if (nb) DRIL_TRY(allreduce_sum(c, b, (size_t)nb, true));
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// buffer
// ---------------------------------------------------------------------------------------
extern "C" int32_t dril_buffer_create(dril_ctx* c, int64_t T, int64_t N, int32_t obs_dim, int32_t act_kind,
                                      int32_t act_dim, dril_buffer** out) {
    DRIL_REQUIRE(c && out && T >= 1 && N >= 1 && obs_dim >= 1 && obs_dim <= DRIL_MAX_OBS_DIM, "bad buffer arguments");
    DRIL_REQUIRE(act_kind == DRIL_ACT_DISCRETE || (act_kind == DRIL_ACT_CONTINUOUS && act_dim >= 1 && act_dim <= DRIL_MAX_ACT_DIM),
                 "bad action space");
    DRIL_CUDA(cudaSetDevice(c->device));
    dril_buffer* b = new dril_buffer();
    b->ctx = c;
    memset(&b->d, 0, sizeof(b->d));
    b->d.T = T; b->d.N = N; b->d.obs_dim = obs_dim; b->d.act_kind = act_kind;
    b->d.act_dim = act_kind == DRIL_ACT_DISCRETE ? 1 : act_dim;
    b->act_elems = b->d.act_dim;
    size_t tn = (size_t)T * N;
    // one slab (one cudaMalloc + one memset) carved into the fields, each 256-byte aligned
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t off = 0, o_obs = off; off += al(tn * obs_dim * 4);
    size_t o_act = off; off += al(tn * b->act_elems * 4);
    size_t o_f[7];
    for (int i = 0; i < 7; ++i) { o_f[i] = off; off += al(tn * 4); }
    size_t o_last = off; off += al((size_t)N * 4);
    size_t o_epl = off; off += al(tn * 4);
    size_t o_flags = off; off += al(tn);
    size_t o_dc = off; off += al((size_t)T * 4);
    DRIL_CUDA(cudaMalloc(&b->slab, off));
    char* base = (char*)b->slab;
    b->d.obs = (float*)(base + o_obs); b->d.actions = base + o_act;
    b->d.rewards = (float*)(base + o_f[0]); b->d.values = (float*)(base + o_f[1]); b->d.logprobs = (float*)(base + o_f[2]);
    b->d.advantages = (float*)(base + o_f[3]); b->d.returns = (float*)(base + o_f[4]); b->d.boot = (float*)(base + o_f[5]);
    b->d.episode_r = (float*)(base + o_f[6]); b->d.last_values = (float*)(base + o_last); b->d.episode_l = (int*)(base + o_epl);
    b->d.flags = (unsigned char*)(base + o_flags); b->d.done_count = (int*)(base + o_dc);
    // reset!(rollout_buffer) zero-fills (rollout_buffer.jl:35-44)
    DRIL_CUDA(cudaMemsetAsync(b->slab, 0, off, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    *out = b;
    return DRIL_OK;
}
extern "C" int32_t dril_buffer_destroy(dril_buffer* b) {
    if (!b) return DRIL_OK;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    cudaFree(b->slab);
    if (b->tcs_slab) cudaFree(b->tcs_slab);
    if (b->dcs_slab) cudaFree(b->dcs_slab);
    delete b;
    return DRIL_OK;
}
static int32_t buffer_field(dril_buffer* b, int32_t field, void** ptr, int64_t* bytes) {
    size_t tn = (size_t)b->d.T * b->d.N;
    switch (field) {
        case DRIL_BUF_OBS: *ptr = b->d.obs; *bytes = tn * b->d.obs_dim * 4; break;
        case DRIL_BUF_ACTIONS: *ptr = b->d.actions; *bytes = tn * b->act_elems * 4; break;
        case DRIL_BUF_REWARDS: *ptr = b->d.rewards; *bytes = tn * 4; break;
        case DRIL_BUF_VALUES: *ptr = b->d.values; *bytes = tn * 4; break;
        case DRIL_BUF_LOGPROBS: *ptr = b->d.logprobs; *bytes = tn * 4; break;
        case DRIL_BUF_ADVANTAGES: *ptr = b->d.advantages; *bytes = tn * 4; break;
        case DRIL_BUF_RETURNS: *ptr = b->d.returns; *bytes = tn * 4; break;
        case DRIL_BUF_FLAGS: *ptr = b->d.flags; *bytes = tn; break;
        case DRIL_BUF_BOOT: *ptr = b->d.boot; *bytes = tn * 4; break;
        case DRIL_BUF_LAST_VALUES: *ptr = b->d.last_values; *bytes = (size_t)b->d.N * 4; break;
        case DRIL_BUF_EPISODE_R: *ptr = b->d.episode_r; *bytes = tn * 4; break;
        case DRIL_BUF_EPISODE_L: *ptr = b->d.episode_l; *bytes = tn * 4; break;
        default: dril_set_error("unknown buffer field %d", field); return DRIL_ERR_INVALID;
    }
    return DRIL_OK;
}
extern "C" int32_t dril_buffer_field_bytes(dril_buffer* b, int32_t field, int64_t* bytes) {
    DRIL_REQUIRE(b && bytes, "NULL argument");
    void* p;
    return buffer_field(b, field, &p, bytes);
}
extern "C" int32_t dril_buffer_download(dril_buffer* b, int32_t field, void* dst, int64_t bytes) {
    DRIL_REQUIRE(b && dst, "NULL argument");
    void* p; int64_t nb;
    DRIL_TRY(buffer_field(b, field, &p, &nb));
    DRIL_REQUIRE(bytes == nb, "field %d is %lld bytes, caller passed %lld", field, (long long)nb, (long long)bytes);
    DRIL_CUDA(cudaSetDevice(b->ctx->device));
    DRIL_CUDA(cudaMemcpyAsync(dst, p, nb, cudaMemcpyDeviceToHost, b->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_buffer_upload(dril_buffer* b, int32_t field, const void* src, int64_t bytes) {
    DRIL_REQUIRE(b && src, "NULL argument");
    void* p; int64_t nb;
    DRIL_TRY(buffer_field(b, field, &p, &nb));
    DRIL_REQUIRE(bytes == nb, "field %d is %lld bytes, caller passed %lld", field, (long long)nb, (long long)bytes);
    DRIL_CUDA(cudaSetDevice(b->ctx->device));
    DRIL_CUDA(cudaMemcpyAsync(p, src, nb, cudaMemcpyHostToDevice, b->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// policy
// ---------------------------------------------------------------------------------------
static inline int pad4(int x) { return (x + 3) & ~3; }
struct LossLaunch { int M4; bool ws; size_t smem; int grid_cap; int splits; bool single; bool mma; bool thin; };
static int32_t plan_loss(dril_policy* p, LossLaunch* out);
static bool ftg_active(const dril_policy* p);

extern "C" int32_t dril_policy_create(dril_ctx* c, int32_t obs_dim, int32_t n_hidden, const int32_t* hidden,
                                      int32_t act_kind, int32_t act_n, int32_t act_start, const float* act_low,
                                      const float* act_high, dril_policy** out) {
    DRIL_REQUIRE(c && out, "NULL argument");
    DRIL_REQUIRE(obs_dim >= 1 && obs_dim <= DRIL_MAX_OBS_DIM, "obs_dim %d out of range", obs_dim);
    DRIL_REQUIRE(n_hidden >= 0 && n_hidden <= DRIL_MAX_HIDDEN_LAYERS, "n_hidden %d out of range", n_hidden);
    DRIL_REQUIRE(act_kind == DRIL_ACT_DISCRETE || act_kind == DRIL_ACT_CONTINUOUS, "bad act_kind");
    DRIL_REQUIRE(act_n >= 1 && (act_kind == DRIL_ACT_DISCRETE ? act_n <= 1024 : act_n <= DRIL_MAX_ACT_DIM), "act_n %d out of range", act_n);
    for (int i = 0; i < n_hidden; ++i) DRIL_REQUIRE(hidden[i] >= 1 && hidden[i] <= 1024, "hidden dim out of range");
    DRIL_CUDA(cudaSetDevice(c->device));
    dril_policy* p = new dril_policy();
    p->ctx = c;
    p->seed = c->seed;
    PolicyDesc& pd = p->pd;
    memset(&pd, 0, sizeof(pd));
    pd.obs_dim = obs_dim; pd.obs_dim_p = pad4(obs_dim);
    pd.act_kind = act_kind; pd.act_n = act_n; pd.act_start = act_start;
    // layer shapes (layers/layer_helpers.jl:27-57): empty hidden_dims -> single Dense(in -> 1)
    pd.n_layers = n_hidden == 0 ? 1 : n_hidden + 1;
    int flat_off = 0, pack_off = 0;
    pd.max_np = 4;
    for (int net = 0; net < 2; ++net) {
        for (int l = 0; l < pd.n_layers; ++l) {
            LayerDesc& L = pd.L[net][l];
            L.K = l == 0 ? obs_dim : hidden[l - 1];
            if (n_hidden == 0) L.N = 1;
            else L.N = l < n_hidden ? hidden[l] : (net == 0 ? act_n : 1);
            L.Kp = pad4(L.K); L.Np = pad4(L.N);
            L.w_off = flat_off; flat_off += L.K * L.N;
            L.b_off = flat_off; flat_off += L.N;
            L.pw_off = pack_off; pack_off += L.Kp * L.Np;
            L.pb_off = pack_off; pack_off += L.Np;
            pd.max_np = std::max(pd.max_np, L.Np);
        }
    }
    if (n_hidden == 0) DRIL_REQUIRE(act_kind == DRIL_ACT_DISCRETE ? act_n == 1 : act_n == 1,
                                    "hidden_dims=[] gives a Dense(in->1) actor (layer_helpers.jl:33); act_n must be 1");
    pd.pack_fwd = pack_off;
    for (int net = 0; net < 2; ++net)
        for (int l = 0; l < pd.n_layers; ++l) { pd.L[net][l].pwt_off = pack_off; pack_off += pd.L[net][l].Kp * pd.L[net][l].Np; }
    pd.pack_total = pack_off;
    pd.log_std_off = -1;
    if (act_kind == DRIL_ACT_CONTINUOUS) { pd.log_std_off = flat_off; flat_off += act_n; }
    pd.n_params = flat_off;
    pd.gpack = pd.pack_fwd + pad4(act_n) + 8;
    for (int j = 0; j < DRIL_MAX_ACT_DIM; ++j) {
        pd.act_low[j] = (act_kind == DRIL_ACT_CONTINUOUS && act_low && j < act_n) ? act_low[j] : -INFINITY;
        pd.act_high[j] = (act_kind == DRIL_ACT_CONTINUOUS && act_high && j < act_n) ? act_high[j] : INFINITY;
    }
    // index maps flat -> packed W, packed Wt, packed gradient
    std::vector<int> f2p(pd.n_params, -1), f2t(pd.n_params, -1), f2g(pd.n_params, -1);
    for (int net = 0; net < 2; ++net)
        for (int l = 0; l < pd.n_layers; ++l) {
            const LayerDesc& L = pd.L[net][l];
            for (int k = 0; k < L.K; ++k)
                for (int n = 0; n < L.N; ++n) {
                    int f = L.w_off + k * L.N + n;   // Lux (out,in) column-major == [in][out]
                    f2p[f] = L.pw_off + k * L.Np + n;
                    f2t[f] = L.pwt_off + n * L.Kp + k;
                    f2g[f] = f2p[f];
                }
            for (int n = 0; n < L.N; ++n) { f2p[L.b_off + n] = L.pb_off + n; f2g[L.b_off + n] = L.pb_off + n; }
        }
    if (act_kind == DRIL_ACT_CONTINUOUS)
        for (int j = 0; j < act_n; ++j) f2g[pd.log_std_off + j] = pd.pack_fwd + j;
    size_t np = pd.n_params;
    DRIL_TRY(dmalloc(&p->flat, np)); DRIL_TRY(dmalloc(&p->m, np)); DRIL_TRY(dmalloc(&p->v, np));
    DRIL_TRY(dmalloc(&p->g, np + 8)); DRIL_TRY(dmalloc(&p->pack, (size_t)pd.pack_total));
    DRIL_TRY(dmalloc(&p->flat2pack, np)); DRIL_TRY(dmalloc(&p->flat2packT, np)); DRIL_TRY(dmalloc(&p->flat2g, np));
    DRIL_TRY(dmalloc(&p->step, 1)); DRIL_TRY(dmalloc(&p->iter_acc, ITER_ACC_N)); DRIL_TRY(dmalloc(&p->ev_acc, 4));
    DRIL_TRY(dmalloc(&p->stop_flag, 1));
    p->gpart_ctas = c->sm_count * 2;   // CTAs per partial plane
    DRIL_TRY(dmalloc(&p->gpart, (size_t)DRIL_GPLANES * p->gpart_ctas * pd.gpack));
    DRIL_CUDA(cudaMemcpy(p->flat2pack, f2p.data(), np * 4, cudaMemcpyHostToDevice));
    DRIL_CUDA(cudaMemcpy(p->flat2packT, f2t.data(), np * 4, cudaMemcpyHostToDevice));
    DRIL_CUDA(cudaMemcpy(p->flat2g, f2g.data(), np * 4, cudaMemcpyHostToDevice));
    DRIL_CUDA(cudaMemset(p->flat, 0, np * 4)); DRIL_CUDA(cudaMemset(p->m, 0, np * 4)); DRIL_CUDA(cudaMemset(p->v, 0, np * 4));
    DRIL_CUDA(cudaMemset(p->g, 0, (np + 8) * 4)); DRIL_CUDA(cudaMemset(p->pack, 0, (size_t)pd.pack_total * 4));
    DRIL_CUDA(cudaMemset(p->step, 0, 8)); DRIL_CUDA(cudaMemset(p->iter_acc, 0, ITER_ACC_N * 8));
    DRIL_CUDA(cudaMemset(p->ev_acc, 0, 32)); DRIL_CUDA(cudaMemset(p->stop_flag, 0, 4));
    DRIL_CUDA(cudaMemset(p->gpart, 0, (size_t)DRIL_GPLANES * p->gpart_ctas * pd.gpack * 4));
    for (int i = 0; i < 3; ++i) DRIL_CUDA(cudaEventCreate(&p->ev[i]));
    {   // gradient partial planes per parameter (must mirror the tile choice in ppo_loss_grad_kernel)
        LossLaunch ll;
        DRIL_TRY(plan_loss(p, &ll));
        p->loss_M4 = ll.M4; p->loss_ws = ll.ws; p->loss_splits = ll.splits; p->plan_single = ll.single ? 1 : 0;
        p->plan_mma = ll.mma ? 1 : 0;
        std::vector<unsigned char> planes(np, 1);
        for (int net = 0; net < 2; ++net)
            for (int l = 0; l < pd.n_layers; ++l) {
                const LayerDesc& L = pd.L[net][l];
                const bool t8 = (ll.M4 % 16) == 0 && (L.Kp % 8) == 0 && (L.Np % 8) == 0;
                const bool mma = ll.mma && mma_layer_ok(L.Kp, L.Np);
                for (int i = 0; i < L.K * L.N; ++i) planes[L.w_off + i] = (unsigned char)(mma ? 1 : (t8 ? 2 : ll.splits));
            }
        DRIL_TRY(dmalloc(&p->f2planes, np));
        DRIL_CUDA(cudaMemcpy(p->f2planes, planes.data(), np, cudaMemcpyHostToDevice));
        std::vector<unsigned char> one_plane(np, 1);
        DRIL_TRY(dmalloc(&p->f2planes_one, np));
        DRIL_CUDA(cudaMemcpy(p->f2planes_one, one_plane.data(), np, cudaMemcpyHostToDevice));
        DRIL_TRY(dmalloc(&p->sq_part, 8192));
        DRIL_TRY(dmalloc(&p->ticket, 1));
        DRIL_CUDA(cudaMemset(p->ticket, 0, 4));
        double ones[2] = {1.0, 1.0};
        DRIL_CUDA(cudaMemcpy(p->iter_acc + 12, ones, 16, cudaMemcpyHostToDevice));
    }
    c->policies.push_back(p);
    *out = p;
    return DRIL_OK;
}
extern "C" int32_t dril_policy_destroy(dril_policy* p) {
    if (!p) return DRIL_OK;
    cudaSetDevice(p->ctx->device);
    cudaStreamSynchronize(p->ctx->stream);
    {
        auto& v = p->ctx->policies;
        v.erase(std::remove(v.begin(), v.end(), p), v.end());
    }
    void* ps[] = {p->flat, p->pack, p->m, p->v, p->g, p->gpart, p->flat2pack, p->flat2packT, p->flat2g, p->step,
                  p->iter_acc, p->ev_acc, p->mbstats, p->adv_partial, p->stop_flag, p->scratch, p->f2planes, p->f2planes_one, p->sq_part,
                  p->ticket, p->ft_tiles, p->ft_recs};
    for (void* q : ps) if (q) cudaFree(q);
    for (int i = 0; i < 3; ++i) if (p->ev[i]) cudaEventDestroy(p->ev[i]);
    for (auto& sl : p->slots) {
        for (int i = 0; i < 4; ++i) if (sl.ev[i]) cudaEventDestroy(sl.ev[i]);
        if (sl.host) cudaFreeHost(sl.host);
    }
    if (p->rec_dev) cudaFree(p->rec_dev);
    delete p;
    return DRIL_OK;
}
extern "C" int32_t dril_policy_num_params(dril_policy* p, int64_t* n) {
    DRIL_REQUIRE(p && n, "NULL argument");
    *n = p->pd.n_params;
    return DRIL_OK;
}
/* 1 when dril_ppo_update / dril_ppo_loss_grad run the tcgen05 loss/grad kernel for this policy; 2 when they run the
 * general-shape kernel with at least one layer on mma.sync 3xTF32 tiles; 0: general-shape kernel, fp32 FMA tiles only */
extern "C" int32_t dril_policy_update_path(dril_policy* p, int32_t* out) {
    DRIL_REQUIRE(p && out, "NULL argument");
    *out = 0;
    if (ftg_active(p) || (g_opt_tc && tc_eligible(p->pd))) { *out = 1; return DRIL_OK; }
    if (p->plan_mma == 1)
        for (int net = 0; net < 2; ++net)
            for (int l = 0; l < p->pd.n_layers; ++l) {
                const LayerDesc& L = p->pd.L[net][l];
                if (mma_layer_ok(L.Kp, L.Np)) *out = 2;
            }
    return DRIL_OK;
}
static int32_t repack(dril_policy* p) {
    Span sp(p->ctx, DRIL_K_POLICY);
    int n = p->pd.n_params;
    repack_kernel<<<(n + 255) / 256, 256, 0, p->ctx->stream>>>(p->flat, p->pack, p->flat2pack, p->flat2packT, n);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}
extern "C" int32_t dril_policy_set_params(dril_policy* p, const float* flat, int64_t n) {
    DRIL_REQUIRE(p && flat, "NULL argument");
    DRIL_REQUIRE(n == p->pd.n_params, "expected %d parameters, got %lld", p->pd.n_params, (long long)n);
    DRIL_CUDA(cudaSetDevice(p->ctx->device));
    DRIL_CUDA(cudaMemcpyAsync(p->flat, flat, n * 4, cudaMemcpyHostToDevice, p->ctx->stream));
    DRIL_TRY(repack(p));
    DRIL_CUDA(cudaStreamSynchronize(p->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_policy_get_params(dril_policy* p, float* flat, int64_t n) {
    DRIL_REQUIRE(p && flat, "NULL argument");
    DRIL_REQUIRE(n == p->pd.n_params, "expected %d parameters, got %lld", p->pd.n_params, (long long)n);
    DRIL_CUDA(cudaSetDevice(p->ctx->device));
    DRIL_CUDA(cudaMemcpyAsync(flat, p->flat, n * 4, cudaMemcpyDeviceToHost, p->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(p->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_policy_get_opt_state(dril_policy* p, float* m, float* v, int64_t n, int64_t* step) {
    DRIL_REQUIRE(p && m && v && step, "NULL argument");
    DRIL_REQUIRE(n == p->pd.n_params, "expected %d parameters, got %lld", p->pd.n_params, (long long)n);
    DRIL_CUDA(cudaSetDevice(p->ctx->device));
    long long s = 0;
    DRIL_CUDA(cudaMemcpyAsync(m, p->m, n * 4, cudaMemcpyDeviceToHost, p->ctx->stream));
    DRIL_CUDA(cudaMemcpyAsync(v, p->v, n * 4, cudaMemcpyDeviceToHost, p->ctx->stream));
    DRIL_CUDA(cudaMemcpyAsync(&s, p->step, 8, cudaMemcpyDeviceToHost, p->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(p->ctx->stream));
    *step = s;
    return DRIL_OK;
}
extern "C" int32_t dril_policy_set_opt_state(dril_policy* p, const float* m, const float* v, int64_t n, int64_t step) {
    DRIL_REQUIRE(p && m && v, "NULL argument");
    DRIL_REQUIRE(n == p->pd.n_params, "expected %d parameters, got %lld", p->pd.n_params, (long long)n);
    DRIL_CUDA(cudaSetDevice(p->ctx->device));
    long long s = step;
    DRIL_CUDA(cudaMemcpyAsync(p->m, m, n * 4, cudaMemcpyHostToDevice, p->ctx->stream));
    DRIL_CUDA(cudaMemcpyAsync(p->v, v, n * 4, cudaMemcpyHostToDevice, p->ctx->stream));
    DRIL_CUDA(cudaMemcpyAsync(p->step, &s, 8, cudaMemcpyHostToDevice, p->ctx->stream));
    // running beta^t of the bias correction: the betas of the last update (Optimisers.Adam defaults (0.9, 0.999), ppo.jl:64-66, before one)
    double pw[2] = {pow(p->beta1, (double)step), pow(p->beta2, (double)step)};
    DRIL_CUDA(cudaMemcpyAsync(p->iter_acc + 12, pw, 16, cudaMemcpyHostToDevice, p->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(p->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_policy_seed(dril_policy* p, uint64_t seed, uint64_t step_index) {
    DRIL_REQUIRE(p, "NULL argument");
    p->seed = seed;
    p->step_index = (uint32_t)step_index;
    return DRIL_OK;
}

// tile width / weight placement for the stand-alone layer application
static int32_t launch_apply(dril_policy* p, ApplyArgs& a) {
    dril_ctx* c = p->ctx;
    const PolicyDesc& pd = p->pd;
    int M4 = 64;
    auto bytes = [&](int m4, bool ws) {
        int ld = m4 + 4;
        return ((size_t)(ws ? pd.pack_fwd : 0) + (size_t)pd.obs_dim_p * ld + (size_t)4 * pd.max_np * ld) * 4;
    };
    bool ws = true;
    while (M4 > 4 && bytes(M4, true) > DRIL_SMEM_MAX && bytes(M4, false) > DRIL_SMEM_MAX) M4 -= 4;
    if (bytes(M4, true) > DRIL_SMEM_MAX) ws = false;
    if (bytes(M4, ws) > DRIL_SMEM_MAX) { dril_set_error("network too wide for shared memory"); return DRIL_ERR_UNSUPPORTED; }
    while (M4 > 4 && (a.B + M4 - 1) / M4 < c->sm_count && M4 > (a.B + c->sm_count - 1) / c->sm_count) M4 -= 4;
    a.M4 = M4; a.weights_smem = ws;
    a.pd = pd; a.pack = p->pack; a.flat = p->flat; a.pseed = p->seed;
    long long tiles = (a.B + M4 - 1) / M4;
    int grid = (int)std::min<long long>(tiles, (long long)c->sm_count * 4);
    Span sp(c, DRIL_K_POLICY);
    if (ws) policy_apply_kernel<true><<<grid, DRIL_THREADS, bytes(M4, ws), c->stream>>>(a);
    else policy_apply_kernel<false><<<grid, DRIL_THREADS, bytes(M4, ws), c->stream>>>(a);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}

// host actions (int64 | float) -> device int32 | float
static int32_t stage_actions(dril_ctx* c, int act_kind, int act_n, const void* host, int64_t count, void* dev) {
    if (act_kind == DRIL_ACT_DISCRETE) {
        std::vector<int> tmp((size_t)count);
        const int64_t* src = (const int64_t*)host;
        for (int64_t i = 0; i < count; ++i) tmp[i] = (int)src[i];
        DRIL_CUDA(cudaMemcpyAsync(dev, tmp.data(), count * 4, cudaMemcpyHostToDevice, c->stream));
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
    } else {
        DRIL_CUDA(cudaMemcpyAsync(dev, host, count * act_n * 4, cudaMemcpyHostToDevice, c->stream));
    }
    return DRIL_OK;
}
static int32_t unstage_actions(dril_ctx* c, int act_kind, int act_n, const void* dev, int64_t count, void* host) {
    if (act_kind == DRIL_ACT_DISCRETE) {
        std::vector<int> tmp((size_t)count);
        DRIL_CUDA(cudaMemcpyAsync(tmp.data(), dev, count * 4, cudaMemcpyDeviceToHost, c->stream));
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
        int64_t* dst = (int64_t*)host;
        for (int64_t i = 0; i < count; ++i) dst[i] = tmp[i];
    } else {
        DRIL_CUDA(cudaMemcpyAsync(host, dev, count * act_n * 4, cudaMemcpyDeviceToHost, c->stream));
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
    }
    return DRIL_OK;
}

static int32_t policy_apply_host(dril_policy* p, int mode, const float* obs, const void* actions_in, int64_t B,
                                 const int64_t* gids, void* actions_out, float* values, float* logprobs, float* entropy) {
    DRIL_REQUIRE(p && obs && B >= 1, "bad arguments");
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const PolicyDesc& pd = p->pd;
    const int ae = pd.act_kind == DRIL_ACT_DISCRETE ? 1 : pd.act_n;
    size_t o_obs = 0, o_act = o_obs + (size_t)B * pd.obs_dim * 4, o_val = o_act + (size_t)B * ae * 4,
           o_lp = o_val + (size_t)B * 4, o_ent = o_lp + (size_t)B * 4, o_gid = (o_ent + (size_t)B * 4 + 7) & ~(size_t)7,
           total = o_gid + (size_t)B * 8;
    DRIL_TRY(ensure_scratch(p, total));
    char* s = (char*)p->scratch;
    DRIL_CUDA(cudaMemcpyAsync(s + o_obs, obs, (size_t)B * pd.obs_dim * 4, cudaMemcpyHostToDevice, c->stream));
    if (mode == 2) { DRIL_REQUIRE(actions_in, "actions is NULL"); DRIL_TRY(stage_actions(c, pd.act_kind, pd.act_n, actions_in, B, s + o_act)); }
    if (gids) DRIL_CUDA(cudaMemcpyAsync(s + o_gid, gids, (size_t)B * 8, cudaMemcpyHostToDevice, c->stream));
    ApplyArgs a;
    memset(&a, 0, sizeof(a));
    a.obs = (const float*)(s + o_obs);
    a.actions_in = mode == 2 ? (s + o_act) : nullptr;
    a.actions_out = (mode == 0 || mode == 1) ? (s + o_act) : nullptr;
    a.gids = gids ? (const long long*)(s + o_gid) : nullptr;
    a.values = (float*)(s + o_val);
    a.logprobs = mode != 3 ? (float*)(s + o_lp) : nullptr;
    a.entropy = mode == 2 ? (float*)(s + o_ent) : nullptr;
    a.B = B; a.mode = mode; a.step = p->step_index;
    DRIL_TRY(launch_apply(p, a));
    if (mode == 0) p->step_index += 1;
    if (values) DRIL_CUDA(cudaMemcpyAsync(values, s + o_val, (size_t)B * 4, cudaMemcpyDeviceToHost, c->stream));
    if (logprobs && mode != 3) DRIL_CUDA(cudaMemcpyAsync(logprobs, s + o_lp, (size_t)B * 4, cudaMemcpyDeviceToHost, c->stream));
    if (entropy && mode == 2) DRIL_CUDA(cudaMemcpyAsync(entropy, s + o_ent, (size_t)B * 4, cudaMemcpyDeviceToHost, c->stream));
    if (actions_out && (mode == 0 || mode == 1)) DRIL_TRY(unstage_actions(c, pd.act_kind, pd.act_n, s + o_act, B, actions_out));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_policy_forward(dril_policy* p, const float* obs, int64_t B, int32_t deterministic,
                                       const int64_t* env_gids, void* actions, float* values, float* logprobs) {
    return policy_apply_host(p, deterministic ? 1 : 0, obs, nullptr, B, env_gids, actions, values, logprobs, nullptr);
}
extern "C" int32_t dril_policy_evaluate(dril_policy* p, const float* obs, const void* actions, int64_t B,
                                        float* values, float* logprobs, float* entropy) {
    return policy_apply_host(p, 2, obs, actions, B, nullptr, nullptr, values, logprobs, entropy);
}
extern "C" int32_t dril_policy_predict_values(dril_policy* p, const float* obs, int64_t B, float* values) {
    return policy_apply_host(p, 3, obs, nullptr, B, nullptr, nullptr, values, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------
// env
// ---------------------------------------------------------------------------------------
static int32_t env_alloc_obs_arrays(dril_env* e);
static int32_t env_restart(dril_env* e);
extern "C" int32_t dril_env_create(dril_ctx* c, int32_t kind, int64_t n_envs, int32_t max_steps, int32_t obs_dim,
                                   int32_t act_start, int64_t gid_offset, const dril_norm_cfg* norm,
                                   int32_t monitor_window, dril_env** out) {
    DRIL_REQUIRE(c && out && n_envs >= 1, "bad env arguments");
    DRIL_REQUIRE(kind >= DRIL_ENV_CARTPOLE && kind <= DRIL_ENV_ACROBOT, "unknown env kind %d", kind);
    DRIL_REQUIRE(n_envs + gid_offset < (1ll << 32), "global env ids must fit 32 bits");
    DRIL_CUDA(cudaSetDevice(c->device));
    dril_env* e = new dril_env();
    e->ctx = c;
    EnvDev& d = e->d;
    memset(&d, 0, sizeof(d));
    memset(&e->nopolicy, 0, sizeof(e->nopolicy));
    d.kind = kind; d.n_envs = n_envs; d.gid_offset = gid_offset; d.seed = c->seed; d.act_start = act_start;
    if (kind == DRIL_ENV_CARTPOLE) { d.obs_dim = 4; d.state_dim = 4; d.act_dim = 0; d.max_steps = max_steps > 0 ? max_steps : 500; }
    else if (kind == DRIL_ENV_PENDULUM) { d.obs_dim = 3; d.state_dim = 2; d.act_dim = 1; d.max_steps = max_steps > 0 ? max_steps : 200; }
    else if (kind == DRIL_ENV_MOUNTAINCAR) { d.obs_dim = 2; d.state_dim = 2; d.act_dim = 0; d.max_steps = max_steps > 0 ? max_steps : 200; }
    else if (kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS) { d.obs_dim = 2; d.state_dim = 2; d.act_dim = 1; d.max_steps = max_steps > 0 ? max_steps : 999; }
    else if (kind == DRIL_ENV_ACROBOT) { d.obs_dim = 6; d.state_dim = 4; d.act_dim = 0; d.max_steps = max_steps > 0 ? max_steps : 500; }
    else {
        DRIL_REQUIRE(obs_dim >= 1 && obs_dim <= DRIL_MAX_OBS_DIM, "synthetic obs_dim %d out of range", obs_dim);
        d.obs_dim = obs_dim; d.state_dim = 0; d.act_dim = 0; d.max_steps = max_steps > 0 ? max_steps : 500;
    }
    d.hist_len = 1; d.frame_dim = d.obs_dim;
    size_t n = (size_t)n_envs;
    DRIL_TRY(dmalloc(&d.state, n * std::max(d.state_dim, 1))); DRIL_TRY(dmalloc(&d.steps, n));
    DRIL_TRY(dmalloc(&d.episode, n)); DRIL_TRY(dmalloc(&d.life, n));
    DRIL_TRY(dmalloc(&d.old_rewards, n));
    DRIL_CUDA(cudaMemset(d.state, 0, n * std::max(d.state_dim, 1) * 4)); DRIL_CUDA(cudaMemset(d.steps, 0, n * 4));
    DRIL_CUDA(cudaMemset(d.episode, 0, n * 4)); DRIL_CUDA(cudaMemset(d.life, 0, n * 4));
    DRIL_CUDA(cudaMemset(d.old_rewards, 0, n * 4));
    d.monitor = monitor_window > 0 ? monitor_window : 0;
    DRIL_TRY(dmalloc(&d.ep_ret, n)); DRIL_TRY(dmalloc(&d.ep_len, n)); DRIL_TRY(dmalloc(&d.roll_sums, 2)); DRIL_TRY(dmalloc(&d.roll_eps, 1));
    DRIL_CUDA(cudaMemset(d.ep_ret, 0, n * 4)); DRIL_CUDA(cudaMemset(d.ep_len, 0, n * 4));
    DRIL_CUDA(cudaMemset(d.roll_sums, 0, 16)); DRIL_CUDA(cudaMemset(d.roll_eps, 0, 8));
    int w = std::max(d.monitor, 1);
    e->ring.window = w;
    DRIL_TRY(dmalloc(&e->ring.ret, (size_t)w)); DRIL_TRY(dmalloc(&e->ring.len, (size_t)w)); DRIL_TRY(dmalloc(&e->ring.head, 1));
    DRIL_CUDA(cudaMemset(e->ring.ret, 0, w * 4)); DRIL_CUDA(cudaMemset(e->ring.len, 0, w * 4)); DRIL_CUDA(cudaMemset(e->ring.head, 0, 8));
    d.normalize = norm ? 1 : 0;
    if (norm) {
        d.training = norm->training; d.norm_obs = norm->norm_obs; d.norm_reward = norm->norm_reward;
        d.clip_obs = norm->clip_obs; d.clip_reward = norm->clip_reward; d.ngamma = norm->gamma; d.eps = norm->epsilon;
    }
    e->max_blocks = c->sm_count * 8;
    DRIL_TRY(dmalloc(&d.ret, n));
    DRIL_TRY(dmalloc(&d.ret_stats, 2)); DRIL_TRY(dmalloc(&d.counts, 2));
    DRIL_TRY(dmalloc(&e->norm_snap_cnt, 2));
    d.roll_moments = nullptr;
    DRIL_CUDA(cudaMemset(d.ret, 0, n * 4));
    {   // RunningMeanStd init: mean 0, var 1, count 0 (normalizeWrapperEnv.jl:13-15); the obs columns in env_alloc_obs_arrays
        float rs[2] = {0.f, 1.f};
        DRIL_CUDA(cudaMemcpy(d.ret_stats, rs, 8, cudaMemcpyHostToDevice));
        DRIL_CUDA(cudaMemset(d.counts, 0, 16));
    }
    DRIL_CUDA(cudaMalloc(&e->compat_actions, n * std::max(d.act_dim, 1) * 4));
    DRIL_TRY(env_alloc_obs_arrays(e));
    *out = e;
    DRIL_TRY(dril_env_reset(e));
    return DRIL_OK;
}
// the arrays sized by obs_dim, (re)allocated for the env's current width: terminal and old observations, the normaliser's
// obs mean / var (mean 0, var 1), its per-CTA partials, the data-parallel moments and exchange buffers, the compat buffer, and
// the observation-history store (filled from the current state)
static int32_t env_alloc_obs_arrays(dril_env* e) {
    dril_ctx* c = e->ctx;
    EnvDev& d = e->d;
    const size_t n = (size_t)d.n_envs, D = (size_t)d.obs_dim;
    for (float** p : {&d.tobs, &d.old_obs, &d.obs_mean, &d.obs_var, &e->norm_snap, &e->compat_obs, &d.hist}) { if (*p) cudaFree(*p); *p = nullptr; }
    for (double** p : {&d.partials, &e->roll_moments, &e->xr}) { if (*p) cudaFree(*p); *p = nullptr; }
    if (e->compat) { dril_buffer_destroy(e->compat); e->compat = nullptr; }
    DRIL_TRY(dmalloc(&d.tobs, n * D)); DRIL_TRY(dmalloc(&d.old_obs, n * D));
    DRIL_CUDA(cudaMemset(d.tobs, 0, n * D * 4)); DRIL_CUDA(cudaMemset(d.old_obs, 0, n * D * 4));
    DRIL_TRY(dmalloc(&d.obs_mean, D)); DRIL_TRY(dmalloc(&d.obs_var, D));
    DRIL_TRY(dmalloc(&d.partials, (size_t)2 * e->max_blocks * (2 * D + 2)));
    DRIL_TRY(dmalloc(&e->roll_moments, (size_t)2 * (D + 1) + 2));     // handed to the kernels only in data-parallel runs
    DRIL_TRY(dmalloc(&e->xr, (size_t)4 + 3 + 2 * (D + 1) + 2));
    DRIL_TRY(dmalloc(&e->norm_snap, (size_t)2 * D + 2));
    {
        std::vector<float> ones(D, 1.0f);
        DRIL_CUDA(cudaMemset(d.obs_mean, 0, D * 4));
        DRIL_CUDA(cudaMemcpy(d.obs_var, ones.data(), D * 4, cudaMemcpyHostToDevice));
    }
    DRIL_TRY(dril_buffer_create(c, 1, d.n_envs, d.obs_dim, d.act_dim == 0 ? DRIL_ACT_DISCRETE : DRIL_ACT_CONTINUOUS,
                                std::max(d.act_dim, 1), &e->compat));
    DRIL_TRY(dmalloc(&e->compat_obs, n * D));
    if (d.hist_len > 1) {
        DRIL_TRY(dmalloc(&d.hist, n * (size_t)(d.hist_len - 1) * d.frame_dim));
        DRIL_TRY(env_restart(e));
    }
    return DRIL_OK;
}
// every env's observation history restarted from its current frame and its action queue restarted (no-op without either)
static int32_t env_restart(dril_env* e) {
    if (!e->d.hist && !e->d.act_delay) return DRIL_OK;
    dril_ctx* c = e->ctx;
    Span sp(c, DRIL_K_ENV);
    const unsigned grid = (unsigned)((e->d.n_envs + 255) / 256);
    if (env_perturbed(e)) env_perturb_restart_kernel<<<grid, 256, 0, c->stream>>>(e->d);   // noisy frames, queues
    else env_hist_fill_kernel<<<grid, 256, 0, c->stream>>>(e->d);
    DRIL_CUDA(cudaGetLastError());
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_destroy(dril_env* e) {
    if (!e) return DRIL_OK;
    cudaSetDevice(e->ctx->device);
    cudaStreamSynchronize(e->ctx->stream);
    // iterations still in flight keep a back-pointer to their env (episode bookkeeping in dril_iteration_result): cleared here
    for (dril_policy* p : e->ctx->policies) {
        if (p->last_env == e) p->last_env = nullptr;
        for (auto& sl : p->slots) if (sl.env == e) sl.env = nullptr;
    }
    EnvDev& d = e->d;
    void* ps[] = {d.state, d.steps, d.episode, d.life, d.tobs, d.old_obs, d.old_rewards, d.ep_ret, d.ep_len, d.roll_sums,
                  d.roll_eps, d.ret, d.obs_mean, d.obs_var, d.ret_stats, d.counts, d.partials, e->ring.ret, e->ring.len,
                  e->ring.head, e->compat_actions, e->compat_obs, e->roll_moments, e->xr, e->norm_snap, e->norm_snap_cnt,
                  d.pval, d.plo, d.phi, d.hist, d.obs_noise, d.act_delay, d.act_q};
    for (void* p : ps) if (p) cudaFree(p);
    dril_buffer_destroy(e->compat);
    delete e;
    return DRIL_OK;
}
extern "C" int32_t dril_env_seed(dril_env* e, uint64_t seed) {
    DRIL_REQUIRE(e, "NULL argument");
    DRIL_CUDA(cudaSetDevice(e->ctx->device));
    e->d.seed = seed;
    DRIL_CUDA(cudaMemsetAsync(e->d.episode, 0, (size_t)e->d.n_envs * 4, e->ctx->stream));
    DRIL_CUDA(cudaMemsetAsync(e->d.life, 0, (size_t)e->d.n_envs * 4, e->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(e->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_reset(dril_env* e) {
    DRIL_REQUIRE(e, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    {
        Span sp(c, DRIL_K_ENV);
        const unsigned grid = (unsigned)((e->d.n_envs + 255) / 256);
        if (env_has_params(env_ks(e))) env_reset_kernel<ENV_KS_ALL | ENV_KS_PARAMS><<<grid, 256, 0, c->stream>>>(e->d);
        else env_reset_kernel<ENV_KS_ALL><<<grid, 256, 0, c->stream>>>(e->d);
        DRIL_CUDA(cudaGetLastError());
    }
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return env_restart(e);
}
extern "C" int32_t dril_env_set_params(dril_env* e, int32_t n_params, const float* lo, const float* hi) {
    DRIL_REQUIRE(e, "NULL argument");
    EnvDev& d = e->d;
    const int np = env_n_params(d.kind);
    DRIL_REQUIRE(np > 0, "env kind %d has no physical parameters", d.kind);
    DRIL_REQUIRE(n_params == np, "env kind %d has %d parameters, got %d", d.kind, np, n_params);
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const size_t n = (size_t)d.n_envs;
    std::vector<float> dflt;
    if (!lo && (e->obs_ks || env_perturbed(e))) {   // observed parameters / history / perturbation stay: back to lo = hi = the defaults
        dflt.resize(n * np);
        for (int k = 0; k < np; ++k) std::fill(dflt.begin() + (size_t)k * n, dflt.begin() + (size_t)(k + 1) * n, env_param_default(d.kind).v[k]);
        lo = hi = dflt.data();
    }
    if (!lo) {   // back to the built-in constants and the default instantiations
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
        e->default_params = false;
        for (float* p : {d.pval, d.plo, d.phi}) if (p) cudaFree(p);
        d.pval = d.plo = d.phi = nullptr;
        d.has_params = 0;
        return DRIL_OK;
    }
    if (!hi) hi = lo;
    for (int k = 0; k < np; ++k) {
        const bool pos = k_env_param_positive[d.kind][k] != 0;
        for (size_t i = 0; i < n; ++i) {
            const float l = lo[(size_t)k * n + i], h = hi[(size_t)k * n + i];
            DRIL_REQUIRE(std::isfinite(l) && std::isfinite(h) && l <= h, "parameter %d of env %zu: range [%g, %g] is not finite with lo <= hi",
                         k, i, (double)l, (double)h);
            DRIL_REQUIRE(pos ? l > 0.f : l >= 0.f, "parameter %d of env %zu: lo %g must be %s 0", k, i, (double)l, pos ? ">" : ">=");
        }
    }
    if (!d.pval) {
        DRIL_TRY(dmalloc(&d.pval, n * DRIL_ENV_MAX_PARAMS));
        DRIL_TRY(dmalloc(&d.plo, n * DRIL_ENV_MAX_PARAMS));
        DRIL_TRY(dmalloc(&d.phi, n * DRIL_ENV_MAX_PARAMS));
    }
    DRIL_CUDA(cudaMemcpyAsync(d.plo, lo, n * np * 4, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(d.phi, hi, n * np * 4, cudaMemcpyHostToDevice, c->stream));
    d.has_params = 1;
    e->default_params = !dflt.empty();
    {
        Span sp(c, DRIL_K_ENV);
        env_params_draw_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d);
        DRIL_CUDA(cudaGetLastError());
    }
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_get_params(dril_env* e, int32_t n_params, float* values) {
    DRIL_REQUIRE(e && values, "NULL argument");
    const EnvDev& d = e->d;
    const int np = env_n_params(d.kind);
    DRIL_REQUIRE(n_params == np, "env kind %d has %d parameters, got %d", d.kind, np, n_params);
    const size_t n = (size_t)d.n_envs;
    if (!d.has_params) {
        for (int k = 0; k < np; ++k) std::fill(values + (size_t)k * n, values + (size_t)(k + 1) * n, env_param_default(d.kind).v[k]);
        return DRIL_OK;
    }
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    DRIL_CUDA(cudaMemcpyAsync(values, d.pval, n * np * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}

// An env with an observation layout option, observation noise or action delay runs the parametrised kernels: without ranges it
// holds lo = hi = the defaults, which it drops again with the last such option.
static int32_t env_hold_default_params(dril_env* e) {
    const bool need = e->obs_ks || env_perturbed(e);
    if ((need && !e->d.has_params) || (!need && e->default_params)) DRIL_TRY(dril_env_set_params(e, env_n_params(e->d.kind), nullptr, nullptr));
    return DRIL_OK;
}
// the observation layout: obs_ks (0, ENV_KS_OBS_PARAMS or ENV_KS_HISTORY), the history's k and frame width, the observation width
// and the obs-sized arrays
static int32_t env_set_obs_layout(dril_env* e, unsigned obs_ks, int hist_len, int frame_dim) {
    EnvDev& d = e->d;
    const int np = env_n_params(d.kind);
    DRIL_CUDA(cudaSetDevice(e->ctx->device));
    DRIL_CUDA(cudaStreamSynchronize(e->ctx->stream));
    e->obs_ks = obs_ks;
    d.hist_len = hist_len;
    d.frame_dim = frame_dim;
    d.obs_dim = frame_dim * hist_len + (obs_ks == ENV_KS_OBS_PARAMS ? np : 0);
    DRIL_TRY(env_hold_default_params(e));
    return env_alloc_obs_arrays(e);
}
extern "C" int32_t dril_env_set_observe_params(dril_env* e, int32_t on) {
    DRIL_REQUIRE(e, "NULL argument");
    EnvDev& d = e->d;
    if (env_n_params(d.kind) == 0) { dril_set_error("env kind %d has no physical parameters to observe", d.kind); return DRIL_ERR_UNSUPPORTED; }
    if (on && e->obs_ks == ENV_KS_HISTORY) { dril_set_error("observe_params cannot be combined with an observation history"); return DRIL_ERR_UNSUPPORTED; }
    if (on && env_perturbed(e)) { dril_set_error("observe_params cannot be combined with observation noise or action delay"); return DRIL_ERR_UNSUPPORTED; }
    DRIL_REQUIRE(!e->observed, "observe_params can only change before the env's first observation");
    if ((on != 0) == (e->obs_ks == ENV_KS_OBS_PARAMS)) return DRIL_OK;
    return env_set_obs_layout(e, on ? ENV_KS_OBS_PARAMS : 0u, 1, env_base_obs_dim(d.kind));
}
extern "C" int32_t dril_env_set_obs_history(dril_env* e, int32_t history_len, int32_t mask_velocities) {
    DRIL_REQUIRE(e, "NULL argument");
    EnvDev& d = e->d;
    const bool on = history_len != 1 || mask_velocities != 0;
    if (env_n_params(d.kind) == 0) { dril_set_error("env kind %d has no observation history", d.kind); return DRIL_ERR_UNSUPPORTED; }
    if (on && e->obs_ks == ENV_KS_OBS_PARAMS) { dril_set_error("an observation history cannot be combined with observe_params"); return DRIL_ERR_UNSUPPORTED; }
    DRIL_REQUIRE(history_len >= 1 && history_len <= DRIL_ENV_MAX_HISTORY, "history_len %d outside [1, %d]", history_len, DRIL_ENV_MAX_HISTORY);
    const int frame_dim = env_frame_dim(d.kind, mask_velocities != 0);
    if (history_len == d.hist_len && frame_dim == d.frame_dim) return DRIL_OK;
    DRIL_REQUIRE(!e->observed, "the observation history can only change before the env's first observation");
    return env_set_obs_layout(e, on ? ENV_KS_HISTORY : 0u, history_len, frame_dim);
}
extern "C" int32_t dril_env_set_obs_noise(dril_env* e, int32_t n_comp, const float* std) {
    DRIL_REQUIRE(e, "NULL argument");
    EnvDev& d = e->d;
    if (env_n_params(d.kind) == 0) { dril_set_error("env kind %d has no observation noise", d.kind); return DRIL_ERR_UNSUPPORTED; }
    if (std && e->obs_ks == ENV_KS_OBS_PARAMS) { dril_set_error("observation noise cannot be combined with observe_params"); return DRIL_ERR_UNSUPPORTED; }
    const int D0 = env_base_obs_dim(d.kind);
    const size_t n = (size_t)d.n_envs;
    if (std) {
        DRIL_REQUIRE(n_comp == D0, "env kind %d has %d observation components, got %d", d.kind, D0, n_comp);
        for (size_t i = 0; i < (size_t)D0 * n; ++i)
            DRIL_REQUIRE(std::isfinite(std[i]) && std[i] >= 0.f, "noise std %g of component %zu, env %zu is not finite and >= 0",
                         (double)std[i], i / n, i % n);
    }
    DRIL_CUDA(cudaSetDevice(e->ctx->device));
    DRIL_CUDA(cudaStreamSynchronize(e->ctx->stream));
    if (!std) {
        if (d.obs_noise) cudaFree(d.obs_noise);
        d.obs_noise = nullptr;
        return env_hold_default_params(e);
    }
    if (!d.obs_noise) DRIL_TRY(dmalloc(&d.obs_noise, (size_t)D0 * n));
    DRIL_CUDA(cudaMemcpy(d.obs_noise, std, (size_t)D0 * n * 4, cudaMemcpyHostToDevice));
    return env_hold_default_params(e);
}
extern "C" int32_t dril_env_set_action_delay(dril_env* e, const int32_t* delay) {
    DRIL_REQUIRE(e, "NULL argument");
    EnvDev& d = e->d;
    if (env_n_params(d.kind) == 0) { dril_set_error("env kind %d has no action delay", d.kind); return DRIL_ERR_UNSUPPORTED; }
    if (delay && e->obs_ks == ENV_KS_OBS_PARAMS) { dril_set_error("action delay cannot be combined with observe_params"); return DRIL_ERR_UNSUPPORTED; }
    const size_t n = (size_t)d.n_envs;
    int max_delay = 0;
    if (delay) {
        for (size_t i = 0; i < n; ++i) {
            DRIL_REQUIRE(delay[i] >= 0 && delay[i] <= DRIL_ENV_MAX_ACTION_DELAY, "delay %d of env %zu outside [0, %d]", delay[i], i,
                         DRIL_ENV_MAX_ACTION_DELAY);
            max_delay = std::max(max_delay, (int)delay[i]);
        }
    }
    DRIL_CUDA(cudaSetDevice(e->ctx->device));
    DRIL_CUDA(cudaStreamSynchronize(e->ctx->stream));
    d.max_delay = max_delay;
    if (!delay) {
        for (void* p : {(void*)d.act_delay, (void*)d.act_q}) if (p) cudaFree(p);
        d.act_delay = nullptr; d.act_q = nullptr;
        return env_hold_default_params(e);
    }
    if (!d.act_delay) {
        DRIL_TRY(dmalloc(&d.act_delay, n));
        DRIL_TRY(dmalloc(&d.act_q, (size_t)DRIL_ENV_MAX_ACTION_DELAY * n));
    }
    std::vector<int32_t> dq(delay, delay + n);   // every queue restarts: the next action fills it
    for (int32_t& v : dq) v |= ENV_DELAY_RESTART;
    DRIL_CUDA(cudaMemcpy(d.act_delay, dq.data(), n * 4, cudaMemcpyHostToDevice));
    return env_hold_default_params(e);
}
extern "C" int32_t dril_env_obs_dim(dril_env* e, int32_t* obs_dim) {
    DRIL_REQUIRE(e && obs_dim, "NULL argument");
    *obs_dim = e->d.obs_dim;
    return DRIL_OK;
}

extern "C" int32_t dril_env_num_envs(dril_env* e, int64_t* n) {
    DRIL_REQUIRE(e && n, "NULL argument");
    *n = e->d.n_envs;
    return DRIL_OK;
}

// Launch the rollout engine. policy may be NULL (compat paths).
// scratch of the deferred-critic rollouts (final observations + the compact list of truncated terminal observations)
static int32_t ensure_tcs(dril_buffer* b) {
    if (b->tcs_slab) return DRIL_OK;
    const size_t cap = (size_t)b->d.T * b->d.N, N = (size_t)b->d.N;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_last = 0, o_tobs = o_last + al(N * 16), o_tidx = o_tobs + al(cap * 16), o_cnt = o_tidx + al(cap * 8);
    DRIL_CUDA(cudaMalloc(&b->tcs_slab, o_cnt + 256));
    char* base = (char*)b->tcs_slab;
    b->tcs.last_obs = (float*)(base + o_last); b->tcs.trunc_obs = (float*)(base + o_tobs);
    b->tcs.trunc_idx = (long long*)(base + o_tidx); b->tcs.trunc_count = (unsigned int*)(base + o_cnt);
    b->tcs.cap = (unsigned int)std::min<size_t>(cap, 0x7fffffffu);
    return DRIL_OK;
}
static int32_t ensure_dcs(dril_buffer* b) {
    if (b->dcs_slab) return DRIL_OK;
    const size_t cap = (size_t)b->d.T * b->d.N, Db = (size_t)b->d.obs_dim * 4, N = (size_t)b->d.N;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_last = 0, o_tobs = o_last + al(N * Db), o_tidx = o_tobs + al(cap * Db), o_cnt = o_tidx + al(cap * 8);
    DRIL_CUDA(cudaMalloc(&b->dcs_slab, o_cnt + 256));
    char* base = (char*)b->dcs_slab;
    b->dcs.last_obs = (float*)(base + o_last); b->dcs.trunc_obs = (float*)(base + o_tobs);
    b->dcs.trunc_idx = (long long*)(base + o_tidx); b->dcs.trunc_count = (unsigned int*)(base + o_cnt);
    b->dcs.cap = (unsigned int)std::min<size_t>(cap, 0x7fffffffu);
    return DRIL_OK;
}

static int32_t launch_rollout(dril_env* e, dril_policy* p, dril_buffer* b, const void* forced_dev, float* obs_out_dev,
                              int T, int base_flags) {
    dril_ctx* c = e->ctx;
    RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.env = e->d; a.buf = b->d;
    const bool has_policy = p != nullptr;
    a.pd = has_policy ? p->pd : e->nopolicy;
    a.pack = has_policy ? p->pack : nullptr;
    a.flat = has_policy ? p->flat : nullptr;
    a.forced = forced_dev; a.obs_out = obs_out_dev;
    a.pseed = has_policy ? p->seed : 0; a.step0 = has_policy ? p->step_index : 0;
    a.T = T;
    int flags = base_flags | (has_policy ? RO_HAS_POLICY : 0);
    const EnvDev& d = e->d;
    const unsigned ks = env_ks(e);
    e->observed = true;
    const bool upd = d.normalize && d.training && (d.norm_obs || d.norm_reward);
    if (upd) flags |= RO_GRID_SYNC;
    const long long N = d.n_envs;
    const bool general_only = (base_flags & RO_DETERMINISTIC) != 0 || b->is_view;   // evaluation / chunked collection
    if (has_policy && !general_only && g_opt_tc_rollout && !d.normalize && !d.has_params && d.kind == DRIL_ENV_CARTPOLE && d.obs_dim == 4 && T > 0 && tc_eligible(a.pd) &&
        T == b->d.T) {
        // tensor-core path: actor-only step loop (64 envs per CTA) + one batched critic pass for values / bootstrap values
        DRIL_TRY(ensure_tcs(b));
        DRIL_CUDA(cudaMemsetAsync(b->tcs.trunc_count, 0, 4, c->stream));
        a.flags = flags; a.M4 = RT_ENVS;
        a.n_tiles = (int)((N + RT_ENVS - 1) / RT_ENVS);
        {
            Span sp(c, DRIL_K_ROLLOUT);
            // at least two tiles per SM: the two-CTAs-per-SM build (64 registers) overlaps two per-step chains
            static const int two_opt = getenv("DRIL_TC_ROLLOUT_2CTA") ? atoi(getenv("DRIL_TC_ROLLOUT_2CTA")) : 1;
            const bool two = two_opt && a.n_tiles >= 2 * c->sm_count;
            const int grid = std::min(a.n_tiles, (two ? 2 : 1) * c->sm_count);
            if (two) rollout_tc_kernel<2><<<grid, RT_THREADS, RT_SMEM_BYTES, c->stream>>>(a, b->tcs);
            else rollout_tc_kernel<1><<<grid, RT_THREADS, RT_SMEM_BYTES, c->stream>>>(a, b->tcs);
            DRIL_CUDA(cudaGetLastError());
        }
        {
            Span sp(c, DRIL_K_ROLLOUT);
            const long long tiles = ((long long)b->d.T * N + N + 127) / 128 + 8;
            const int grid = (int)std::min<long long>(tiles, 3ll * c->sm_count);
            critic_values_tc_kernel<<<grid, CV_THREADS, CV_SMEM_BYTES, c->stream>>>(a.pd, a.pack, b->d, b->tcs);
            DRIL_CUDA(cudaGetLastError());
        }
        return DRIL_OK;
    }
    if (has_policy && g_opt_syn_rollout && !general_only && T > 0 && syn_rollout_eligible(a.pd, d)) {      // (evaluation / chunked collection: general kernel)
        // synthetic env + small policy: one thread per env, everything in registers (rollout_syn.cuh)
        int hp = 0;
        for (int net = 0; net < 2; ++net)
            for (int l = 0; l + 1 < a.pd.n_layers; ++l) hp = std::max(hp, a.pd.L[net][l].Np);
        const int HP = hp <= 8 ? 8 : 16, NH = a.pd.n_layers - 1;
        const int E = (HP == 8 && g_opt_syn_rollout == 2) ? 2 : 1;          // envs per thread: two only on request (measured slower: registers halve the occupancy)
        const int threads = N >= 512ll * c->sm_count ? 128 : (N >= 64ll * c->sm_count ? 64 : 32);
        const int grid = (int)((N + (long long)threads * E - 1) / ((long long)threads * E));
        const size_t smem = (size_t)syn_smem_layout((d.obs_dim + 3) & ~3, HP, NH).total * sizeof(float);
        a.flags = flags; a.M4 = threads; a.n_tiles = grid;
        Span sp(c, DRIL_K_ROLLOUT);
        if (HP == 8 && NH == 1 && E == 2) rollout_syn_kernel<8, 1, 2><<<grid, threads, smem, c->stream>>>(a);
        else if (HP == 8 && E == 2) rollout_syn_kernel<8, 2, 2><<<grid, threads, smem, c->stream>>>(a);
        else if (HP == 8 && NH == 1) rollout_syn_kernel<8, 1, 1><<<grid, threads, smem, c->stream>>>(a);
        else if (HP == 8) rollout_syn_kernel<8, 2, 1><<<grid, threads, smem, c->stream>>>(a);
        else if (NH == 1) rollout_syn_kernel<16, 1, 1><<<grid, threads, smem, c->stream>>>(a);
        else rollout_syn_kernel<16, 2, 1><<<grid, threads, smem, c->stream>>>(a);
        DRIL_CUDA(cudaGetLastError());
        return DRIL_OK;
    }
    static const int env_nofast = getenv("DRIL_ROLLOUT_NO_FAST") ? atoi(getenv("DRIL_ROLLOUT_NO_FAST")) : 0;
    if (has_policy && !upd && !env_nofast && !(base_flags & RO_DETERMINISTIC) && d.kind != DRIL_ENV_SYNTHETIC && a.pd.act_n <= RF_MAX_OUT - 1 && T > 0 &&
        (a.pd.act_kind == DRIL_ACT_DISCRETE || a.pd.act_n == 1)) {
        // fast path: state in registers, one tile per CTA, K-split output layers
        static const int f_ctas = getenv("DRIL_FAST_CTAS_PER_SM") ? atoi(getenv("DRIL_FAST_CTAS_PER_SM")) : 2;
        const long long want = (long long)c->sm_count * std::max(f_ctas, 1);
        int M4 = (int)std::min<long long>(64, ((N + want - 1) / want + 3) & ~3ll);
        M4 = std::max(M4, 8);
        if (M4 > 32) M4 = 64; else if (M4 > 16) M4 = 32; else if (M4 > 8) M4 = 16; else M4 = 8;   // threads % M4 == 0
        int tiles = 2 * (a.pd.max_np >> 2) * (M4 >> 2);
        // many envs per SM: the rollout is throughput bound -> 64-env tiles, 8x8 register tiles
        // (1 B of shared-memory traffic per FMA instead of 2), several CTAs per SM
        static const int f_t8 = getenv("DRIL_FAST_TILES8") ? atoi(getenv("DRIL_FAST_TILES8")) : -1;
        const bool t8 = f_t8 >= 0 ? (f_t8 != 0 && M4 >= 16) : (M4 == 64 && N >= 96ll * c->sm_count);
        if (t8) { flags |= RO_TILES_8X8; tiles = 2 * (a.pd.max_np >> 3) * (M4 >> 3); }
        int threads = std::min(DRIL_THREADS, std::max(128, (tiles + 31) & ~31));
        const int tq = std::max(32, M4);
        threads = std::min(DRIL_THREADS, (threads + tq - 1) / tq * tq);
        static const int f_threads = getenv("DRIL_FAST_THREADS") ? atoi(getenv("DRIL_FAST_THREADS")) : 0;
        if (f_threads >= tq && f_threads <= DRIL_THREADS && f_threads % tq == 0) threads = f_threads;
        bool ws = true;
        const int hist_rows = (env_history(ks) ? d.obs_dim - d.frame_dim : 0) + (d.act_delay ? d.max_delay : 0);   // + action queues
        auto tot = [&](int m4, int th, bool w) { return rollout_fast_smem_layout(a.pd, m4, th, w, hist_rows).total; };
        if (tot(M4, threads, true) > DRIL_SMEM_MAX) ws = false;
        while (M4 > 8 && tot(M4, threads, ws) > DRIL_SMEM_MAX) M4 >>= 1;
        if (tot(M4, threads, ws) <= DRIL_SMEM_MAX) {
            a.M4 = M4; a.flags = flags | (ws ? RO_WEIGHTS_SMEM : 0);
            a.n_tiles = (int)((N + M4 - 1) / M4);
            Span sp(c, DRIL_K_ROLLOUT);
            void* args[] = {(void*)&a};
            DRIL_CUDA(cudaLaunchKernel(rollout_fast_fn(ws, ks), dim3(a.n_tiles), dim3(threads), args, tot(M4, threads, ws), c->stream));
            return DRIL_OK;
        }
    }
    // tile width: the per-step critical path (state load -> forward -> sample -> dynamics) is latency
    // bound, so small batches are cut into ~4 CTAs per SM that overlap each other's phases; at most
    // 64 envs per tile, shrink until shared memory fits
    // shapes the general tcgen05 kernels cover (update_ftg.cuh): only the actor runs inside the step loop; V(s_t), V(terminal_obs)
    // and V(new_obs) come from one batched critic pass over the stored (normalised) observations afterwards
    const bool defer = has_policy && g_opt_defer_critic && g_opt_ftg && ftg_eligible(a.pd) && !b->is_view && T == b->d.T && T > 0 &&
                       !(base_flags & RO_DETERMINISTIC);
    if (defer) {
        DRIL_TRY(ensure_dcs(b));
        DRIL_CUDA(cudaMemsetAsync(b->dcs.trunc_count, 0, 4, c->stream));
        a.dc = b->dcs;
        flags |= RO_DEFER_CRITIC;
    }
    // the batched critic pass behind a deferred-critic step loop
    auto launch_critic = [&]() -> int32_t {
        Span sp2(c, DRIL_K_ROLLOUT);
        const FtgLayout lay = ftg_layout(a.pd);
        const long long tiles = ((long long)b->d.T * N + N + 63) / 64 + 8;
        const int cgrid = (int)std::min<long long>(tiles, (long long)c->sm_count);
        if (a.pd.n_layers - 1 == 2) critic_values_ftg_kernel<2><<<cgrid, FTG_THREADS, (size_t)lay.total, c->stream>>>(a.pd, a.pack, b->d, b->dcs, lay);
        else critic_values_ftg_kernel<3><<<cgrid, FTG_THREADS, (size_t)lay.total, c->stream>>>(a.pd, a.pack, b->d, b->dcs, lay);
        DRIL_CUDA(cudaGetLastError());
        return DRIL_OK;
    };
    // enough envs for a 128-env tile per SM: the actor's layers on tcgen05 inside the step loop (rollout_gtc.cuh)
    if (defer && g_opt_tc_actor && N >= 64ll * c->sm_count) {
        const size_t body = rollout_smem_layout(a.pd, d.obs_dim, d.act_dim, GTC_ENVS, false, true, false, true).total;
        const GtcLayout gl = gtc_layout(a.pd);
        const size_t smem_g = body + (size_t)gl.total;
        if (smem_g <= (size_t)DRIL_SMEM_MAX - 2048) {
            a.M4 = GTC_ENVS; a.flags = flags;
            a.n_tiles = (int)((N + GTC_ENVS - 1) / GTC_ENVS);
            int grid = a.n_tiles, body_i = (int)body;
            void* fn = rollout_gtc_fn(a.pd.n_layers - 1, ks, a.pd.act_n);
            void* args[] = {(void*)&a, (void*)&gl, (void*)&body_i};
            {
                Span sp(c, DRIL_K_ROLLOUT);
                if (flags & RO_GRID_SYNC) {
                    int per_sm = 0;
                    DRIL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, DRIL_THREADS, smem_g));
                    DRIL_REQUIRE(per_sm >= 1, "rollout kernel does not fit on an SM");
                    grid = std::min(grid, std::min(per_sm * c->sm_count, e->max_blocks));
                    DRIL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(DRIL_THREADS), args, smem_g, c->stream));
                } else {
                    grid = std::min(grid, 4 * c->sm_count);
                    DRIL_CUDA(cudaLaunchKernel(fn, dim3(grid), dim3(DRIL_THREADS), args, smem_g, c->stream));
                }
            }
            return launch_critic();
        }
    }
    static const int env_ctas = getenv("DRIL_ROLLOUT_CTAS_PER_SM") ? atoi(getenv("DRIL_ROLLOUT_CTAS_PER_SM")) : 4;
    static const int env_threads = getenv("DRIL_ROLLOUT_THREADS") ? atoi(getenv("DRIL_ROLLOUT_THREADS")) : 0;
    const long long want_ctas = (long long)c->sm_count * std::max(env_ctas, 1);
    int M4 = (int)std::min<long long>(64, ((N + want_ctas - 1) / want_ctas + 3) & ~3ll);
    M4 = std::max(M4, 4);
    bool ws = has_policy;
    auto total = [&](int m4, bool w) { return rollout_smem_layout(a.pd, d.obs_dim, d.act_dim, m4, w, has_policy, !defer).total; };
    while (M4 > 4 && total(M4, ws) > DRIL_SMEM_MAX && total(M4, false) > DRIL_SMEM_MAX) M4 -= 4;
    if (total(M4, ws) > DRIL_SMEM_MAX) ws = false;
    if (total(M4, ws) > DRIL_SMEM_MAX) { dril_set_error("network too wide for the rollout kernel's shared memory"); return DRIL_ERR_UNSUPPORTED; }
    // weights that leave no room for a reasonable tile are streamed from L2 instead
    if (ws && M4 < 32 && N >= 32ll * c->sm_count && total(64, false) <= DRIL_SMEM_MAX) { ws = false; M4 = 64; }
    // wide nets whose weights stream from L2 anyway: 64-env tiles with the wide layers on mma.sync 3xTF32 tiles
    // (mma_tiles.cuh) once there are enough envs to give every SM such a tile
    if (has_policy && !ws && g_opt_mma && N >= 64ll * c->sm_count && total(64, false) <= DRIL_SMEM_MAX) {
        bool any = false;
        for (int net = 0; net < 2; ++net)
            for (int l = 0; l < a.pd.n_layers; ++l) {
                const LayerDesc& L = a.pd.L[net][l];
                any = any || mma_layer_ok(L.Kp, L.Np);
            }
        if (any) { M4 = 64; flags |= RO_MMA; }
        // critic deferred: the actor's activations alone leave room for 128-env tiles, i.e. one tile per SM and step at C3's
        // 16 384 envs instead of two 64-env tiles in sequence (the per-step env / statistics phases are per tile)
        if (any && defer && N >= 96ll * c->sm_count && total(128, false) <= DRIL_SMEM_MAX) M4 = 128;
    }
    if (ws) flags |= RO_WEIGHTS_SMEM;
    a.M4 = M4; a.flags = flags;
    a.n_tiles = (int)((N + M4 - 1) / M4);
    size_t smem = total(M4, ws);
    int grid = a.n_tiles;
    // block size: enough threads for the 4x4 thread-tiles of the widest layer of both nets
    int threads = DRIL_THREADS;
    if (has_policy) {
        int tiles = 2 * (a.pd.max_np >> 2) * (M4 >> 2);
        threads = std::min(DRIL_THREADS, std::max(128, (tiles + 31) & ~31));
    } else {
        threads = std::min(DRIL_THREADS, std::max(64, (M4 + 31) & ~31));
    }
    if (env_threads >= 32 && env_threads <= DRIL_THREADS) threads = env_threads & ~31;
    threads = std::max(threads, (M4 + 31) & ~31);
    Span sp(c, has_policy ? DRIL_K_ROLLOUT : DRIL_K_ENV);
    if (flags & RO_GRID_SYNC) {
        int per_sm = 0;
        DRIL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rollout_fn(ws, ks), threads, smem));
        DRIL_REQUIRE(per_sm >= 1, "rollout kernel does not fit on an SM");
        grid = std::min(grid, std::min(per_sm * c->sm_count, e->max_blocks));
        void* args[] = {(void*)&a};
        DRIL_CUDA(cudaLaunchCooperativeKernel(rollout_fn(ws, ks), dim3(grid), dim3(threads), args, smem, c->stream));
    } else {
        void* args[] = {(void*)&a};
        DRIL_CUDA(cudaLaunchKernel(rollout_fn(ws, ks), dim3(grid), dim3(threads), args, smem, c->stream));
    }
    if (defer) return launch_critic();
    return DRIL_OK;
}

static int32_t launch_monitor_finalize(dril_env* e, dril_buffer* b) {
    if (!e->d.monitor) return DRIL_OK;
    Span sp(e->ctx, DRIL_K_MONITOR);
    monitor_finalize_kernel<<<1, 1024, 0, e->ctx->stream>>>(e->ring, b->d.flags, b->d.episode_r, b->d.episode_l,
                                                            b->d.done_count, b->d.T, b->d.N);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}

extern "C" int32_t dril_env_observe(dril_env* e, float* obs_out) {
    DRIL_REQUIRE(e && obs_out, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    DRIL_TRY(launch_rollout(e, nullptr, e->compat, nullptr, e->compat_obs, 0, RO_INITIAL_OBSERVE | RO_WRITE_OBS_OUT));
    DRIL_CUDA(cudaMemcpyAsync(obs_out, e->compat_obs, (size_t)e->d.n_envs * e->d.obs_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}

extern "C" int32_t dril_env_step(dril_env* e, const void* actions, float* rewards, uint8_t* terminated, uint8_t* truncated,
                                 float* terminal_obs, float* episode_r, int64_t* episode_l) {
    DRIL_REQUIRE(e && actions && rewards && terminated && truncated, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const EnvDev& d = e->d;
    const int64_t N = d.n_envs;
    DRIL_TRY(stage_actions(c, d.act_dim == 0 ? DRIL_ACT_DISCRETE : DRIL_ACT_CONTINUOUS, d.act_dim, actions, N, e->compat_actions));
    DRIL_CUDA(cudaMemsetAsync(e->compat->d.done_count, 0, 4, c->stream));
    DRIL_CUDA(cudaMemsetAsync(d.roll_sums, 0, 16, c->stream));
    DRIL_CUDA(cudaMemsetAsync(d.roll_eps, 0, 8, c->stream));
    DRIL_TRY(launch_rollout(e, nullptr, e->compat, e->compat_actions, nullptr, 1, 0));
    DRIL_TRY(launch_monitor_finalize(e, e->compat));
    std::vector<uint8_t> flags((size_t)N);
    DRIL_CUDA(cudaMemcpyAsync(rewards, e->compat->d.rewards, N * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(flags.data(), e->compat->d.flags, N, cudaMemcpyDeviceToHost, c->stream));
    if (terminal_obs) DRIL_CUDA(cudaMemcpyAsync(terminal_obs, d.tobs, (size_t)N * d.obs_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    if (episode_r) DRIL_CUDA(cudaMemcpyAsync(episode_r, e->compat->d.episode_r, N * 4, cudaMemcpyDeviceToHost, c->stream));
    std::vector<int> el;
    if (episode_l) { el.resize((size_t)N); DRIL_CUDA(cudaMemcpyAsync(el.data(), e->compat->d.episode_l, N * 4, cudaMemcpyDeviceToHost, c->stream)); }
    unsigned long long eps = 0;
    DRIL_CUDA(cudaMemcpyAsync(&eps, d.roll_eps, 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    e->total_episodes += (int64_t)eps;
    for (int64_t i = 0; i < N; ++i) {
        terminated[i] = flags[i] & 1; truncated[i] = (flags[i] >> 1) & 1;
        if (episode_l) episode_l[i] = (flags[i] & 3) ? el[i] : 0;
        if (episode_r && !(flags[i] & 3)) episode_r[i] = 0.f;
    }
    return DRIL_OK;
}

extern "C" int32_t dril_env_get_state(dril_env* e, float* state, int32_t* steps) {
    DRIL_REQUIRE(e, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    if (state && e->d.state_dim) DRIL_CUDA(cudaMemcpyAsync(state, e->d.state, (size_t)e->d.n_envs * e->d.state_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    if (steps) DRIL_CUDA(cudaMemcpyAsync(steps, e->d.steps, (size_t)e->d.n_envs * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_set_state(dril_env* e, const float* state, const int32_t* steps) {
    DRIL_REQUIRE(e, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    if (state && e->d.state_dim) DRIL_CUDA(cudaMemcpyAsync(e->d.state, state, (size_t)e->d.n_envs * e->d.state_dim * 4, cudaMemcpyHostToDevice, c->stream));
    if (steps) DRIL_CUDA(cudaMemcpyAsync(e->d.steps, steps, (size_t)e->d.n_envs * 4, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return env_restart(e);
}
extern "C" int32_t dril_env_get_norm_stats(dril_env* e, float* obs_mean, float* obs_var, int64_t* obs_count,
                                           float* ret_mean, float* ret_var, int64_t* ret_count) {
    DRIL_REQUIRE(e, "NULL argument");
    DRIL_REQUIRE(e->d.normalize, "env has no NormalizeWrapperEnv");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    float rs[2]; long long cnt[2];
    if (obs_mean) DRIL_CUDA(cudaMemcpyAsync(obs_mean, e->d.obs_mean, e->d.obs_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    if (obs_var) DRIL_CUDA(cudaMemcpyAsync(obs_var, e->d.obs_var, e->d.obs_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(rs, e->d.ret_stats, 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(cnt, e->d.counts, 16, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    if (ret_mean) *ret_mean = rs[0];
    if (ret_var) *ret_var = rs[1];
    if (obs_count) *obs_count = cnt[0];
    if (ret_count) *ret_count = cnt[1];
    return DRIL_OK;
}
extern "C" int32_t dril_env_set_norm_stats(dril_env* e, const float* obs_mean, const float* obs_var, int64_t obs_count,
                                           float ret_mean, float ret_var, int64_t ret_count) {
    DRIL_REQUIRE(e && obs_mean && obs_var, "NULL argument");
    DRIL_REQUIRE(e->d.normalize, "env has no NormalizeWrapperEnv");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    float rs[2] = {ret_mean, ret_var}; long long cnt[2] = {obs_count, ret_count};
    DRIL_CUDA(cudaMemcpyAsync(e->d.obs_mean, obs_mean, e->d.obs_dim * 4, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(e->d.obs_var, obs_var, e->d.obs_dim * 4, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(e->d.ret_stats, rs, 8, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(e->d.counts, cnt, 16, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_set_training(dril_env* e, int32_t training) {
    DRIL_REQUIRE(e, "NULL argument");
    e->d.training = training ? 1 : 0;
    return DRIL_OK;
}
extern "C" int32_t dril_env_set_scaling(dril_env* e, int32_t on, const float* obs_low, const float* obs_high, const float* act_low,
                                        const float* act_high) {
    DRIL_REQUIRE(e, "NULL argument");
    // frames change with the mapping: an observation history restarts from the mapped frame
    if (!on) { e->d.scaling = 0; return env_restart(e); }
    DRIL_REQUIRE(obs_low && obs_high && act_low && act_high, "NULL bounds");
    // ScalingWrapperEnv needs Box observation and action spaces (scalingWrapperEnv.jl:22): of the built-in envs that is Pendulum
    DRIL_REQUIRE(e->d.kind == DRIL_ENV_PENDULUM || e->d.kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS,
                 "ScalingWrapperEnv: Box observation and action spaces required (pendulum, mountaincar_continuous)");
    // observed parameters (dril_env_set_observe_params) pass through raw: the bounds cover the base observation only (with
    // masked velocities (dril_env_set_obs_history) too: the kept components use their own bounds)
    const int D0 = env_base_obs_dim(e->d.kind);
    DRIL_REQUIRE(D0 <= 4 && e->d.act_dim == 1, "ScalingWrapperEnv: obs_dim <= 4, act_dim == 1");
    for (int j = 0; j < D0; ++j) {
        e->d.sc_obs_f[j] = 2.0f / (obs_high[j] - obs_low[j]);                     // :37-39
        e->d.sc_obs_o[j] = obs_low[j];
    }
    e->d.sc_act_f = 2.0f / (act_high[0] - act_low[0]);                            // :42-44
    e->d.sc_act_o = act_low[0];
    e->d.scaling = 1;
    return env_restart(e);
}
extern "C" int32_t dril_env_get_original(dril_env* e, float* obs_out, float* rewards_out) {
    DRIL_REQUIRE(e, "NULL argument");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    if (obs_out) DRIL_CUDA(cudaMemcpyAsync(obs_out, e->d.old_obs, (size_t)e->d.n_envs * e->d.obs_dim * 4, cudaMemcpyDeviceToHost, c->stream));
    if (rewards_out) DRIL_CUDA(cudaMemcpyAsync(rewards_out, e->d.old_rewards, (size_t)e->d.n_envs * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_env_monitor_stats(dril_env* e, float* ep_rew_mean, float* ep_len_mean, int64_t* n_in_window,
                                          int64_t* total_episodes) {
    DRIL_REQUIRE(e, "NULL argument");
    DRIL_REQUIRE(e->d.monitor, "env has no MonitorWrapperEnv");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    int w = e->ring.window;
    std::vector<float> r((size_t)w); std::vector<int> l((size_t)w);
    long long head = 0;
    DRIL_CUDA(cudaMemcpyAsync(r.data(), e->ring.ret, w * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(l.data(), e->ring.len, w * 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(&head, e->ring.head, 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    long long cnt = std::min<long long>(head, w);
    float sr = 0.f; double sl = 0;
    for (long long i = 0; i < cnt; ++i) { sr += r[i]; sl += l[i]; }   // mean(::CircularBuffer{Float32})
    if (ep_rew_mean) *ep_rew_mean = cnt ? sr / (float)cnt : NAN;
    if (ep_len_mean) *ep_len_mean = cnt ? (float)(sl / (double)cnt) : NAN;
    if (n_in_window) *n_in_window = cnt;
    if (total_episodes) *total_episodes = e->total_episodes;
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// rollout / GAE
// ---------------------------------------------------------------------------------------
static int32_t check_compat(dril_env* e, dril_policy* p, dril_buffer* b) {
    DRIL_REQUIRE(e && p && b, "NULL argument");
    DRIL_REQUIRE(e->ctx == p->ctx && e->ctx == b->ctx, "env, policy and buffer must share a ctx");
    DRIL_REQUIRE(b->d.N == e->d.n_envs, "buffer has %lld envs, env has %lld", b->d.N, e->d.n_envs);
    DRIL_REQUIRE(b->d.obs_dim == e->d.obs_dim && p->pd.obs_dim == e->d.obs_dim, "obs_dim mismatch");
    DRIL_REQUIRE(b->d.act_kind == p->pd.act_kind, "action kind mismatch between buffer and policy");
    if (p->pd.act_kind == DRIL_ACT_CONTINUOUS) DRIL_REQUIRE(b->d.act_dim == p->pd.act_n, "act_dim mismatch");
    if (e->d.kind == DRIL_ENV_CARTPOLE) DRIL_REQUIRE(p->pd.act_kind == DRIL_ACT_DISCRETE && p->pd.act_n == 2, "CartPole needs Discrete(2)");
    if (e->d.kind == DRIL_ENV_PENDULUM) DRIL_REQUIRE(p->pd.act_kind == DRIL_ACT_CONTINUOUS && p->pd.act_n == 1, "Pendulum needs Box (1,)");
    if (e->d.kind == DRIL_ENV_MOUNTAINCAR) DRIL_REQUIRE(p->pd.act_kind == DRIL_ACT_DISCRETE && p->pd.act_n == 3, "MountainCar needs Discrete(3)");
    if (e->d.kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS)
        DRIL_REQUIRE(p->pd.act_kind == DRIL_ACT_CONTINUOUS && p->pd.act_n == 1, "MountainCarContinuous needs Box (1,)");
    if (e->d.kind == DRIL_ENV_ACROBOT) DRIL_REQUIRE(p->pd.act_kind == DRIL_ACT_DISCRETE && p->pd.act_n == 3, "Acrobot needs Discrete(3)");
    return DRIL_OK;
}

// Data-parallel runs (SURVEY §8e): every rank normalises its own env shard during a rollout; afterwards the ranks merge the
// rollout's (count, mean, M2) over ALL shards into the statistics they started the rollout with (Chan merge of
// normalizeWrapperEnv.jl:37-48), so every rollout begins with identical statistics on every rank, and the Monitor sums
// (episode returns / lengths / count of the rollout) become global.
static bool dp_norm_active(const dril_env* e) {
    return e->ctx->nranks > 1 && e->d.normalize && e->d.training && (e->d.norm_obs || e->d.norm_reward);
}
static int dp_xr_count(const dril_env* e) { return 3 + 2 * (e->d.obs_dim + 1) + 2; }
static int32_t dp_rollout_begin(dril_env* e) {
    dril_ctx* c = e->ctx;
    e->d.roll_moments = nullptr;
    if (!dp_norm_active(e)) return DRIL_OK;
    e->d.roll_moments = e->roll_moments;
    norm_snapshot_kernel<<<1, 64, 0, c->stream>>>(e->d, e->norm_snap, e->norm_snap_cnt);
    DRIL_CUDA(cudaGetLastError());
    c->launches += 1;
    return DRIL_OK;
}
static int32_t dp_rollout_pack(dril_env* e) {
    dril_ctx* c = e->ctx;
    if (c->nranks == 1) return DRIL_OK;
    norm_monitor_pack_kernel<<<1, 64, 0, c->stream>>>(e->d, e->xr + 4, e->norm_snap, e->norm_snap_cnt, 2 * (e->d.obs_dim + 1) + 2);
    DRIL_CUDA(cudaGetLastError());
    c->launches += 1;
    return DRIL_OK;
}
static int32_t dp_rollout_merge(dril_env* e) {
    dril_ctx* c = e->ctx;
    if (c->nranks == 1) return DRIL_OK;
    norm_monitor_merge_kernel<<<1, 64, 0, c->stream>>>(e->d, e->xr + 4, e->norm_snap, e->norm_snap_cnt, dp_norm_active(e) ? 1 : 0);
    DRIL_CUDA(cudaGetLastError());
    c->launches += 1;
    return DRIL_OK;
}

static int32_t rollout_async(dril_env* e, dril_policy* p, dril_buffer* b, const void* forced_dev) {
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaMemsetAsync(b->d.done_count, 0, (size_t)b->d.T * 4, c->stream));
    DRIL_CUDA(cudaMemsetAsync(e->d.roll_sums, 0, 16, c->stream));
    DRIL_CUDA(cudaMemsetAsync(e->d.roll_eps, 0, 8, c->stream));
    DRIL_TRY(dp_rollout_begin(e));
    DRIL_TRY(launch_rollout(e, p, b, forced_dev, nullptr, (int)b->d.T, RO_INITIAL_OBSERVE | RO_FOLD_NEXT_OBSERVE));
    p->step_index += (uint32_t)b->d.T;
    return DRIL_OK;
}

extern "C" int32_t dril_rollout_collect(dril_env* e, dril_policy* p, dril_buffer* b, const void* forced_actions, float* fps_out) {
    DRIL_TRY(check_compat(e, p, b));
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    void* forced_dev = nullptr;
    if (forced_actions) {
        size_t cnt = (size_t)b->d.T * b->d.N;
        DRIL_TRY(ensure_scratch(p, cnt * b->act_elems * 4));
        DRIL_TRY(stage_actions(c, b->d.act_kind, b->d.act_dim, forced_actions, cnt, p->scratch));
        forced_dev = p->scratch;
    }
    DRIL_CUDA(cudaEventRecord(p->ev[0], c->stream));
    DRIL_TRY(rollout_async(e, p, b, forced_dev));
    DRIL_CUDA(cudaEventRecord(p->ev[1], c->stream));
    if (c->nranks > 1) {
        DRIL_TRY(dp_rollout_pack(e));
        DRIL_TRY(allreduce_small(c, nullptr, 0, e->xr + 4, dp_xr_count(e)));
        DRIL_TRY(dp_rollout_merge(e));
    }
    DRIL_TRY(launch_monitor_finalize(e, b));
    unsigned long long eps = 0;
    DRIL_CUDA(cudaMemcpyAsync(&eps, e->d.roll_eps, 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    e->total_episodes += (int64_t)eps;
    float ms = 0.f;
    DRIL_CUDA(cudaEventElapsedTime(&ms, p->ev[0], p->ev[1]));
    if (fps_out) *fps_out = (float)((double)b->d.T * b->d.N / (ms * 1e-3));
    return DRIL_OK;
}


// rows [t0, t0 + tc) of a buffer as a buffer of tc steps (pointers into the same slab; last_values shared)
static dril_buffer buffer_view(dril_buffer* b, long long t0, long long tc) {
    dril_buffer v = *b;
    const long long N = b->d.N;
    const size_t r0 = (size_t)t0 * N;
    v.d.T = tc;
    v.d.obs += r0 * b->d.obs_dim;
    v.d.actions = (char*)b->d.actions + r0 * b->act_elems * 4;
    v.d.rewards += r0; v.d.values += r0; v.d.logprobs += r0; v.d.advantages += r0; v.d.returns += r0; v.d.boot += r0;
    v.d.episode_r += r0; v.d.episode_l += r0; v.d.flags += r0; v.d.done_count += t0;
    v.is_view = true; v.tcs_slab = nullptr; v.dcs_slab = nullptr;
    return v;
}

/* Steps [t_begin, t_begin + t_count) of a rollout into rows [t_begin, ...) of the buffer: collect_trajectories
 * (buffers/trajectory.jl:22-78) run in chunks so that on_step callbacks (:34-39) see the advancing env and can stop the
 * collection mid-rollout.  start != 0 begins a rollout: per-rollout counters zeroed and the observe() before the loop (:32),
 * which precedes the first on_step hook, so it can be requested on its own with t_count = 0.  The bootstrap values of the
 * last chunk are the rollout's.  Follow with dril_gae once t_begin + t_count == n_steps. */
extern "C" int32_t dril_rollout_collect_steps(dril_env* e, dril_policy* p, dril_buffer* b, int64_t t_begin, int64_t t_count,
                                              int32_t start, const void* forced_actions) {
    DRIL_TRY(check_compat(e, p, b));
    DRIL_REQUIRE(t_begin >= 0 && t_count >= 0 && t_begin + t_count <= b->d.T, "steps [%lld, %lld) outside the buffer's %lld steps",
                 (long long)t_begin, (long long)(t_begin + t_count), b->d.T);
    DRIL_REQUIRE(t_count >= 1 || start, "nothing to do");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    dril_buffer v = buffer_view(b, t_begin, std::max<int64_t>(t_count, 1));
    void* forced_dev = nullptr;
    if (forced_actions && t_count > 0) {
        const size_t cnt = (size_t)t_count * b->d.N;
        DRIL_TRY(ensure_scratch(p, cnt * b->act_elems * 4));
        DRIL_TRY(stage_actions(c, b->d.act_kind, b->d.act_dim, forced_actions, cnt, p->scratch));
        forced_dev = p->scratch;
    }
    if (start) {
        DRIL_CUDA(cudaMemsetAsync(b->d.done_count, 0, (size_t)b->d.T * 4, c->stream));
        DRIL_CUDA(cudaMemsetAsync(e->d.roll_sums, 0, 16, c->stream));
        DRIL_CUDA(cudaMemsetAsync(e->d.roll_eps, 0, 8, c->stream));
    }
    const bool obs_stats = e->d.normalize && e->d.training && e->d.norm_obs;
    if (t_count > 0 || (start && obs_stats))
        DRIL_TRY(launch_rollout(e, t_count > 0 ? p : nullptr, &v, forced_dev, nullptr, (int)t_count, (start ? RO_INITIAL_OBSERVE : 0) | RO_FOLD_NEXT_OBSERVE));
    p->step_index += (uint32_t)t_count;
    if (t_count > 0 && t_begin + t_count == b->d.T) {
        DRIL_TRY(launch_monitor_finalize(e, b));
        unsigned long long eps = 0;
        DRIL_CUDA(cudaMemcpyAsync(&eps, e->d.roll_eps, 8, cudaMemcpyDeviceToHost, c->stream));
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
        e->total_episodes += (int64_t)eps;
    } else {
        DRIL_CUDA(cudaStreamSynchronize(c->stream));
    }
    return DRIL_OK;
}

/* evaluate_agent (src/evaluation.jl:54-143) with the episode loop on the device: reset!(env), then the policy (mode of the
 * distribution when deterministic) steps all envs in chunks of `chunk_steps` fused steps; after every chunk ONE device -> host
 * copy brings the chunk's done flags and episode records, and finished episodes are appended in the reference's order
 * (step by step, env index within a step) until n_eval_episodes are collected.  Episode returns / lengths are the
 * MonitorWrapperEnv records when the env is monitored (evaluation.jl:110-113), else the sums of the step rewards the
 * outermost wrapper returned (:114-117).  The env is left where the last chunk ended (up to chunk_steps - 1 steps past the
 * reference's stopping point). */
extern "C" int32_t dril_evaluate(dril_env* e, dril_policy* p, int64_t n_eval_episodes, int32_t deterministic, int32_t chunk_steps,
                                 float* episode_rewards, int64_t* episode_lengths, int64_t* n_collected, int64_t* env_steps) {
    DRIL_REQUIRE(e && p && episode_rewards && episode_lengths, "NULL argument");
    DRIL_REQUIRE(e->ctx == p->ctx, "env and policy must share a ctx");
    DRIL_REQUIRE(n_eval_episodes >= 1 && chunk_steps >= 1, "n_eval_episodes and chunk_steps must be positive");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const long long N = e->d.n_envs;
    const int K = chunk_steps;
    dril_buffer* b = nullptr;
    DRIL_TRY(dril_buffer_create(c, K, N, e->d.obs_dim, p->pd.act_kind, p->pd.act_kind == DRIL_ACT_DISCRETE ? 1 : p->pd.act_n, &b));
    int32_t st = check_compat(e, p, b);
    std::vector<unsigned char> flags((size_t)K * N);
    std::vector<float> er((size_t)K * N), rew((size_t)K * N);
    std::vector<int> el((size_t)K * N);
    std::vector<float> cur_r((size_t)N, 0.f);
    std::vector<long long> cur_l((size_t)N, 0);
    long long got = 0, steps = 0;
    const bool mon = e->d.monitor != 0;
    if (st == DRIL_OK) st = dril_env_reset(e);
    for (long long chunk = 0; st == DRIL_OK && got < n_eval_episodes; ++chunk) {
        if (chunk > 100000) { dril_set_error("dril_evaluate: no episode finished in %lld steps", steps); st = DRIL_ERR_INVALID; break; }
        cudaMemsetAsync(b->d.done_count, 0, (size_t)K * 4, c->stream);
        cudaMemsetAsync(e->d.roll_sums, 0, 16, c->stream);
        cudaMemsetAsync(e->d.roll_eps, 0, 8, c->stream);
        if ((st = launch_rollout(e, p, b, nullptr, nullptr, K, (chunk == 0 ? RO_INITIAL_OBSERVE : 0) | RO_FOLD_NEXT_OBSERVE |
                                 (deterministic ? RO_DETERMINISTIC : 0)))) break;
        p->step_index += (uint32_t)K;
        if ((st = launch_monitor_finalize(e, b))) break;
        unsigned long long eps = 0;
        cudaMemcpyAsync(flags.data(), b->d.flags, flags.size(), cudaMemcpyDeviceToHost, c->stream);
        if (mon) {
            cudaMemcpyAsync(er.data(), b->d.episode_r, er.size() * 4, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(el.data(), b->d.episode_l, el.size() * 4, cudaMemcpyDeviceToHost, c->stream);
        } else {
            cudaMemcpyAsync(rew.data(), b->d.rewards, rew.size() * 4, cudaMemcpyDeviceToHost, c->stream);
        }
        cudaMemcpyAsync(&eps, e->d.roll_eps, 8, cudaMemcpyDeviceToHost, c->stream);
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { dril_set_error("CUDA failure in dril_evaluate: %s", cudaGetErrorString(cudaGetLastError())); st = DRIL_ERR_CUDA; break; }
        e->total_episodes += (int64_t)eps;
        for (int t = 0; t < K && got < n_eval_episodes; ++t) {
            steps += 1;
            for (long long n = 0; n < N; ++n) {
                const size_t i = (size_t)t * N + n;
                if (!mon) { cur_r[n] += rew[i]; cur_l[n] += 1; }
                if ((flags[i] & 3) && got < n_eval_episodes) {
                    episode_rewards[got] = mon ? er[i] : cur_r[n];
                    episode_lengths[got] = mon ? (int64_t)el[i] : (int64_t)cur_l[n];
                    ++got;
                    cur_r[n] = 0.f; cur_l[n] = 0;
                }
            }
        }
    }
    dril_buffer_destroy(b);
    if (n_collected) *n_collected = got;
    if (env_steps) *env_steps = steps;
    return st;
}

/* sync_normalization_stats! zeroes the discounted-return accumulators of the receiving env (normalizeWrapperEnv.jl:306) */
extern "C" int32_t dril_env_zero_returns(dril_env* e) {
    DRIL_REQUIRE(e, "NULL argument");
    DRIL_CUDA(cudaSetDevice(e->ctx->device));
    if (e->d.ret) DRIL_CUDA(cudaMemsetAsync(e->d.ret, 0, (size_t)e->d.n_envs * 4, e->ctx->stream));
    DRIL_CUDA(cudaStreamSynchronize(e->ctx->stream));
    return DRIL_OK;
}

// ev_acc4 (optional, zeroed by the caller): the explained-variance moments are accumulated in the same pass
static int32_t gae_async(dril_ctx* c, const BufDev& d, float gamma, float lambda, double* ev_acc4 = nullptr) {
    Span sp(c, DRIL_K_GAE);
    gae_kernel<<<(unsigned)((d.N + 255) / 256), 256, 0, c->stream>>>(d.rewards, d.values, d.flags, d.boot, d.last_values,
                                                                    d.advantages, d.returns, d.T, d.N, gamma, lambda, ev_acc4);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}
extern "C" int32_t dril_gae(dril_buffer* b, float gamma, float lambda) {
    DRIL_REQUIRE(b, "NULL argument");
    DRIL_CUDA(cudaSetDevice(b->ctx->device));
    DRIL_TRY(gae_async(b->ctx, b->d, gamma, lambda));
    DRIL_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return DRIL_OK;
}
extern "C" int32_t dril_gae_raw(dril_ctx* c, const float* rewards, const float* values, const uint8_t* terminated,
                                const uint8_t* truncated, const float* boot, const float* last_values, int64_t T, int64_t N,
                                float gamma, float lambda, float* advantages, float* returns) {
    DRIL_REQUIRE(c && rewards && values && terminated && truncated && boot && last_values && advantages && returns, "NULL argument");
    DRIL_REQUIRE(T >= 1 && N >= 1, "empty buffer");
    dril_buffer* b = nullptr;
    DRIL_TRY(dril_buffer_create(c, T, N, 1, DRIL_ACT_DISCRETE, 1, &b));
    size_t tn = (size_t)T * N;
    std::vector<uint8_t> flags(tn);
    for (size_t i = 0; i < tn; ++i) flags[i] = (terminated[i] ? 1 : 0) | (truncated[i] ? 2 : 0);
    int32_t st = DRIL_OK;
    do {
        if ((st = dril_buffer_upload(b, DRIL_BUF_REWARDS, rewards, tn * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_VALUES, values, tn * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_FLAGS, flags.data(), tn))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_BOOT, boot, tn * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_LAST_VALUES, last_values, (size_t)N * 4))) break;
        if ((st = dril_gae(b, gamma, lambda))) break;
        if ((st = dril_buffer_download(b, DRIL_BUF_ADVANTAGES, advantages, tn * 4))) break;
        if ((st = dril_buffer_download(b, DRIL_BUF_RETURNS, returns, tn * 4))) break;
    } while (0);
    dril_buffer_destroy(b);
    return st;
}

// ---------------------------------------------------------------------------------------
// update
// ---------------------------------------------------------------------------------------
static UpdateHyper to_hyper(const dril_ppo_hyper* h) {
    UpdateHyper u;
    u.clip_range = h->clip_range; u.clip_range_vf = h->clip_range_vf; u.ent_coef = h->ent_coef; u.vf_coef = h->vf_coef;
    u.max_grad_norm = h->max_grad_norm; u.target_kl = h->target_kl; u.normalize_advantage = h->normalize_advantage;
    u.lr = h->learning_rate; u.beta1 = h->adam_beta1; u.beta2 = h->adam_beta2; u.adam_eps = h->adam_eps;
    return u;
}
static FeistelKey make_feistel(long long n_total, uint64_t epoch_counter, int rank, uint64_t seed) {
    FeistelKey fk;
    uint32_t k[4];
    philox4x32((uint32_t)epoch_counter, (uint32_t)rank, 0u, DRIL_TAG_SHUFFLE, seed, k);
    for (int i = 0; i < 4; ++i) fk.k[i] = k[i];
    int bits = 0;
    unsigned long long v = (unsigned long long)(n_total - 1);
    while (v) { ++bits; v >>= 1; }
    bits = std::max(bits, 2);
    fk.half_bits = (bits + 1) / 2;
    fk.half_mask = (1u << fk.half_bits) - 1u;
    return fk;
}

static int32_t plan_loss(dril_policy* p, LossLaunch* out) {
    const PolicyDesc& pd = p->pd;
    // widest tile (<= 128 samples, multiple of 16 so the 8x8 paths apply) that fits; weights in
    // shared memory when there is room for at least a 32-sample tile next to them
    int M4 = 128;
    bool ws = true, single = false;
    auto total = [&](int m4, bool w, bool sn = false, bool thin = false) { return loss_smem_layout(pd, m4, w, sn, thin).total; };
    while (M4 > 16 && total(M4, true) > DRIL_SMEM_MAX) M4 -= 16;
    if (total(M4, true) > DRIL_SMEM_MAX || M4 < 32) {
        ws = false; M4 = 128;
        while (M4 > 16 && total(M4, false) > DRIL_SMEM_MAX) M4 -= 16;
        // wide nets (weights streamed from L2): when both nets' activations do not fit a 128-sample tile, process the
        // nets in two passes with shared activation rows -> wider tile, weights read less often per sample, and
        // thread-tile counts that divide the block evenly
        if (M4 < 128 && (p->plan_single >= 0 ? p->plan_single : g_opt_single_net)) {
            int Ms = 128;
            while (Ms > 16 && total(Ms, false, true) > DRIL_SMEM_MAX) Ms -= 16;
            if (Ms > M4 && total(Ms, false, true) <= DRIL_SMEM_MAX) { single = true; M4 = Ms; }
        }
    }
    if (total(M4, ws, single) > DRIL_SMEM_MAX) { dril_set_error("network too wide for the loss kernel's shared memory"); return DRIL_ERR_UNSUPPORTED; }
    out->M4 = M4; out->ws = ws; out->single = single; out->smem = total(M4, ws, single);
    out->mma = (M4 % 16) == 0 && M4 >= 32 && (p->plan_mma >= 0 ? p->plan_mma : g_opt_mma) != 0;
    // MMA layers stream their weights from L2; the remaining (thin) layers' weights are staged in shared memory if they fit
    out->thin = out->mma && !ws && loss_thin_floats(pd) > 0 && loss_thin_floats(pd) < pd.pack_total / 2 &&
                total(M4, ws, single, true) <= DRIL_SMEM_MAX;
    if (out->thin) out->smem = total(M4, ws, single, true);
    int splits = 1;
    while (splits < DRIL_GPLANES && (M4 / (splits * 2)) % 4 == 0 && M4 / (splits * 2) >= 4) splits *= 2;
    out->splits = splits;
    int per_sm = 0;
    if (ws) DRIL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_loss_grad_kernel<true>, DRIL_THREADS, out->smem));
    else DRIL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_loss_grad_kernel<false>, DRIL_THREADS, out->smem));
    per_sm = std::max(1, std::min(per_sm, 2));
    out->grid_cap = std::min(per_sm * p->ctx->sm_count, p->gpart_ctas);
    return DRIL_OK;
}

// per-sample records of the whole buffer (update_ft.cuh): one streaming pass per update, read by every epoch's permute kernel
static int32_t ensure_ft_recs(dril_policy* p, const BufDev& bd, long long n_total) {
    dril_ctx* c = p->ctx;
    const int stride = ft_rec_stride(bd.obs_dim, bd.act_dim);
    const size_t need = (size_t)n_total * stride;
    if (p->ft_recs_floats < need) {
        if (p->ft_recs) { DRIL_CUDA(cudaStreamSynchronize(c->stream)); cudaFree(p->ft_recs); }
        p->ft_recs = nullptr; p->ft_recs_floats = 0;
        DRIL_CUDA(cudaMalloc((void**)&p->ft_recs, need * 4));
        p->ft_recs_floats = need;
    }
    p->ft_rec_stride = stride;
    return DRIL_OK;
}
static int32_t ensure_ft_tiles(dril_policy* p, size_t bytes) {
    dril_ctx* c = p->ctx;
    if (p->ft_tiles_bytes < bytes) {
        if (p->ft_tiles) { DRIL_CUDA(cudaStreamSynchronize(c->stream)); cudaFree(p->ft_tiles); }
        p->ft_tiles = nullptr; p->ft_tiles_bytes = 0;
        DRIL_CUDA(cudaMalloc((void**)&p->ft_tiles, bytes));
        p->ft_tiles_bytes = bytes;
    }
    return DRIL_OK;
}
static int32_t ft_pack_records(dril_policy* p, const BufDev& bd, long long n_total) {
    dril_ctx* c = p->ctx;
    DRIL_TRY(ensure_ft_recs(p, bd, n_total));
    const int stride = p->ft_rec_stride;
    const int grid = (int)std::max<long long>(1, std::min<long long>((n_total + 255) / 256, (long long)c->sm_count * 8));
    Span sp(c, DRIL_K_PERMUTE);
    ft_pack_records_kernel<<<grid, 256, 0, c->stream>>>(bd, n_total, stride, p->ft_recs);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}
// update_ft.cuh path: the samples of one epoch (all its minibatches) as shuffled, contiguous tile records
static bool ft_active(const dril_policy* p) { return g_opt_tc && g_opt_ft && tc_eligible(p->pd) && !(g_opt_ftg == 2 && ftg_eligible(p->pd)); }
// update_ftg.cuh path (general shapes); option "ftg" = 2 prefers it over update_ft.cuh where both apply
static bool ftg_active(const dril_policy* p) {
    if (!g_opt_ftg || !ftg_eligible(p->pd)) return false;
    if (g_opt_ftg == 2) return true;
    return !(g_opt_tc && tc_eligible(p->pd));
}
static const void* ftg_kernel(const PolicyDesc& pd) {
    const int L = pd.n_layers - 1, cont = pd.act_kind == DRIL_ACT_CONTINUOUS ? 1 : 0, n = pd.act_n;
    if (L == 2) {
        if (cont) return n == 1 ? (const void*)ppo_loss_grad_ftg_kernel<2, 1, 1> : (const void*)ppo_loss_grad_ftg_kernel<2, 1, 2>;
        if (n > 2) return n == 3 ? (const void*)ppo_loss_grad_ftg_kernel<2, 0, 3> : (const void*)ppo_loss_grad_ftg_kernel<2, 0, 4>;
        return n == 1 ? (const void*)ppo_loss_grad_ftg_kernel<2, 0, 1> : (const void*)ppo_loss_grad_ftg_kernel<2, 0, 2>;
    }
    if (cont) return n == 1 ? (const void*)ppo_loss_grad_ftg_kernel<3, 1, 1> : (const void*)ppo_loss_grad_ftg_kernel<3, 1, 2>;
    if (n > 2) return n == 3 ? (const void*)ppo_loss_grad_ftg_kernel<3, 0, 3> : (const void*)ppo_loss_grad_ftg_kernel<3, 0, 4>;
    return n == 1 ? (const void*)ppo_loss_grad_ftg_kernel<3, 0, 1> : (const void*)ppo_loss_grad_ftg_kernel<3, 0, 2>;
}
static int32_t ftg_stage_epoch(dril_policy* p, const BufDev& bd, const FeistelKey& fk, long long n_total, long long batch_size, int identity) {
    dril_ctx* c = p->ctx;
    const int n_mb = (int)((n_total + batch_size - 1) / batch_size);
    const int tpm = (int)((std::min<long long>(batch_size, n_total) + 63) / 64);
    const int cont = p->pd.act_kind == DRIL_ACT_CONTINUOUS ? 1 : 0;
    const int rf = ftg_rec_floats(p->pd.obs_dim, cont, p->pd.act_n);
    const size_t bytes = (size_t)n_mb * tpm * rf * 4;
    DRIL_TRY(ensure_ft_tiles(p, bytes));
    p->ft_tiles_per_mb = tpm; p->ft_batch = batch_size;
    const long long slots = (long long)n_mb * tpm * 64;
    const int grid = (int)std::max<long long>(1, std::min<long long>((slots + 255) / 256, (long long)c->sm_count * 8));
    Span sp(c, DRIL_K_PERMUTE);
    ftg_permute_kernel<<<grid, 256, 0, c->stream>>>(p->ft_recs, p->ft_rec_stride, bd.obs_dim, fk, n_total, batch_size, n_mb, tpm, identity,
                                                    p->pd.act_start, p->pd.act_n, cont, rf, reinterpret_cast<float*>(p->ft_tiles));
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}
static int32_t ft_stage_epoch(dril_policy* p, const BufDev& bd, const FeistelKey& fk, long long n_total, long long batch_size, int identity) {
    dril_ctx* c = p->ctx;
    const int n_mb = (int)((n_total + batch_size - 1) / batch_size);
    const int tpm = (int)((std::min<long long>(batch_size, n_total) + FT_TS - 1) / FT_TS);
    const size_t bytes = (size_t)n_mb * tpm * FT_TILE_BYTES;
    DRIL_TRY(ensure_ft_tiles(p, bytes));
    p->ft_tiles_per_mb = tpm; p->ft_batch = batch_size;
    const long long slots = (long long)n_mb * tpm * FT_TS;
    const int grid = (int)std::max<long long>(1, std::min<long long>((slots + 255) / 256, (long long)c->sm_count * 8));
    Span sp(c, DRIL_K_PERMUTE);
    ft_permute_kernel<<<grid, 256, 0, c->stream>>>(p->ft_recs, p->ft_rec_stride, fk, n_total, batch_size, n_mb, tpm, identity, p->pd.act_start,
                                                   p->pd.act_n, p->ft_tiles);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}

// ALL epochs of an update staged by one launch (both tcgen05 paths), which also leaves the per-minibatch advantage moments in
// p->adv_partial (layout of adv_stats_kernel with `bpm` blocks per minibatch).  *staged = false (nothing launched) when the tile
// records of all epochs would not fit the memory budget: the caller then stages epoch by epoch.
static int32_t ft_stage_epochs(dril_policy* p, const BufDev& bd, const FeistelKeys& fks, int ne, long long n_total, long long batch_size, int bpm,
                               bool* staged) {
    dril_ctx* c = p->ctx;
    *staged = false;
    const bool ftg = ftg_active(p);
    const int n_mb = (int)((n_total + batch_size - 1) / batch_size);
    const int tpm = (int)((std::min<long long>(batch_size, n_total) + 63) / 64);
    const int cont = p->pd.act_kind == DRIL_ACT_CONTINUOUS ? 1 : 0;
    const int rf = ftg_rec_floats(p->pd.obs_dim, cont, p->pd.act_n);
    const size_t tile_bytes = ftg ? (size_t)rf * 4 : (size_t)FT_TILE_BYTES;
    const long long epoch_tiles = (long long)n_mb * tpm;
    const size_t bytes = (size_t)ne * epoch_tiles * tile_bytes;
    static const size_t budget = (getenv("DRIL_STAGE_ALL_MB") ? (size_t)atoll(getenv("DRIL_STAGE_ALL_MB")) : 8192) << 20;
    if (bytes > budget) return DRIL_OK;
    DRIL_TRY(ensure_ft_tiles(p, bytes));
    p->ft_tiles_per_mb = tpm; p->ft_batch = batch_size;
    Span sp(c, DRIL_K_PERMUTE);
    const dim3 grid(bpm, n_mb, ne);
    if (ftg) ftg_permute_epochs_kernel<<<grid, 256, 0, c->stream>>>(p->ft_recs, p->ft_rec_stride, bd.obs_dim, fks, n_total, batch_size, tpm, p->pd.act_start,
                                                                   p->pd.act_n, cont, rf, reinterpret_cast<float*>(p->ft_tiles), epoch_tiles, p->adv_partial);
    else ft_permute_epochs_kernel<<<grid, 256, 0, c->stream>>>(p->ft_recs, p->ft_rec_stride, fks, n_total, batch_size, tpm, p->pd.act_start, p->pd.act_n,
                                                               p->ft_tiles, epoch_tiles, p->adv_partial);
    DRIL_CUDA(cudaGetLastError());
    *staged = true;
    return DRIL_OK;
}

// one minibatch: loss/grad kernel -> reduce -> (allreduce) -> clip + Adam
static int32_t minibatch_step(dril_policy* p, const BufDev& bd, const Minibatch& mb, const double* mbstats_dev,
                              const UpdateHyper& hp, const LossLaunch& ll, bool apply, int apply_stats) {
    dril_ctx* c = p->ctx;
    const PolicyDesc& pd = p->pd;
    LossArgs a;
    memset(&a, 0, sizeof(a));
    a.pd = pd; a.buf = bd; a.pack = p->pack; a.flat = p->flat; a.mbstats = mbstats_dev; a.gpart = p->gpart;
    a.stop_flag = p->stop_flag; a.mb = mb; a.hp = hp; a.M4 = ll.M4; a.weights_smem = ll.ws;
    a.half_stride = p->gpart_ctas; a.small_splits = ll.splits; a.single_net = ll.single ? 1 : 0;
    a.use_mma = ll.mma ? 1 : 0; a.stage_thin = ll.thin ? 1 : 0;
    const bool ftg = ftg_active(p);
    const bool tc = ftg || (g_opt_tc && tc_eligible(pd));
    const bool ft = !ftg && tc && g_opt_ft;
    const int tile_m = (ft || ftg) ? FT_TS : (tc ? TC_M : ll.M4);
    long long tiles = (mb.count + tile_m - 1) / tile_m;
    int grid = (int)std::max<long long>(1, std::min<long long>(tiles, tc ? std::min(c->sm_count, p->gpart_ctas) : ll.grid_cap));
    const unsigned char* planes_dev = tc ? p->f2planes_one : p->f2planes;
    AdamArgs aa;
    aa.g = p->g; aa.flat = p->flat; aa.m = p->m; aa.v = p->v; aa.pack = p->pack; aa.flat2pack = p->flat2pack;
    aa.flat2packT = p->flat2packT; aa.step = p->step; aa.iter_acc = p->iter_acc; aa.stop_flag = p->stop_flag;
    aa.global_count = mb.global_count; aa.hp = hp; aa.n_params = pd.n_params; aa.apply_stats = apply_stats;
    const int n = pd.n_params + 6;
    const int fgrid = (n + RA_PARAMS_PER_BLOCK - 1) / RA_PARAMS_PER_BLOCK;
    const bool fused = apply && c->nranks == 1;
    const bool p2p = apply && c->nranks > 1 && c->p2p_enabled && n <= c->p2p.n_slots;
    // tensor-core path: reduction (+ peer-memory exchange) + clip + Adam run as the tail of the loss/grad kernel
    const bool tail = tc && g_opt_tail && (fused || p2p) && grid <= c->sm_count && grid <= P2P_MAX_CTA;
    {
        Span sp(c, DRIL_K_LOSS_GRAD);
        if (tc) {
            TailArgs tl;
            memset(&tl, 0, sizeof(tl));
            tl.mode = tail ? (fused ? 1 : 2) : 0;
            tl.flat2g = p->flat2g; tl.f2planes = planes_dev; tl.stats_off = pd.pack_fwd + pd.act_n; tl.sq_part = p->sq_part;
            tl.adam = aa;
            if (p2p) tl.pp = c->p2p;
            if (ftg) {
                FtgArgs fa;
                fa.tiles = p->ft_tiles;
                fa.tile0 = p->ft_epoch_tile0 + (mb.start / std::max<long long>(1, p->ft_batch)) * p->ft_tiles_per_mb;
                fa.lay = ftg_layout(pd);
                const void* fn = ftg_kernel(pd);
                void* args[] = {(void*)&a, (void*)&tl, (void*)&fa};
                if (tail) DRIL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(FTG_THREADS), args, (size_t)fa.lay.total, c->stream));
                else DRIL_CUDA(cudaLaunchKernel(fn, dim3(grid), dim3(FTG_THREADS), args, (size_t)fa.lay.total, c->stream));
            } else if (ft) {
                // tile records of this minibatch: written by ft_stage_epoch before the epoch's first step
                FtArgs fa;
                memset(&fa, 0, sizeof(fa));
                fa.tiles = p->ft_tiles;
                fa.tile0 = p->ft_epoch_tile0 + (mb.start / std::max<long long>(1, p->ft_batch)) * p->ft_tiles_per_mb;
                const void* fn = pd.act_n == 1 ? (const void*)ppo_loss_grad_ft_kernel<1> : (const void*)ppo_loss_grad_ft_kernel<2>;
                void* args[] = {(void*)&a, (void*)&tl, (void*)&fa};
                if (tail) DRIL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(FT_THREADS), args, FT_SMEM_BYTES, c->stream));
                else DRIL_CUDA(cudaLaunchKernel(fn, dim3(grid), dim3(FT_THREADS), args, FT_SMEM_BYTES, c->stream));
            } else if (tail) {
                void* args[] = {(void*)&a, (void*)&tl};
                DRIL_CUDA(cudaLaunchCooperativeKernel((const void*)ppo_loss_grad_tc_kernel, dim3(grid), dim3(TC_THREADS), args,
                                                      TC_SMEM_BYTES, c->stream));
            } else {
                ppo_loss_grad_tc_kernel<<<grid, TC_THREADS, TC_SMEM_BYTES, c->stream>>>(a, tl);
            }
        }
        else if (ll.ws) ppo_loss_grad_kernel<true><<<grid, DRIL_THREADS, ll.smem, c->stream>>>(a);
        else ppo_loss_grad_kernel<false><<<grid, DRIL_THREADS, ll.smem, c->stream>>>(a);
        DRIL_CUDA(cudaGetLastError());
    }
    if (tail) return DRIL_OK;
    {
        // reduction over CTAs / planes (+ norm, clip, Adam in the same kernel on a single GPU; + publication
        // of this rank's gradient to its peers on the peer-memory path)
        Span sp(c, fused ? DRIL_K_ADAM : DRIL_K_GRAD_REDUCE);
        reduce_adam_kernel<<<fgrid, 1024, 0, c->stream>>>(p->gpart, grid, p->gpart_ctas, pd.gpack, p->flat2g, planes_dev,
                                                         pd.pack_fwd + pd.act_n, p->sq_part, p->ticket, aa,
                                                         fused ? 1 : (p2p ? 2 : 0), p2p ? c->p2p.local_gbuf : nullptr,
                                                         p2p ? c->p2p.n_slots : 0, p2p ? c->p2p.local_seq : nullptr,
                                                         p2p ? c->p2p.local_flag : nullptr);
        DRIL_CUDA(cudaGetLastError());
    }
    if (fused) return DRIL_OK;
    if (p2p) {
        // cross-rank sum over NVLink peer memory + norm, clip, Adam
        Span sp(c, DRIL_K_ALLREDUCE);
        p2p_sum_adam_kernel<<<(n + 1023) / 1024, 1024, 0, c->stream>>>(c->p2p, p->sq_part, p->ticket, aa);
        DRIL_CUDA(cudaGetLastError());
        return DRIL_OK;
    }
    DRIL_TRY(allreduce_sum(c, p->g, (size_t)pd.n_params + 6, false));
    if (apply) {
        Span sp(c, DRIL_K_ADAM);
        adam_finalize_kernel<<<1, 1024, 0, c->stream>>>(aa);
        DRIL_CUDA(cudaGetLastError());
    }
    return DRIL_OK;
}

// update_ft.cuh, persistent mode: the n_mb * ne minibatch steps of `ne` staged epochs in ONE cooperative launch (reduction, peer
// exchange, clip, KL stop and Adam in the kernel's tail; a grid barrier between steps).  *done = false when the conditions of the
// fused tail do not hold (the caller then steps minibatch by minibatch).
static int32_t ft_persistent_update(dril_policy* p, const BufDev& bd, const UpdateHyper& hp, const LossLaunch& ll, int n_mb, int ne, long long n_total,
                                    long long batch_size, bool* done) {
    dril_ctx* c = p->ctx;
    const PolicyDesc& pd = p->pd;
    *done = false;
    const int n = pd.n_params + 6;
    const bool fused = c->nranks == 1;
    const bool p2p = c->nranks > 1 && c->p2p_enabled && n <= c->p2p.n_slots;
    const long long tiles = (std::min<long long>(batch_size, n_total) + FT_TS - 1) / FT_TS;
    const int grid = (int)std::max<long long>(1, std::min<long long>(tiles, std::min(c->sm_count, p->gpart_ctas)));
    // single GPU only by default: with the peer exchange inside the step loop an 8-GPU run stopped making progress (2 and 4 GPUs
    // pass; not understood yet), so data-parallel updates keep one launch per minibatch step unless "persistent" is 2
    if (!g_opt_persistent || (c->nranks > 1 && g_opt_persistent < 2) || !g_opt_tail || !(fused || p2p) || grid > c->sm_count ||
        grid > P2P_MAX_CTA || n_mb * ne < 2) return DRIL_OK;
    LossArgs a;
    memset(&a, 0, sizeof(a));
    a.pd = pd; a.buf = bd; a.pack = p->pack; a.flat = p->flat; a.mbstats = p->mbstats; a.gpart = p->gpart;
    a.stop_flag = p->stop_flag; a.hp = hp; a.M4 = ll.M4; a.weights_smem = ll.ws;
    a.half_stride = p->gpart_ctas; a.small_splits = ll.splits; a.single_net = ll.single ? 1 : 0;
    a.use_mma = ll.mma ? 1 : 0; a.stage_thin = ll.thin ? 1 : 0;
    a.mb.n_total = n_total; a.mb.start = 0; a.mb.count = std::min<long long>(batch_size, n_total);
    a.mb.global_count = (double)a.mb.count * c->nranks; a.mb.identity = 0;
    AdamArgs aa;
    aa.g = p->g; aa.flat = p->flat; aa.m = p->m; aa.v = p->v; aa.pack = p->pack; aa.flat2pack = p->flat2pack;
    aa.flat2packT = p->flat2packT; aa.step = p->step; aa.iter_acc = p->iter_acc; aa.stop_flag = p->stop_flag;
    aa.global_count = a.mb.global_count; aa.hp = hp; aa.n_params = pd.n_params; aa.apply_stats = 1;
    TailArgs tl;
    memset(&tl, 0, sizeof(tl));
    tl.mode = fused ? 1 : 2;
    tl.flat2g = p->flat2g; tl.f2planes = p->f2planes_one; tl.stats_off = pd.pack_fwd + pd.act_n; tl.sq_part = p->sq_part;
    tl.adam = aa;
    if (p2p) tl.pp = c->p2p;
    FtArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.tiles = p->ft_tiles; fa.tile0 = 0;
    fa.n_steps = n_mb * ne; fa.n_mb = n_mb; fa.tpm = p->ft_tiles_per_mb; fa.nranks = c->nranks;
    fa.batch = batch_size; fa.n_total = n_total; fa.epoch_tiles = (long long)n_mb * p->ft_tiles_per_mb; fa.mbstats0 = p->mbstats;
    const void* fn = pd.act_n == 1 ? (const void*)ppo_loss_grad_ft_kernel<1> : (const void*)ppo_loss_grad_ft_kernel<2>;
    void* args[] = {(void*)&a, (void*)&tl, (void*)&fa};
    Span sp(c, DRIL_K_LOSS_GRAD);
    DRIL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(FT_THREADS), args, FT_SMEM_BYTES, c->stream));
    *done = true;
    return DRIL_OK;
}

static int32_t ensure_mbstats(dril_policy* p, int n_mb, int blocks_per_mb) {
    if (p->mbstats_cap >= n_mb) return DRIL_OK;
    if (p->mbstats) cudaFree(p->mbstats);
    if (p->adv_partial) cudaFree(p->adv_partial);
    p->mbstats = nullptr; p->adv_partial = nullptr; p->mbstats_cap = 0;
    DRIL_TRY(dmalloc(&p->mbstats, (size_t)n_mb * 2));
    DRIL_TRY(dmalloc(&p->adv_partial, (size_t)n_mb * 64 * 2));
    p->mbstats_cap = n_mb;
    return DRIL_OK;
}

// extra / n_extra: a second small fp64 array summed over ranks together with the first batch of advantage moments
static int32_t update_async(dril_policy* p, dril_buffer* b, const dril_ppo_hyper* h, int epochs, int64_t batch_size,
                            uint64_t shuffle_seed, uint64_t epoch_counter, double* extra = nullptr, int n_extra = 0) {
    dril_ctx* c = p->ctx;
    const long long n_total = b->d.T * b->d.N;
    DRIL_REQUIRE(batch_size >= 1, "batch_size must be positive");
    DRIL_REQUIRE(epochs >= 0, "epochs must be non-negative");
    const int n_mb = (int)((n_total + batch_size - 1) / batch_size);
    const UpdateHyper hp = to_hyper(h);
    p->beta1 = (double)h->adam_beta1; p->beta2 = (double)h->adam_beta2;
    LossLaunch ll;
    DRIL_TRY(plan_loss(p, &ll));
    const int bpm = (int)std::max<long long>(1, std::min<long long>(64, (std::min<long long>(batch_size, n_total) + 2047) / 2048));
    if (ftg_active(p) || ft_active(p)) DRIL_TRY(ft_pack_records(p, b->d, n_total));
    DRIL_CUDA(cudaMemsetAsync(p->iter_acc, 0, 12 * 8, c->stream));   // [12],[13] carry beta^t across iterations
    DRIL_CUDA(cudaMemsetAsync(p->stop_flag, 0, 4, c->stream));
    // minibatch advantage moments of up to DRIL_MAX_EPOCHS_BATCHED epochs per launch / allreduce
    for (int e0 = 0; e0 < epochs; e0 += DRIL_MAX_EPOCHS_BATCHED) {
        const int ne = std::min(DRIL_MAX_EPOCHS_BATCHED, epochs - e0);
        DRIL_TRY(ensure_mbstats(p, n_mb * ne, bpm));
        FeistelKeys fks;
        for (int e = 0; e < ne; ++e) fks.k[e] = make_feistel(n_total, epoch_counter + e0 + e, c->rank, shuffle_seed);
        for (int e = ne; e < DRIL_MAX_EPOCHS_BATCHED; ++e) fks.k[e] = fks.k[0];
        // tcgen05 paths: the tile records of all `ne` epochs and the advantage moments come from one launch
        bool staged_all = false;
        if (ftg_active(p) || ft_active(p)) DRIL_TRY(ft_stage_epochs(p, b->d, fks, ne, n_total, batch_size, bpm, &staged_all));
        if (hp.normalize_advantage) {
            if (!staged_all) {
                Span sp(c, DRIL_K_ADV_STATS);
                adv_stats_kernel<<<dim3(bpm, n_mb, ne), 256, 0, c->stream>>>(b->d.advantages, n_total, batch_size, fks, 0, p->adv_partial);
                DRIL_CUDA(cudaGetLastError());
            }
            {
                Span sp(c, DRIL_K_ADV_STATS);
                adv_stats_finalize_kernel<<<(n_mb * ne * 2 + 127) / 128, 128, 0, c->stream>>>(p->adv_partial, bpm, n_mb * ne, p->mbstats);
                DRIL_CUDA(cudaGetLastError());
            }
            DRIL_TRY(allreduce_small(c, p->mbstats, n_mb * ne * 2, extra, n_extra));
            n_extra = 0;
        }
        if (staged_all && ft_active(p)) {
            bool done = false;
            DRIL_TRY(ft_persistent_update(p, b->d, hp, ll, n_mb, ne, n_total, batch_size, &done));
            if (done) continue;
        }
        for (int e = 0; e < ne; ++e) {
            if (staged_all) p->ft_epoch_tile0 = (long long)e * n_mb * p->ft_tiles_per_mb;
            else {
                p->ft_epoch_tile0 = 0;
                if (ftg_active(p)) DRIL_TRY(ftg_stage_epoch(p, b->d, fks.k[e], n_total, batch_size, 0));
                else if (ft_active(p)) DRIL_TRY(ft_stage_epoch(p, b->d, fks.k[e], n_total, batch_size, 0));
            }
            for (int i = 0; i < n_mb; ++i) {
                Minibatch mb;
                mb.n_total = n_total; mb.start = (long long)i * batch_size;
                mb.count = std::min<long long>(batch_size, n_total - mb.start);
                mb.global_count = (double)mb.count * c->nranks;
                mb.fk = fks.k[e]; mb.identity = 0;
                DRIL_TRY(minibatch_step(p, b->d, mb, p->mbstats + 2 * ((size_t)e * n_mb + i), hp, ll, true, 1));
            }
        }
    }
    p->ft_epoch_tile0 = 0;
    if (n_extra) DRIL_TRY(allreduce_small(c, nullptr, 0, extra, n_extra));   // no advantage moments were exchanged
    return DRIL_OK;
}

static int32_t ev_async(dril_policy* p, dril_buffer* b) {
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaMemsetAsync(p->ev_acc, 0, 32, c->stream));
    Span sp(c, DRIL_K_EXPLAINED_VAR);
    long long n = b->d.T * b->d.N;
    int grid = (int)std::min<long long>((n + 255) / 256, (long long)c->sm_count * 8);
    explained_variance_kernel<<<grid, 256, 0, c->stream>>>(b->d.values, b->d.returns, n, p->ev_acc);
    DRIL_CUDA(cudaGetLastError());
    return DRIL_OK;
}
static int32_t ev_finish(dril_policy* p, long long n_local, float* out) {
    dril_ctx* c = p->ctx;
    DRIL_TRY(allreduce_sum(c, p->ev_acc, 4, true));
    double acc[4];
    DRIL_CUDA(cudaMemcpyAsync(acc, p->ev_acc, 32, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    double n = (double)n_local * c->nranks;
    double var_d = (acc[1] - acc[0] * acc[0] / n) / (n - 1.0);
    double var_r = (acc[3] - acc[2] * acc[2] / n) / (n - 1.0);
    *out = (float)(1.0 - var_d / var_r);
    return DRIL_OK;
}
extern "C" int32_t dril_explained_variance(dril_buffer* b, float* out) {
    DRIL_REQUIRE(b && out, "NULL argument");
    dril_ctx* c = b->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    double* acc = nullptr;
    DRIL_TRY(dmalloc(&acc, 4));
    DRIL_CUDA(cudaMemsetAsync(acc, 0, 32, c->stream));
    long long n = b->d.T * b->d.N;
    {
        Span sp(c, DRIL_K_EXPLAINED_VAR);
        int grid = (int)std::min<long long>((n + 255) / 256, (long long)c->sm_count * 8);
        explained_variance_kernel<<<grid, 256, 0, c->stream>>>(b->d.values, b->d.returns, n, acc);
    }
    double h[4];
    DRIL_CUDA(cudaMemcpyAsync(h, acc, 32, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(acc);
    double dn = (double)n;
    *out = (float)(1.0 - ((h[1] - h[0] * h[0] / dn) / (dn - 1.0)) / ((h[3] - h[2] * h[2] / dn) / (dn - 1.0)));
    return DRIL_OK;
}

static int32_t collect_iter_stats(dril_policy* p, dril_iter_stats* s, bool with_rollout) {
    dril_ctx* c = p->ctx;
    double acc[ITER_ACC_N];
    int stop = 0;
    DRIL_CUDA(cudaMemcpyAsync(acc, p->iter_acc, ITER_ACC_N * 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaMemcpyAsync(&stop, p->stop_flag, 4, cudaMemcpyDeviceToHost, c->stream));
    double rs[2] = {0, 0};
    unsigned long long eps = 0;
    if (with_rollout && p->last_env) {
        DRIL_CUDA(cudaMemcpyAsync(rs, p->last_env->d.roll_sums, 16, cudaMemcpyDeviceToHost, c->stream));
        DRIL_CUDA(cudaMemcpyAsync(&eps, p->last_env->d.roll_eps, 8, cudaMemcpyDeviceToHost, c->stream));
    }
    int p2p_err = 0;
    if (c->p2p_enabled) DRIL_CUDA(cudaMemcpyAsync(&p2p_err, c->p2p.err, 4, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    if (p2p_err) { dril_set_error("peer-memory allreduce timed out waiting for a peer rank"); return DRIL_ERR_NCCL; }
    memset(s, 0, sizeof(*s));
    double n = acc[9];
    // means over the iteration's applied minibatches; empty -> NaN like mean(Float32[]) (ppo.jl:257-263)
    s->policy_loss = (float)(acc[0] / n); s->value_loss = (float)(acc[1] / n); s->entropy_loss = (float)(acc[2] / n);
    s->clip_fraction = (float)(acc[3] / n); s->approx_kl_div = (float)(acc[4] / n); s->entropy = (float)(acc[5] / n);
    s->ratio = (float)(acc[6] / n); s->loss = (float)(acc[7] / n);
    s->grad_norm = (float)(acc[8] / acc[10]);
    s->n_minibatch_steps = (int32_t)n;
    s->kl_stopped = stop;
    s->learning_rate = p->last_lr;
    s->episodes = (int64_t)eps; s->episode_return_sum = rs[0]; s->episode_length_sum = rs[1];
    s->ep_rew_mean = NAN; s->ep_len_mean = NAN;      // the monitor window is reported by dril_iteration_result only
    return DRIL_OK;
}

extern "C" int32_t dril_ppo_update(dril_policy* p, dril_buffer* b, const dril_ppo_hyper* h, int32_t epochs,
                                   int64_t batch_size, uint64_t shuffle_seed, uint64_t epoch_counter, dril_iter_stats* stats_out) {
    DRIL_REQUIRE(p && b && h, "NULL argument");
    DRIL_REQUIRE(p->ctx == b->ctx, "policy and buffer must share a ctx");
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    p->last_lr = h->learning_rate;
    DRIL_CUDA(cudaEventRecord(p->ev[1], c->stream));
    DRIL_TRY(update_async(p, b, h, epochs, batch_size, shuffle_seed, epoch_counter));
    DRIL_CUDA(cudaEventRecord(p->ev[2], c->stream));
    DRIL_TRY(ev_async(p, b));
    dril_iter_stats s;
    dril_env* keep = p->last_env;
    p->last_env = nullptr;
    DRIL_TRY(collect_iter_stats(p, &s, false));
    p->last_env = keep;
    DRIL_TRY(ev_finish(p, b->d.T * b->d.N, &s.explained_variance));
    float ms = 0.f;
    DRIL_CUDA(cudaEventElapsedTime(&ms, p->ev[1], p->ev[2]));
    s.update_ms = ms;
    if (stats_out) *stats_out = s;
    return DRIL_OK;
}

// Every allocation the first iterations would otherwise make lazily (result slots, pinned records, sample / tile records,
// advantage-moment buffers, deferred-critic scratch).  Data-parallel hosts call it on every rank and then synchronise the ranks
// BEFORE the first iteration: a rank that is still inside cudaMalloc / cudaMallocHost while a peer's GPU already spins in a
// peer-memory exchange waiting for it can stall for a long time (driver calls may need every peer-mapped device).
extern "C" int32_t dril_iteration_prepare(dril_env* e, dril_policy* p, dril_buffer* b, int32_t epochs, int64_t batch_size) {
    DRIL_TRY(check_compat(e, p, b));
    DRIL_REQUIRE(batch_size >= 1 && epochs >= 0, "bad prepare arguments");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    for (int si = 0; si < DRIL_RESULT_SLOTS; ++si) {
        dril_policy::Slot& sl = p->slots[si];
        if (!sl.host) {
            DRIL_CUDA(cudaMallocHost(&sl.host, sizeof(IterRecord)));
            for (int i = 0; i < 4; ++i) DRIL_CUDA(cudaEventCreate(&sl.ev[i]));
        }
    }
    if (!p->rec_dev) DRIL_CUDA(cudaMalloc(&p->rec_dev, sizeof(IterRecord) * DRIL_RESULT_SLOTS));
    const long long n_total = b->d.T * b->d.N;
    const int n_mb = (int)((n_total + batch_size - 1) / batch_size);
    const int ne = std::max(1, std::min<int>(DRIL_MAX_EPOCHS_BATCHED, epochs));
    const int bpm = (int)std::max<long long>(1, std::min<long long>(64, (std::min<long long>(batch_size, n_total) + 2047) / 2048));
    DRIL_TRY(ensure_mbstats(p, n_mb * ne, bpm));
    if (ftg_active(p) || ft_active(p)) {
        DRIL_TRY(ensure_ft_recs(p, b->d, n_total));
        const int tpm = (int)((std::min<long long>(batch_size, n_total) + 63) / 64);
        const int cont = p->pd.act_kind == DRIL_ACT_CONTINUOUS ? 1 : 0;
        const size_t tile_bytes = ftg_active(p) ? (size_t)ftg_rec_floats(p->pd.obs_dim, cont, p->pd.act_n) * 4 : (size_t)FT_TILE_BYTES;
        const size_t budget = (getenv("DRIL_STAGE_ALL_MB") ? (size_t)atoll(getenv("DRIL_STAGE_ALL_MB")) : 8192) << 20;
        const size_t all = (size_t)ne * n_mb * tpm * tile_bytes;
        DRIL_TRY(ensure_ft_tiles(p, all <= budget ? all : (size_t)n_mb * tpm * tile_bytes));
    }
    if (!e->d.normalize && e->d.kind == DRIL_ENV_CARTPOLE && tc_eligible(p->pd)) DRIL_TRY(ensure_tcs(b));
    if (ftg_eligible(p->pd)) DRIL_TRY(ensure_dcs(b));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    return DRIL_OK;
}

extern "C" int32_t dril_ppo_iteration_async(dril_env* e, dril_policy* p, dril_buffer* b, const dril_ppo_hyper* h,
                                            int32_t epochs, int64_t batch_size, uint64_t shuffle_seed, uint64_t epoch_counter) {
    DRIL_TRY(check_compat(e, p, b));
    DRIL_REQUIRE(h, "hyper is NULL");
    dril_ctx* c = e->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const int si = (int)(p->slot_tail % DRIL_RESULT_SLOTS);
    dril_policy::Slot& sl = p->slots[si];
    if (p->slot_tail - p->slot_head >= DRIL_RESULT_SLOTS) {
        // results are optional: the oldest unread one is dropped (its record must have landed before the slot is reused)
        DRIL_CUDA(cudaEventSynchronize(sl.ev[3]));
        if (sl.env) sl.env->total_episodes += (int64_t)sl.host->roll_eps;
        p->slot_head += 1;
    }
    if (!sl.host) {
        DRIL_CUDA(cudaMallocHost(&sl.host, sizeof(IterRecord)));
        for (int i = 0; i < 4; ++i) DRIL_CUDA(cudaEventCreate(&sl.ev[i]));
    }
    if (!p->rec_dev) DRIL_CUDA(cudaMalloc(&p->rec_dev, sizeof(IterRecord) * DRIL_RESULT_SLOTS));
    sl.env = e; sl.n_local = b->d.T * b->d.N; sl.lr = h->learning_rate;
    p->last_env = e; p->last_buf = b; p->last_lr = h->learning_rate;
    DRIL_CUDA(cudaEventRecord(sl.ev[0], c->stream));
    DRIL_TRY(rollout_async(e, p, b, nullptr));
    // data-parallel: explained-variance moments, Monitor sums and the rollout's normaliser moments travel in ONE small fp64
    // exchange together with the first batch of minibatch advantage moments
    const bool dp = c->nranks > 1;
    double* ev = dp ? e->xr : p->ev_acc;
    DRIL_CUDA(cudaMemsetAsync(ev, 0, 32, c->stream));
    DRIL_TRY(gae_async(c, b->d, h->gamma, h->gae_lambda, ev));   // + explained-variance moments (ppo.jl:256)
    DRIL_TRY(launch_monitor_finalize(e, b));
    if (dp) DRIL_TRY(dp_rollout_pack(e));
    DRIL_CUDA(cudaEventRecord(sl.ev[1], c->stream));
    DRIL_TRY(update_async(p, b, h, epochs, batch_size, shuffle_seed, epoch_counter, ev, dp ? 4 + dp_xr_count(e) : 4));
    if (dp) DRIL_TRY(dp_rollout_merge(e));
    DRIL_CUDA(cudaEventRecord(sl.ev[2], c->stream));
    {
        IterRecordSrc src;
        src.acc = p->iter_acc; src.ev = ev; src.roll_sums = e->d.roll_sums; src.roll_eps = e->d.roll_eps;
        src.stop = p->stop_flag; src.p2p_err = c->p2p_enabled ? c->p2p.err : nullptr; src.ring = e->ring;
        src.has_ring = e->d.monitor ? 1 : 0;
        Span sp(c, DRIL_K_MONITOR);
        iter_record_kernel<<<1, 32, 0, c->stream>>>(src, p->rec_dev + si);
        DRIL_CUDA(cudaGetLastError());
    }
    DRIL_CUDA(cudaMemcpyAsync(sl.host, p->rec_dev + si, sizeof(IterRecord), cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaEventRecord(sl.ev[3], c->stream));
    p->slot_tail += 1;
    return DRIL_OK;
}
extern "C" int32_t dril_iteration_result(dril_policy* p, dril_iter_stats* stats_out) {
    DRIL_REQUIRE(p && stats_out, "NULL argument");
    DRIL_REQUIRE(p->slot_head < p->slot_tail, "no iteration in flight");
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    dril_policy::Slot& sl = p->slots[p->slot_head % DRIL_RESULT_SLOTS];
    p->slot_head += 1;
    DRIL_CUDA(cudaEventSynchronize(sl.ev[3]));
    const IterRecord& r = *sl.host;
    if (r.p2p_err) { dril_set_error("peer-memory allreduce timed out waiting for a peer rank"); return DRIL_ERR_NCCL; }
    dril_iter_stats s;
    memset(&s, 0, sizeof(s));
    const double n = r.acc[9];
    // means over the iteration's applied minibatches; empty -> NaN like mean(Float32[]) (ppo.jl:257-263)
    s.policy_loss = (float)(r.acc[0] / n); s.value_loss = (float)(r.acc[1] / n); s.entropy_loss = (float)(r.acc[2] / n);
    s.clip_fraction = (float)(r.acc[3] / n); s.approx_kl_div = (float)(r.acc[4] / n); s.entropy = (float)(r.acc[5] / n);
    s.ratio = (float)(r.acc[6] / n); s.loss = (float)(r.acc[7] / n);
    s.grad_norm = (float)(r.acc[8] / r.acc[10]);
    s.n_minibatch_steps = (int32_t)n;
    s.kl_stopped = r.stop;
    s.learning_rate = sl.lr;
    s.episodes = (int64_t)r.roll_eps; s.episode_return_sum = r.roll_sums[0]; s.episode_length_sum = r.roll_sums[1];
    {
        const double nn = (double)sl.n_local * c->nranks;
        const double var_d = (r.ev[1] - r.ev[0] * r.ev[0] / nn) / (nn - 1.0);
        const double var_r = (r.ev[3] - r.ev[2] * r.ev[2] / nn) / (nn - 1.0);
        s.explained_variance = (float)(1.0 - var_d / var_r);
    }
    s.ep_rew_mean = r.ring_rew_mean; s.ep_len_mean = r.ring_len_mean; s.episodes_in_window = r.ring_count;
    float ms = 0.f;
    DRIL_CUDA(cudaEventElapsedTime(&ms, sl.ev[0], sl.ev[1])); s.rollout_ms = ms;
    DRIL_CUDA(cudaEventElapsedTime(&ms, sl.ev[1], sl.ev[2])); s.update_ms = ms;
    if (sl.env) sl.env->total_episodes += s.episodes;
    *stats_out = s;
    return DRIL_OK;
}

// ---------------------------------------------------------------------------------------
// parity entries on host minibatches
// ---------------------------------------------------------------------------------------
extern "C" int32_t dril_ppo_loss_grad(dril_policy* p, const float* obs, const void* actions, const float* advantages,
                                      const float* returns, const float* old_logprobs, const float* old_values, int64_t B,
                                      const dril_ppo_hyper* h, float* loss, float* stats7, float* grads) {
    DRIL_REQUIRE(p && obs && actions && advantages && returns && old_logprobs && old_values && h, "NULL argument");
    DRIL_REQUIRE(B >= 1, "empty minibatch");
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    const PolicyDesc& pd = p->pd;
    dril_buffer* b = nullptr;
    DRIL_TRY(dril_buffer_create(c, 1, B, pd.obs_dim, pd.act_kind, pd.act_kind == DRIL_ACT_DISCRETE ? 1 : pd.act_n, &b));
    int32_t st = DRIL_OK;
    do {
        if ((st = dril_buffer_upload(b, DRIL_BUF_OBS, obs, (size_t)B * pd.obs_dim * 4))) break;
        if ((st = stage_actions(c, pd.act_kind, pd.act_n, actions, B, b->d.actions))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_ADVANTAGES, advantages, B * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_RETURNS, returns, B * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_LOGPROBS, old_logprobs, B * 4))) break;
        if ((st = dril_buffer_upload(b, DRIL_BUF_VALUES, old_values, B * 4))) break;
        const UpdateHyper hp = to_hyper(h);
        LossLaunch ll;
        if ((st = plan_loss(p, &ll))) break;
        if ((st = ensure_mbstats(p, 1, 64))) break;
        cudaMemsetAsync(p->stop_flag, 0, 4, c->stream);
        FeistelKey fk = make_feistel(B, 0, 0, 0);
        int bpm = (int)std::max<int64_t>(1, std::min<int64_t>(64, (B + 2047) / 2048));
        FeistelKeys fks;
        for (int e = 0; e < DRIL_MAX_EPOCHS_BATCHED; ++e) fks.k[e] = fk;
        adv_stats_kernel<<<dim3(bpm, 1, 1), 256, 0, c->stream>>>(b->d.advantages, B, B, fks, 1, p->adv_partial);
        adv_stats_finalize_kernel<<<1, 128, 0, c->stream>>>(p->adv_partial, bpm, 1, p->mbstats);
        c->launches += 2;
        Minibatch mb;
        mb.n_total = B; mb.start = 0; mb.count = B; mb.global_count = (double)B; mb.fk = fk; mb.identity = 1;
        if ((ftg_active(p) || ft_active(p)) && (st = ft_pack_records(p, b->d, B))) break;
        if (ftg_active(p)) { if ((st = ftg_stage_epoch(p, b->d, fk, B, B, 1))) break; }
        else if (ft_active(p) && (st = ft_stage_epoch(p, b->d, fk, B, B, 1))) break;
        if ((st = minibatch_step(p, b->d, mb, p->mbstats, hp, ll, false, 0))) break;
        std::vector<float> g((size_t)pd.n_params + 6);
        cudaMemcpyAsync(g.data(), p->g, g.size() * 4, cudaMemcpyDeviceToHost, c->stream);
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { dril_set_error("CUDA failure in dril_ppo_loss_grad: %s", cudaGetErrorString(cudaGetLastError())); st = DRIL_ERR_CUDA; break; }
        const float* s6 = g.data() + pd.n_params;
        float invB = (float)(1.0 / (double)B);
        float p_loss = s6[0] * invB, v_loss = s6[1] * invB, ent = s6[2] * invB;
        if (stats7) {
            stats7[0] = p_loss; stats7[1] = v_loss; stats7[2] = -ent; stats7[3] = s6[3] * invB; stats7[4] = s6[4] * invB;
            stats7[5] = ent; stats7[6] = s6[5] * invB;
        }
        if (loss) *loss = p_loss + h->ent_coef * (-ent) + h->vf_coef * v_loss;
        if (grads) memcpy(grads, g.data(), (size_t)pd.n_params * 4);
    } while (0);
    dril_buffer_destroy(b);
    return st;
}

extern "C" int32_t dril_optimizer_step(dril_policy* p, const float* grads, int64_t n, const dril_ppo_hyper* h, float* grad_norm) {
    DRIL_REQUIRE(p && grads && h, "NULL argument");
    DRIL_REQUIRE(n == p->pd.n_params, "expected %d gradients, got %lld", p->pd.n_params, (long long)n);
    dril_ctx* c = p->ctx;
    DRIL_CUDA(cudaSetDevice(c->device));
    DRIL_CUDA(cudaMemcpyAsync(p->g, grads, n * 4, cudaMemcpyHostToDevice, c->stream));
    DRIL_CUDA(cudaMemsetAsync(p->stop_flag, 0, 4, c->stream));
    AdamArgs aa;
    aa.g = p->g; aa.flat = p->flat; aa.m = p->m; aa.v = p->v; aa.pack = p->pack; aa.flat2pack = p->flat2pack;
    aa.flat2packT = p->flat2packT; aa.step = p->step; aa.iter_acc = p->iter_acc; aa.stop_flag = p->stop_flag;
    aa.global_count = 1.0; aa.hp = to_hyper(h); aa.n_params = p->pd.n_params; aa.apply_stats = 0;
    {
        Span sp(c, DRIL_K_ADAM);
        adam_finalize_kernel<<<1, 1024, 0, c->stream>>>(aa);
        DRIL_CUDA(cudaGetLastError());
    }
    double acc8 = 0;
    DRIL_CUDA(cudaMemcpyAsync(&acc8, p->iter_acc + 8, 8, cudaMemcpyDeviceToHost, c->stream));
    DRIL_CUDA(cudaStreamSynchronize(c->stream));
    if (grad_norm) *grad_norm = (float)acc8;
    return DRIL_OK;
}

#ifdef TC_TRACE
extern "C" int32_t dril_debug_rt_trace(long long* out) {
    DRIL_CUDA(cudaDeviceSynchronize());
    DRIL_CUDA(cudaMemcpyFromSymbol(out, g_rt_trace, sizeof(long long) * 4 * 8 * 8));
    return DRIL_OK;
}
extern "C" int32_t dril_debug_tc_trace(long long* out) {
    DRIL_CUDA(cudaDeviceSynchronize());
    DRIL_CUDA(cudaMemcpyFromSymbol(out, g_tc_trace, sizeof(long long) * 2 * 32 * 16));
    return DRIL_OK;
}
#endif
