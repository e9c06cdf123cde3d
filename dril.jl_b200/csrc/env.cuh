// Batched classic-control dynamics (device functions).
//
// The reference takes CartPole / Pendulum from the un-vendored ClassicControlEnvironments.jl
// (call sites README.md:50,76; benchmark/bench_utils.jl:14,20); these follow the Gymnasium
// CartPole-v1 / Pendulum-v1 / MountainCar-v0 / MountainCarContinuous-v0 / Acrobot-v1 equations
// exactly as restated in oracle/envs.py and oracle/classic_envs.py.  Every fp32 operation uses a round-to-nearest intrinsic
// (never contracted into FMA) and sin/cos are the correctly rounded fp32 values (fp64 evaluation,
// one rounding), so replayed action sequences reproduce the oracle bit for bit.
//
// This file is the only place that branches on the env kind.  The kernels take the set of kinds
// they are built for as a template argument (ENV_KS_*): the instantiations for CartPole, Pendulum
// and the synthetic env contain exactly the code they had before MountainCar and Acrobot existed
// (Acrobot's RK4 step and 6-wide observation do not enter their register budget).
#pragma once
#include "common.cuh"

#define ENV_MAX_STATE 4
#define ENV_KS_CLASSIC ((1u << DRIL_ENV_CARTPOLE) | (1u << DRIL_ENV_PENDULUM) | (1u << DRIL_ENV_SYNTHETIC))
#define ENV_KS_ALL (ENV_KS_CLASSIC | (1u << DRIL_ENV_MOUNTAINCAR) | (1u << DRIL_ENV_MOUNTAINCAR_CONTINUOUS) | (1u << DRIL_ENV_ACROBOT))

// kind-set bits beyond the kinds: ENV_KS_PARAMS = per-env physical parameters (below); ENV_KS_OBS_PARAMS (only together with
// ENV_KS_PARAMS) = observations [base observation | the running episode's parameter values in table order]; ENV_KS_HISTORY
// (only together with ENV_KS_PARAMS) = observations [f_{t-k+1} | ... | f_t], the last k frames (env_frame), k = hist_len;
// ENV_KS_PERTURB (only together with ENV_KS_PARAMS, not with ENV_KS_OBS_PARAMS) = observation noise and action delay (below)
#define ENV_KS_PARAMS (1u << 16)
#define ENV_KS_OBS_PARAMS (1u << 17)
#define ENV_KS_HISTORY (1u << 18)
#define ENV_KS_PERTURB (1u << 19)

__host__ __device__ constexpr bool env_in(unsigned ks, int kind) { return (ks >> kind) & 1u; }
__host__ __device__ constexpr bool env_obs_params(unsigned ks) { return (ks & ENV_KS_OBS_PARAMS) != 0; }
__host__ __device__ constexpr bool env_history(unsigned ks) { return (ks & ENV_KS_HISTORY) != 0; }
__host__ __device__ constexpr bool env_perturb(unsigned ks) { return (ks & ENV_KS_PERTURB) != 0; }
__host__ __device__ constexpr int env_n_params(int kind) {
    return kind == DRIL_ENV_CARTPOLE || kind == DRIL_ENV_ACROBOT ? 6
         : kind == DRIL_ENV_PENDULUM ? 4
         : kind == DRIL_ENV_MOUNTAINCAR || kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS ? 2 : 0;
}
// observation components of a state-based kind without its parameters
__host__ __device__ constexpr int env_base_obs_dim(int kind) {
    return kind == DRIL_ENV_CARTPOLE ? 4 : kind == DRIL_ENV_PENDULUM ? 3 : kind == DRIL_ENV_ACROBOT ? 6 : 2;
}
// blocks of four observation components a kernel built for the kinds `ks` handles (Acrobot: 6 components; with
// ENV_KS_OBS_PARAMS both parametrised kind sets hold a kind of base + parameter width > 8: CartPole 10, Acrobot 12; with
// ENV_KS_HISTORY the blocks of one frame, at most 6 components, which the kernels assemble into the k-frame stack)
__host__ __device__ constexpr int env_obs_blocks(unsigned ks) {
    return env_obs_params(ks) ? 3 : (env_in(ks, DRIL_ENV_ACROBOT) || env_history(ks) ? 2 : 1);
}
// components of one frame of an env with an observation history: the base observation, or with mask_velocities its
// non-velocity components (CartPole (x, theta), Pendulum (cos, sin), MountainCar(Continuous) (position), Acrobot
// (cos th1, sin th1, cos th2, sin th2))
__host__ __device__ constexpr int env_frame_dim(int kind, bool mask_velocities) {
    return !mask_velocities ? env_base_obs_dim(kind)
         : kind == DRIL_ENV_ACROBOT ? 4 : kind == DRIL_ENV_CARTPOLE || kind == DRIL_ENV_PENDULUM ? 2 : 1;
}
// the kind set whose instantiation serves env kind `kind`
__host__ __device__ constexpr unsigned env_kind_set(int kind) { return env_in(ENV_KS_CLASSIC, kind) ? ENV_KS_CLASSIC : ENV_KS_ALL; }

__device__ __forceinline__ void sincos_rn(float th, float* s, float* c) {
    double sd, cd;
    sincos((double)th, &sd, &cd);
    *s = (float)sd;
    *c = (float)cd;
}

// observation components 4b .. 4b+3 of a state-based env (zero beyond obs_dim)
template <unsigned KS>
__device__ __forceinline__ void env_raw_obs_block(int kind, const float* st, int b, float* o) {
    if (env_in(KS, DRIL_ENV_ACROBOT) && kind == DRIL_ENV_ACROBOT) {   // (cos th1, sin th1, cos th2, sin th2 | w1, w2)
        if (b == 0) {
            sincos_rn(st[0], &o[1], &o[0]);
            sincos_rn(st[1], &o[3], &o[2]);
        } else {
            o[0] = st[2]; o[1] = st[3]; o[2] = 0.f; o[3] = 0.f;
        }
    } else if ((env_in(KS, DRIL_ENV_MOUNTAINCAR) && kind == DRIL_ENV_MOUNTAINCAR) ||
               (env_in(KS, DRIL_ENV_MOUNTAINCAR_CONTINUOUS) && kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS)) {   // (position, velocity)
        o[0] = st[0]; o[1] = st[1]; o[2] = 0.f; o[3] = 0.f;
    } else if (kind == DRIL_ENV_CARTPOLE) {
        o[0] = st[0]; o[1] = st[1]; o[2] = st[2]; o[3] = st[3];
    } else {  // pendulum: (cos th, sin th, thdot)
        float s, c;
        sincos_rn(st[0], &s, &c);
        o[0] = c; o[1] = s; o[2] = st[1]; o[3] = 0.f;
    }
}

// ---------------------------------------------------------------------------------------
// Observation noise and action delay (ENV_KS_PERTURB; dril_b200.h has the rules).  Component j of the base observation of env n
// in its episode e after s steps of it is o_j + sigma[j][n] z_j, z_j a standard normal of Philox block (gid, e, 2 s + j / 4,
// DRIL_TAG_OBS_NOISE) word pair (j / 2) % 2 through Box-Muller in fp64 with one rounding to fp32 (like sincos_rn: the fp64 value
// is far closer to the fp32 result than fp32's rounding steps, so oracle/env_perturb.py reproduces it bit for bit).  The noise is
// added to the raw observation, before Scaling and the velocity mask.
// ---------------------------------------------------------------------------------------
// whose observation a kernel builds: env n, in its episode e (the index of its reset draw), after s steps of that episode
struct EnvObsAt { long long n; uint32_t e, s; };
template <unsigned KS>
__device__ __forceinline__ EnvObsAt env_obs_at(const EnvDev& env, long long n) {
    if (!env_perturb(KS)) return {};
    return {n, env.episode[n] - 1u, (uint32_t)env.steps[n]};
}
// o[0 .. 3] (raw components 4b .. 4b+3) plus their noise; components beyond the base width and those with sigma 0 are untouched
__device__ __forceinline__ void env_obs_noise_block(const EnvDev& env, const EnvObsAt& at, int b, float* o) {
    if (!env.obs_noise) return;
    const int D0 = env_base_obs_dim(env.kind);
    uint32_t x[4];
    philox4x32((uint32_t)(env.gid_offset + at.n), at.e, 2u * at.s + (uint32_t)b, DRIL_TAG_OBS_NOISE, env.seed, x);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        if (4 * b + 2 * p >= D0) break;
        const float sg0 = env.obs_noise[(size_t)(4 * b + 2 * p) * env.n_envs + at.n];
        const float sg1 = 4 * b + 2 * p + 1 < D0 ? env.obs_noise[(size_t)(4 * b + 2 * p + 1) * env.n_envs + at.n] : 0.f;
        if (sg0 == 0.f && sg1 == 0.f) continue;
        const double r = sqrt(__dmul_rn(-2.0, log((double)u01_f32_open(x[2 * p]))));
        double sn, cs;
        sincos(__dmul_rn(6.283185307179586, (double)u01_f32(x[2 * p + 1])), &sn, &cs);
        if (sg0 != 0.f) o[2 * p] = __fadd_rn(o[2 * p], __fmul_rn(sg0, (float)__dmul_rn(r, cs)));
        if (sg1 != 0.f) o[2 * p + 1] = __fadd_rn(o[2 * p + 1], __fmul_rn(sg1, (float)__dmul_rn(r, sn)));
    }
}
// ... out of line for the all-kinds instantiations: inlined, the fp64 draw makes ptxas spill 232 bytes in the all-kinds fast
// kernel (128 registers); out of line it spills in the CartPole / Pendulum one, so those keep it inline
__device__ __noinline__ void env_obs_noise_block_call(const EnvDev& env, const EnvObsAt& at, int b, float* o) {
    env_obs_noise_block(env, at, b, o);
}
template <unsigned KS>
__device__ __forceinline__ void env_obs_noise(const EnvDev& env, const EnvObsAt& at, int b, float* o) {
    if (env_in(KS, DRIL_ENV_ACROBOT)) env_obs_noise_block_call(env, at, b, o);
    else env_obs_noise_block(env, at, b, o);
}
// the action env n applies this step: `a` (the env-space action it chose, a Discrete index as a float) enters its queue q (rows
// of stride `stride`, oldest first) and the one chosen d steps earlier leaves it.  *dq = d | ENV_DELAY_RESTART after a restart:
// the first action then fills the queue.
#define ENV_DELAY_RESTART 8
__device__ __forceinline__ float env_delay_action(int* dq, float* q, size_t stride, float a) {
    const int d = *dq & 7;
    float out = a;
    if (*dq & ENV_DELAY_RESTART) {
        for (int i = 0; i < d; ++i) q[(size_t)i * stride] = a;
        *dq = d;
    } else if (d > 0) {
        out = q[0];
        for (int i = 0; i + 1 < d; ++i) q[(size_t)i * stride] = q[(size_t)(i + 1) * stride];
        q[(size_t)(d - 1) * stride] = a;
    }
    return out;
}

// observation block b as the wrappers above the env see it: raw, or mapped to [-1, 1] by ScalingWrapperEnv.observe
// (scalingWrapperEnv.jl:72-75,94-99: `(x - offset) * scale - 1`, three separate fp32 roundings; Box/Box envs of
// obs_dim <= 4 only, so block 0).
// ENV_KS_OBS_PARAMS: components D0 .. D0+P-1 (D0 = env_base_obs_dim, P = env_n_params) are par[0 .. P-1], raw; the blocks
// straddle the boundary (Acrobot's block 1 is (w1, w2, p0, p1)), and Scaling maps only the D0 base components.
// ENV_KS_PERTURB: plus the noise of `at`.
template <unsigned KS>
__device__ __forceinline__ void env_obs_block(const EnvDev& env, const float* st, int b, float* o, const float* par = nullptr,
                                              const EnvObsAt& at = {}) {
    if (env_obs_params(KS)) {
        const int D0 = env_base_obs_dim(env.kind), P = env_n_params(env.kind);
        if (4 * b < D0) {
            env_raw_obs_block<KS>(env.kind, st, b, o);
            if (env.scaling && b == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < D0) o[j] = __fsub_rn(__fmul_rn(__fsub_rn(o[j], env.sc_obs_o[j]), env.sc_obs_f[j]), 1.0f);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int k = 0; k < DRIL_ENV_MAX_PARAMS; ++k)   // a select per (j, k): no dynamic index into the register array
                if (k < P && 4 * b + j == D0 + k) o[j] = par[k];
        }
        return;
    }
    env_raw_obs_block<KS>(env.kind, st, b, o);
    if (env_perturb(KS)) env_obs_noise<KS>(env, at, b, o);
    if (env.scaling && b == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < env.obs_dim) o[j] = __fsub_rn(__fmul_rn(__fsub_rn(o[j], env.sc_obs_o[j]), env.sc_obs_f[j]), 1.0f);
    }
}
// ---------------------------------------------------------------------------------------
// Observation history (ENV_KS_HISTORY).  The observation of env n at step t is the stack [f_{t-k+1} | ... | f_t], oldest
// first; a frame is env_frame of the state.  The k-1 older frames live in a history store of H = (k-1) * F rows (component j
// of the stack in row j, one column per env): env.hist in global memory, or a shared-memory copy in the fast kernel.  It
// moves once per env step (env_hist_push, before the reset) and is refilled with the new frame after every reset
// (env_hist_fill); every observation only reads it.
// ---------------------------------------------------------------------------------------
#define ENV_MAX_FRAME 6
// f[0 .. frame_dim-1]: the base observation as the wrappers below Normalize see it (raw, or mapped by Scaling), without its
// velocity components when frame_dim says so (env_frame_dim); the components beyond frame_dim are unspecified.  ENV_KS_PERTURB:
// with the noise of `at` (before Scaling and the mask)
template <unsigned KS>
__device__ __forceinline__ void env_frame(const EnvDev& env, const float* st, float* f, const EnvObsAt& at = {}) {
    env_raw_obs_block<KS>(env.kind, st, 0, f);
    if (env_perturb(KS)) env_obs_noise<KS>(env, at, 0, f);
    if (env.scaling) {
        const int D0 = env_base_obs_dim(env.kind);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < D0) f[j] = __fsub_rn(__fmul_rn(__fsub_rn(f[j], env.sc_obs_o[j]), env.sc_obs_f[j]), 1.0f);
    }
    if (env_in(KS, DRIL_ENV_ACROBOT) && env.kind == DRIL_ENV_ACROBOT) {
        f[4] = st[2]; f[5] = st[3];
        if (env_perturb(KS)) {
            float w[4] = {f[4], f[5], 0.f, 0.f};
            env_obs_noise<KS>(env, at, 1, w);
            f[4] = w[0]; f[5] = w[1];
        }
    } else if (env.kind == DRIL_ENV_CARTPOLE && env.frame_dim < 4) {
        f[1] = f[2];   // (x, theta)
    }
}
// stack component rows [0, H) of one env in a history store with row stride `stride`: f (the frame an action was chosen on)
// enters as the newest of the older frames, the oldest leaves
__device__ __forceinline__ void env_hist_push(float* h, size_t stride, int H, int F, const float* f) {
    for (int j = 0; j + F < H; ++j) h[(size_t)j * stride] = h[(size_t)(j + F) * stride];
#pragma unroll
    for (int j = 0; j < ENV_MAX_FRAME; ++j)
        if (j < F && H > 0) h[(size_t)(H - F + j) * stride] = f[j];
}
// ... every older frame = f (reset padding: before an episode's first observation the frames are that observation)
__device__ __forceinline__ void env_hist_fill(float* h, size_t stride, int H, int F, const float* f) {
    for (int j0 = 0; j0 < H; j0 += F) {
#pragma unroll
        for (int j = 0; j < ENV_MAX_FRAME; ++j)
            if (j < F) h[(size_t)(j0 + j) * stride] = f[j];
    }
}

// ScalingWrapperEnv.act! (scalingWrapperEnv.jl:77-80,112-115): `(a + 1) / scale + offset` before the wrapped env's act!
__device__ __forceinline__ float env_unscale_action(const EnvDev& env, float a) {
    return env.scaling ? __fadd_rn(__fdiv_rn(__fadd_rn(a, 1.0f), env.sc_act_f), env.sc_act_o) : a;
}

template <unsigned KS = ENV_KS_CLASSIC>
__device__ __forceinline__ void env_reset_state(int kind, uint32_t gid, uint32_t episode, unsigned long long seed,
                                                float* st) {
    uint32_t x[4];
    philox4x32(gid, episode, 0u, DRIL_TAG_RESET, seed, x);
    if (kind == DRIL_ENV_CARTPOLE) {
#pragma unroll
        for (int k = 0; k < 4; ++k) st[k] = __fadd_rn(-0.05f, __fmul_rn(0.1f, u01_f32(x[k])));
    } else if (kind == DRIL_ENV_PENDULUM) {
        st[0] = __fadd_rn(-3.14159274101257324f, __fmul_rn(6.28318548202514648f, u01_f32(x[0])));
        st[1] = __fadd_rn(-1.0f, __fmul_rn(2.0f, u01_f32(x[1])));
        st[2] = 0.f; st[3] = 0.f;
    } else if ((env_in(KS, DRIL_ENV_MOUNTAINCAR) && kind == DRIL_ENV_MOUNTAINCAR) ||
               (env_in(KS, DRIL_ENV_MOUNTAINCAR_CONTINUOUS) && kind == DRIL_ENV_MOUNTAINCAR_CONTINUOUS)) {
        st[0] = __fadd_rn(-0.6f, __fmul_rn(0.2f, u01_f32(x[0])));
        st[1] = 0.f; st[2] = 0.f; st[3] = 0.f;
    } else if (env_in(KS, DRIL_ENV_ACROBOT) && kind == DRIL_ENV_ACROBOT) {
#pragma unroll
        for (int k = 0; k < 4; ++k) st[k] = __fadd_rn(-0.1f, __fmul_rn(0.2f, u01_f32(x[k])));
    }
}

// ---------------------------------------------------------------------------------------
// Per-env physical parameters (dril_b200.h has the table).  Every step below takes the constants of the table from `p`, in table
// order: the kernels built for ENV_KS_PARAMS pass the env's values for the running episode, the default instantiations pass
// env_param_default as compile-time constants, which the compiler folds into the code of a step with the constants written in.
// Each derived coefficient is one fixed fp32 sequence, restated in oracle/env_params.py, that gives Gymnasium's constant bit
// for bit at the default values.
// ---------------------------------------------------------------------------------------
__host__ __device__ constexpr bool env_has_params(unsigned ks) { return (ks & ENV_KS_PARAMS) != 0; }
// the parametrised kind set whose instantiation serves env kind `kind` (the synthetic env has no parameters)
__host__ __device__ constexpr unsigned env_param_kind_set(int kind) {
    return (env_kind_set(kind) & ~(1u << DRIL_ENV_SYNTHETIC)) | ENV_KS_PARAMS;
}
// ... and the one that also observes the parameters
__host__ __device__ constexpr unsigned env_obs_param_kind_set(int kind) { return env_param_kind_set(kind) | ENV_KS_OBS_PARAMS; }
// ... and the one with an observation history (an env with history always runs with parameters: lo = hi = the defaults
// without ranges)
__host__ __device__ constexpr unsigned env_hist_kind_set(int kind) { return env_param_kind_set(kind) | ENV_KS_HISTORY; }
// ... and the ones with observation noise or action delay (parametrised like a history), without and with a history
__host__ __device__ constexpr unsigned env_perturb_kind_set(int kind) { return env_param_kind_set(kind) | ENV_KS_PERTURB; }
__host__ __device__ constexpr unsigned env_hist_perturb_kind_set(int kind) { return env_hist_kind_set(kind) | ENV_KS_PERTURB; }

// the defaults of the table (Gymnasium's constants), by kind
struct EnvParams { float v[DRIL_ENV_MAX_PARAMS]; };
__host__ __device__ constexpr EnvParams env_param_default(int kind) {
    constexpr EnvParams k_env_param_default[6] = {
        {{9.8f, 1.0f, 0.1f, 0.5f, 10.0f, 0.02f}},        // cartpole: gravity masscart masspole length force_mag tau
        {{10.0f, 1.0f, 1.0f, 0.05f}},                     // pendulum: g m l dt
        {},                                               // synthetic
        {{0.001f, 0.0025f}},                              // mountaincar: force gravity
        {{0.0015f, 0.0025f}},                             // mountaincar_continuous: power gravity
        {{1.0f, 1.0f, 1.0f, 0.5f, 0.5f, 1.0f}}};          // acrobot: link_length_1 link_mass_1 link_mass_2 link_com_pos_1 link_com_pos_2 link_moi
    return k_env_param_default[kind];
}
// whether a value must be > 0 (1) or >= 0 (0)
static const int k_env_param_positive[6][DRIL_ENV_MAX_PARAMS] = {
    {0, 1, 1, 1, 0, 1}, {0, 1, 1, 1}, {}, {0, 0}, {0, 0}, {1, 1, 1, 1, 1, 1}};

// the values of env n's episode `episode`: lo + (hi - lo) * u, u from Philox (gid, episode, k / 4, DRIL_TAG_ENV_PARAMS) word
// k % 4; written to par and env.pval
__device__ __forceinline__ void env_draw_params(const EnvDev& env, long long n, uint32_t gid, uint32_t episode, float* par) {
    const int np = env_n_params(env.kind);
    const long long N = env.n_envs;
    uint32_t x[4];
#pragma unroll
    for (int k = 0; k < DRIL_ENV_MAX_PARAMS; ++k) {
        if (k < np) {
            if ((k & 3) == 0) philox4x32(gid, episode, (uint32_t)(k >> 2), DRIL_TAG_ENV_PARAMS, env.seed, x);
            const float lo = env.plo[(size_t)k * N + n], hi = env.phi[(size_t)k * N + n];
            par[k] = __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), u01_f32(x[k & 3])));
            env.pval[(size_t)k * N + n] = par[k];
        }
    }
}
__device__ __forceinline__ void env_load_params(const EnvDev& env, long long n, float* par) {
    const int np = env_n_params(env.kind);
#pragma unroll
    for (int k = 0; k < DRIL_ENV_MAX_PARAMS; ++k) par[k] = k < np ? env.pval[(size_t)k * env.n_envs + n] : 0.f;
}

// CartPole-v1: p = (gravity, masscart, masspole, length, force_mag, tau); total_mass = masspole + masscart,
// polemass_length = masspole * length
struct CartPoleCoef { float gravity, masspole, length, force_mag, tau, total_mass, pml; };
__device__ __forceinline__ CartPoleCoef cartpole_coef(const float* p) {
    const float gravity = p[0], masscart = p[1], masspole = p[2], length = p[3], force_mag = p[4], tau = p[5];
    return {gravity, masspole, length, force_mag, tau, __fadd_rn(masspole, masscart), __fmul_rn(masspole, length)};
}
// Euler step with the (correctly rounded) sin/cos of the pole angle supplied by the caller.
// a01: 0 = push left, 1 = push right. Returns reward; sets terminated.
__device__ __forceinline__ float cartpole_step_sc(float* st, int a01, float sinth, float costh, const CartPoleCoef& C, bool* terminated) {
    const float THETA_THR = 0.20943951023931953f, X_THR = 2.4f, FOUR_THIRDS = 1.3333333333333333f;
    float x = st[0], x_dot = st[1], th = st[2], th_dot = st[3];
    float force = (a01 == 1) ? C.force_mag : -C.force_mag;
    float temp = __fdiv_rn(__fadd_rn(force, __fmul_rn(__fmul_rn(C.pml, __fmul_rn(th_dot, th_dot)), sinth)), C.total_mass);
    float den = __fmul_rn(C.length, __fsub_rn(FOUR_THIRDS, __fdiv_rn(__fmul_rn(C.masspole, __fmul_rn(costh, costh)), C.total_mass)));
    float thetaacc = __fdiv_rn(__fsub_rn(__fmul_rn(C.gravity, sinth), __fmul_rn(costh, temp)), den);
    float xacc = __fsub_rn(temp, __fdiv_rn(__fmul_rn(__fmul_rn(C.pml, thetaacc), costh), C.total_mass));
    float xn = __fadd_rn(x, __fmul_rn(C.tau, x_dot));
    float xdn = __fadd_rn(x_dot, __fmul_rn(C.tau, xacc));
    float thn = __fadd_rn(th, __fmul_rn(C.tau, th_dot));
    float thdn = __fadd_rn(th_dot, __fmul_rn(C.tau, thetaacc));
    st[0] = xn; st[1] = xdn; st[2] = thn; st[3] = thdn;
    *terminated = (xn < -X_THR) || (xn > X_THR) || (thn < -THETA_THR) || (thn > THETA_THR);
    return 1.0f;
}
__device__ __forceinline__ float cartpole_step(float* st, int a01, const CartPoleCoef& C, bool* terminated) {
    float sinth, costh;
    sincos_rn(st[2], &sinth, &costh);
    return cartpole_step_sc(st, a01, sinth, costh, C, terminated);
}

// Pendulum-v1: p = (g, m, l, dt); thdot += (3 g / (2 l) * sin th + 3 / (m l^2) * u) * dt with the coefficients
// c_sin = (3 g) / (2 l) and c_u = 3 / (m (l l))
struct PendulumCoef { float c_sin, c_u, dt; };
__device__ __forceinline__ PendulumCoef pendulum_coef(const float* p) {
    const float g = p[0], m = p[1], l = p[2], dt = p[3];
    return {__fdiv_rn(__fmul_rn(3.0f, g), __fmul_rn(2.0f, l)), __fdiv_rn(3.0f, __fmul_rn(m, __fmul_rn(l, l))), dt};
}
// ... at the defaults, as compile-time constants (15, 3, 0.05: every product and quotient is exact there).  The compiler does
// not fold __fdiv_rn of constants, so the default instantiations take these instead of pendulum_coef of the defaults.
__host__ __device__ constexpr PendulumCoef pendulum_default_coef() {
    constexpr EnvParams d = env_param_default(DRIL_ENV_PENDULUM);
    return {(3.0f * d.v[0]) / (2.0f * d.v[2]), 3.0f / (d.v[1] * (d.v[2] * d.v[2])), d.v[3]};
}
// u: env-space torque (clipped again like Gymnasium)
__device__ __forceinline__ float pendulum_step(float* st, float u, const PendulumCoef& C) {
    const float MAX_SPEED = 8.0f, MAX_TORQUE = 2.0f;
    const float PI = 3.14159274101257324f, TWO_PI = 6.28318548202514648f;
    u = fminf(fmaxf(u, -MAX_TORQUE), MAX_TORQUE);
    float th = st[0], thdot = st[1];
    float xp = __fadd_rn(th, PI);
    float an = __fsub_rn(__fsub_rn(xp, __fmul_rn(TWO_PI, floorf(__fdiv_rn(xp, TWO_PI)))), PI);
    float cost = __fadd_rn(__fadd_rn(__fmul_rn(an, an), __fmul_rn(0.1f, __fmul_rn(thdot, thdot))),
                           __fmul_rn(0.001f, __fmul_rn(u, u)));
    float sinth, costh;
    sincos_rn(th, &sinth, &costh);
    float nthdot = __fadd_rn(thdot, __fmul_rn(__fadd_rn(__fmul_rn(C.c_sin, sinth), __fmul_rn(C.c_u, u)), C.dt));
    nthdot = fminf(fmaxf(nthdot, -MAX_SPEED), MAX_SPEED);
    float nth = __fadd_rn(th, __fmul_rn(nthdot, C.dt));
    st[0] = nth; st[1] = nthdot;
    return -cost;
}

// MountainCar-v0 / MountainCarContinuous-v0 after the velocity increment dv: clip, move, clip, left wall, goal test
__device__ __forceinline__ void mountaincar_move(float* st, float dv, float goal, bool* terminated) {
    const float MAX_SPEED = 0.07f, MIN_POS = -1.2f, MAX_POS = 0.6f;
    float vel = fminf(fmaxf(__fadd_rn(st[1], dv), -MAX_SPEED), MAX_SPEED);
    const float pos = fminf(fmaxf(__fadd_rn(st[0], vel), MIN_POS), MAX_POS);
    if (pos == MIN_POS && vel < 0.f) vel = 0.f;
    st[0] = pos; st[1] = vel;
    *terminated = pos >= goal && vel >= 0.f;
}
// MountainCar-v0: p = (force, gravity); idx 0 = push left, 1 = none, 2 = push right.  Returns reward -1.
__device__ __forceinline__ float mountaincar_step(float* st, int idx, const float* p, bool* terminated) {
    float s, c;
    sincos_rn(__fmul_rn(3.0f, st[0]), &s, &c);
    mountaincar_move(st, __fadd_rn(__fmul_rn((float)(idx - 1), p[0]), __fmul_rn(c, -p[1])), 0.5f, terminated);
    return -1.0f;
}
// MountainCarContinuous-v0: p = (power, gravity); a = env-space force (clipped to [-1, 1] for the dynamics, not for the reward)
__device__ __forceinline__ float mountaincar_continuous_step(float* st, float a, const float* p, bool* terminated) {
    const float f = fminf(fmaxf(a, -1.0f), 1.0f);
    float s, c;
    sincos_rn(__fmul_rn(3.0f, st[0]), &s, &c);
    mountaincar_move(st, __fsub_rn(__fmul_rn(f, p[0]), __fmul_rn(p[1], c)), 0.45f, terminated);
    return __fsub_rn(*terminated ? 100.0f : 0.0f, __fmul_rn(__fmul_rn(a, a), 0.1f));
}

// Acrobot-v1: p = (l1, m1, m2, lc1, lc2, I) with I1 = I2 = I (link_moi) and g = 9.8.  The book dynamics f(s) for torque a as
//   d1 = ((m1 lc1^2 + m2 ((l1^2 + lc2^2) + (2 l1) lc2 c2)) + I) + I       d2 = m2 (lc2^2 + (l1 lc2) c2) + I
//   phi2 = ((m2 lc2) g) cos(th1 + th2 - pi/2)
//   phi1 = (((-h w2^2) s2 - ((2 h) (w2 w1)) s2) + ((m1 lc1 + m2 l1) g) cos(th1 - pi/2)) + phi2,   h = m2 (l1 lc2)
//   al2 = (((a + (d2 / d1) phi1) - (h w1^2) s2) - phi2) / ((m2 lc2^2 + I) - d2^2 / d1)      al1 = -(d2 al2 + phi1) / d1
// with every coefficient rounded once in the order written (at the defaults: 0.25, 1.25, 1, 1, 1, 0.25, 0.5, 0.5, 1, 4.9f, 14.7f,
// 1.25; (m1 lc1 + m2 l1) g = 1.5 * 9.8f rounded once)
struct AcrobotCoef { float a1, p, k, m2, i, l2, q, h, h2, g_lc2, g_12, j; };
__device__ __forceinline__ AcrobotCoef acrobot_coef(const float* p) {
    const float l1 = p[0], m1 = p[1], m2 = p[2], lc1 = p[3], lc2 = p[4], moi = p[5];
    AcrobotCoef c;
    c.a1 = __fmul_rn(m1, __fmul_rn(lc1, lc1));
    c.p = __fadd_rn(__fmul_rn(l1, l1), __fmul_rn(lc2, lc2));
    c.k = __fmul_rn(__fmul_rn(2.0f, l1), lc2);
    c.m2 = m2;
    c.i = moi;
    c.l2 = __fmul_rn(lc2, lc2);
    c.q = __fmul_rn(l1, lc2);
    c.h = __fmul_rn(m2, c.q);
    c.h2 = __fmul_rn(2.0f, c.h);
    c.g_lc2 = __fmul_rn(__fmul_rn(m2, lc2), 9.8f);
    c.g_12 = __fmul_rn(__fadd_rn(__fmul_rn(m1, lc1), __fmul_rn(m2, l1)), 9.8f);
    c.j = __fadd_rn(__fmul_rn(m2, c.l2), moi);
    return c;
}
__device__ __forceinline__ void acrobot_dsdt(const float* s, float a, const AcrobotCoef& C, float* ds) {
    const float HALF_PI = 1.57079637050628662f;
    const float th1 = s[0], th2 = s[1], w1 = s[2], w2 = s[3];
    float s2, c2, sp, cp2, cp1;
    sincos_rn(th2, &s2, &c2);
    const float d1 = __fadd_rn(__fadd_rn(__fadd_rn(C.a1, __fmul_rn(C.m2, __fadd_rn(C.p, __fmul_rn(C.k, c2)))), C.i), C.i);
    const float d2 = __fadd_rn(__fmul_rn(C.m2, __fadd_rn(C.l2, __fmul_rn(C.q, c2))), C.i);
    sincos_rn(__fsub_rn(__fadd_rn(th1, th2), HALF_PI), &sp, &cp2);
    const float phi2 = __fmul_rn(C.g_lc2, cp2);
    sincos_rn(__fsub_rn(th1, HALF_PI), &sp, &cp1);
    const float phi1 = __fadd_rn(__fadd_rn(__fsub_rn(__fmul_rn(__fmul_rn(-C.h, __fmul_rn(w2, w2)), s2),
                                                     __fmul_rn(__fmul_rn(C.h2, __fmul_rn(w2, w1)), s2)),
                                           __fmul_rn(C.g_12, cp1)), phi2);
    const float num = __fsub_rn(__fsub_rn(__fadd_rn(a, __fmul_rn(__fdiv_rn(d2, d1), phi1)), __fmul_rn(__fmul_rn(C.h, __fmul_rn(w1, w1)), s2)), phi2);
    const float al2 = __fdiv_rn(num, __fsub_rn(C.j, __fdiv_rn(__fmul_rn(d2, d2), d1)));
    const float al1 = __fdiv_rn(-__fadd_rn(__fmul_rn(d2, al2), phi1), d1);
    ds[0] = w1; ds[1] = w2; ds[2] = al1; ds[3] = al2;
}
// ... at the defaults, for the default instantiations: acrobot_dsdt with the products by m2 = 1, 2 l1 lc2 = 1 and 2 h = 1 left
// out (they are exact).  This is the one step kept twice: the compiler does not remove __fmul_rn(1, x), so acrobot_dsdt with the
// defaults as constants is not the code of these dynamics (16 more instructions per RK4 step), and turning those three products
// into plain ones changes the code of the parametrised instantiations.
__device__ __forceinline__ void acrobot_dsdt_default(const float* s, float a, float* ds) {
    const float HALF_PI = 1.57079637050628662f, G_LC2 = 4.90000009536743164f, G_12 = 14.7000007629394531f;
    const float th1 = s[0], th2 = s[1], w1 = s[2], w2 = s[3];
    float s2, c2, sp, cp2, cp1;
    sincos_rn(th2, &s2, &c2);
    const float d1 = __fadd_rn(__fadd_rn(__fadd_rn(0.25f, __fadd_rn(1.25f, c2)), 1.0f), 1.0f);
    const float d2 = __fadd_rn(__fadd_rn(0.25f, __fmul_rn(0.5f, c2)), 1.0f);
    sincos_rn(__fsub_rn(__fadd_rn(th1, th2), HALF_PI), &sp, &cp2);
    const float phi2 = __fmul_rn(G_LC2, cp2);
    sincos_rn(__fsub_rn(th1, HALF_PI), &sp, &cp1);
    const float phi1 = __fadd_rn(__fadd_rn(__fsub_rn(__fmul_rn(__fmul_rn(-0.5f, __fmul_rn(w2, w2)), s2), __fmul_rn(__fmul_rn(w2, w1), s2)),
                                           __fmul_rn(G_12, cp1)), phi2);
    const float num = __fsub_rn(__fsub_rn(__fadd_rn(a, __fmul_rn(__fdiv_rn(d2, d1), phi1)), __fmul_rn(__fmul_rn(0.5f, __fmul_rn(w1, w1)), s2)), phi2);
    const float al2 = __fdiv_rn(num, __fsub_rn(1.25f, __fdiv_rn(__fmul_rn(d2, d2), d1)));
    const float al1 = __fdiv_rn(-__fadd_rn(__fmul_rn(d2, al2), phi1), d1);
    ds[0] = w1; ds[1] = w2; ds[2] = al1; ds[3] = al2;
}
// Gymnasium's wrap(x, -pi, pi): subtract / add 2 pi until inside (a non-finite angle, only reachable through set_state, is
// left as it is instead of looping forever)
__device__ __forceinline__ float acrobot_wrap(float x) {
    const float PI = 3.14159274101257324f, TWO_PI = 6.28318548202514648f;
    if (!isfinite(x)) return x;
    while (x > PI) x = __fsub_rn(x, TWO_PI);
    while (x < -PI) x = __fadd_rn(x, TWO_PI);
    return x;
}
// Acrobot-v1: idx 0 / 1 / 2 = torque -1 / 0 / +1 held over one RK4 step of dt = 0.2 of the dynamics dsdt(s, a, ds).  Returns
// reward 0 on termination, else -1.
template <class Dsdt>
__device__ __forceinline__ float acrobot_step(float* st, int idx, const Dsdt& dsdt, bool* terminated) {
    const float DT = 0.2f, DT2 = 0.1f, DT6 = 0.0333333350718021393f;
    const float MAX_VEL_1 = 12.5663709640502930f, MAX_VEL_2 = 28.2743339538574219f;
    const float a = (float)(idx - 1);
    float k1[4], k2[4], k3[4], k4[4], y[4];
    dsdt(st, a, k1);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = __fadd_rn(st[i], __fmul_rn(DT2, k1[i]));
    dsdt(y, a, k2);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = __fadd_rn(st[i], __fmul_rn(DT2, k2[i]));
    dsdt(y, a, k3);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = __fadd_rn(st[i], __fmul_rn(DT, k3[i]));
    dsdt(y, a, k4);
#pragma unroll
    for (int i = 0; i < 4; ++i)
        y[i] = __fadd_rn(st[i], __fmul_rn(DT6, __fadd_rn(__fadd_rn(__fadd_rn(k1[i], __fmul_rn(2.0f, k2[i])), __fmul_rn(2.0f, k3[i])), k4[i])));
    st[0] = acrobot_wrap(y[0]);
    st[1] = acrobot_wrap(y[1]);
    st[2] = fminf(fmaxf(y[2], -MAX_VEL_1), MAX_VEL_1);
    st[3] = fminf(fmaxf(y[3], -MAX_VEL_2), MAX_VEL_2);
    float s, c1, c12;
    sincos_rn(st[0], &s, &c1);
    sincos_rn(__fadd_rn(st[1], st[0]), &s, &c12);
    *terminated = __fsub_rn(-c1, c12) > 1.0f;
    return *terminated ? 0.0f : -1.0f;
}

// Synthetic env (SURVEY §8d C5): obs block b of lifetime step `life`
__device__ __forceinline__ void synthetic_obs_block(uint32_t gid, uint32_t life, int b, unsigned long long seed, float o[4]) {
    uint32_t x[4];
    philox4x32(gid, life, (uint32_t)b, DRIL_TAG_SYN_OBS, seed, x);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = __fadd_rn(-1.0f, __fmul_rn(2.0f, u01_f32(x[j])));
}
__device__ __forceinline__ float synthetic_step(uint32_t gid, uint32_t life, unsigned long long seed, bool* terminated) {
    uint32_t x[4];
    philox4x32(gid, life, 0u, DRIL_TAG_SYN_DYN, seed, x);
    *terminated = u01_f32(x[1]) < 0.005f;
    return u01_f32(x[0]);
}

// env_step tests the kinds of KS in the order CartPole, Pendulum, MountainCar, MountainCarContinuous, Acrobot, synthetic; the
// last kind of KS in that order is taken without a test
__host__ __device__ constexpr int env_last_kind(unsigned ks) {
    return env_in(ks, DRIL_ENV_SYNTHETIC) ? DRIL_ENV_SYNTHETIC
         : env_in(ks, DRIL_ENV_ACROBOT) ? DRIL_ENV_ACROBOT
         : env_in(ks, DRIL_ENV_MOUNTAINCAR_CONTINUOUS) ? DRIL_ENV_MOUNTAINCAR_CONTINUOUS
         : env_in(ks, DRIL_ENV_MOUNTAINCAR) ? DRIL_ENV_MOUNTAINCAR
         : env_in(ks, DRIL_ENV_PENDULUM) ? DRIL_ENV_PENDULUM : DRIL_ENV_CARTPOLE;
}
template <unsigned KS, int K>
__device__ __forceinline__ bool env_is(int kind) { return env_in(KS, K) && (K == env_last_kind(KS) || kind == K); }

// one step of env n: a_disc = env-space action of a Discrete env, a_cont = the Box env's action as the wrappers above it hand it
// over (read only for Box envs), life = the synthetic env's lifetime step counter (read and advanced for that kind only).
// par: the env's parameter values, which the ENV_KS_PARAMS instantiations step with; the others step with the defaults.
// Returns the reward; sets terminated.
template <unsigned KS>
__device__ __forceinline__ float env_step(const EnvDev& env, float* st, long long n, int a_disc, const float* a_cont, uint32_t* life,
                                          bool* terminated, const float* par = nullptr) {
    constexpr bool P = env_has_params(KS);
    if (env_is<KS, DRIL_ENV_CARTPOLE>(env.kind)) {
        constexpr EnvParams D = env_param_default(DRIL_ENV_CARTPOLE);
        return cartpole_step(st, a_disc - env.act_start, cartpole_coef(P ? par : D.v), terminated);
    }
    if (env_is<KS, DRIL_ENV_PENDULUM>(env.kind)) {
        constexpr PendulumCoef D = pendulum_default_coef();
        return pendulum_step(st, env_unscale_action(env, *a_cont), P ? pendulum_coef(par) : D);
    }
    if (env_is<KS, DRIL_ENV_MOUNTAINCAR>(env.kind)) {
        constexpr EnvParams D = env_param_default(DRIL_ENV_MOUNTAINCAR);
        return mountaincar_step(st, a_disc - env.act_start, P ? par : D.v, terminated);
    }
    if (env_is<KS, DRIL_ENV_MOUNTAINCAR_CONTINUOUS>(env.kind)) {
        constexpr EnvParams D = env_param_default(DRIL_ENV_MOUNTAINCAR_CONTINUOUS);
        return mountaincar_continuous_step(st, env_unscale_action(env, *a_cont), P ? par : D.v, terminated);
    }
    if (env_is<KS, DRIL_ENV_ACROBOT>(env.kind)) {
        const int idx = a_disc - env.act_start;
        if (!P) return acrobot_step(st, idx, acrobot_dsdt_default, terminated);
        const AcrobotCoef C = acrobot_coef(par);
        return acrobot_step(st, idx, [&C](const float* s, float a, float* ds) { acrobot_dsdt(s, a, C, ds); }, terminated);
    }
    *life = env.life[n];
    const float r = synthetic_step((uint32_t)(env.gid_offset + n), *life, env.seed, terminated);
    *life += 1;
    env.life[n] = *life;
    return r;
}
