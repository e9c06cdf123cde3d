// Shared device/host definitions for libdril_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/dril_b200.h"

#define DRIL_MAX_LAYERS (DRIL_MAX_HIDDEN_LAYERS + 1)
#define DRIL_THREADS 256

// ---------------------------------------------------------------------------------------
// error handling (never throws across the C boundary)
// ---------------------------------------------------------------------------------------
void dril_set_error(const char* fmt, ...);

#define DRIL_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            dril_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__, \
                           cudaGetErrorString(_e));                                             \
            return DRIL_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)

#define DRIL_REQUIRE(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            dril_set_error(__VA_ARGS__);        \
            return DRIL_ERR_INVALID;            \
        }                                       \
    } while (0)

#define DRIL_TRY(expr)                  \
    do {                                \
        int32_t _s = (expr);            \
        if (_s != DRIL_OK) return _s;   \
    } while (0)

// ---------------------------------------------------------------------------------------
// descriptors passed by value to kernels
// ---------------------------------------------------------------------------------------
struct LayerDesc {
    int K, N;        // logical in/out
    int Kp, Np;      // padded to multiples of 4
    int w_off, b_off;    // offsets in the flat (ComponentVector-order) parameter vector
    int pw_off, pb_off;  // offsets in the packed buffer: W [Kp][Np] (zero padded), bias [Np]
    int pwt_off;         // offset in the packed buffer of Wt [Np][Kp]
};

struct PolicyDesc {
    int obs_dim, obs_dim_p;
    int n_layers;  // dense layers per net (hidden + output)
    int act_kind, act_n, act_start;
    int n_params;
    int log_std_off;   // flat offset (continuous) or -1
    int pack_fwd;      // floats of the forward part of the packed buffer (all W + bias, both nets)
    int pack_total;    // forward part + all Wt
    int gpack;         // floats of a packed gradient partial: pack_fwd + act_n (log_std) + 8 (stats)
    int max_np;        // widest padded layer output
    LayerDesc L[2][DRIL_MAX_LAYERS];  // [0]=actor_head, [1]=critic_head
    float act_low[DRIL_MAX_ACT_DIM], act_high[DRIL_MAX_ACT_DIM];
};

struct EnvDev {
    int kind, obs_dim, state_dim, max_steps, act_start, act_dim;
    long long n_envs, gid_offset;
    unsigned long long seed;
    float* state;               // [state_dim][n]
    int* steps;                 // [n]
    unsigned int* episode;      // [n] reset counter (RNG)
    unsigned int* life;         // [n] lifetime step counter (synthetic RNG)
    // MonitorWrapperEnv
    int monitor;                // window (0 = off)
    float* ep_ret;              // [n]
    int* ep_len;                // [n]
    double* roll_sums;          // [2]: sum episode return, sum episode length over this rollout
    unsigned long long* roll_eps;  // [1]: episodes this rollout
    // NormalizeWrapperEnv
    int normalize, training, norm_obs, norm_reward;
    float clip_obs, clip_reward, ngamma, eps;
    float* ret;                 // [n] discounted return accumulator
    float* obs_mean;            // [obs_dim]
    float* obs_var;             // [obs_dim]
    float* ret_stats;           // [2] mean, var
    long long* counts;          // [2] obs_count, ret_count
    double* partials;           // [2 parity][max_blocks][2*obs_dim + 2]
    double* roll_moments;       // [2 * (obs_dim + 1) + 2]: this rollout's sums / sums of squares per normalised column
                                // (obs dims, discounted return) and the obs / return sample counts (data-parallel merge)
    // ScalingWrapperEnv (scalingWrapperEnv.jl:14-49): per-env wrapper BELOW Monitor / Normalize; factors pre-computed on the host
    int scaling;
    float sc_obs_f[4], sc_obs_o[4];   // obs' = (obs - offset) * factor - 1
    float sc_act_f, sc_act_o;         // env action = (a + 1) / factor + offset
    float* tobs;                // [n][obs_dim] raw terminal observations scratch
    float* old_obs;             // [n][obs_dim] raw obs of the last observe (compat path)
    float* old_rewards;         // [n]
    // per-env physical parameters (env.cuh); null unless dril_env_set_params gave ranges
    int has_params;
    float* pval;                // [DRIL_ENV_MAX_PARAMS][n] values of the running episode
    float* plo;                 // [DRIL_ENV_MAX_PARAMS][n] ranges
    float* phi;
    // observation history (env.cuh, ENV_KS_HISTORY); hist_len 1 and hist null unless dril_env_set_obs_history turned it on.
    // frame_dim < the kind's base width means velocity-free frames.  (16 bytes: the offsets behind EnvDev in RolloutArgs keep
    // their 16-byte alignment, and with it the existing kernels' code.)
    int hist_len, frame_dim;
    float* hist;                // [(hist_len - 1) * frame_dim][n] the older frames of the stack, oldest first
    // observation noise and action delay (env.cuh, ENV_KS_PERTURB); each null while off.  (32 bytes: 16-byte alignment kept.)
    float* obs_noise;           // [base obs dim][n] standard deviations
    int* act_delay;             // [n] delay d | ENV_DELAY_RESTART while the queue waits for its first action
    float* act_q;               // [DRIL_ENV_MAX_ACTION_DELAY][n] the queued env-space actions, oldest first
    int max_delay;              // the largest d (rows of the fast kernel's shared-memory queue)
    int pad_;
};

struct BufDev {
    long long T, N;
    int obs_dim, act_kind, act_dim;
    float* obs;
    void* actions;
    float *rewards, *values, *logprobs, *advantages, *returns, *boot, *last_values, *episode_r;
    int* episode_l;
    unsigned char* flags;
    int* done_count;  // [T]
};

// ---------------------------------------------------------------------------------------
// Philox4x32-10 — the normative stream of oracle/philox.py
// ---------------------------------------------------------------------------------------
#define DRIL_TAG_RESET 1u
#define DRIL_TAG_SAMPLE 2u
#define DRIL_TAG_SYN_OBS 3u
#define DRIL_TAG_SHUFFLE 4u
#define DRIL_TAG_SYN_DYN 5u
#define DRIL_TAG_ENV_PARAMS 6u
#define DRIL_TAG_OBS_NOISE 7u

__host__ __device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                     unsigned long long seed, uint32_t out[4]) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        unsigned long long p0 = 0xD2511F53ull * c0;
        unsigned long long p1 = 0xCD9E8D57ull * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__host__ __device__ __forceinline__ float u01_f32(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
__host__ __device__ __forceinline__ float u01_f32_open(uint32_t x) {
    return ((float)(x >> 8) + 1.0f) * 5.9604644775390625e-08f;
}
__host__ __device__ __forceinline__ double u01_f64(uint32_t x0, uint32_t x1) {
    unsigned long long bits = ((unsigned long long)x0 << 21) | (unsigned long long)(x1 >> 11);
    return (double)bits * 1.1102230246251565e-16;
}

// keyed bijection on [0,n): 4-round Feistel + cycle walking (oracle/philox.py feistel_permute)
struct FeistelKey {
    uint32_t k[4];
    int half_bits;
    uint32_t half_mask;
};

__host__ __device__ __forceinline__ uint32_t feistel_round(uint32_t r, uint32_t key, uint32_t mask) {
    uint32_t h = r + key;
    h *= 0x9E3779B1u;
    h ^= h >> 15;
    h *= 0x85EBCA77u;
    h ^= h >> 13;
    return h & mask;
}

__host__ __device__ __forceinline__ long long feistel_permute(long long i, long long n, const FeistelKey& fk) {
    unsigned long long x = (unsigned long long)i;
    do {
        uint32_t l = (uint32_t)(x >> fk.half_bits) & fk.half_mask;
        uint32_t r = (uint32_t)x & fk.half_mask;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t nl = r;
            r = l ^ feistel_round(r, fk.k[q], fk.half_mask);
            l = nl;
        }
        x = ((unsigned long long)l << fk.half_bits) | r;
    } while (x >= (unsigned long long)n);
    return (long long)x;
}

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
// tanh with ~1e-7 absolute error from ex2.approx + fast divide (Lux tanh on fp32 is
// itself a ~1 ulp polynomial; the tolerance budget is 1e-6 on values, 1e-5 on logprobs).
// tanh(x) = 1 - 2 / (1 + e^(2x)) in five instructions (FMUL, MUFU.EX2, FADD, MUFU.RCP, FFMA); absolute error ~1e-7.
// x -> +inf: e = inf, rcp = 0, result 1; x -> -inf: e = 0, result -1.
__device__ __forceinline__ float fast_tanh(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));      // 2 * log2(e)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// deterministic block sum of `v` over DRIL_THREADS threads; result valid in all threads.
// scratch: >= 32 elements of shared memory; contains two __syncthreads.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    T r = 0;
    int nw = (blockDim.x + 31) >> 5;
    for (int i = 0; i < nw; ++i) r += scratch[i];
    return r;
}
#endif
