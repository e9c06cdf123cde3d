// Automatic domain randomisation (dril_env_set_adr, include/dril_b200.h): two device passes between a rollout and the next
// one.  They work entirely through the parameter ranges plo / phi, which every reset draws from, and through the rollout
// buffer the Monitor filled; no rollout kernel knows about ADR.
//   adr_scan_kernel    attributes the episodes that ended in the rollout (flags / episode_r) to boundary slots and writes the
//                      rollout's per-slot return sums and counts (fixed-order block partials, summed by the last block)
//   adr_update_kernel  adds them to the accumulators, moves the boundaries whose buffers are full, and writes the next round's
//                      ranges of the parameters under ADR (every block decides redundantly, the last block commits)
#pragma once
#include "common.cuh"
#include "env.cuh"

#define ADR_THREADS 256
#define ADR_MAX_SLOTS (2 * DRIL_ENV_MAX_PARAMS)

// the configuration (by value in the launches)
struct AdrCfg {
    int n;                                        // |J|: parameters under ADR, slots 2 i + side
    int idx[DRIL_ENV_MAX_PARAMS];                 // table index of the i-th parameter
    float init_lo[DRIL_ENV_MAX_PARAMS], init_hi[DRIL_ENV_MAX_PARAMS];
    float limit_lo[DRIL_ENV_MAX_PARAMS], limit_hi[DRIL_ENV_MAX_PARAMS];
    float delta[DRIL_ENV_MAX_PARAMS];
    float p_boundary, t_low, t_high;
    long long m;                                  // episodes per slot before a decision
};
// the state (device memory; identical on every rank)
struct AdrState {
    float lo[DRIL_ENV_MAX_PARAMS], hi[DRIL_ENV_MAX_PARAMS];
    double sum[ADR_MAX_SLOTS];
    long long cnt[ADR_MAX_SLOTS];
    long long round;
    unsigned ticket[2];                           // finished CTAs of the running scan / update launch (0 between launches)
};
// per-env attribution words
struct AdrEnv {
    unsigned* ep_mark;                            // [n] episode counter at the end of the previous round
    int* run_slot;                                // [n] slot of the episode that was running then (-1: none)
};

// the slot of env gid during round r: -1 for a plain env
__device__ __forceinline__ int adr_slot(const AdrCfg& c, unsigned long long seed, uint32_t gid, long long round) {
    uint32_t x[4];
    philox4x32(gid, (uint32_t)round, 0u, DRIL_TAG_ADR, seed, x);
    if (!(u01_f32(x[0]) < c.p_boundary)) return -1;
    return (int)(x[1] % (uint32_t)(2 * c.n));
}

// env n's ranges of the ADR parameters for a round in which it has `slot`: [lo_i, hi_i], the slot's side pinned
__device__ __forceinline__ void adr_write_rows(const AdrCfg& c, const float* lo, const float* hi, int slot, const EnvDev& env,
                                               long long n) {
    const size_t N = (size_t)env.n_envs;
    for (int i = 0; i < c.n; ++i) {
        float l = lo[i], h = hi[i];
        if (slot == 2 * i) h = l;
        else if (slot == 2 * i + 1) l = h;
        env.plo[(size_t)c.idx[i] * N + n] = l;
        env.phi[(size_t)c.idx[i] * N + n] = h;
    }
}

struct AdrRanges { float lo[DRIL_ENV_MAX_PARAMS], hi[DRIL_ENV_MAX_PARAMS]; };
// The ranges r of `round`, written from the host:
//   ADR_WRITE_OFF    without boundary envs (turning ADR off); the attribution words are left alone
//   ADR_WRITE_ON     with the round's boundary envs (turning ADR on, round 0): ep_mark = the reset counter, run_slot = the slot
//                    (the running episodes are redrawn from these ranges next)
//   ADR_WRITE_RESEED with the boundary envs under a new seed (dril_env_seed): ep_mark = the reset counter, run_slot = -1 (the
//                    episodes running now drew their parameters under the old assignment and are not counted)
enum { ADR_WRITE_OFF = 0, ADR_WRITE_ON = 1, ADR_WRITE_RESEED = 2 };
__global__ void __launch_bounds__(ADR_THREADS) adr_write_kernel(const __grid_constant__ AdrCfg c, const __grid_constant__ AdrRanges r,
                                                                EnvDev env, AdrEnv ae, long long round, int mode) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= env.n_envs) return;
    const int slot = mode != ADR_WRITE_OFF ? adr_slot(c, env.seed, (uint32_t)(env.gid_offset + n), round) : -1;
    adr_write_rows(c, r.lo, r.hi, slot, env, n);
    if (mode != ADR_WRITE_OFF) { ae.ep_mark[n] = env.episode[n]; ae.run_slot[n] = mode == ADR_WRITE_ON ? slot : -1; }
}

// Attribution (thread per env, coalesced across envs, the env's T rows column-wise from the last): the k-th of env n's d done
// rows ends episode episode[n] - 1 - d + k; it counts for the current round's slot if that index is >= ep_mark[n], else for
// run_slot[n].  part: [gridDim.x][2 S] (sums | counts) per CTA; the last CTA writes roll[2 S] = their sum in CTA order.
__global__ void __launch_bounds__(ADR_THREADS) adr_scan_kernel(const __grid_constant__ AdrCfg c, AdrState* st, EnvDev env, AdrEnv ae,
                                                               const unsigned char* __restrict__ flags,
                                                               const float* __restrict__ episode_r, long long T,
                                                               double* __restrict__ part, double* __restrict__ roll) {
    __shared__ double s_sum[ADR_THREADS / 32][ADR_MAX_SLOTS];
    __shared__ int s_cnt[ADR_THREADS / 32][ADR_MAX_SLOTS];
    __shared__ bool s_last;
    const int S = 2 * c.n, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long N = env.n_envs, n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int slot_a = -1, slot_b = -1, cnt_a = 0, cnt_b = 0;     // the current round's slot, run_slot
    double sum_a = 0.0, sum_b = 0.0;
    if (n < N) {
        const long long round = st->round;
        const unsigned ep = env.episode[n], mark = ae.ep_mark[n];
        slot_a = adr_slot(c, env.seed, (uint32_t)(env.gid_offset + n), round);
        slot_b = ae.run_slot[n];
        long long e = (long long)ep - 1;                     // the running episode
        for (int t = (int)T - 1; t >= 0; --t) {
            if (flags[(size_t)t * N + n] & 3) {
                --e;
                const double r = (double)episode_r[(size_t)t * N + n];
                if (e >= (long long)mark) { sum_a += r; cnt_a += 1; }
                else { sum_b += r; cnt_b += 1; }
            }
        }
        if ((long long)ep - 1 >= (long long)mark) ae.run_slot[n] = slot_a;
        ae.ep_mark[n] = ep;
    }
    for (int s = 0; s < S; ++s) {
        double v = (slot_a == s ? sum_a : 0.0) + (slot_b == s ? sum_b : 0.0);
        int k = (slot_a == s ? cnt_a : 0) + (slot_b == s ? cnt_b : 0);
        v = warp_sum(v);
        k = __reduce_add_sync(0xffffffffu, k);
        if (lane == 0) { s_sum[w][s] = v; s_cnt[w][s] = k; }
    }
    __syncthreads();
    if (threadIdx.x < S) {
        double v = 0.0;
        long long k = 0;
        for (int i = 0; i < ADR_THREADS / 32; ++i) { v += s_sum[i][threadIdx.x]; k += s_cnt[i][threadIdx.x]; }
        part[(size_t)blockIdx.x * 2 * S + threadIdx.x] = v;
        part[(size_t)blockIdx.x * 2 * S + S + threadIdx.x] = (double)k;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&st->ticket[0], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int v = w; v < 2 * S; v += ADR_THREADS / 32) {
        double a = 0.0;
        for (unsigned b = lane; b < gridDim.x; b += 32) a += __ldcg(part + (size_t)b * 2 * S + v);
        a = warp_sum(a);
        if (lane == 0) roll[v] = a;
    }
    if (threadIdx.x == 0) st->ticket[0] = 0u;
}

// The decision of one round from the state and the rollout's (rank-summed) roll[2 S]: new lo / hi; sums / counts after it
__device__ __forceinline__ void adr_decide(const AdrCfg& c, const AdrState* st, const double* roll, float* lo, float* hi,
                                           double* sum, long long* cnt) {
    const int S = 2 * c.n;
    for (int i = 0; i < c.n; ++i) { lo[i] = st->lo[i]; hi[i] = st->hi[i]; }
    for (int s = 0; s < S; ++s) {
        sum[s] = st->sum[s] + roll[s];
        cnt[s] = st->cnt[s] + (long long)(roll[S + s] + 0.5);
        if (cnt[s] < c.m) continue;
        const double mean = sum[s] / (double)cnt[s];
        const int i = s >> 1;
        if (mean >= (double)c.t_high) {            // widen
            if (s & 1) hi[i] = fminf(c.limit_hi[i], __fadd_rn(st->hi[i], c.delta[i]));
            else lo[i] = fmaxf(c.limit_lo[i], __fsub_rn(st->lo[i], c.delta[i]));
        } else if (mean <= (double)c.t_low) {      // narrow, never inside the initial range
            if (s & 1) hi[i] = fmaxf(c.init_hi[i], __fsub_rn(st->hi[i], c.delta[i]));
            else lo[i] = fminf(c.init_lo[i], __fadd_rn(st->lo[i], c.delta[i]));
        }
        sum[s] = 0.0;
        cnt[s] = 0;
    }
}

__global__ void __launch_bounds__(ADR_THREADS) adr_update_kernel(const __grid_constant__ AdrCfg c, AdrState* st, EnvDev env,
                                                                 const double* __restrict__ roll) {
    __shared__ float s_lo[DRIL_ENV_MAX_PARAMS], s_hi[DRIL_ENV_MAX_PARAMS];
    __shared__ long long s_round;
    __shared__ bool s_last;
    if (threadIdx.x == 0) {
        double sum[ADR_MAX_SLOTS];
        long long cnt[ADR_MAX_SLOTS];
        adr_decide(c, st, roll, s_lo, s_hi, sum, cnt);
        s_round = st->round + 1;
    }
    __syncthreads();
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n < env.n_envs) adr_write_rows(c, s_lo, s_hi, adr_slot(c, env.seed, (uint32_t)(env.gid_offset + n), s_round), env, n);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&st->ticket[1], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    // every other CTA has read the state: commit
    double sum[ADR_MAX_SLOTS];
    long long cnt[ADR_MAX_SLOTS];
    float lo[DRIL_ENV_MAX_PARAMS], hi[DRIL_ENV_MAX_PARAMS];
    adr_decide(c, st, roll, lo, hi, sum, cnt);
    for (int i = 0; i < c.n; ++i) { st->lo[i] = lo[i]; st->hi[i] = hi[i]; }
    for (int s = 0; s < 2 * c.n; ++s) { st->sum[s] = sum[s]; st->cnt[s] = cnt[s]; }
    st->round = s_round;
    st->ticket[1] = 0u;
}
