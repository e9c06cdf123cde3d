// Fused rollout engine: observe -> normalise -> actor/critic forward -> sample -> to_env ->
// env step -> monitor / normaliser statistics -> auto-reset, for n_steps, written straight
// into the device-resident rollout buffer.  One persistent kernel per rollout.
//
// Replaces the n_steps loop of collect_trajectories (buffers/trajectory.jl:33-76) together
// with NormalizeWrapperEnv.observe/act! (environment_wrappers/normalizeWrapperEnv.jl:123-165),
// MonitorWrapperEnv.act! (monitorWrapperEnv.jl:44-60), MultiThreadedParallelEnv.act!
// (multithreadedParallelEnv.jl:47-74), the layer call (layers/layer_forward.jl:3-39) and the
// batch-of-1 bootstrap predict_values calls (trajectory.jl:57-70).
//
// Work decomposition: a CTA owns tiles of M consecutive envs.  Without a training
// NormalizeWrapperEnv the envs are independent for the whole rollout, so the grid is one
// tile per CTA and there is no inter-CTA communication.  With running statistics every step
// needs the batch moments over ALL envs before rewards / the next observation can be
// normalised: the kernel is then launched cooperatively and uses one grid barrier per step
// (the reward-return moments of step t and the observation moments of observe t+1 share it).
#pragma once
#include <cooperative_groups.h>

#include "env.cuh"
#include "mlp.cuh"

namespace cg = cooperative_groups;

enum {
    RO_HAS_POLICY = 1,        // run the actor-critic (fused rollout); off: compat act!/observe
    RO_INITIAL_OBSERVE = 2,   // the observe() before the loop (trajectory.jl:32) updates obs stats
    RO_FOLD_NEXT_OBSERVE = 4, // the observe() after each act! (trajectory.jl:45) is folded into the step
    RO_WEIGHTS_SMEM = 8,
    RO_GRID_SYNC = 16,        // training normaliser: cooperative launch + grid barrier per step
    RO_WRITE_OBS_OUT = 32,    // compat observe: write normalised obs to obs_out
    RO_TILES_8X8 = 64,        // throughput mode (many envs per SM): 8x8 register tiles in the hidden layers
    RO_MMA = 128,             // general kernel, tile width multiple of 16: wide layers on mma.sync 3xTF32 tiles
    RO_DETERMINISTIC = 256,   // general kernel: mode of the distribution instead of a sample (evaluate_agent, evaluation.jl:54-143)
    RO_DEFER_CRITIC = 512     // general kernel: only the actor runs in the step loop; V(s_t), V(terminal_obs) and V(new_obs) are
                              // evaluated afterwards by one batched critic pass over the (normalised) observations it stored
};

// observations whose values are evaluated after the rollout (RO_DEFER_CRITIC): what the policy saw, i.e. already normalised
struct DeferredCritic {
    float* last_obs;          // [N][D] observation after the final step
    float* trunc_obs;         // [cap][D] terminal observations of truncated steps
    long long* trunc_idx;     // [cap] buffer sample index of each entry
    unsigned int* trunc_count;
    unsigned int cap;
};

struct RolloutArgs {
    EnvDev env;
    BufDev buf;
    PolicyDesc pd;
    const float* pack;       // packed parameters (global)
    const float* flat;       // flat parameters (log_std)
    const void* forced;      // forced actions [T][N] int32 | [T][N][A] float, or null
    float* obs_out;          // compat observe output [N][D]
    unsigned long long pseed;
    unsigned int step0;
    int T, M4, n_tiles, flags;
    DeferredCritic dc;
};

struct RolloutSmem {
    int ld, raw_rows;
    size_t w, raw, x, acta, actc, envact, stat, part, total;  // float offsets (part: bytes offset for doubles)
};

// critic = false (RO_DEFER_CRITIC): no critic activations, which leaves room for 128-env tiles with wide nets
// tca (rollout_gtc.cuh): the actor's layers run on tcgen05 out of their own image region behind `total`; only the output rows
// (<= 8 actions / action dims) are kept here
__host__ __device__ inline RolloutSmem rollout_smem_layout(const PolicyDesc& pd, int obs_dim, int act_dim, int M4,
                                                           bool weights_smem, bool has_policy, bool critic = true, bool tca = false) {
    RolloutSmem s;
    s.ld = M4 + 4;
    int Dp = (obs_dim + 3) & ~3;
    s.raw_rows = Dp + 4;
    size_t o = 0;
    s.w = o; o += (weights_smem && has_policy) ? (size_t)pd.pack_fwd : 0;
    s.raw = o; o += (size_t)s.raw_rows * s.ld;
    s.x = o; o += (size_t)Dp * s.ld;
    s.acta = o; o += has_policy ? (tca ? (size_t)8 * s.ld : (size_t)2 * pd.max_np * s.ld) : 0;
    s.actc = o; o += (has_policy && critic) ? (size_t)2 * pd.max_np * s.ld : 0;
    int adp = act_dim < 1 ? 1 : act_dim;
    s.envact = o; o += (size_t)adp * s.ld;
    s.stat = o; o += (size_t)4 * Dp + 8;
    o = (o + 3) & ~(size_t)3;
    s.part = o * sizeof(float);                       // doubles: [2*D+2] accumulators + 64 scratch + 4 counts
    s.total = s.part + (size_t)(2 * obs_dim + 2 + 64 + 4) * sizeof(double);
    return s;
}

// Chan/Welford merge exactly as RunningMeanStd.update_from_moments! (normalizeWrapperEnv.jl:28-50), fp32.
__device__ __forceinline__ void rms_merge(float& mean, float& var, long long count, float bm, float bv, long long bc) {
    if (count == 0) {
        mean = bm; var = bv;
    } else {
        float delta = __fsub_rn(bm, mean);
        long long total = count + bc;
        float fc = (float)count, fb = (float)bc, ft = (float)total;
        float new_mean = __fadd_rn(mean, __fdiv_rn(__fmul_rn(delta, fb), ft));
        float m_a = __fmul_rn(var, fc);
        float m_b = __fmul_rn(bv, fb);
        float m2 = __fadd_rn(__fadd_rn(m_a, m_b),
                             __fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(delta, delta), fc), fb), ft));
        mean = new_mean;
        var = __fdiv_rn(m2, ft);
    }
}

// Data-parallel normaliser merge after a rollout (SURVEY §8e): xr holds, summed over ranks, [roll return sum, roll length sum,
// roll episodes | per column (obs dims, return): sum, sum of squares | obs samples, return samples] of this rollout; the running
// statistics become snap (+) global batch with the Chan merge of normalizeWrapperEnv.jl:28-50, identically on every rank.
__global__ void norm_monitor_merge_kernel(EnvDev env, const double* __restrict__ xr, const float* __restrict__ snap, const long long* __restrict__ snap_cnt,
                                          int do_norm) {
    const int D = env.obs_dim, t = threadIdx.x;
    if (t == 0) {
        env.roll_sums[0] = xr[0]; env.roll_sums[1] = xr[1];
        *env.roll_eps = (unsigned long long)(xr[2] + 0.5);
    }
    if (!do_norm) return;
    const double* mom = xr + 3;
    const double n_obs = mom[2 * (D + 1)], n_ret = mom[2 * (D + 1) + 1];
    for (int d = t; d < D; d += blockDim.x) {
        if (n_obs > 0.0) {
            const double bm = mom[2 * d] / n_obs;
            double bv = mom[2 * d + 1] / n_obs - bm * bm;
            if (bv < 0.0) bv = 0.0;
            float m = snap[d], v = snap[D + d];
            rms_merge(m, v, snap_cnt[0], (float)bm, (float)bv, (long long)(n_obs + 0.5));
            env.obs_mean[d] = m; env.obs_var[d] = v;
        }
    }
    if (t == 0) {
        if (n_ret > 0.0) {
            const double bm = mom[2 * D] / n_ret;
            double bv = mom[2 * D + 1] / n_ret - bm * bm;
            if (bv < 0.0) bv = 0.0;
            float m = snap[2 * D], v = snap[2 * D + 1];
            rms_merge(m, v, snap_cnt[1], (float)bm, (float)bv, (long long)(n_ret + 0.5));
            env.ret_stats[0] = m; env.ret_stats[1] = v;
        }
        env.counts[0] = snap_cnt[0] + (long long)(n_obs + 0.5);
        env.counts[1] = snap_cnt[1] + (long long)(n_ret + 0.5);
    }
}
__global__ void norm_monitor_pack_kernel(EnvDev env, double* __restrict__ xr, float* __restrict__ snap, long long* __restrict__ snap_cnt, int n_mom) {
    const int t = threadIdx.x;
    if (t == 0) { xr[0] = env.roll_sums[0]; xr[1] = env.roll_sums[1]; xr[2] = (double)*env.roll_eps; }
    for (int i = t; i < n_mom; i += blockDim.x) xr[3 + i] = env.roll_moments ? env.roll_moments[i] : 0.0;
}
__global__ void norm_snapshot_kernel(EnvDev env, float* __restrict__ snap, long long* __restrict__ snap_cnt) {
    const int D = env.obs_dim, t = threadIdx.x;
    for (int d = t; d < D; d += blockDim.x) { snap[d] = env.obs_mean[d]; snap[D + d] = env.obs_var[d]; }
    if (t == 0) { snap[2 * D] = env.ret_stats[0]; snap[2 * D + 1] = env.ret_stats[1]; snap_cnt[0] = env.counts[0]; snap_cnt[1] = env.counts[1]; }
    for (int i = t; i < 2 * (D + 1) + 2; i += blockDim.x) env.roll_moments[i] = 0.0;
}

__device__ __forceinline__ float normalize_obs_val(float x, float mean, float var, float eps, float clip) {
    float v = __fdiv_rn(__fsub_rn(x, mean), __fsqrt_rn(__fadd_rn(var, eps)));
    return fminf(fmaxf(v, -clip), clip);
}

// column sums (double) of rows [0,rows) of sRaw over the valid samples of this tile, accumulated
// into acc[2*c], acc[2*c+1] (sum, sum of squares) by a fixed warp per column => deterministic.
__device__ __forceinline__ void tile_column_sums(const float* sRaw, int ld, int row0, int rows, int col0, int nvalid,
                                                 double* acc) {
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int r = warp; r < rows; r += nw) {
        double s = 0.0, q = 0.0;
        for (int e = lane; e < nvalid; e += 32) {
            double v = (double)sRaw[(size_t)(row0 + r) * ld + e];
            s += v; q += v * v;
        }
        s = warp_sum(s); q = warp_sum(q);
        if (lane == 0) { acc[2 * (col0 + r)] += s; acc[2 * (col0 + r) + 1] += q; }
    }
}

// the layer forward of the step loop: fp32 FMA / mma.sync tiles out of the ping-pong activation buffers (mlp.cuh); the tcgen05
// actor of rollout_gtc.cuh is the other implementation of this call
struct MlpForward {
    __device__ __forceinline__ int operator()(const PolicyDesc& pd, const float* __restrict__ Wbase, const float* sX, float* sActA, float* sActC,
                                              int M4, int ld, int net_mask, bool use_mma) const {
        return mlp_forward_pingpong(pd, Wbase, sX, sActA, sActC, M4, ld, net_mask, use_mma);
    }
};

// KS: the env kinds this instantiation serves (env.cuh)
template <bool WS, bool TCA, unsigned KS, class Fwd>
__device__ __forceinline__ void rollout_body(const RolloutArgs& a, float* smem, Fwd& fwd) {
    const EnvDev& env = a.env;
    const BufDev& buf = a.buf;
    const PolicyDesc& pd = a.pd;
    const bool has_policy = a.flags & RO_HAS_POLICY;
    const bool defer = (a.flags & RO_DEFER_CRITIC) != 0;
    const bool grid_sync = a.flags & RO_GRID_SYNC;
    const bool use_mma = (a.flags & RO_MMA) != 0;
    const int D = env.obs_dim, Dp = (D + 3) & ~3;
    const int M4 = a.M4;
    const long long N = env.n_envs;
    const RolloutSmem L = rollout_smem_layout(pd, D, env.act_dim, M4, WS, has_policy, !(a.flags & RO_DEFER_CRITIC), TCA);
    const int ld = L.ld;
    float* sRaw = smem + L.raw;
    float* sX = smem + L.x;
    float* sActA = smem + L.acta;
    float* sActC = smem + L.actc;
    float* sEnvAct = smem + L.envact;
    float* sMean = smem + L.stat;        // [Dp]
    float* sVar = sMean + Dp;            // [Dp]
    float* sNewMean = sVar + Dp;         // [Dp]
    float* sNewVar = sNewMean + Dp;      // [Dp]
    float* sRet = sNewVar + Dp;          // [0] ret_mean [1] ret_var
    double* sAcc = reinterpret_cast<double*>(reinterpret_cast<char*>(smem) + L.part);  // [2*D+2]
    double* sScratch = sAcc + 2 * D + 2;                                                // [64]
    long long* sCnt = reinterpret_cast<long long*>(sScratch + 64);                      // obs_count, ret_count
    const int tid = threadIdx.x;
    const int ncol = D + 1;  // obs columns + the discounted-return column
    const bool upd_obs = env.normalize && env.training && env.norm_obs;
    const bool upd_ret = env.normalize && env.training && env.norm_reward;

    // WS: weights staged in shared memory (L.w == 0; address space known at compile time -> LDS)
    const float* __restrict__ Wbase = WS ? smem : a.pack;
    if (WS) {
        const float4* src = reinterpret_cast<const float4*>(a.pack);
        float4* dst = reinterpret_cast<float4*>(smem);
        for (int i = tid; i < pd.pack_fwd / 4; i += blockDim.x) dst[i] = src[i];
    }
    for (int d = tid; d < Dp; d += blockDim.x) {
        sMean[d] = (env.normalize && d < D) ? env.obs_mean[d] : 0.f;
        sVar[d] = (env.normalize && d < D) ? env.obs_var[d] : 1.f;
    }
    if (tid == 0) {
        sRet[0] = env.normalize ? env.ret_stats[0] : 0.f;
        sRet[1] = env.normalize ? env.ret_stats[1] : 1.f;
        sCnt[0] = env.normalize ? env.counts[0] : 0;
        sCnt[1] = env.normalize ? env.counts[1] : 0;
    }
    for (int i = tid; i < 2 * ncol; i += blockDim.x) sAcc[i] = 0.0;
    __syncthreads();

    int parity = 0;
    // merge this step's batch moments (all CTAs compute the same values in the same order)
    auto reduce_and_merge = [&](bool do_obs, bool do_ret) {
        double* mine = env.partials + ((size_t)parity * gridDim.x + blockIdx.x) * (2 * ncol);
        for (int i = tid; i < 2 * ncol; i += blockDim.x) { mine[i] = sAcc[i]; }
        __threadfence();
        cg::this_grid().sync();
        const double* all = env.partials + (size_t)parity * gridDim.x * (2 * ncol);
        int warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
        for (int c = warp; c < 2 * ncol; c += nw) {
            double s = 0.0;
            for (int b = lane; b < (int)gridDim.x; b += 32) s += all[(size_t)b * (2 * ncol) + c];
            s = warp_sum(s);
            if (lane == 0) sAcc[c] = s;
        }
        __syncthreads();
        // data-parallel runs: this rollout's batch moments are also accumulated on their own, so that after the rollout the ranks
        // can merge (count, mean, M2) of the GLOBAL batch into the statistics they all started the rollout with
        if (env.roll_moments && blockIdx.x == 0) {
            for (int c = tid; c < 2 * ncol; c += blockDim.x) {
                const bool is_ret = (c >> 1) == D;
                if (is_ret ? do_ret : do_obs) env.roll_moments[c] += sAcc[c];
            }
            if (tid == 0) {
                if (do_obs) env.roll_moments[2 * ncol] += (double)N;
                if (do_ret) env.roll_moments[2 * ncol + 1] += (double)N;
            }
        }
        double dn = (double)N;
        if (do_obs) {
            for (int d = tid; d < D; d += blockDim.x) {
                double bm = sAcc[2 * d] / dn;
                double bv = sAcc[2 * d + 1] / dn - bm * bm;
                if (bv < 0.0) bv = 0.0;
                float m = sMean[d], v = sVar[d];
                rms_merge(m, v, sCnt[0], (float)bm, (float)bv, N);
                sNewMean[d] = m; sNewVar[d] = v;
            }
        }
        if (do_ret && tid == 0) {
            double bm = sAcc[2 * D] / dn;
            double bv = sAcc[2 * D + 1] / dn - bm * bm;
            if (bv < 0.0) bv = 0.0;
            float m = sRet[0], v = sRet[1];
            rms_merge(m, v, sCnt[1], (float)bm, (float)bv, N);
            sRet[0] = m; sRet[1] = v;
        }
        __syncthreads();
        if (tid == 0) {
            if (do_obs) sCnt[0] += N;
            if (do_ret) sCnt[1] += N;
        }
        for (int i = tid; i < 2 * ncol; i += blockDim.x) sAcc[i] = 0.0;
        parity ^= 1;
        __syncthreads();
    };
    auto commit_obs_stats = [&]() {
        for (int d = tid; d < D; d += blockDim.x) { sMean[d] = sNewMean[d]; sVar[d] = sNewVar[d]; }
        __syncthreads();
    };

    // raw observation of every env of a tile -> sRaw rows [0,D) (feature-major); zero padding.
    auto tile_raw_obs = [&](long long n0, int nvalid) {
        if (env.kind == DRIL_ENV_SYNTHETIC) {
            int nb = Dp >> 2;
            for (int i = tid; i < nb * M4; i += blockDim.x) {
                int b = i / M4, e = i - b * M4;
                float o[4] = {0.f, 0.f, 0.f, 0.f};
                if (e < nvalid) synthetic_obs_block((uint32_t)(env.gid_offset + n0 + e), env.life[n0 + e], b, env.seed, o);
#pragma unroll
                for (int j = 0; j < 4; ++j) sRaw[(size_t)(4 * b + j) * ld + e] = (4 * b + j < D) ? o[j] : 0.f;
            }
        } else if (env_history(KS)) {   // [older frames from the history store | the frame of the current state]
            if (tid < M4) {
                const int F = env.frame_dim, H = D - F;
                const bool v = tid < nvalid;
                float f[ENV_MAX_FRAME] = {};
                if (v) {
                    float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * N + n0 + tid];
                    env_frame<KS>(env, st, f, env_obs_at<KS>(env, n0 + tid));
                }
                for (int j = 0; j < H; ++j) sRaw[(size_t)j * ld + tid] = v ? env.hist[(size_t)j * N + n0 + tid] : 0.f;
#pragma unroll
                for (int j = 0; j < ENV_MAX_FRAME; ++j) if (j < F) sRaw[(size_t)(H + j) * ld + tid] = f[j];
                for (int j = D; j < Dp; ++j) sRaw[(size_t)j * ld + tid] = 0.f;
            }
        } else {
            if (tid < M4) {
#pragma unroll
                for (int b = 0; b < env_obs_blocks(KS); ++b) {
                    float o[4] = {0.f, 0.f, 0.f, 0.f};
                    if (tid < nvalid) {
                        float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                        for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * N + n0 + tid];
                        if (env_obs_params(KS)) {   // the running episode's values (after an auto-reset: the new draw)
                            float par[DRIL_ENV_MAX_PARAMS];
                            env_load_params(env, n0 + tid, par);
                            env_obs_block<KS>(env, st, b, o, par);
                        } else {
                            env_obs_block<KS>(env, st, b, o, nullptr, env_obs_at<KS>(env, n0 + tid));
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) if (4 * b + j < Dp) sRaw[(size_t)(4 * b + j) * ld + tid] = o[j];
                }
            }
        }
        __syncthreads();
    };
    // normalise sRaw -> sX with (mean,var); optionally also record old_obs
    auto tile_normalize = [&](const float* mean, const float* var, int nvalid) {
        for (int i = tid; i < Dp * M4; i += blockDim.x) {
            int d = i / M4, e = i - d * M4;
            float x = sRaw[(size_t)d * ld + e];
            if (env.normalize && env.norm_obs && d < D && e < nvalid)
                x = normalize_obs_val(x, mean[d], var[d], env.eps, env.clip_obs);
            sX[(size_t)d * ld + e] = x;
        }
        __syncthreads();
    };

    // ---------------- the observe() before the loop -----------------------------------------
    if ((a.flags & RO_INITIAL_OBSERVE) && upd_obs) {
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
            long long n0 = (long long)tile * M4;
            int nvalid = (int)min((long long)M4, N - n0);
            tile_raw_obs(n0, nvalid);
            tile_column_sums(sRaw, ld, 0, D, 0, nvalid, sAcc);
            __syncthreads();
        }
        reduce_and_merge(true, false);
        commit_obs_stats();
    }
    if (a.flags & RO_WRITE_OBS_OUT) {  // compat observe(): normalised obs out, raw obs cached
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
            long long n0 = (long long)tile * M4;
            int nvalid = (int)min((long long)M4, N - n0);
            tile_raw_obs(n0, nvalid);
            tile_normalize(sMean, sVar, nvalid);
            for (int i = tid; i < nvalid * D; i += blockDim.x) {
                int e = i / D, d = i - e * D;
                a.obs_out[(size_t)n0 * D + i] = sX[(size_t)d * ld + e];
                if (env.old_obs) env.old_obs[(size_t)n0 * D + i] = sRaw[(size_t)d * ld + e];
            }
            __syncthreads();
        }
    }

    // ---------------- n_steps ---------------------------------------------------------------
    for (int t = 0; t < a.T; ++t) {
        const size_t row = (size_t)t * N;
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
            long long n0 = (long long)tile * M4;
            int nvalid = (int)min((long long)M4, N - n0);
            const bool mine = tid < nvalid;
            const long long n = n0 + tid;
            int fin = 0;
            if (has_policy) {
                // observe: raw -> normalised -> buffer
                tile_raw_obs(n0, nvalid);
                tile_normalize(sMean, sVar, nvalid);
                for (int i = tid; i < nvalid * D; i += blockDim.x) {
                    int e = i / D, d = i - e * D;
                    buf.obs[(row + n0) * D + i] = sX[(size_t)d * ld + e];
                }
                // actor + critic forward (critic deferred: actor only)
                fin = fwd(pd, Wbase, sX, sActA, sActC, M4, ld, defer ? 1 : 3, use_mma);
            }
            // sample / replay action, log-prob, value; hand the env-space action to the step
            int a_disc = 0;
            if (mine) {
                const uint32_t gid = (uint32_t)(env.gid_offset + n);
                if (has_policy) {
                    const float* z = sActA + (size_t)fin * pd.max_np * ld + tid;
                    float value = defer ? 0.f : sActC[(size_t)fin * pd.max_np * ld + tid];
                    float logp;
                    if (pd.act_kind == DRIL_ACT_DISCRETE) {
                        int mode = 0, forced_v = 0;
                        double u = 0.0;
                        if (a.forced) { mode = 2; forced_v = reinterpret_cast<const int*>(a.forced)[row + n]; }
                        else if (a.flags & RO_DETERMINISTIC) mode = 1;
                        else {
                            uint32_t x[4];
                            philox4x32(gid, a.step0 + (uint32_t)t, 0u, DRIL_TAG_SAMPLE, a.pseed, x);
                            u = u01_f64(x[0], x[1]);
                        }
                        HeadOut h = categorical_head(z, ld, pd.act_n, pd.act_start, mode, u, forced_v, false);
                        logp = h.logp;
                        a_disc = h.action_idx;
                        reinterpret_cast<int*>(buf.actions)[row + n] = a_disc;
                    } else {
                        const int A = pd.act_n;
                        float ls_sum = 0.f, dss = 0.f;
                        for (int j = 0; j < A; ++j) {
                            float mean = z[(size_t)j * ld];
                            float ls = a.flat[pd.log_std_off + j];
                            float act;
                            if (a.forced) act = reinterpret_cast<const float*>(a.forced)[(row + n) * A + j];
                            else if (a.flags & RO_DETERMINISTIC) act = mean;            // mode(DiagGaussian) = mean (diagGaussian.jl:40-47)
                            else act = __fadd_rn(mean, __fmul_rn(expf(ls), sample_normal(gid, a.step0 + (uint32_t)t, j, a.pseed)));
                            float diff = act - mean;
                            dss += diff * diff * expf(-2.0f * ls);
                            ls_sum += ls;
                            reinterpret_cast<float*>(buf.actions)[(row + n) * A + j] = act;   // raw, unclamped (trajectory.jl:48)
                            sEnvAct[(size_t)j * ld + tid] = fminf(fmaxf(act, pd.act_low[j]), pd.act_high[j]);  // ClampAdapter
                        }
                        logp = -0.5f * (2.0f * ls_sum + dss + (float)A * DRIL_LOG2PI);
                    }
                    if (!defer) buf.values[row + n] = value;
                    buf.logprobs[row + n] = logp;
                } else {  // compat act!: actions are given in env space
                    if (env.act_dim == 0) a_disc = reinterpret_cast<const int*>(a.forced)[row + n];
                    else for (int j = 0; j < env.act_dim; ++j)
                        sEnvAct[(size_t)j * ld + tid] = reinterpret_cast<const float*>(a.forced)[(row + n) * env.act_dim + j];
                }
            }
            // env step + monitor + auto-reset (thread per env)
            if (mine) {
                const uint32_t gid = (uint32_t)(env.gid_offset + n);
                float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * N + n];
                int steps = env.steps[n];
                bool term = false;
                float r;
                uint32_t life = 0;
                float par[DRIL_ENV_MAX_PARAMS];
                if (env_has_params(KS)) env_load_params(env, n, par);
                EnvObsAt at = env_obs_at<KS>(env, n);
                if (env_history(KS)) {                          // the frame the action was chosen on enters the history
                    float f[ENV_MAX_FRAME];
                    env_frame<KS>(env, st, f, at);
                    env_hist_push(env.hist + n, (size_t)N, D - env.frame_dim, env.frame_dim, f);
                }
                if (env_perturb(KS) && env.act_delay) {         // the action chosen d steps earlier
                    const float ad = env_delay_action(env.act_delay + n, env.act_q + n, (size_t)N, env.act_dim ? sEnvAct[tid] : (float)a_disc);
                    if (env.act_dim) sEnvAct[tid] = ad; else a_disc = (int)ad;
                }
                r = env_step<KS>(env, st, n, a_disc, sEnvAct + tid, &life, &term, par);
                steps += 1;
                at.s = (uint32_t)steps;
                const bool trunc = steps >= env.max_steps;
                const bool done = term || trunc;
                buf.flags[row + n] = (unsigned char)((term ? 1 : 0) | (trunc ? 2 : 0));
                buf.rewards[row + n] = r;                       // raw for now; normalised after the barrier
                if (env.old_rewards) env.old_rewards[n] = r;
                if (env.monitor) {                              // monitorWrapperEnv.jl:44-60 (raw rewards)
                    float er = __fadd_rn(env.ep_ret[n], r);
                    int el = env.ep_len[n] + 1;
                    if (done) {
                        buf.episode_r[row + n] = er;
                        buf.episode_l[row + n] = el;
                        atomicAdd(&buf.done_count[t], 1);
                        atomicAdd(&env.roll_sums[0], (double)er);
                        atomicAdd(&env.roll_sums[1], (double)el);
                        atomicAdd(env.roll_eps, 1ull);
                        er = 0.f; el = 0;
                    }
                    env.ep_ret[n] = er; env.ep_len[n] = el;
                }
                if (trunc) {                                    // terminal_observation iff truncated
                    if (env.kind == DRIL_ENV_SYNTHETIC) {
                        for (int b = 0; b < (Dp >> 2); ++b) {
                            float o[4];
                            synthetic_obs_block(gid, life, b, env.seed, o);
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (4 * b + j < D) env.tobs[(size_t)n * D + 4 * b + j] = o[j];
                        }
                    } else if (env_history(KS)) {             // the stack that ends in the ended episode's final frame
                        const int F = env.frame_dim, H = D - F;
                        float f[ENV_MAX_FRAME];
                        env_frame<KS>(env, st, f, at);
                        for (int j = 0; j < H; ++j) env.tobs[(size_t)n * D + j] = env.hist[(size_t)j * N + n];
#pragma unroll
                        for (int j = 0; j < ENV_MAX_FRAME; ++j) if (j < F) env.tobs[(size_t)n * D + H + j] = f[j];
                    } else {
#pragma unroll
                        for (int b = 0; b < env_obs_blocks(KS); ++b) {
                            float o[4];
                            env_obs_block<KS>(env, st, b, o, par, at);   // the ended episode's values: drawn anew below
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (4 * b + j < D) env.tobs[(size_t)n * D + 4 * b + j] = o[j];
                        }
                    }
                }
                if (done) {                                     // reset!(env_i)
                    uint32_t ep = env.episode[n];
                    env_reset_state<KS>(env.kind, gid, ep, env.seed, st);
                    if (env_has_params(KS)) env_draw_params(env, n, gid, ep, par);
                    if (env_history(KS)) {
                        float f[ENV_MAX_FRAME];
                        env_frame<KS>(env, st, f, EnvObsAt{n, ep, 0u});
                        env_hist_fill(env.hist + n, (size_t)N, D - env.frame_dim, env.frame_dim, f);
                    }
                    if (env_perturb(KS) && env.act_delay) env.act_delay[n] |= ENV_DELAY_RESTART;
                    env.episode[n] = ep + 1;
                    steps = 0;
                }
#pragma unroll
                for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) env.state[(size_t)k * N + n] = st[k];
                env.steps[n] = steps;
                if (upd_ret) {                                  // update_reward_stats! (normalizeWrapperEnv.jl:167-171)
                    float ret = __fadd_rn(__fmul_rn(env.ret[n], env.ngamma), r);
                    sRaw[(size_t)Dp * ld + tid] = ret;
                    env.ret[n] = done ? 0.f : ret;              // zeroed after the statistics saw it (:153-156)
                } else if (env.normalize && done) {
                    env.ret[n] = 0.f;
                }
            }
            __syncthreads();
            if (grid_sync) {
                if (upd_ret) tile_column_sums(sRaw, ld, Dp, 1, D, nvalid, sAcc);
                if (upd_obs && (a.flags & RO_FOLD_NEXT_OBSERVE)) {
                    __syncthreads();
                    tile_raw_obs(n0, nvalid);                   // post-reset observation = next observe()
                    tile_column_sums(sRaw, ld, 0, D, 0, nvalid, sAcc);
                }
                __syncthreads();
            }
        }
        if (grid_sync) reduce_and_merge(upd_obs && (a.flags & RO_FOLD_NEXT_OBSERVE), upd_ret);

        // after the barrier: reward normalisation, truncation bootstrap values
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
            long long n0 = (long long)tile * M4;
            int nvalid = (int)min((long long)M4, N - n0);
            const bool mine = tid < nvalid;
            const long long n = n0 + tid;
            int trunc = 0;
            if (mine) {
                trunc = (buf.flags[row + n] >> 1) & 1;
                if (env.normalize && env.norm_reward) {         // normalize_rewards! (:188-197)
                    float r = buf.rewards[row + n];
                    r = __fdiv_rn(r, __fsqrt_rn(__fadd_rn(sRet[1], env.eps)));
                    buf.rewards[row + n] = fminf(fmaxf(r, -env.clip_reward), env.clip_reward);
                }
            }
            int any_trunc = __syncthreads_or(trunc);
            if (any_trunc) {
                // terminal observations are normalised with the statistics BEFORE the next observe's update
                for (int i = tid; i < Dp * M4; i += blockDim.x) {
                    int d = i / M4, e = i - d * M4;
                    float x = 0.f;
                    if (d < D && e < nvalid && ((buf.flags[row + n0 + e] >> 1) & 1)) {
                        x = env.tobs[(size_t)(n0 + e) * D + d];
                        if (env.normalize && env.norm_obs) {
                            x = normalize_obs_val(x, sMean[d], sVar[d], env.eps, env.clip_obs);
                            if (!has_policy) env.tobs[(size_t)(n0 + e) * D + d] = x;   // compat: infos["terminal_observation"]
                        }
                    }
                    sX[(size_t)d * ld + e] = x;
                }
                __syncthreads();
                if (has_policy && defer) {                      // V(terminal_obs) later: keep the normalised terminal observation
                    if (mine && trunc) {
                        const unsigned int k = atomicAdd(a.dc.trunc_count, 1u);
                        if (k < a.dc.cap) {
                            for (int d = 0; d < D; ++d) a.dc.trunc_obs[(size_t)k * D + d] = sX[(size_t)d * ld + tid];
                            a.dc.trunc_idx[k] = (long long)(row + n);
                        }
                    }
                    __syncthreads();
                } else if (has_policy) {                        // V(terminal_obs), trajectory.jl:57-61
                    int f = fwd(pd, Wbase, sX, sActA, sActC, M4, ld, 2, use_mma);
                    if (mine && trunc) buf.boot[row + n] = sActC[(size_t)f * pd.max_np * ld + tid];
                    __syncthreads();
                }
            }
        }
        if (grid_sync && upd_obs && (a.flags & RO_FOLD_NEXT_OBSERVE)) commit_obs_stats();
    }

    // ---------------- V(new_obs) after the final step (trajectory.jl:65-70) ----------------
    if (has_policy && a.T > 0) {
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
            long long n0 = (long long)tile * M4;
            int nvalid = (int)min((long long)M4, N - n0);
            tile_raw_obs(n0, nvalid);
            tile_normalize(sMean, sVar, nvalid);
            if (defer) {
                for (int i = tid; i < nvalid * D; i += blockDim.x) {
                    int e = i / D, d = i - e * D;
                    a.dc.last_obs[(size_t)n0 * D + i] = sX[(size_t)d * ld + e];
                }
                __syncthreads();
                continue;
            }
            int f = fwd(pd, Wbase, sX, sActA, sActC, M4, ld, 2, use_mma);
            if (tid < nvalid) buf.last_values[n0 + tid] = sActC[(size_t)f * pd.max_np * ld + tid];
            __syncthreads();
        }
    }
    if (env.normalize && blockIdx.x == 0) {
        for (int d = tid; d < D; d += blockDim.x) { env.obs_mean[d] = sMean[d]; env.obs_var[d] = sVar[d]; }
        if (tid == 0) { env.ret_stats[0] = sRet[0]; env.ret_stats[1] = sRet[1]; env.counts[0] = sCnt[0]; env.counts[1] = sCnt[1]; }
    }
}

template <bool WS, unsigned KS>
__global__ void __launch_bounds__(DRIL_THREADS) rollout_kernel(const __grid_constant__ RolloutArgs a) {
    extern __shared__ float4 smem4[];
    MlpForward fwd;
    rollout_body<WS, false, KS>(a, reinterpret_cast<float*>(smem4), fwd);
}

// ---------------------------------------------------------------------------------------
// Fast path of the fused rollout (the common case): every state-based env, no running-statistics
// update (no NormalizeWrapperEnv, or one in eval mode), one tile of envs per CTA.
//   * env state, step counters and monitor accumulators stay in registers for all n_steps
//     (no global round trip on the per-step critical path);
//   * the output layers (hidden -> n_actions | act_dim, hidden -> 1) are K-split over all threads
//     and reduced through shared memory, and the env-owning thread goes straight from the reduced
//     logits to sampling and the dynamics step: 2 + n_hidden barriers per step;
//   * per-step results are written straight into the time-major buffer (coalesced rows).
// Semantics identical to rollout_kernel (same reference citations).
// ---------------------------------------------------------------------------------------
#define RF_MAX_OUT 9   // actor outputs (<= 8) + value

struct RolloutFastSmem {
    int ld, slices;
    size_t w, x, acta, actc, part, stat, hist, total;   // float offsets; total in bytes
};

// hist_rows: rows of the tile's observation-history store (ENV_KS_HISTORY) and action queues (ENV_KS_PERTURB), 0 otherwise
__host__ __device__ inline RolloutFastSmem rollout_fast_smem_layout(const PolicyDesc& pd, int M4, int threads, bool weights_smem,
                                                                   int hist_rows = 0) {
    RolloutFastSmem s;
    s.ld = M4 + 4;
    s.slices = threads / M4;
    size_t o = 0;
    s.w = o; o += weights_smem ? (size_t)pd.pack_fwd : 0;
    s.x = o; o += (size_t)pd.obs_dim_p * s.ld;
    s.acta = o; o += (size_t)2 * pd.max_np * s.ld;
    s.actc = o; o += (size_t)2 * pd.max_np * s.ld;
    s.part = o; o += (size_t)s.slices * RF_MAX_OUT * s.ld;
    s.stat = o; o += (size_t)2 * pd.obs_dim_p + 4;
    s.hist = o; o += (size_t)hist_rows * s.ld;
    s.total = ((o + 3) & ~(size_t)3) * sizeof(float);
    return s;
}

template <bool WS, unsigned KS>
__global__ void __launch_bounds__(DRIL_THREADS) rollout_fast_kernel(const __grid_constant__ RolloutArgs a) {
    constexpr int OW = 4 * env_obs_blocks(KS);   // observation components held per env
    extern __shared__ float4 smem4[];
    float* smem = reinterpret_cast<float*>(smem4);
    const EnvDev& env = a.env;
    const BufDev& buf = a.buf;
    const PolicyDesc& pd = a.pd;
    const int D = env.obs_dim, Dp = pd.obs_dim_p, M4 = a.M4, NL = pd.n_layers;
    const long long N = env.n_envs;
    // ENV_KS_HISTORY: the tile's history store in shared memory for the whole rollout, rows [0, H), written back at the end;
    // ENV_KS_PERTURB with delays: the tile's action queues likewise, rows [H, H + QR)
    const int F = env_history(KS) ? env.frame_dim : 0, H = env_history(KS) ? D - F : 0;
    const int QR = env_perturb(KS) && env.act_delay ? env.max_delay : 0;
    const RolloutFastSmem L = rollout_fast_smem_layout(pd, M4, blockDim.x, WS, H + QR);
    const int ld = L.ld, S = L.slices;
    float* sX = smem + L.x;
    float* sActA = smem + L.acta;
    float* sActC = smem + L.actc;
    float* sPart = smem + L.part;
    float* sMean = smem + L.stat;
    float* sVar = sMean + Dp;
    float* sHist = smem + L.hist;
    float* sQ = sHist + (size_t)H * L.ld;
    const int tid = threadIdx.x;
    const float* __restrict__ Wbase = WS ? smem : a.pack;
    if (WS) {
        const float4* src = reinterpret_cast<const float4*>(a.pack);
        float4* dst = reinterpret_cast<float4*>(smem);
        for (int i = tid; i < pd.pack_fwd / 4; i += blockDim.x) dst[i] = src[i];
    }
    for (int d = tid; d < Dp; d += blockDim.x) {
        sMean[d] = (env.normalize && d < D) ? env.obs_mean[d] : 0.f;
        sVar[d] = (env.normalize && d < D) ? env.obs_var[d] : 1.f;
    }
    const bool norm_obs = env.normalize && env.norm_obs;
    const float ret_scale_var = env.normalize ? env.ret_stats[1] : 1.f;

    const long long n0 = (long long)blockIdx.x * M4;
    const int nvalid = (int)min((long long)M4, N - n0);
    const bool mine = tid < nvalid;
    const long long n = n0 + tid;
    const uint32_t gid = (uint32_t)(env.gid_offset + n);
    // per-env state in registers
    float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
    int steps = 0, ep_len = 0;
    float ep_ret = 0.f;
    uint32_t episode = 0;
    float eparam[DRIL_ENV_MAX_PARAMS] = {};   // parameter values of the running episode (ENV_KS_PARAMS)
    int dq = 0;                                // delay | ENV_DELAY_RESTART (ENV_KS_PERTURB)
    if (mine) {
#pragma unroll
        for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * N + n];
        steps = env.steps[n];
        episode = env.episode[n];
        if (env_has_params(KS)) env_load_params(env, n, eparam);
        if (env.monitor) { ep_ret = env.ep_ret[n]; ep_len = env.ep_len[n]; }
        for (int j = 0; j < H; ++j) sHist[(size_t)j * ld + tid] = env.hist[(size_t)j * N + n];
        if (QR > 0) {
            dq = env.act_delay[n];
            for (int j = 0; j < QR; ++j) sQ[(size_t)j * ld + tid] = env.act_q[(size_t)j * N + n];
        }
    }
    // output-layer split: thread (e = tid % M4, ks = tid / M4) covers k in [ks*Kc, ks*Kc + Kc)
    const LayerDesc& Lao = pd.L[0][NL - 1];
    const LayerDesc& Lco = pd.L[1][NL - 1];
    const int Kout = Lao.K;
    const int Kc = (Kout + S - 1) / S;
    const int oe = tid % M4, oks = tid / M4;
    const int A = pd.act_n;
    __syncthreads();

    // write the (normalised) observation of the register state into sX and optionally the buffer
    auto stage_obs = [&](float* obs_row /* nullable global [D] */) {
        if (env_history(KS)) {   // older frames straight from sHist, the newest from the registers: no D-wide register array
            if (tid < M4) {
                float f[ENV_MAX_FRAME] = {};
                if (mine) env_frame<KS>(env, st, f, EnvObsAt{n, episode - 1u, (uint32_t)steps});
                for (int j = 0; j < H; ++j) {
                    float x = mine ? sHist[(size_t)j * ld + tid] : 0.f;
                    if (mine && norm_obs) x = normalize_obs_val(x, sMean[j], sVar[j], env.eps, env.clip_obs);
                    if (obs_row) obs_row[j] = x;
                    sX[(size_t)j * ld + tid] = x;
                }
#pragma unroll
                for (int j = 0; j < ENV_MAX_FRAME; ++j) {
                    if (j < F) {
                        float x = f[j];
                        if (mine && norm_obs) x = normalize_obs_val(x, sMean[H + j], sVar[H + j], env.eps, env.clip_obs);
                        if (obs_row) obs_row[H + j] = x;
                        sX[(size_t)(H + j) * ld + tid] = x;
                    }
                }
                for (int j = D; j < Dp; ++j) sX[(size_t)j * ld + tid] = 0.f;
            }
            __syncthreads();
            return;
        }
        if (tid < M4) {
            float o[OW] = {};
            if (mine) {
#pragma unroll
                for (int b = 0; b < OW / 4; ++b) env_obs_block<KS>(env, st, b, o + 4 * b, eparam, EnvObsAt{n, episode - 1u, (uint32_t)steps});
                if (norm_obs) {
#pragma unroll
                    for (int j = 0; j < OW; ++j) if (j < D) o[j] = normalize_obs_val(o[j], sMean[j], sVar[j], env.eps, env.clip_obs);
                }
                if (obs_row) {
                    if (D == 4) *reinterpret_cast<float4*>(obs_row) = make_float4(o[0], o[1], o[2], o[3]);
                    else {
#pragma unroll
                        for (int j = 0; j < OW; ++j) if (j < D) obs_row[j] = o[j];
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < OW; ++j) if (j < Dp) sX[(size_t)j * ld + tid] = o[j];
        }
        __syncthreads();
    };
    // hidden layers (all but the output layer) of the selected nets; returns the buffer parity of the
    // last hidden activation (or -1 if the network has no hidden layer: the input is sX)
    auto hidden_forward = [&](int net_mask) -> int {
        const size_t bufsz = (size_t)pd.max_np * ld;
        for (int l = 0; l < NL - 1; ++l) {
            const float* ia = l == 0 ? sX : sActA + ((l - 1) & 1) * bufsz;
            const float* ic = l == 0 ? sX : sActC + ((l - 1) & 1) * bufsz;
            if (a.flags & RO_TILES_8X8)
                dense_layer_auto(pd, Wbase, l, ia, ic, sActA + (l & 1) * bufsz, sActC + (l & 1) * bufsz, M4, ld, net_mask);
            else
                dense_layer(pd, Wbase, l, ia, ic, sActA + (l & 1) * bufsz, sActC + (l & 1) * bufsz, M4, ld, net_mask);
            __syncthreads();
        }
        return NL >= 2 ? ((NL - 2) & 1) : -1;
    };
    // K-split partial sums of the output layers -> sPart[(ks*RF_MAX_OUT + j)*ld + e]; j < A actor, j == A critic
    auto output_partials = [&](int par, int net_mask) {
        const size_t bufsz = (size_t)pd.max_np * ld;
        const float* ha = par < 0 ? sX : sActA + par * bufsz;
        const float* hc = par < 0 ? sX : sActC + par * bufsz;
        if (oks < S) {
            float acc[RF_MAX_OUT];
#pragma unroll
            for (int j = 0; j < RF_MAX_OUT; ++j) acc[j] = 0.f;
            const int k0 = oks * Kc, k1 = min(Kout, k0 + Kc);
            const float* wa = Wbase + Lao.pw_off;
            const float* wc = Wbase + Lco.pw_off;
            if (A <= 2) {          // the common case (CartPole: 2 actions, Pendulum: 1 mean): no predicated-off work
                for (int k = k0; k < k1; ++k) {
                    if (net_mask & 1) {
                        const float h = ha[(size_t)k * ld + oe];
                        acc[0] = fmaf(h, wa[k * Lao.Np], acc[0]);
                        acc[1] = fmaf(h, wa[k * Lao.Np + 1], acc[1]);     // padded column (zero weights) when A == 1
                    }
                    if (net_mask & 2) acc[RF_MAX_OUT - 1] = fmaf(hc[(size_t)k * ld + oe], wc[k * Lco.Np], acc[RF_MAX_OUT - 1]);
                }
            } else {
                for (int k = k0; k < k1; ++k) {
                    if (net_mask & 1) {
                        const float h = ha[(size_t)k * ld + oe];
#pragma unroll
                        for (int j = 0; j < RF_MAX_OUT - 1; ++j) if (j < A) acc[j] = fmaf(h, wa[k * Lao.Np + j], acc[j]);
                    }
                    if (net_mask & 2) acc[RF_MAX_OUT - 1] = fmaf(hc[(size_t)k * ld + oe], wc[k * Lco.Np], acc[RF_MAX_OUT - 1]);
                }
            }
#pragma unroll
            for (int j = 0; j < RF_MAX_OUT - 1; ++j) if (j < A) sPart[((size_t)oks * RF_MAX_OUT + j) * ld + oe] = acc[j];
            sPart[((size_t)oks * RF_MAX_OUT + RF_MAX_OUT - 1) * ld + oe] = acc[RF_MAX_OUT - 1];
        }
        __syncthreads();
    };
    auto reduce_out = [&](int j, int which /*0 actor j, 1 critic*/) -> float {
        const int jj = which ? RF_MAX_OUT - 1 : j;
        float s = 0.f;
        for (int ks = 0; ks < S; ++ks) s += sPart[((size_t)ks * RF_MAX_OUT + jj) * ld + tid];
        return s + (which ? Wbase[Lco.pb_off] : Wbase[Lao.pb_off + j]);
    };

    for (int t = 0; t < a.T; ++t) {
        const size_t row = (size_t)t * N;
        stage_obs(mine ? buf.obs + (row + n) * D : nullptr);
        const int par = hidden_forward(3);
        output_partials(par, 3);
        int trunc_i = 0;
        float tobs[OW] = {};
        if (mine) {
            const float value = reduce_out(0, 1);
            float z[RF_MAX_OUT - 1];
#pragma unroll
            for (int j = 0; j < RF_MAX_OUT - 1; ++j) z[j] = j < A ? reduce_out(j, 0) : -INFINITY;
            float logp;
            int a_disc = 0;
            float a_cont = 0.f;
            if (pd.act_kind == DRIL_ACT_DISCRETE) {
                float m = z[0];
#pragma unroll
                for (int j = 1; j < RF_MAX_OUT - 1; ++j) if (j < A) m = fmaxf(m, z[j]);
                float ex[RF_MAX_OUT - 1];
                float ssum = 0.f;
#pragma unroll
                for (int j = 0; j < RF_MAX_OUT - 1; ++j) { ex[j] = j < A ? expf(z[j] - m) : 0.f; if (j < A) ssum += ex[j]; }
                int idx = A - 1;
                if (a.forced) {
                    idx = reinterpret_cast<const int*>(a.forced)[row + n] - pd.act_start;
                    idx = idx < 0 ? 0 : (idx >= A ? A - 1 : idx);
                } else {
                    uint32_t x[4];
                    philox4x32(gid, a.step0 + (uint32_t)t, 0u, DRIL_TAG_SAMPLE, a.pseed, x);
                    const double u = u01_f64(x[0], x[1]);
                    float cum = 0.f;
                    bool found = false;
#pragma unroll
                    for (int j = 0; j < RF_MAX_OUT - 1; ++j) {
                        if (j < A) {
                            cum += ex[j] / ssum;                 // fp32 cumsum vs Float64 u (categorical.jl:45-47)
                            if (!found && (double)cum >= u) { idx = j; found = true; }
                        }
                    }
                }
                float pe = ex[0];
#pragma unroll
                for (int j = 1; j < RF_MAX_OUT - 1; ++j) if (j == idx) pe = ex[j];
                logp = logf(pe / ssum);
                a_disc = idx + pd.act_start;
                reinterpret_cast<int*>(buf.actions)[row + n] = a_disc;
            } else {
                float ls_sum = 0.f, dss = 0.f;
#pragma unroll
                for (int j = 0; j < RF_MAX_OUT - 1; ++j) {
                    if (j < A) {
                        const float mean = z[j];
                        const float ls = a.flat[pd.log_std_off + j];
                        float act;
                        if (a.forced) act = reinterpret_cast<const float*>(a.forced)[(row + n) * A + j];
                        else act = __fadd_rn(mean, __fmul_rn(expf(ls), sample_normal(gid, a.step0 + (uint32_t)t, j, a.pseed)));
                        const float diff = act - mean;
                        dss += diff * diff * expf(-2.0f * ls);
                        ls_sum += ls;
                        reinterpret_cast<float*>(buf.actions)[(row + n) * A + j] = act;          // raw, unclamped (trajectory.jl:48)
                        if (j == 0) a_cont = fminf(fmaxf(act, pd.act_low[0]), pd.act_high[0]);    // ClampAdapter
                    }
                }
                logp = -0.5f * (2.0f * ls_sum + dss + (float)A * DRIL_LOG2PI);
            }
            buf.values[row + n] = value;
            buf.logprobs[row + n] = logp;
            // env step + monitor + auto-reset
            bool term = false;
            float r;
            uint32_t life = 0;
            if (env_history(KS)) {                               // the frame the action was chosen on enters the history
                float f[ENV_MAX_FRAME];
                env_frame<KS>(env, st, f, EnvObsAt{n, episode - 1u, (uint32_t)steps});
                env_hist_push(sHist + tid, (size_t)ld, H, F, f);
            }
            if (QR > 0) {                                        // the action chosen d steps earlier
                const float ad = env_delay_action(&dq, sQ + tid, (size_t)ld, pd.act_kind == DRIL_ACT_DISCRETE ? (float)a_disc : a_cont);
                if (pd.act_kind == DRIL_ACT_DISCRETE) a_disc = (int)ad; else a_cont = ad;
            }
            r = env_step<KS & ~(1u << DRIL_ENV_SYNTHETIC)>(env, st, n, a_disc, &a_cont, &life, &term, eparam);   // (no synthetic env here)
            steps += 1;
            const bool trunc = steps >= env.max_steps;
            const bool done = term || trunc;
            buf.flags[row + n] = (unsigned char)((term ? 1 : 0) | (trunc ? 2 : 0));
            float rn = r;
            if (env.normalize && env.norm_reward) {              // eval-mode normaliser: frozen statistics
                rn = __fdiv_rn(r, __fsqrt_rn(__fadd_rn(ret_scale_var, env.eps)));
                rn = fminf(fmaxf(rn, -env.clip_reward), env.clip_reward);
            }
            buf.rewards[row + n] = rn;
            if (env.monitor) {
                ep_ret = __fadd_rn(ep_ret, r);
                ep_len += 1;
                if (done) {
                    buf.episode_r[row + n] = ep_ret;
                    buf.episode_l[row + n] = ep_len;
                    atomicAdd(&buf.done_count[t], 1);
                    atomicAdd(&env.roll_sums[0], (double)ep_ret);
                    atomicAdd(&env.roll_sums[1], (double)ep_len);
                    atomicAdd(env.roll_eps, 1ull);
                    ep_ret = 0.f; ep_len = 0;
                }
            }
            if (trunc && env_history(KS)) {   // the stack ending in the ended episode's final frame, staged like ENV_KS_OBS_PARAMS
                trunc_i = 1;
                float f[ENV_MAX_FRAME];
                env_frame<KS>(env, st, f, EnvObsAt{n, episode - 1u, (uint32_t)steps});
                for (int j = 0; j < H; ++j) {
                    float x = sHist[(size_t)j * ld + tid];
                    if (norm_obs) x = normalize_obs_val(x, sMean[j], sVar[j], env.eps, env.clip_obs);
                    sX[(size_t)j * ld + tid] = x;
                }
#pragma unroll
                for (int j = 0; j < ENV_MAX_FRAME; ++j) {
                    if (j < F) {
                        float x = f[j];
                        if (norm_obs) x = normalize_obs_val(x, sMean[H + j], sVar[H + j], env.eps, env.clip_obs);
                        sX[(size_t)(H + j) * ld + tid] = x;
                    }
                }
            } else if (trunc) {
                trunc_i = 1;
#pragma unroll
                for (int b = 0; b < OW / 4; ++b)   // before the redraw below
                    env_obs_block<KS>(env, st, b, tobs + 4 * b, eparam, EnvObsAt{n, episode - 1u, (uint32_t)steps});
                if (norm_obs) {
#pragma unroll
                    for (int j = 0; j < OW; ++j) if (j < D) tobs[j] = normalize_obs_val(tobs[j], sMean[j], sVar[j], env.eps, env.clip_obs);
                }
                if (env_obs_params(KS)) {   // staged now (this step's forward has read sX): 12 components live across the redraw
#pragma unroll                             // and the barrier would spill
                    for (int j = 0; j < OW; ++j) if (j < Dp) sX[(size_t)j * ld + tid] = tobs[j];
                }
            }
            if (done) {
                env_reset_state<KS>(env.kind, gid, episode, env.seed, st);
                if (env_has_params(KS)) env_draw_params(env, n, gid, episode, eparam);
                if (env_history(KS)) {
                    float f[ENV_MAX_FRAME];
                    env_frame<KS>(env, st, f, EnvObsAt{n, episode, 0u});
                    env_hist_fill(sHist + tid, (size_t)ld, H, F, f);
                }
                if (env_perturb(KS)) dq |= ENV_DELAY_RESTART;
                episode += 1;
                steps = 0;
                if (env.normalize) env.ret[n] = 0.f;             // normalizeWrapperEnv.jl:153-156
            }
        }
        // V(terminal_obs) for truncated envs (trajectory.jl:57-61): rare, CTA-uniform branch
        if (__syncthreads_or(trunc_i)) {
            if (tid < M4 && env_history(KS)) {
                if (!trunc_i) for (int j = 0; j < Dp; ++j) sX[(size_t)j * ld + tid] = 0.f;
            } else if (tid < M4) {
#pragma unroll
                for (int j = 0; j < OW; ++j)
                    if (j < Dp && !(env_obs_params(KS) && trunc_i)) sX[(size_t)j * ld + tid] = trunc_i ? tobs[j] : 0.f;
            }
            __syncthreads();
            const int p2 = hidden_forward(2);
            output_partials(p2, 2);
            if (mine && trunc_i) buf.boot[row + n] = reduce_out(0, 1);
            __syncthreads();
        }
    }
    // V(new_obs) after the final step (trajectory.jl:65-70)
    if (a.T > 0) {
        stage_obs(nullptr);
        const int p2 = hidden_forward(2);
        output_partials(p2, 2);
        if (mine) buf.last_values[n] = reduce_out(0, 1);
    }
    if (mine) {
#pragma unroll
        for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) env.state[(size_t)k * N + n] = st[k];
        env.steps[n] = steps;
        env.episode[n] = episode;
        if (env.monitor) { env.ep_ret[n] = ep_ret; env.ep_len[n] = ep_len; }
        for (int j = 0; j < H; ++j) env.hist[(size_t)j * N + n] = sHist[(size_t)j * ld + tid];
        if (QR > 0) {
            env.act_delay[n] = dq;
            for (int j = 0; j < QR; ++j) env.act_q[(size_t)j * N + n] = sQ[(size_t)j * ld + tid];
        }
    }
}

// the observation history of every env restarted from its current state (ENV_KS_HISTORY): reset, set_state, Scaling turned
// on, or the history turned on
__global__ void env_hist_fill_kernel(EnvDev env) {
    long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= env.n_envs) return;
    float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * env.n_envs + n];
    float f[ENV_MAX_FRAME];
    env_frame<ENV_KS_ALL>(env, st, f);
    env_hist_fill(env.hist + n, (size_t)env.n_envs, (env.hist_len - 1) * env.frame_dim, env.frame_dim, f);
}

// the action queues of every env restarted, and its observation history refilled from its current (noisy) frame
// (ENV_KS_PERTURB): reset, set_state, Scaling changed, or delays / the history set
__global__ void env_perturb_restart_kernel(EnvDev env) {
    constexpr unsigned KS = ENV_KS_ALL | ENV_KS_PARAMS | ENV_KS_PERTURB;
    long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= env.n_envs) return;
    if (env.act_delay) env.act_delay[n] |= ENV_DELAY_RESTART;
    if (!env.hist) return;
    float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) st[k] = env.state[(size_t)k * env.n_envs + n];
    float f[ENV_MAX_FRAME];
    env_frame<KS>(env, st, f, env_obs_at<KS>(env, n));
    env_hist_fill(env.hist + n, (size_t)env.n_envs, (env.hist_len - 1) * env.frame_dim, env.frame_dim, f);
}

// ---------------------------------------------------------------------------------------
// Stand-alone layer application on an arbitrary batch (compat / evaluation path):
//   mode 0: sample (layer call, layer_forward.jl:3-39)    mode 1: deterministic (mode.(ds))
//   mode 2: evaluate_actions (layer_methods.jl:28-55)     mode 3: predict_values (:57-61)
// ---------------------------------------------------------------------------------------
struct ApplyArgs {
    PolicyDesc pd;
    const float* pack;
    const float* flat;
    const float* obs;        // [B][D]
    const void* actions_in;  // mode 2
    const long long* gids;   // optional sample-stream ids
    void* actions_out;       // int32 [B] | float [B][A]
    float *values, *logprobs, *entropy;
    long long B;
    unsigned long long pseed;
    unsigned int step;
    int mode, M4, weights_smem;
};

template <bool WS>
__global__ void __launch_bounds__(DRIL_THREADS) policy_apply_kernel(const __grid_constant__ ApplyArgs a) {
    extern __shared__ float4 smem4[];
    float* smem = reinterpret_cast<float*>(smem4);
    const PolicyDesc& pd = a.pd;
    const int D = pd.obs_dim, Dp = pd.obs_dim_p, M4 = a.M4, ld = M4 + 4;
    float* sX = smem + (WS ? pd.pack_fwd : 0);
    float* sActA = sX + (size_t)Dp * ld;
    float* sActC = sActA + (size_t)2 * pd.max_np * ld;
    const int tid = threadIdx.x;
    const float* __restrict__ Wbase = WS ? smem : a.pack;
    if (WS) {
        const float4* src = reinterpret_cast<const float4*>(a.pack);
        float4* dst = reinterpret_cast<float4*>(smem);
        for (int i = tid; i < pd.pack_fwd / 4; i += blockDim.x) dst[i] = src[i];
    }
    const long long n_tiles = (a.B + M4 - 1) / M4;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        long long n0 = tile * M4;
        int nvalid = (int)min((long long)M4, a.B - n0);
        __syncthreads();
        for (int i = tid; i < Dp * M4; i += blockDim.x) {
            int e = i / Dp, d = i - e * Dp;
            sX[(size_t)d * ld + e] = (e < nvalid && d < D) ? a.obs[(size_t)(n0 + e) * D + d] : 0.f;
        }
        __syncthreads();
        int fin = mlp_forward_pingpong(pd, Wbase, sX, sActA, sActC, M4, ld, a.mode == 3 ? 2 : 3);
        if (tid < nvalid) {
            long long n = n0 + tid;
            float value = sActC[(size_t)fin * pd.max_np * ld + tid];
            if (a.values) a.values[n] = value;
            if (a.mode != 3) {
                const float* z = sActA + (size_t)fin * pd.max_np * ld + tid;
                uint32_t gid = (uint32_t)(a.gids ? a.gids[n] : n);
                float logp, ent;
                if (pd.act_kind == DRIL_ACT_DISCRETE) {
                    int mode = a.mode == 0 ? 0 : (a.mode == 1 ? 1 : 2);
                    double u = 0.0;
                    int forced_v = 0;
                    if (mode == 0) {
                        uint32_t x[4];
                        philox4x32(gid, a.step, 0u, DRIL_TAG_SAMPLE, a.pseed, x);
                        u = u01_f64(x[0], x[1]);
                    } else if (mode == 2) forced_v = reinterpret_cast<const int*>(a.actions_in)[n];
                    HeadOut h = categorical_head(z, ld, pd.act_n, pd.act_start, mode, u, forced_v, a.entropy != nullptr);
                    logp = h.logp; ent = h.entropy;
                    if (a.actions_out) reinterpret_cast<int*>(a.actions_out)[n] = h.action_idx;
                } else {
                    const int A = pd.act_n;
                    float ls_sum = 0.f, dss = 0.f;
                    for (int j = 0; j < A; ++j) {
                        float mean = z[(size_t)j * ld];
                        float ls = a.flat[pd.log_std_off + j];
                        float act;
                        if (a.mode == 2) act = reinterpret_cast<const float*>(a.actions_in)[n * A + j];
                        else if (a.mode == 1) act = mean;
                        else act = __fadd_rn(mean, __fmul_rn(expf(ls), sample_normal(gid, a.step, j, a.pseed)));
                        float diff = act - mean;
                        dss += diff * diff * expf(-2.0f * ls);
                        ls_sum += ls;
                        if (a.actions_out) reinterpret_cast<float*>(a.actions_out)[n * A + j] = act;
                    }
                    logp = -0.5f * (2.0f * ls_sum + dss + (float)A * DRIL_LOG2PI);
                    ent = 0.5f * (float)A * (1.0f + DRIL_LOG2PI) + ls_sum;
                }
                if (a.logprobs) a.logprobs[n] = logp;
                if (a.entropy) a.entropy[n] = ent;
            }
        }
    }
}

// env reset (reset!(env)): new episode for every env, monitor/normaliser accumulators zeroed (and, for KS with ENV_KS_PARAMS,
// the new episode's parameter values drawn).
template <unsigned KS>
__global__ void env_reset_kernel(EnvDev env) {
    long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= env.n_envs) return;
    float st[ENV_MAX_STATE] = {0.f, 0.f, 0.f, 0.f};
    uint32_t ep = env.episode[n];
    env_reset_state<ENV_KS_ALL>(env.kind, (uint32_t)(env.gid_offset + n), ep, env.seed, st);
    if (env_has_params(KS)) {
        float par[DRIL_ENV_MAX_PARAMS];
        env_draw_params(env, n, (uint32_t)(env.gid_offset + n), ep, par);
    }
    env.episode[n] = ep + 1;
#pragma unroll
    for (int k = 0; k < ENV_MAX_STATE; ++k) if (k < env.state_dim) env.state[(size_t)k * env.n_envs + n] = st[k];
    env.steps[n] = 0;
    if (env.monitor) { env.ep_ret[n] = 0.f; env.ep_len[n] = 0; }
    if (env.normalize) env.ret[n] = 0.f;
}

// new ranges (dril_env_set_params): the running episode takes the values its own (gid, episode) draws from them
__global__ void env_params_draw_kernel(EnvDev env) {
    long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= env.n_envs) return;
    float par[DRIL_ENV_MAX_PARAMS];
    env_draw_params(env, n, (uint32_t)(env.gid_offset + n), env.episode[n] - 1u, par);
}
