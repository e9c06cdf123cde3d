// Tensor-core variant of the fused rollout for the reference's default CartPole setup (hidden_dims = [64, 64],
// Discrete(<= 2), obs_dim = 4, no normaliser): the n_steps loop of collect_trajectories (buffers/trajectory.jl:25-73,
// rollout_buffer.jl:46-90) with the actor's 64x64 layer on tcgen05.mma (3xTF32, same split as update_tc.cuh).
//
// The per-step chain (observe -> actor -> sample -> dynamics) is latency bound, so it is cut to the minimum:
//  * only the ACTOR runs inside the step loop.  Values are not needed to choose actions: V(s_t), the bootstrap value of
//    the final observation and V(terminal_obs) of truncated steps (trajectory.jl:57-70) are computed afterwards in one
//    batched tensor-core pass over all n_steps x n_envs observations (critic_values_tc_kernel);
//  * 32 envs per CTA (128 CTAs for 4096 envs), sixteen threads per env (warp w owns hidden features 4w..4w+3 of all 32
//    envs, its slices of W0/b0/b1/W2 stay in registers) that all keep the env state in registers.  A warp can only
//    reach the TMEM lane quadrant warp % 4, which is also its scheduler, so both MMA operands come from shared memory
//    (SS mode) and only four warps copy the 32x64 accumulator back to shared memory: the CUDA-core work is spread over
//    all four schedulers instead of one;
//  * everything that does not depend on the sampled action is done while the MMAs run, one role per warp: the Euler step
//    for BOTH pushes (in CartPole the new positions, the termination test and the reset are action independent, only
//    the two velocities differ), the Philox uniform, the start state of the env's next episode, the correctly rounded
//    fp64 sin/cos of the next pole angle (one step ahead), and the buffer/monitor bookkeeping of the previous step.
//    After the logits only softmax -> compare -> select remains;
//  * per step: layer 0 (K = 4) on CUDA cores -> hi/lo to TMEM -> 24 tcgen05.mma (M = 128 rows, 64 used; N = 64; K = 8)
//    -> tanh + output layer partials -> softmax, Philox inverse-CDF sample, log-prob, dynamics, monitor, auto-reset.
#pragma once
#include "rollout.cuh"
#include <cuda_fp16.h>
#include "update_tc.cuh"

#define RT_ENVS 32
#define RT_THREADS 512
#define RT_COL_D 0
#define RT_COL_HI 64
#define RT_COL_LO 128
#define RT_TMEM_COLS 64
#define RT_OFF_WT_HI 0           // W1^T hi / lo, K-major no-swizzle images (B operand)
#define RT_OFF_WT_LO 16384
// rollout kernel: H0 hi / lo as K-major no-swizzle A operand images.  The M = 64 instruction reads 8 row groups
// (16 KB) from each base but only rows 0..31 (8 KB) hold envs: the images are packed 8 KB apart and the reads of the
// unused rows run over whatever follows (their accumulator rows are never read).
#define RT_OFF_A_HI 32768
#define RT_OFF_A_LO 40960
#define RT_OFF_SMALL 49152
#define RT_SMALL_FLOATS 4096
#define RT_SMEM_BYTES (RT_OFF_SMALL + RT_SMALL_FLOATS * 4 + 1024)   // the M = 64 instruction reads 8 row groups (16 KB) per image
#define CV_OFF_SMALL 32768       // critic kernel: small arrays right after the W1 images
#define CV_SMALL_FLOATS 1024
#define CV_SMEM_BYTES (CV_OFF_SMALL + CV_SMALL_FLOATS * 4 + 1024)

struct TcRolloutScratch {
    float* last_obs;          // [N][4] observation after the final step
    float* trunc_obs;         // [cap][4] terminal observations of truncated steps
    long long* trunc_idx;     // [cap] buffer sample index of each entry
    unsigned int* trunc_count;
    unsigned int cap;
};

#ifdef TC_TRACE
__device__ long long g_rt_trace[4][8][8];     // [feature quarter][step - 8][point], CTA 0, lane 0 of the quarter's first warp
#define RT_MARK(pt) do { if (blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 5 || warp == 6 || warp == 7) && t >= 8 && t < 16) g_rt_trace[warp == 0 ? 0 : warp - 4][t - 8][pt] = clock64(); } while (0)
#else
#define RT_MARK(pt) do { } while (0)
#endif
__device__ __forceinline__ void rt_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float* r) {
    uint32_t u[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]), "=r"(u[9]),
                   "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = __uint_as_float(u[j]);
}


// fp16 split used by the rollout kernel's MMAs: x = hi + lo with hi = fp16(x), lo = fp16(x - hi) (22 significant bits;
// fp16 subnormals keep tiny values to an absolute 3e-8).  Safe here because both operands are bounded: H0 = tanh(.)
// and the layer weights (|w| < 65504).  Products hi*hi + lo*hi + hi*lo on kind::f16 with fp32 accumulation: K = 16 per
// instruction, i.e. half the instructions of the 3xTF32 scheme at the same accuracy.
__device__ __forceinline__ void rt_split_f16(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}
// [R][C] fp16 matrix in the no-swizzle K-major core layout: cores of 8 rows x 8 columns (16-byte rows), ordered [r/8][c/8]
__device__ __forceinline__ int rt_core_index_f16(int r, int c, int C) { return ((r >> 3) * (C >> 3) + (c >> 3)) * 64 + (r & 7) * 8 + (c & 7); }
__device__ __forceinline__ void rt_stage_w1_f16(const float* __restrict__ pack, const LayerDesc& L1, unsigned char* sm, int tid, int nthreads) {
    __half* hi_img = reinterpret_cast<__half*>(sm + RT_OFF_WT_HI);
    __half* lo_img = reinterpret_cast<__half*>(sm + RT_OFF_WT_LO);
    for (int i = tid; i < 64 * 64; i += nthreads) {
        const int k = i >> 6, n = i & 63;
        __half hi, lo;
        rt_split_f16(pack[L1.pw_off + i], hi, lo);
        hi_img[rt_core_index_f16(n, k, 64)] = hi;
        lo_img[rt_core_index_f16(n, k, 64)] = lo;
    }
}
__device__ __forceinline__ void rt_mma_f16_ss(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d),
                 "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}

// MINB = 2: register budget of two resident CTAs per SM (64 registers per thread): used when every SM has at least two tiles, so
// that two per-step latency chains overlap (throughput regime, C4); MINB = 1 keeps the shortest chain for one tile per SM (C2)
template <int MINB>
__global__ void __launch_bounds__(RT_THREADS, MINB) rollout_tc_kernel(const __grid_constant__ RolloutArgs a, const TcRolloutScratch sc) {
    extern __shared__ __align__(1024) unsigned char rt_smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    const EnvDev& env = a.env;
    const BufDev& buf = a.buf;
    const PolicyDesc& pd = a.pd;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int lane = tid & 31;
    const uint32_t raw = tc_smem_u32(rt_smem_raw);
    const uint32_t sm_base = (raw + 1023u) & ~1023u;
    unsigned char* sm = rt_smem_raw + (sm_base - raw);
    __half* sAhi = reinterpret_cast<__half*>(sm + RT_OFF_A_HI);
    __half* sAlo = reinterpret_cast<__half*>(sm + RT_OFF_A_LO);
    float* sSmall = reinterpret_cast<float*>(sm + RT_OFF_SMALL);
    float* sD = sSmall;                 // [32][68] pre-activations of the hidden layer (copied out of TMEM)
    float* sPart = sD + 32 * 68;        // [16 feature groups][32][2] partial logits
    float* sCand = sPart + 1024;        // [32][8] next-state candidates: xn, thn, xd(0), thd(0), xd(1), thd(1)
    float* sReset = sCand + 256;        // [32][8] state of the env's next episode + sin/cos of its pole angle
    float* sSCn = sReset + 256;         // [32][2] sin/cos of the next pole angle if the episode continues
    double* sU = reinterpret_cast<double*>(sSCn + 64);   // [32] uniform of the step's action sample
    float* sState = reinterpret_cast<float*>(sU + 32);   // [32][4] current env state (owned by the decision warp)
    float* sSCcur = sState + 128;       // [32][2] sin/cos of the current pole angle
    int* sNeed = reinterpret_cast<int*>(sSCcur + 64);    // [32] episode whose start state must be prepared, or -1
    const LayerDesc& L0 = pd.L[0][0];
    const LayerDesc& L1 = pd.L[0][1];
    const LayerDesc& L2 = pd.L[0][2];
    rt_stage_w1_f16(a.pack, L1, sm, tid, RT_THREADS);
    const int e = lane;                               // env slot == row of the MMA == TMEM lane
    const int fg = warp, f0 = fg * 4;                 // this thread's 4 hidden features
    // this thread's slices of the thin layers live in registers for the whole rollout
    float w0r[4][4], b0r[4], b1r[4], w2r[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int d = 0; d < 4; ++d) w0r[d][j] = a.pack[L0.pw_off + d * 64 + f0 + j];
        b0r[j] = a.pack[L0.pb_off + f0 + j];
        b1r[j] = a.pack[L1.pb_off + f0 + j];
        w2r[j][0] = a.pack[L2.pw_off + (f0 + j) * 4];
        w2r[j][1] = a.pack[L2.pw_off + (f0 + j) * 4 + 1];
    }
    const float b2_0 = a.pack[L2.pb_off], b2_1 = a.pack[L2.pb_off + 1];
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(RT_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);
    const uint32_t idesc = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(64 >> 4) << 24);   // kind::f16: F16 x F16 -> F32, M = 64, N = 64, K-major
    const long long N = env.n_envs;
    const int A = pd.act_n;
    const float TAU = 0.02f;
    const int a_off = rt_core_index_f16(e, f0, 64);                // K-major no-swizzle core layout: row e, columns f0..f0+3 (8 bytes)
    // roles in the MMA window (warps on different schedulers)
    const bool r_cand = warp == 10, r_philox = warp == 2, r_reset = warp == 3, r_sin = warp == 7, r_cos = warp == 11, r_dec = warp == 6;
    // M = 64: accumulator row i sits in TMEM lane 32 * (i / 16) + i % 16, so envs 0..15 are in quadrant 0 (warps 0, 4, 8, 12)
    // and envs 16..31 in quadrant 1 (warps 1, 5, 9, 13), lanes 0..15 of each
    const bool r_copy = (warp & 3) < 2;
    uint32_t nbar = 0;
    for (long long tile = blockIdx.x; tile * RT_ENVS < N; tile += gridDim.x) {
        const long long n = tile * RT_ENVS + e;
        const bool mine = n < N;
        const uint32_t gid = (uint32_t)(env.gid_offset + n);
        // the decision warp owns the env: state, counters, monitor accumulators; everybody else reads sState
        float st[4] = {0.f, 0.f, 0.f, 0.f};
        int steps = 0, ep_len = 0;
        float ep_ret = 0.f;
        uint32_t episode = 0;
        struct Pending { float pe, ssum, ep_ret; float4 tobs; int idx, ep_len, t; bool term, trunc, live; } pend;
        pend.live = false; pend.pe = pend.ssum = 1.f; pend.ep_ret = 0.f; pend.tobs = make_float4(0.f, 0.f, 0.f, 0.f);
        pend.idx = 0; pend.ep_len = 0; pend.t = 0; pend.term = pend.trunc = false;
        // bookkeeping of a finished step (log-prob, buffer row, monitor, truncation list): done one step late, while the
        // next step's MMAs run, so that it is off the per-step critical path
        auto flush = [&]() {
            if (!pend.live) return;
            const size_t r = (size_t)pend.t * N + n;
            reinterpret_cast<int*>(buf.actions)[r] = pend.idx + pd.act_start;
            buf.logprobs[r] = A == 1 ? 0.f : logf(pend.pe / pend.ssum);
            buf.flags[r] = (unsigned char)((pend.term ? 1 : 0) | (pend.trunc ? 2 : 0));
            buf.rewards[r] = 1.0f;
            if (env.monitor && (pend.term || pend.trunc)) {
                buf.episode_r[r] = pend.ep_ret;
                buf.episode_l[r] = pend.ep_len;
                atomicAdd(&buf.done_count[pend.t], 1);
                atomicAdd(&env.roll_sums[0], (double)pend.ep_ret);
                atomicAdd(&env.roll_sums[1], (double)pend.ep_len);
                atomicAdd(env.roll_eps, 1ull);
            }
            if (pend.trunc) {                                             // V(terminal_obs) is evaluated by the critic pass
                const unsigned int k = atomicAdd(sc.trunc_count, 1u);
                if (k < sc.cap) {
                    *reinterpret_cast<float4*>(sc.trunc_obs + (size_t)k * 4) = pend.tobs;
                    sc.trunc_idx[k] = (long long)r;
                }
            }
            pend.live = false;
        };
        if (r_dec) {
            if (mine) {
#pragma unroll
                for (int k = 0; k < 4; ++k) st[k] = env.state[(size_t)k * N + n];
                steps = env.steps[n];
                episode = env.episode[n];
                if (env.monitor) { ep_ret = env.ep_ret[n]; ep_len = env.ep_len[n]; }
            }
            float s_, c_;
            sincos_rn(st[2], &s_, &c_);
            *reinterpret_cast<float4*>(sState + e * 4) = make_float4(st[0], st[1], st[2], st[3]);
            *reinterpret_cast<float2*>(sSCcur + e * 2) = make_float2(s_, c_);
            sNeed[e] = (int)episode;
        }
        __syncthreads();
        for (int t = 0; t < a.T; ++t) {
            const size_t row = (size_t)t * N;
            RT_MARK(0);
            const float4 s4 = *reinterpret_cast<const float4*>(sState + e * 4);
            // ---- layer 0 (own 4 features) -> hi/lo -> A operand images in shared memory -----------------------------------
            {
                __half hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float h = fmaf(s4.w, w0r[3][j], fmaf(s4.z, w0r[2][j], fmaf(s4.y, w0r[1][j], fmaf(s4.x, w0r[0][j], b0r[j]))));
                    rt_split_f16(fast_tanh(h), hi[j], lo[j]);
                }
                __half2 h01 = __halves2half2(hi[0], hi[1]), h23 = __halves2half2(hi[2], hi[3]);
                __half2 l01 = __halves2half2(lo[0], lo[1]), l23 = __halves2half2(lo[2], lo[3]);
                uint2 uh, ul;
                uh.x = *reinterpret_cast<uint32_t*>(&h01); uh.y = *reinterpret_cast<uint32_t*>(&h23);
                ul.x = *reinterpret_cast<uint32_t*>(&l01); ul.y = *reinterpret_cast<uint32_t*>(&l23);
                *reinterpret_cast<uint2*>(sAhi + a_off) = uh;
                *reinterpret_cast<uint2*>(sAlo + a_off) = ul;
            }
            RT_MARK(1);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            // ---- H1pre = H0 W1 on the tensor cores (both operands from shared memory) ---------------------------------------
            if (warp == 0 && tc_elect_one()) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int ps = 0; ps < 3; ++ps) {
                    const uint32_t aimg = sm_base + (ps == 1 ? RT_OFF_A_LO : RT_OFF_A_HI);
                    const uint32_t bimg = sm_base + (ps == 2 ? RT_OFF_WT_LO : RT_OFF_WT_HI);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)          // K = 16 per instruction: two 16-byte cores, 128 B apart; row groups 1 KB apart
                        rt_mma_f16_ss(tb + RT_COL_D, tc_desc(aimg + kk * 256, 128, 1024, 0), tc_desc(bimg + kk * 256, 128, 1024, 0), idesc,
                                      (ps | kk) ? 1u : 0u);
                }
                tc_commit(&bar);
            }
            RT_MARK(2);
            // ---- while the MMAs run: everything that does not depend on the action, one role per warp --------------------
            if (r_cand) {
                // Euler step for BOTH pushes: positions, termination and the reset do not depend on the action
                const float2 scv = *reinterpret_cast<const float2*>(sSCcur + e * 2);
                constexpr EnvParams D = env_param_default(DRIL_ENV_CARTPOLE);
                const CartPoleCoef C = cartpole_coef(D.v);
                float s0[4] = {s4.x, s4.y, s4.z, s4.w}, s1[4] = {s4.x, s4.y, s4.z, s4.w};
                bool t0, t1;
                cartpole_step_sc(s0, 0, scv.x, scv.y, C, &t0);
                cartpole_step_sc(s1, 1, scv.x, scv.y, C, &t1);
                *reinterpret_cast<float4*>(sCand + e * 8) = make_float4(s0[0], s0[2], s0[1], s0[3]);     // xn, thn, xd(0), thd(0)
                *reinterpret_cast<float2*>(sCand + e * 8 + 4) = make_float2(s1[1], s1[3]);              // xd(1), thd(1)
            } else if (r_philox) {
                uint32_t x[4];
                philox4x32(gid, a.step0 + (uint32_t)t, 0u, DRIL_TAG_SAMPLE, a.pseed, x);
                sU[e] = u01_f64(x[0], x[1]);
            } else if (r_reset) {
                const int ep = sNeed[e];
                if (ep >= 0) {                            // start state of the env's next episode and sin/cos of its pole angle
                    float rs[4], s_, c_;
                    env_reset_state(env.kind, gid, (uint32_t)ep, env.seed, rs);
                    sincos_rn(rs[2], &s_, &c_);
                    *reinterpret_cast<float4*>(sReset + e * 8) = make_float4(rs[0], rs[1], rs[2], rs[3]);
                    *reinterpret_cast<float2*>(sReset + e * 8 + 4) = make_float2(s_, c_);
                }
            } else if (r_sin || r_cos) {
                // correctly rounded sin / cos of the next pole angle (if no reset); the two fp64 evaluations are dependent
                // chains of slow instructions, so they run on two warps
                const double th = (double)__fadd_rn(s4.z, __fmul_rn(TAU, s4.w));
                sSCn[e * 2 + (r_cos ? 1 : 0)] = (float)(r_cos ? cos(th) : sin(th));
            } else if (r_dec) {
                if (mine) *reinterpret_cast<float4*>(buf.obs + (row + n) * 4) = s4;
                flush();
            }
            RT_MARK(3);
            // ---- warps 0/4/8/12 copy the accumulator (16 columns each) out of TMEM -----------------------------------------
            if (r_copy) {
                tc_wait(&bar, nbar & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                float d[16];
                const int c0 = (warp >> 2) * 16, qd = warp & 3;
                tc_ld16(tb + ((uint32_t)(qd * 32) << 16) + RT_COL_D + c0, d);
                if (lane < 16) {
                    float* dst = sD + (qd * 16 + lane) * 68 + c0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(d[j], d[j + 1], d[j + 2], d[j + 3]);
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            }
            ++nbar;
            RT_MARK(4);
            __syncthreads();
            // ---- H1 = tanh(. + b1), partial logits over the own 4 features --------------------------------------------------
            {
                const float4 z = *reinterpret_cast<const float4*>(sD + e * 68 + f0);
                const float h0 = fast_tanh(z.x + b1r[0]), h1 = fast_tanh(z.y + b1r[1]), h2 = fast_tanh(z.z + b1r[2]), h3 = fast_tanh(z.w + b1r[3]);
                const float p0 = fmaf(h3, w2r[3][0], fmaf(h2, w2r[2][0], fmaf(h1, w2r[1][0], h0 * w2r[0][0])));
                const float p1 = fmaf(h3, w2r[3][1], fmaf(h2, w2r[2][1], fmaf(h1, w2r[1][1], h0 * w2r[0][1])));
                *reinterpret_cast<float2*>(sPart + (fg * 32 + e) * 2) = make_float2(p0, p1);
            }
            RT_MARK(5);
            __syncthreads();
            RT_MARK(6);
            // ---- the decision warp: logits, softmax, inverse-CDF sample, select the pre-computed next state / reset -----------
            if (r_dec && mine) {
                int forced_a = 0;
                if (a.forced) forced_a = reinterpret_cast<const int*>(a.forced)[row + n];
                // logits: fixed-order tree over the 16 partials (4 independent chains)
                float za[4] = {0.f, 0.f, 0.f, 0.f}, zb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const float2 pp = *reinterpret_cast<const float2*>(sPart + (k * 32 + e) * 2);
                    za[k & 3] += pp.x; zb[k & 3] += pp.y;
                }
                const float z0 = b2_0 + ((za[0] + za[1]) + (za[2] + za[3]));
                const float z1 = b2_1 + ((zb[0] + zb[1]) + (zb[2] + zb[3]));
                int idx = 0;
                float pe = 1.f, ssum = 1.f;
                if (A > 1) {
                    const float m = fmaxf(z0, z1);
                    const float e0 = expf(z0 - m), e1 = expf(z1 - m);
                    ssum = e0 + e1;
                    idx = 1;
                    if (a.forced) {
                        idx = forced_a - pd.act_start;
                        idx = idx < 0 ? 0 : (idx > 1 ? 1 : idx);
                    } else {
                        const float cum0 = e0 / ssum;                    // fp32 cumsum vs Float64 u (categorical.jl:45-47)
                        if ((double)cum0 >= sU[e]) idx = 0;
                    }
                    pe = idx == 0 ? e0 : e1;
                }
                RT_MARK(7);
                const float4 c4 = *reinterpret_cast<const float4*>(sCand + e * 8);
                const float2 c2 = *reinterpret_cast<const float2*>(sCand + e * 8 + 4);
                st[0] = c4.x; st[2] = c4.y;
                st[1] = idx == 1 ? c2.x : c4.z;
                st[3] = idx == 1 ? c2.y : c4.w;
                const bool term = (st[0] < -2.4f) || (st[0] > 2.4f) || (st[2] < -0.20943951023931953f) || (st[2] > 0.20943951023931953f);
                steps += 1;
                const bool trunc = steps >= env.max_steps;
                const bool done = term || trunc;
                if (env.monitor) { ep_ret = __fadd_rn(ep_ret, 1.0f); ep_len += 1; }
                pend.live = true; pend.t = t; pend.idx = idx; pend.pe = pe; pend.ssum = ssum; pend.term = term; pend.trunc = trunc;
                pend.ep_ret = ep_ret; pend.ep_len = ep_len;
                if (trunc) pend.tobs = make_float4(st[0], st[1], st[2], st[3]);
                float2 scn;
                if (done) {
                    if (env.monitor) { ep_ret = 0.f; ep_len = 0; }
                    const float4 r4 = *reinterpret_cast<const float4*>(sReset + e * 8);
                    scn = *reinterpret_cast<const float2*>(sReset + e * 8 + 4);
                    st[0] = r4.x; st[1] = r4.y; st[2] = r4.z; st[3] = r4.w;
                    episode += 1;
                    steps = 0;
                    sNeed[e] = (int)episode;
                } else {
                    scn = *reinterpret_cast<const float2*>(sSCn + e * 2);
                    sNeed[e] = -1;
                }
                *reinterpret_cast<float4*>(sState + e * 4) = make_float4(st[0], st[1], st[2], st[3]);
                *reinterpret_cast<float2*>(sSCcur + e * 2) = scn;
            }
            __syncthreads();
        }
        if (r_dec) {
            flush();
            if (mine) {
                *reinterpret_cast<float4*>(sc.last_obs + (size_t)n * 4) = make_float4(st[0], st[1], st[2], st[3]);
#pragma unroll
                for (int k = 0; k < 4; ++k) env.state[(size_t)k * N + n] = st[k];
                env.steps[n] = steps;
                env.episode[n] = episode;
                if (env.monitor) { env.ep_ret[n] = ep_ret; env.ep_len[n] = ep_len; }
            }
        }
        __syncthreads();                              // the next tile reuses the shared arrays
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(RT_TMEM_COLS));
}

// ---------------------------------------------------------------------------------------------------------
// Batched critic: values of all T*N buffer observations, of the N final observations (bootstrap, trajectory.jl:65-70)
// and of the terminal observations of truncated steps (trajectory.jl:57-61).  128 samples per tile, two threads per
// sample (32 hidden features each), hidden layer on tcgen05 (fp16 hi/lo).  3 CTAs per SM (128 TMEM columns each).
// ---------------------------------------------------------------------------------------------------------
#define CV_THREADS 256
#define CV_TMEM_COLS 128         // D 0..63 | packed hi operand 64..95 | packed lo operand 96..127: three CTAs per SM (registers: 85)
#define CV_COL_HI 64
#define CV_COL_LO 96
__global__ void __launch_bounds__(CV_THREADS, 3) critic_values_tc_kernel(const PolicyDesc pd, const float* __restrict__ pack, BufDev buf,
                                                                        const TcRolloutScratch sc) {
    extern __shared__ __align__(1024) unsigned char rt_smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const uint32_t raw = tc_smem_u32(rt_smem_raw);
    const uint32_t sm_base = (raw + 1023u) & ~1023u;
    unsigned char* sm = rt_smem_raw + (sm_base - raw);
    float* sSmall = reinterpret_cast<float*>(sm + CV_OFF_SMALL);
    float* sW0 = sSmall;
    float* sb0 = sW0 + 256;
    float* sb1 = sb0 + 64;
    float* sW2 = sb1 + 64;
    float* sb2 = sW2 + 256;
    float* sPart = sb2 + 8;         // [2 halves][128]
    const LayerDesc& L0 = pd.L[1][0];
    const LayerDesc& L1 = pd.L[1][1];
    const LayerDesc& L2 = pd.L[1][2];
    rt_stage_w1_f16(pack, L1, sm, tid, CV_THREADS);
    for (int i = tid; i < 256; i += CV_THREADS) { sW0[i] = pack[L0.pw_off + i]; sW2[i] = pack[L2.pw_off + i]; }
    if (tid < 64) { sb0[tid] = pack[L0.pb_off + tid]; sb1[tid] = pack[L1.pb_off + tid]; }
    if (tid < 4) sb2[tid] = pack[L2.pb_off + tid];
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(CV_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);
    const int m = tid & 127, half = (warp >> 2) & 1, f0 = half * 32;
    const uint32_t my = tb + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t idesc = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // kind::f16, M = 128, N = 64
    const long long TN = buf.T * buf.N;
    const unsigned int ntr = min(*sc.trunc_count, sc.cap);
    const long long total = TN + buf.N + (long long)ntr;
    const long long n_tiles = (total + 127) / 128;
    uint32_t nbar = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long v = tile * 128 + m;
        const bool valid = v < total;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        float* dst = nullptr;
        if (valid) {
            if (v < TN) { x = *reinterpret_cast<const float4*>(buf.obs + v * 4); dst = buf.values + v; }
            else if (v < TN + buf.N) { x = *reinterpret_cast<const float4*>(sc.last_obs + (v - TN) * 4); dst = buf.last_values + (v - TN); }
            else { const long long k = v - TN - buf.N; x = *reinterpret_cast<const float4*>(sc.trunc_obs + k * 4); dst = buf.boot + sc.trunc_idx[k]; }
        }
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 8) {
            float h[8];
            {
                const float4 ba = *reinterpret_cast<const float4*>(sb0 + f0 + c0);
                const float4 bb = *reinterpret_cast<const float4*>(sb0 + f0 + c0 + 4);
                h[0] = ba.x; h[1] = ba.y; h[2] = ba.z; h[3] = ba.w; h[4] = bb.x; h[5] = bb.y; h[6] = bb.z; h[7] = bb.w;
            }
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const float xd = d == 0 ? x.x : (d == 1 ? x.y : (d == 2 ? x.z : x.w));
                const float4 w0 = *reinterpret_cast<const float4*>(sW0 + d * 64 + f0 + c0);
                const float4 w1 = *reinterpret_cast<const float4*>(sW0 + d * 64 + f0 + c0 + 4);
                h[0] = fmaf(xd, w0.x, h[0]); h[1] = fmaf(xd, w0.y, h[1]); h[2] = fmaf(xd, w0.z, h[2]); h[3] = fmaf(xd, w0.w, h[3]);
                h[4] = fmaf(xd, w1.x, h[4]); h[5] = fmaf(xd, w1.y, h[5]); h[6] = fmaf(xd, w1.z, h[6]); h[7] = fmaf(xd, w1.w, h[7]);
            }
            // fp16 hi/lo split (bounded operands, see rt_split_f16); A operand in TMEM: two consecutive K elements per 32-bit
            // column, feature k of the hi / lo operand in packed column k / 2
            uint32_t ph[4], pl[4];
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                __half a_h, a_l, b_h, b_l;
                rt_split_f16(fast_tanh(h[j]), a_h, a_l);
                rt_split_f16(fast_tanh(h[j + 1]), b_h, b_l);
                const __half2 vh = __halves2half2(a_h, b_h), vl = __halves2half2(a_l, b_l);
                ph[j >> 1] = *reinterpret_cast<const uint32_t*>(&vh);
                pl[j >> 1] = *reinterpret_cast<const uint32_t*>(&vl);
            }
            asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(my + CV_COL_HI + ((f0 + c0) >> 1)), "r"(ph[0]), "r"(ph[1]),
                         "r"(ph[2]), "r"(ph[3]) : "memory");
            asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(my + CV_COL_LO + ((f0 + c0) >> 1)), "r"(pl[0]), "r"(pl[1]),
                         "r"(pl[2]), "r"(pl[3]) : "memory");
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 0 && tc_elect_one()) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int ps = 0; ps < 3; ++ps) {
                const uint32_t acol = tb + (ps == 1 ? CV_COL_LO : CV_COL_HI);
                const uint32_t bimg = sm_base + (ps == 2 ? RT_OFF_WT_LO : RT_OFF_WT_HI);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)          // K = 16: features 16 kk .. 16 kk + 15 = 8 packed columns
                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(
                                     tb + RT_COL_D),
                                 "r"(acol + kk * 8), "l"(tc_desc(bimg + kk * 256, 128, 1024, 0)), "r"(idesc),
                                 "r"((ps | kk) ? 1u : 0u) : "memory");
            }
            tc_commit(&bar);
        }
        tc_wait(&bar, nbar & 1u);
        ++nbar;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        {
            float h1[32];
            tc_ld32(my + RT_COL_D + f0, h1);
            float p0 = 0.f;
#pragma unroll
            for (int k = 0; k < 32; ++k) p0 = fmaf(fast_tanh(h1[k] + sb1[f0 + k]), sW2[(f0 + k) * 4], p0);
            sPart[half * 128 + m] = p0;
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (half == 0 && valid) *dst = sb2[0] + (sPart[m] + sPart[128 + m]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(CV_TMEM_COLS));
}
