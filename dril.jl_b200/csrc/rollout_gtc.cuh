// General rollout kernel with the ACTOR on tcgen05 (critic deferred, rollout.cuh RO_DEFER_CRITIC): the step loop, env stepping,
// Monitor / Normalize statistics and grid barriers are rollout_body (rollout.cuh) unchanged; only the layer forward of a
// 128-env tile is replaced.  Same formulation as the general loss/grad kernel's forward half (update_ftg.cuh): features on
// TMEM lanes, the tile's 128 envs on TMEM columns, every layer one GEMM
//     Hpre_l [width_l][128] = (C2 W_l)^T [width_l][width_{l-1}] · H_{l-1} [width_{l-1}][128]
// on kind::f16 with fp16 hi / lo splits of both operands (hi·hi + lo·hi + hi·lo, fp32 accumulation in TMEM: 22 bits), layer 0
// included (x image with a ones row carries the bias), tanh's 2·log2(e) folded into the weight images.  Weight images of the
// actor (W_1.., [W_0; b_0]) stay resident in shared memory for the whole rollout; ONE activation image buffer is reused by all
// layers (a layer's MMAs have completed before its epilogue overwrites their B operand) and ends as the fp32 tile of the last
// hidden layer, from which the thin output layer (<= 4 outputs) is evaluated on CUDA cores.
// Replaces the mma.sync tiles of mlp.cuh in the step loop for the shapes update_ftg.cuh covers (2-3 hidden layers of 64 / 128).
// Reference: the layer call of collect_trajectories (layers/layer_forward.jl:3-39, layer_helpers.jl:27-57).
#pragma once
#include "rollout.cuh"
#include "update_ftg.cuh"

#define GTC_ENVS 128
#define GTC_HS_LD 132

struct GtcLayout {             // byte offsets from the 1024-aligned start of the image region
    int w[3];                  // [l - 1] images (hi, lo) of C2 * W_l, l = 1 .. L-1
    int w0a;                   // images (hi, lo) of C2 * [W_0; b_0; 0]^T: rows = features of layer 0, 16 columns
    int h;                     // activation images (hi, lo) [width][128 envs] of the current layer / fp32 [width L-1][132] at the end
    int ximg;                  // x images (hi, lo): 16 rows x 128 envs
    int wout;                  // output layer [width L-1][NO] floats + bias [NO]
    int part;                  // output-layer partials [2 halves][NO outputs][128]
    int total;
};
// output columns the kernel stages: 2, or 4 for Discrete(3 | 4)
__host__ __device__ inline int gtc_nout(const PolicyDesc& pd) { return pd.act_n > 2 ? 4 : 2; }
__host__ __device__ inline GtcLayout gtc_layout(const PolicyDesc& pd) {
    GtcLayout s;
    const int L = pd.n_layers - 1;
    int o = 0;
    auto take = [&](int bytes) { const int r = o; o += (bytes + 127) & ~127; return r; };
    for (int l = 0; l < 3; ++l) s.w[l] = 0;
    for (int l = 1; l < L; ++l) s.w[l - 1] = take(2 * pd.L[0][l].N * pd.L[0][l - 1].N * 2);
    s.w0a = take(2 * pd.L[0][0].N * 16 * 2);
    int hb = 0;
    for (int l = 0; l + 1 < L; ++l) hb = hb > 2 * pd.L[0][l].N * GTC_ENVS * 2 ? hb : 2 * pd.L[0][l].N * GTC_ENVS * 2;
    const int last = pd.L[0][L - 1].N * GTC_HS_LD * 4;
    s.h = take(hb > last ? hb : last);
    s.ximg = take(2 * 16 * GTC_ENVS * 2);
    const int no = gtc_nout(pd);
    s.wout = take((pd.L[0][L - 1].N * no + 4) * 4);
    s.part = take(2 * no * GTC_ENVS * 4);
    s.total = o + 1024;
    return s;
}

// 16-byte row (8 consecutive envs starting at c, c % 8 == 0) of feature row r of a [rows][128] fp16 image, no-swizzle core layout
__device__ __forceinline__ uint32_t gtc_row_off(int r, int c) { return (uint32_t)((((r >> 3) * 16 + (c >> 3)) << 7) + ((r & 7) << 4)); }

template <int L, int NO>
struct GtcForward {
    unsigned char* sm;         // image region (generic pointer)
    uint32_t sm_base;          // its shared-space address
    GtcLayout ly;
    uint64_t* barM;
    uint32_t tb;               // TMEM base
    uint32_t n_mma;
    int wd[L], fl[L];
    float bsc[L];
    int D, A;

    // actor outputs of the tile whose normalised observations are in sX [Dp][ld] -> sActA rows [j][ld]; returns buffer index 0
    __device__ __forceinline__ int operator()(const PolicyDesc& pd, const float* __restrict__, const float* sX, float* sActA, float*, int, int ld,
                                              int, bool) {
        const int tid = threadIdx.x;
        const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
        const int q = warp & 3, sg = warp >> 2;
        const uint32_t my = tb + ((uint32_t)(q * 32) << 16);
        __half* sXimg = reinterpret_cast<__half*>(sm + ly.ximg);
        // ---- x of the tile's 128 envs -> fp16 hi / lo rows 0 .. D-1 of the x images (row D is the constant ones row) ------------
        for (int i = tid; i < GTC_ENVS * D; i += blockDim.x) {
            const int m = i & (GTC_ENVS - 1), d = i >> 7;
            const float x = fminf(fmaxf(sX[(size_t)d * ld + m], -65504.f), 65504.f);
            const __half h = __float2half_rn(x);
            const int idx = ((d >> 3) * 16 + (m >> 3)) * 64 + (d & 7) * 8 + (m & 7);
            sXimg[idx] = h;
            sXimg[16 * GTC_ENVS + idx] = __float2half_rn(x - __half2float(h));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        float* Hs = reinterpret_cast<float*>(sm + ly.h);
#pragma unroll
        for (int l = 0; l < L; ++l) {
            if (warp == 0 && tc_elect_one()) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (l == 0) {
                    const uint32_t id = ft_idesc(wd[0], GTC_ENVS, 0, 1);
#pragma unroll
                    for (int ps = 0; ps < 3; ++ps)
                        ft_mma(tb, tc_desc(sm_base + ly.w0a + (ps == 1 ? wd[0] * 32 : 0), 128, 256, 0),
                               tc_desc(sm_base + ly.ximg + (ps == 2 ? 16 * GTC_ENVS * 2 : 0), 2048, 128, 0), id, ps ? 1u : 0u);
                } else {
                    const int K = wd[l - 1], N = wd[l];
                    const uint32_t id = ft_idesc(N, GTC_ENVS, 0, 1);
#pragma unroll
                    for (int ps = 0; ps < 3; ++ps) {
                        const uint32_t ai = sm_base + ly.w[l - 1] + (ps == 1 ? N * K * 2 : 0), bi = sm_base + ly.h + (ps == 2 ? K * GTC_ENVS * 2 : 0);
                        for (int kk = 0; kk < (K >> 4); ++kk)
                            ft_mma(tb, tc_desc(ai + kk * 256, 128, (K >> 3) * 128, 0), tc_desc(bi + kk * 4096, 2048, 128, 0), id, (ps || kk) ? 1u : 0u);
                    }
                }
                tc_commit(barM);
            }
            tc_wait(barM, n_mma & 1u); ++n_mma;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // epilogue: this thread's feature, its sample group's 64 envs in chunks of 16 (lanes 16..31 of a quadrant hold no
            // feature of a 64-wide layer, but the warp-wide TMEM loads need every lane)
            {
                unsigned char* ph = sm + ly.h;
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) {
                    const int c0 = 64 * sg + 16 * c4;
                    float v[16];
                    ft_ld16(my + c0, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (fl[l] >= 0) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = ft_tanh_scaled(v[j] + bsc[l]);
                        if (l + 1 < L) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                uint4 vh, vl;
                                ft_split2(v[8 * c], v[8 * c + 1], vh.x, vl.x); ft_split2(v[8 * c + 2], v[8 * c + 3], vh.y, vl.y);
                                ft_split2(v[8 * c + 4], v[8 * c + 5], vh.z, vl.z); ft_split2(v[8 * c + 6], v[8 * c + 7], vh.w, vl.w);
                                const uint32_t off = gtc_row_off(fl[l], c0 + 8 * c);
                                *reinterpret_cast<uint4*>(ph + off) = vh;
                                *reinterpret_cast<uint4*>(ph + wd[l] * GTC_ENVS * 2 + off) = vl;
                            }
                        } else {
                            float* hr = Hs + fl[l] * GTC_HS_LD + c0;
#pragma unroll
                            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(hr + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                        }
                    }
                }
            }
            if (l + 1 < L) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
        }
        // ---- output layer (<= NO outputs) on CUDA cores: the feature range is split over the two halves of the block ------------
        {
            const float* sWout = reinterpret_cast<const float*>(sm + ly.wout);
            float* sPart = reinterpret_cast<float*>(sm + ly.part);
            const int m = tid & (GTC_ENVS - 1), half = (tid >> 7) & 1, per = wd[L - 1] >> 1;
            if (tid < 2 * GTC_ENVS) {
                const float* hp = Hs + (half * per) * GTC_HS_LD + m;
                if constexpr (NO == 2) {
                    float p0 = 0.f, p1 = 0.f;
                    for (int n = 0; n < per; ++n) {
                        const float hv = hp[n * GTC_HS_LD];
                        const float2 w = *reinterpret_cast<const float2*>(sWout + 2 * (half * per + n));
                        p0 = fmaf(hv, w.x, p0); p1 = fmaf(hv, w.y, p1);
                    }
                    sPart[(half * 2 + 0) * GTC_ENVS + m] = p0;
                    sPart[(half * 2 + 1) * GTC_ENVS + m] = p1;
                } else {
                    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
                    for (int n = 0; n < per; ++n) {
                        const float hv = hp[n * GTC_HS_LD];
                        const float4 w = *reinterpret_cast<const float4*>(sWout + 4 * (half * per + n));
                        p0 = fmaf(hv, w.x, p0); p1 = fmaf(hv, w.y, p1); p2 = fmaf(hv, w.z, p2); p3 = fmaf(hv, w.w, p3);
                    }
                    sPart[(half * 4 + 0) * GTC_ENVS + m] = p0;
                    sPart[(half * 4 + 1) * GTC_ENVS + m] = p1;
                    sPart[(half * 4 + 2) * GTC_ENVS + m] = p2;
                    sPart[(half * 4 + 3) * GTC_ENVS + m] = p3;
                }
            }
            __syncthreads();
            if (tid < GTC_ENVS) {
#pragma unroll
                for (int j = 0; j < NO; ++j)
                    if (j < A) sActA[(size_t)j * ld + tid] = sWout[NO * wd[L - 1] + j] + (sPart[j * GTC_ENVS + tid] + sPart[(NO + j) * GTC_ENVS + tid]);
            }
            __syncthreads();
        }
        return 0;
    }
};

// KS: env kinds served (env.cuh); NO: output columns staged (gtc_nout)
template <int L, unsigned KS, int NO>
__global__ void __launch_bounds__(DRIL_THREADS, 1) rollout_gtc_kernel(const __grid_constant__ RolloutArgs a, const __grid_constant__ GtcLayout ly,
                                                                      const int body_bytes) {
    extern __shared__ __align__(1024) unsigned char gtc_smem_raw[];
    __shared__ __align__(8) uint64_t barM;
    __shared__ uint32_t tmem_base_s;
    constexpr int net = 0;
    const PolicyDesc& pd = a.pd;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int lane = tid & 31, q = warp & 3;
    const uint32_t raw = tc_smem_u32(gtc_smem_raw);
    const uint32_t sm_base = (raw + (uint32_t)body_bytes + 1023u) & ~1023u;       // image region behind rollout_body's arrays
    unsigned char* sm = gtc_smem_raw + (sm_base - raw);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(GTC_ENVS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&barM)));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    GtcForward<L, NO> fwd;
    fwd.sm = sm; fwd.sm_base = sm_base; fwd.ly = ly; fwd.barM = &barM; fwd.n_mma = 0; fwd.D = pd.obs_dim; fwd.A = pd.act_n;
#pragma unroll
    for (int l = 0; l < L; ++l) {
        fwd.wd[l] = pd.L[net][l].N;
        fwd.fl[l] = fwd.wd[l] == 128 ? 32 * q + lane : (lane < 16 ? 16 * q + lane : -1);
    }
    // ---- the actor's weights: images of C2 * W_l (l >= 1), of C2 * [W_0; b_0]^T, output layer in fp32 -----------------------------
#pragma unroll
    for (int l = 1; l < L; ++l) {
        const LayerDesc& Ll = pd.L[net][l];
        const int K = fwd.wd[l - 1], N = fwd.wd[l], KB = K >> 3;
        __half* hi = reinterpret_cast<__half*>(sm + ly.w[l - 1]);
        __half* lo = hi + N * K;
        for (int i0 = tid * 4; i0 < K * N; i0 += blockDim.x * 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(a.pack + Ll.pw_off + i0);
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
            const int k = i0 / N, nb = i0 - k * N;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = nb + j;
                const float w = fminf(fmaxf(wv[j] * FT_C2, -65504.f), 65504.f);
                const __half h = __float2half_rn(w);
                const int idx = ((n >> 3) * KB + (k >> 3)) * 64 + (n & 7) * 8 + (k & 7);
                hi[idx] = h;
                lo[idx] = __float2half_rn(w - __half2float(h));
            }
        }
    }
    {
        const LayerDesc& L0 = pd.L[net][0];
        __half* hi = reinterpret_cast<__half*>(sm + ly.w0a);
        __half* lo = hi + fwd.wd[0] * 16;
        for (int i = tid; i < fwd.wd[0] * 16; i += blockDim.x) {
            const int k = i >> 4, d = i & 15;
            float w = d < fwd.D ? a.pack[L0.pw_off + d * L0.Np + k] : (d == fwd.D ? a.pack[L0.pb_off + k] : 0.f);
            w = fminf(fmaxf(w * FT_C2, -65504.f), 65504.f);
            const __half h = __float2half_rn(w);
            const int idx = ((k >> 3) * 2 + (d >> 3)) * 64 + (k & 7) * 8 + (d & 7);
            hi[idx] = h;
            lo[idx] = __float2half_rn(w - __half2float(h));
        }
    }
    {
        const LayerDesc& Lout = pd.L[net][L];
        float* sWout = reinterpret_cast<float*>(sm + ly.wout);
        for (int i = tid; i < fwd.wd[L - 1]; i += blockDim.x) {
            sWout[NO * i] = a.pack[Lout.pw_off + i * Lout.Np];
            sWout[NO * i + 1] = fwd.A > 1 ? a.pack[Lout.pw_off + i * Lout.Np + 1] : 0.f;
            if (NO == 4) {
                sWout[NO * i + 2] = fwd.A > 2 ? a.pack[Lout.pw_off + i * Lout.Np + 2] : 0.f;
                sWout[NO * i + 3] = fwd.A > 3 ? a.pack[Lout.pw_off + i * Lout.Np + 3] : 0.f;
            }
        }
        if (tid < NO) sWout[NO * fwd.wd[L - 1] + tid] = tid < fwd.A ? a.pack[Lout.pb_off + tid] : 0.f;
    }
    {
        __half* sXimg = reinterpret_cast<__half*>(sm + ly.ximg);
        for (int i = tid; i < 2 * 16 * GTC_ENVS; i += blockDim.x) {
            const int e = i & (16 * GTC_ENVS - 1), d = ((e >> 10) << 3) + ((e >> 3) & 7);
            sXimg[i] = __float2half_rn((i < 16 * GTC_ENVS && d == fwd.D) ? 1.0f : 0.f);
        }
    }
#pragma unroll
    for (int l = 1; l < L; ++l) fwd.bsc[l] = fwd.fl[l] >= 0 ? a.pack[pd.L[net][l].pb_off + fwd.fl[l]] * FT_C2 : 0.f;
    fwd.bsc[0] = 0.f;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    fwd.tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);

    rollout_body<false, true, KS>(a, reinterpret_cast<float*>(gtc_smem_raw), fwd);

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(fwd.tb), "r"(GTC_ENVS));
}
