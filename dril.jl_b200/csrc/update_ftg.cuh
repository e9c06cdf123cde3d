// General-shape features-on-lanes tcgen05 loss/grad kernel: two or three tanh hidden layers of width 64 or 128 per net,
// obs_dim <= 15, Discrete(n <= 4) or Box actions of dimension <= 2 — e.g. BASELINE config C3, Pendulum with
// hidden_dims = [128, 128, 64] and a diagonal Gaussian (layers/layer_helpers.jl:27-57, DRiLDistributions/diagGaussian.jl:13-47,
// loss functor algorithms/ppo.jl:365-407).  Same formulation as update_ft.cuh (features on TMEM lanes, samples on columns,
// fp16 hi/lo operands on kind::f16, one no-swizzle image per matrix for both GEMM orientations), generalised:
//   * one net per pass (a 128-wide layer needs all 128 lanes: M = 128, row i <-> lane i; a 64-wide layer is an M = 64
//     accumulator, row i <-> lane 32 (i / 16) + i % 16, half of the threads idle in its element-wise phases);
//   * 16 warps work on ONE 64-sample tile (warp = lane quadrant x sample quarter), phases strictly in sequence:
//       G0 (prefetched) -> A0 -> G1 -> A1 [-> G2 -> A2] -> output layer + loss head -> dZ_last -> {dH, dW} -> dZ ... -> dZ_0 sums
//     with every GEMM of the chain on the tensor cores:  forward  H_l^pre = W_l^T H_{l-1}   (A = W_l image, K-major),
//                                                          dH_{l-1} = W_l dZ_l              (A = the same image, MN-major),
//                                                          dW_l     = H_{l-1} dZ_l^T        (A = H_{l-1} image, K-major);
//   * the dW_l accumulators stay in TMEM over all tiles of the pass.  The deltas are scaled by ONE power of two per CTA and
//     pass, fixed at the first tile with a non-zero gradient such that its largest |dZ_last| bound sits at 2^2; a later
//     tile whose scaled bound would reach 2^14 lowers the scale to sit where the first tile sat and multiplies the dW
//     accumulators and scaled sums by the exact ratio (fp16 ends at 65504); everything is unscaled exactly when the
//     partial plane is written;
//   * shared memory: weight images of the pass (W_1.., W_0 with the bias row), one image buffer per hidden layer but
//     the last (H_l, later reused for dZ_l), one buffer for the last layer's fp32 tile / delta image, two tile records.
// The kernel ends with the cooperative tail of update_tc.cuh.  Tile records of all epochs are written by one launch of
// ftg_permute_epochs_kernel (DataLoader shuffle, ppo.jl:188-195, + minibatch advantage moments) and fetched with
// cp.async.bulk one tile ahead.
#pragma once
#include "update_ft.cuh"

#define FTG_THREADS 512
#define FTG_COL_D 0
#define FTG_COL_D0 64
#define FTG_COL_G 128          // stashes of 1 - H_l^2, 64 columns per hidden layer but the last
#define FTG_COL_DW 256         // dW_l accumulators, 128 columns each (l = 1, 2)
#define FTG_TMEM_COLS 512
#define FTG_MAX_OBS 15

struct FtgLayout {             // byte offsets inside the dynamic shared memory (1024-aligned base), all multiples of 128
    int w[3];                  // [l - 1] images (hi, lo) of C2 * W_l, l = 1 .. L-1: rows n (width l), columns k (width l - 1)
    int w0a;                   // images (hi, lo) of C2 * [W_0; b_0; 0]^T: rows k (width 0), 16 columns
    int h[2];                  // image buffers (hi, lo) of H_l, l = 0 .. L-2 (later dZ_l)
    int last;                  // fp32 tile [width L-1][68] of the last hidden layer, then its delta images
    int rec;                   // two tile records
    int ximg;                  // x images (hi, lo) of the next tile: 16 rows x 64 samples
    int part;                  // [8 feature slices][64 samples] float4 output-layer partials
    int dout;                  // [64 samples] float4: dL/dout (<= 4) per sample
    int small;                 // output-layer weights [width L-1] float2 (float4 for Discrete(3 | 4)), bias, reduction scratch
    int total;
    int rec_floats;
};
struct FtgArgs {
    const unsigned char* tiles;
    long long tile0;
    FtgLayout lay;
};

__host__ __device__ inline int ftg_rec_floats(int obs_dim, int cont, int act_n) { return 64 * (((obs_dim + 3) & ~3) + 4 + (cont ? act_n : 1)); }
__host__ inline FtgLayout ftg_layout(const PolicyDesc& pd) {
    FtgLayout s;
    const int L = pd.n_layers - 1;
    int o = 0;
    auto take = [&](int bytes) { const int r = o; o += (bytes + 127) & ~127; return r; };
    int wd[3];
    for (int l = 0; l < L; ++l) wd[l] = std::max(pd.L[0][l].N, pd.L[1][l].N);
    for (int l = 0; l < 3; ++l) s.w[l] = 0;
    for (int l = 1; l < L; ++l) s.w[l - 1] = take(2 * wd[l] * wd[l - 1] * 2);
    s.w0a = take(2 * wd[0] * 16 * 2);
    s.h[0] = s.h[1] = 0;
    for (int l = 0; l + 1 < L; ++l) s.h[l] = take(2 * wd[l] * 64 * 2);
    s.last = take(std::max(wd[L - 1] * 68 * 4, 2 * wd[L - 1] * 64 * 2));
    s.rec_floats = ftg_rec_floats(pd.obs_dim, pd.act_kind == DRIL_ACT_CONTINUOUS, pd.act_n);
    s.rec = take(2 * s.rec_floats * 4);
    s.ximg = take(2 * 2048);
    s.part = take(8 * 64 * 16);
    s.dout = take(64 * 16);
    // W_out [128] float2 | bias, bounds | thin-sum scratch [4 sample quarters][8][128]; Discrete(3 | 4): W_out [128] float4 and the
    // four output biases behind the bound / dmax / head-sum slots (ftg_pass)
    const bool wide = pd.act_kind == DRIL_ACT_DISCRETE && pd.act_n > 2;
    s.small = take((wide ? 128 * 16 + 128 : 128 * 8 + 64) + 4 * 8 * 128 * 4);
    s.total = o + 1024;
    return s;
}

// The epoch's samples in shuffled order as contiguous records of 64: x [64][Dp] | advantage | old log-prob | return | old value |
// action (index int / act_n floats, [j][64]).  Slot r of minibatch mb; returns the sample's advantage.
__device__ __forceinline__ float ftg_permute_slot(const float* __restrict__ recs, int stride, int D, const FeistelKey& fk, long long n_total,
                                                  long long batch_size, long long per, long long mb, long long r, int identity, int act_start,
                                                  int act_n, int cont, int rec_floats, float* __restrict__ out, bool& valid) {
    const int Dp = (D + 3) & ~3, A = cont ? act_n : 1;
    const long long pos = mb * batch_size + r, s = mb * per + r;
    valid = r < batch_size && pos < n_total;
    float* blk = out + (s >> 6) * rec_floats;
    const int j = (int)(s & 63);
    long long sidx = 0;
    if (valid) sidx = identity ? pos : feistel_permute(pos, n_total, fk);
    const float* rp = recs + sidx * stride;                       // obs (Dp) | action (A) | adv, logp, ret, val: sample record (update_ft.cuh)
    for (int d4 = 0; d4 < Dp; d4 += 4)
        *reinterpret_cast<float4*>(blk + j * Dp + d4) = valid ? *reinterpret_cast<const float4*>(rp + d4) : make_float4(0.f, 0.f, 0.f, 0.f);
    float* sc = blk + 64 * Dp;
    const float adv = valid ? rp[Dp + A] : 0.f;
    sc[j] = adv;
    sc[64 + j] = valid ? rp[Dp + A + 1] : 0.f;
    sc[128 + j] = valid ? rp[Dp + A + 2] : 0.f;
    sc[192 + j] = valid ? rp[Dp + A + 3] : 0.f;
    if (cont) {
        for (int a = 0; a < act_n; ++a) sc[256 + a * 64 + j] = valid ? rp[Dp + a] : 0.f;
    } else {
        int ai = valid ? __float_as_int(rp[Dp]) - act_start : 0;
        ai = ai < 0 ? 0 : (ai >= act_n ? act_n - 1 : ai);
        reinterpret_cast<int*>(sc)[256 + j] = ai;
    }
    return adv;
}
__global__ void __launch_bounds__(256) ftg_permute_kernel(const float* __restrict__ recs, int stride, int D, const FeistelKey fk, long long n_total,
                                                          long long batch_size, int n_mb, int tiles_per_mb, int identity, int act_start, int act_n,
                                                          int cont, int rec_floats, float* __restrict__ out) {
    const long long per = (long long)tiles_per_mb * 64;
    const long long slots = per * n_mb;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += (long long)gridDim.x * blockDim.x) {
        const long long mb = s / per;
        bool valid;
        ftg_permute_slot(recs, stride, D, fk, n_total, batch_size, per, mb, s - mb * per, identity, act_start, act_n, cont, rec_floats, out, valid);
    }
}
// all epochs of an update in one launch + the minibatch advantage moments (see ft_permute_epochs_kernel, update_ft.cuh)
__global__ void __launch_bounds__(256) ftg_permute_epochs_kernel(const float* __restrict__ recs, int stride, int D, const __grid_constant__ FeistelKeys fks,
                                                                 long long n_total, long long batch_size, int tiles_per_mb, int act_start, int act_n,
                                                                 int cont, int rec_floats, float* __restrict__ out, long long epoch_tiles,
                                                                 double* __restrict__ partial, const PermuteTail pt) {
    __shared__ double scratch[32];
    const FeistelKey& fk = fks.k[blockIdx.z];
    const long long per = (long long)tiles_per_mb * 64, mb = blockIdx.y;
    float* o = out + (size_t)blockIdx.z * epoch_tiles * rec_floats;
    double sm = 0, sq = 0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < per; r += (long long)gridDim.x * blockDim.x) {
        bool valid;
        const float adv = ftg_permute_slot(recs, stride, D, fk, n_total, batch_size, per, mb, r, 0, act_start, act_n, cont, rec_floats, o, valid);
        if (valid) { sm += (double)adv; sq += (double)adv * (double)adv; }
    }
    sm = block_sum(sm, scratch); sq = block_sum(sq, scratch);
    if (threadIdx.x == 0) {
        double* pp = partial + (((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 2;
        pp[0] = sm; pp[1] = sq;
    }
    permute_epochs_finish(pt, partial);
}

__device__ __forceinline__ void ftg_st16(uint32_t taddr, const float* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])), "r"(__float_as_uint(r[2])), "r"(__float_as_uint(r[3])),
                 "r"(__float_as_uint(r[4])), "r"(__float_as_uint(r[5])), "r"(__float_as_uint(r[6])), "r"(__float_as_uint(r[7])),
                 "r"(__float_as_uint(r[8])), "r"(__float_as_uint(r[9])), "r"(__float_as_uint(r[10])), "r"(__float_as_uint(r[11])),
                 "r"(__float_as_uint(r[12])), "r"(__float_as_uint(r[13])), "r"(__float_as_uint(r[14])), "r"(__float_as_uint(r[15])) : "memory");
}

// HEAD: 0 discrete actor, 1 Gaussian actor, 2 critic
template <int L, int HEAD, int NOUT>
__device__ __forceinline__ void ftg_pass(const LossArgs& a, const FtgArgs& fa, unsigned char* sm, uint32_t sm_base, uint32_t tb, uint64_t* bars,
                                         uint32_t& n_rec, uint32_t& n_g0, uint32_t& n_mma, uint32_t& n_w, float adv_mean, float adv_den, float invB, float* stats,
                                         float* gp) {
    const PolicyDesc& pd = a.pd;
    const FtgLayout& ly = fa.lay;
    constexpr int net = HEAD == 2 ? 1 : 0;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int lane = tid & 31, q = warp & 3, sg = warp >> 2;
    const int m0 = 16 * sg;                       // this thread's samples of the tile: m0 .. m0 + 15
    const int ms = tid & 63, slice = tid >> 6;    // sample role: sample, feature slice (8 slices)
    const bool issuer = warp == 0;
    int wd[L];
#pragma unroll
    for (int l = 0; l < L; ++l) wd[l] = pd.L[net][l].N;
    int fl[L];                                    // this thread's feature of layer l, or -1
#pragma unroll
    for (int l = 0; l < L; ++l) fl[l] = wd[l] == 128 ? 32 * q + lane : (lane < 16 ? 16 * q + lane : -1);
    const uint32_t my = tb + ((uint32_t)(q * 32) << 16);
    const int D = pd.obs_dim, Dp = (D + 3) & ~3;
    uint64_t* barL = bars;          // [2] tile records
    uint64_t* barG0 = bars + 2;     // G0 of the next tile
    uint64_t* barM = bars + 3;      // the GEMM(s) a phase waits for
    uint64_t* barW = bars + 4;      // dW GEMMs (image buffers may be overwritten)
    constexpr bool W4 = NOUT > 2;                             // Discrete(3 | 4): four output columns
    float* sSmall = reinterpret_cast<float*>(sm + ly.small);
    float2* sWout = reinterpret_cast<float2*>(sSmall);        // [width L-1] output-layer weights (columns 0, 1)
    float4* sWout4 = reinterpret_cast<float4*>(sSmall);       // W4: [width L-1] output-layer weights (columns 0 .. 3)
    float* sMisc = sSmall + (W4 ? 512 : 256);                 // [0..1] output bias (W4: [16..19]), [2] |W_out| bound, [4..7] per-warp
                                                              // dmax of the head warps, [8..15] end-of-pass head sums
    float* sBout = W4 ? sMisc + 16 : sMisc;
    float* sThin = sSmall + (W4 ? 544 : 272);                 // [4 sample quarters][8 sums][128] end-of-pass scratch
    float* Hs = reinterpret_cast<float*>(sm + ly.last);
    float4* sPart = reinterpret_cast<float4*>(sm + ly.part);
    float4* sDout = reinterpret_cast<float4*>(sm + ly.dout);
    __half* sXimg = reinterpret_cast<__half*>(sm + ly.ximg);
    const LayerDesc& Lout = pd.L[net][L];
    // ---- stage this net's weights ---------------------------------------------------------------------------------
    __syncthreads();
#pragma unroll
    for (int l = 1; l < L; ++l) {
        const LayerDesc& Ll = pd.L[net][l];
        const int K = wd[l - 1], N = wd[l], KB = K >> 3;
        __half* hi = reinterpret_cast<__half*>(sm + ly.w[l - 1]);
        __half* lo = hi + N * K;
        for (int i0 = tid * 4; i0 < K * N; i0 += FTG_THREADS * 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(a.pack + Ll.pw_off + i0);      // packed [k][n], n contiguous
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
            const int k = i0 / N, nb = i0 - k * N;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = nb + j;
                float w = fminf(fmaxf(wv[j] * FT_C2, -65504.f), 65504.f);
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
        __half* lo = hi + wd[0] * 16;
        for (int i = tid; i < wd[0] * 16; i += FTG_THREADS) {
            const int k = i >> 4, d = i & 15;
            float w = d < D ? a.pack[L0.pw_off + d * L0.Np + k] : (d == D ? a.pack[L0.pb_off + k] : 0.f);
            w = fminf(fmaxf(w * FT_C2, -65504.f), 65504.f);
            const __half h = __float2half_rn(w);
            const int idx = ((k >> 3) * 2 + (d >> 3)) * 64 + (k & 7) * 8 + (d & 7);
            hi[idx] = h;
            lo[idx] = __float2half_rn(w - __half2float(h));
        }
    }
    if (W4) {
        for (int i = tid; i < wd[L - 1]; i += FTG_THREADS) {
            const float* w = a.pack + Lout.pw_off + i * Lout.Np;
            sWout4[i] = make_float4(w[0], w[1], w[2], NOUT > 3 ? w[3] : 0.f);
        }
        if (tid < 4) sBout[tid] = tid < NOUT ? a.pack[Lout.pb_off + tid] : 0.f;
    } else {
        for (int i = tid; i < wd[L - 1]; i += FTG_THREADS)
            sWout[i] = make_float2(a.pack[Lout.pw_off + i * Lout.Np], NOUT > 1 ? a.pack[Lout.pw_off + i * Lout.Np + 1] : 0.f);
        if (tid < 2) sMisc[tid] = tid < NOUT ? a.pack[Lout.pb_off + tid] : 0.f;
    }
    for (int i = tid; i < 2 * 1024; i += FTG_THREADS) {       // x images: rows > obs_dim zero, row obs_dim of the hi image = 1 (bias)
        const int e = i & 1023, d = ((e >> 9) << 3) + ((e >> 3) & 7);
        sXimg[i] = __float2half_rn((i < 1024 && d == D) ? 1.0f : 0.f);
    }
    // per-thread slices of the thin layers
    float bsc[L];                                                  // C2 * b_l of this thread's feature (l >= 1)
#pragma unroll
    for (int l = 1; l < L; ++l) bsc[l] = fl[l] >= 0 ? a.pack[pd.L[net][l].pb_off + fl[l]] * FT_C2 : 0.f;
    bsc[0] = 0.f;
    const int flast = fl[L - 1];
    const float wo0 = flast >= 0 ? a.pack[Lout.pw_off + flast * Lout.Np] : 0.f;
    const float wo1 = (flast >= 0 && NOUT > 1) ? a.pack[Lout.pw_off + flast * Lout.Np + 1] : 0.f;
    const float wo2 = (flast >= 0 && NOUT > 2) ? a.pack[Lout.pw_off + flast * Lout.Np + 2] : 0.f;
    const float wo3 = (flast >= 0 && NOUT > 3) ? a.pack[Lout.pw_off + flast * Lout.Np + 3] : 0.f;
    __syncthreads();
    if (tid < 32) {                                                // bound of the output-layer weight row sums
        float wb = 0.f;
        for (int i = tid; i < wd[L - 1]; i += 32) {
            if (W4) { const float4 w = sWout4[i]; wb = fmaxf(wb, ((fabsf(w.x) + fabsf(w.y)) + fabsf(w.z)) + fabsf(w.w)); }
            else wb = fmaxf(wb, fabsf(sWout[i].x) + fabsf(sWout[i].y));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wb = fmaxf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
        if (tid == 0) sMisc[2] = wb;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const float wbound = sMisc[2];

    // persistent per-thread gradient sums (scaled like the deltas they come from)
    float accb[L];
#pragma unroll
    for (int l = 0; l < L; ++l) accb[l] = 0.f;
    float accW0[FTG_MAX_OBS + 1];
#pragma unroll
    for (int d = 0; d < FTG_MAX_OBS + 1; ++d) accW0[d] = 0.f;
    float accWo0 = 0.f, accWo1 = 0.f, accWo2 = 0.f, accWo3 = 0.f;  // dW_out[flast][0..3] (unscaled)
    float accbo0 = 0.f, accbo1 = 0.f, accls0 = 0.f, accls1 = 0.f;  // head threads: output bias / log_std gradient sums
    float accbo2 = 0.f, accbo3 = 0.f;
    float S = 1.0f, invS = 1.0f;                                   // delta scale of the pass
    bool s_fixed = false;

    const long long n_tiles = (a.mb.count + 63) / 64;
    const int nt = (long long)blockIdx.x < n_tiles ? (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
    const int rec_bytes = ly.rec_floats * 4;
    const unsigned char* rec0 = fa.tiles + (size_t)fa.tile0 * rec_bytes;
    auto load_tile = [&](int it, uint32_t slot) {
        const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
        const uint32_t dst = sm_base + ly.rec + slot * rec_bytes;
        const uint32_t bar = tc_smem_u32(barL + slot);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(rec_bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(rec0 + (size_t)tile * rec_bytes), "r"(rec_bytes), "r"(bar) : "memory");
    };
    auto build_x = [&](uint32_t slot) {               // x of the record in `slot` -> rows 0 .. obs_dim-1 of the x images
        const float* r = reinterpret_cast<const float*>(sm + ly.rec + slot * rec_bytes);
        for (int i = tid; i < 64 * D; i += FTG_THREADS) {
            const int m = i & 63, d = i >> 6;
            const float x = fminf(fmaxf(r[m * Dp + d], -65504.f), 65504.f);
            const __half h = __float2half_rn(x);
            const int idx = ((d >> 3) * 8 + (m >> 3)) * 64 + (d & 7) * 8 + (m & 7);
            sXimg[idx] = h;
            sXimg[1024 + idx] = __float2half_rn(x - __half2float(h));
        }
    };
    auto issue_g0 = [&]() {
        const uint32_t id = ft_idesc(wd[0], 64, 0, 1);
#pragma unroll
        for (int ps = 0; ps < 3; ++ps)
            ft_mma(tb + FTG_COL_D0, tc_desc(sm_base + ly.w0a + (ps == 1 ? wd[0] * 32 : 0), 128, 256, 0),
                   tc_desc(sm_base + ly.ximg + (ps == 2 ? 2048 : 0), 1024, 128, 0), id, ps ? 1u : 0u);
        tc_commit(barG0);
    };
    // one GEMM with the three hi/lo products: a_img / b_img = byte offsets of the hi images, *_lo = distance to the lo image,
    // steps = K / 16, a_step / b_step = descriptor advance per K step
    auto gemm3 = [&](uint32_t d_col, uint32_t idesc, uint32_t a_img, uint32_t a_lo, uint32_t a_step, uint32_t a_lbo, uint32_t a_sbo,
                     uint32_t b_img, uint32_t b_lo, uint32_t b_step, uint32_t b_lbo, uint32_t b_sbo, int steps, bool accumulate) {
#pragma unroll
        for (int ps = 0; ps < 3; ++ps) {
            const uint32_t ai = sm_base + a_img + (ps == 1 ? a_lo : 0), bi = sm_base + b_img + (ps == 2 ? b_lo : 0);
            for (int kk = 0; kk < steps; ++kk)
                ft_mma(tb + d_col, tc_desc(ai + kk * a_step, a_lbo, a_sbo, 0), tc_desc(bi + kk * b_step, b_lbo, b_sbo, 0), idesc,
                       (accumulate || ps || kk) ? 1u : 0u);
        }
    };
    // forward GEMM of layer l: D = W_l^T-image (K-major A) x H_{l-1} image (MN-major B)
    auto issue_fwd = [&](int l) {
        const int K = wd[l - 1], N = wd[l];
        gemm3(FTG_COL_D, ft_idesc(N, 64, 0, 1), ly.w[l - 1], N * K * 2, 256, 128, (K >> 3) * 128, ly.h[l - 1], K * 128, 2048, 1024, 128, K >> 4, false);
        tc_commit(barM);
    };
    // dH_{l-1} = W_l dZ_l (A = W_l image MN-major, B = dZ_l image MN-major) and dW_l += H_{l-1} dZ_l^T (A, B K-major)
    auto issue_bwd = [&](int l, uint32_t z_img, bool first_tile) {
        const int K = wd[l - 1], N = wd[l];
        gemm3(FTG_COL_D, ft_idesc(K, 64, 1, 1), ly.w[l - 1], N * K * 2, 2 * (K >> 3) * 128, (K >> 3) * 128, 128, z_img, N * 128, 2048, 1024, 128, N >> 4, false);
        tc_commit(barM);
        gemm3(FTG_COL_DW + (l - 1) * 128, ft_idesc(K, N, 0, 0), ly.h[l - 1], K * 128, 256, 128, 1024, z_img, N * 128, 256, 128, 1024, 4, !first_tile);
        tc_commit(barW);
    };

    uint32_t rslot = n_rec & 1u;
    if (nt > 0) {
        if (tid == 0) load_tile(0, rslot);
        tc_wait(barL + rslot, (n_rec >> 1) & 1u);
        build_x(rslot);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (issuer && tc_elect_one()) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            issue_g0();
        }
    }
    for (int it = 0; it < nt; ++it) {
        rslot = n_rec & 1u;
        const float* rec = reinterpret_cast<const float*>(sm + ly.rec + rslot * rec_bytes);
        const float* sc = rec + 64 * Dp;
        if (tid == 0 && it + 1 < nt) load_tile(it + 1, rslot ^ 1u);
        tc_wait(barG0, n_g0 & 1u); ++n_g0;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- forward: A_l (tanh, images, derivative stash) and G_{l+1} ----------------------------------------------------
#pragma unroll
        for (int l = 0; l < L; ++l) {
            float v[16];
            ft_ld16(my + (l == 0 ? FTG_COL_D0 : FTG_COL_D) + m0, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = ft_tanh_scaled(v[j] + bsc[l]);
            if (l + 1 < L) {
                if (fl[l] >= 0) {
                    unsigned char* ph = sm + ly.h[l];
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint4 vh, vl;
                        ft_split2(v[8 * c], v[8 * c + 1], vh.x, vl.x); ft_split2(v[8 * c + 2], v[8 * c + 3], vh.y, vl.y);
                        ft_split2(v[8 * c + 4], v[8 * c + 5], vh.z, vl.z); ft_split2(v[8 * c + 6], v[8 * c + 7], vh.w, vl.w);
                        const uint32_t off = ft_row_off(fl[l], m0 + 8 * c);
                        *reinterpret_cast<uint4*>(ph + off) = vh;
                        *reinterpret_cast<uint4*>(ph + wd[l] * 128 + off) = vl;
                    }
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = fmaf(-v[j], v[j], 1.0f);
                ftg_st16(my + FTG_COL_G + l * 64 + m0, v);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncthreads();
                if (issuer && tc_elect_one()) {
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    issue_fwd(l + 1);
                }
                tc_wait(barM, n_mma & 1u); ++n_mma;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            } else {
                // last hidden layer: fp32 tile for the output layer, H kept in D for the delta phase
                if (fl[l] >= 0) {
                    float* hr = Hs + fl[l] * FT_HS_LD + m0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(hr + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
                ftg_st16(my + FTG_COL_D + m0, v);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                __syncthreads();
            }
        }
        // ---- output layer partials: thread <-> (sample ms, feature slice) -------------------------------------------------
        {
            const int per = wd[L - 1] >> 3;
            float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
            const float* hp = Hs + (slice * per) * FT_HS_LD + ms;
            for (int n = 0; n < per; ++n) {
                const float hv = hp[n * FT_HS_LD];
                if (W4) {
                    const float4 w = sWout4[slice * per + n];
                    p0 = fmaf(hv, w.x, p0); p1 = fmaf(hv, w.y, p1); p2 = fmaf(hv, w.z, p2); p3 = fmaf(hv, w.w, p3);
                } else {
                    const float2 w = sWout[slice * per + n];
                    p0 = fmaf(hv, w.x, p0);
                    if (NOUT > 1) p1 = fmaf(hv, w.y, p1);
                }
            }
            sPart[slice * 64 + ms] = make_float4(p0, p1, p2, p3);
        }
        __syncthreads();
        // ---- loss head: one thread per sample (warps 0 and 1) ----------------------------------------------------------------
        if (tid < 64) {
            constexpr int NA = W4 ? 4 : 2;
            float out[NA];
#pragma unroll
            for (int j = 0; j < NA; ++j) out[j] = sBout[j];
#pragma unroll
            for (int sl = 0; sl < 8; ++sl) {
                const float4 p = sPart[sl * 64 + ms];
                out[0] += p.x; out[1] += p.y;
                if (W4) { out[2] += p.z; out[3] += p.w; }
            }
            const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
            const bool valid = tile * 64 + ms < a.mb.count;
            float dout[NA];
#pragma unroll
            for (int j = 0; j < NA; ++j) dout[j] = 0.f;
            if (HEAD == 2) {
                const float ret = sc[128 + ms], ov = sc[192 + ms];
                const float v_raw = out[0];
                float v = v_raw;
                bool v_pass = true;
                if (a.hp.clip_range_vf >= 0.f) {
                    const float dlt = v_raw - ov;
                    v_pass = dlt >= -a.hp.clip_range_vf && dlt <= a.hp.clip_range_vf;
                    v = ov + fminf(fmaxf(dlt, -a.hp.clip_range_vf), a.hp.clip_range_vf);
                }
                const float verr = v - ret;
                dout[0] = (valid && v_pass) ? a.hp.vf_coef * 2.0f * verr * invB : 0.f;
                if (valid) stats[1] += verr * verr;
            } else {
                float adv = sc[ms];
                if (valid && a.hp.normalize_advantage) adv = (adv - adv_mean) / adv_den;
                const float olp = sc[64 + ms];
                float logp = 0.f, ent = 0.f;
                float pj[NA], lpj[NA], diff[NA], vi[NA];
#pragma unroll
                for (int j = 0; j < NA; ++j) { pj[j] = 0.f; lpj[j] = 0.f; diff[j] = 0.f; vi[j] = 0.f; }
                int aidx = 0;
                if (HEAD == 0) {
                    aidx = reinterpret_cast<const int*>(sc)[256 + ms];
                    int jmax = 0;
                    float mx = out[0];
                    if (NOUT > 1 && out[1] > mx) { mx = out[1]; jmax = 1; }
                    if (NOUT > 2 && out[2] > mx) { mx = out[2]; jmax = 2; }
                    if (NOUT > 3 && out[3] > mx) { mx = out[3]; jmax = 3; }
                    float ex[NA], s = 0.f;
#pragma unroll
                    for (int j = 0; j < NOUT; ++j) { ex[j] = j == jmax ? 1.0f : expf(out[j] - mx); s += ex[j]; }
                    float hsum = 0.f;
#pragma unroll
                    for (int j = 0; j < NOUT; ++j) {
                        pj[j] = ex[j] / s; lpj[j] = logf(pj[j]); hsum += pj[j] * lpj[j];
                        if (j == aidx) logp = lpj[j];
                    }
                    ent = -hsum;
                } else {
                    float ls_sum = 0.f, dss = 0.f;
#pragma unroll
                    for (int j = 0; j < NOUT; ++j) {
                        const float ls = a.flat[pd.log_std_off + j];
                        vi[j] = expf(-2.0f * ls);
                        diff[j] = sc[256 + j * 64 + ms] - out[j];
                        dss += diff[j] * diff[j] * vi[j];
                        ls_sum += ls;
                    }
                    logp = -0.5f * (2.0f * ls_sum + dss + (float)NOUT * DRIL_LOG2PI);
                    ent = 0.5f * (float)NOUT * (1.0f + DRIL_LOG2PI) + ls_sum;
                }
                const float log_ratio = logp - olp;
                const float ratio = expf(log_ratio);
                const float rc = fminf(fmaxf(ratio, 1.0f - a.hp.clip_range), 1.0f + a.hp.clip_range);
                const float s1 = ratio * adv, s2 = rc * adv;
                const float g_logp = (!valid || s2 < s1) ? 0.f : -invB * adv * ratio;       // min(s1, s2): ties -> s1
                const float g_ent = valid ? -a.hp.ent_coef * invB : 0.f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) {
                    if (HEAD == 0) dout[j] = g_logp * ((j == aidx ? 1.0f : 0.0f) - pj[j]) + g_ent * (-pj[j] * (lpj[j] + ent));
                    else {
                        dout[j] = g_logp * diff[j] * vi[j];
                        const float dls = g_logp * (-1.0f + diff[j] * diff[j] * vi[j]) + g_ent;      // d/dlog_std_j
                        if (j == 0) accls0 += dls; else accls1 += dls;
                    }
                }
                if (valid) {
                    stats[0] += -fminf(s1, s2);
                    stats[2] += ent;
                    stats[3] += (ratio != rc) ? 1.0f : 0.0f;
                    stats[4] += ratio - 1.0f - log_ratio;
                    stats[5] += ratio;
                }
            }
            accbo0 += dout[0]; accbo1 += dout[1];
            if (W4) { accbo2 += dout[2]; accbo3 += dout[3]; }
            sDout[ms] = make_float4(dout[0], dout[1], W4 ? dout[2] : 0.f, W4 ? dout[3] : 0.f);
            float dmax = fmaxf(fabsf(dout[0]), fabsf(dout[1]));
            if (W4) dmax = fmaxf(dmax, fmaxf(fabsf(dout[2]), fabsf(dout[3])));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
            if (lane == 0) sMisc[4 + warp] = dmax;
        }
        __syncthreads();
        // ---- dZ_{L-1} = (W_out dout) .* (1 - H^2), scaled -> delta images (over the fp32 tile); bias / W_out sums -------------
        {
            const float bound = fmaxf(sMisc[4], sMisc[5]) * wbound * (float)NOUT;
            float z[16];
            ft_ld16(my + FTG_COL_D + m0, z);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            // the pass's delta scale: fixed at the first tile with a non-zero gradient; a later tile whose bound would reach 2^14
            // moves it down to sit where the first tile sat, and the dW accumulators in TMEM and the scaled register sums are
            // multiplied by the exact ratio of the two powers of two (the previous tile's dW GEMMs completed at barW, this
            // tile's are issued after the barrier that follows the delta images).  The decision is CTA-uniform; its shared
            // memory loads were issued before the TMEM load above.
            if (bound > 0.f && bound < 3.0e38f && (!s_fixed || bound * S >= 16384.0f)) {
                int E = ((__float_as_int(bound) >> 23) & 255) - 127;              // bound < 2^(E + 1)
                E = E < -100 ? -100 : (E > 100 ? 100 : E);
                if (s_fixed) {
                    const int d = (128 - (__float_as_int(S) >> 23)) - E;          // S = 2^(1 - E_old): S_new / S_old = 2^d, -200 <= d <= 0
                    const float r1 = __int_as_float((d / 2 + 127) << 23), r2 = __int_as_float((d - d / 2 + 127) << 23);
#pragma unroll
                    for (int l = 1; l < L; ++l) ft_rescale_tmem(my + FTG_COL_DW + (l - 1) * 128 + sg * (wd[l] >> 2), wd[l] >> 2, r1, r2);
#pragma unroll
                    for (int l = 0; l < L; ++l) accb[l] = (accb[l] * r1) * r2;
#pragma unroll
                    for (int k = 0; k < FTG_MAX_OBS + 1; ++k) accW0[k] = (accW0[k] * r1) * r2;
                }
                S = __int_as_float((1 - E + 127) << 23);                          // S * bound < 2^2
                invS = __int_as_float((E - 1 + 127) << 23);
                s_fixed = true;
            }
            const float ws0 = wo0 * S, ws1 = wo1 * S, ws2 = wo2 * S, ws3 = wo3 * S;
            float sb = 0.f, sw0 = 0.f, sw1 = 0.f, sw2 = 0.f, sw3 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float4 d = sDout[m0 + j];
                const float h = z[j];
                sw0 = fmaf(h, d.x, sw0);
                if (NOUT > 1) sw1 = fmaf(h, d.y, sw1);
                if (NOUT > 2) sw2 = fmaf(h, d.z, sw2);
                if (NOUT > 3) sw3 = fmaf(h, d.w, sw3);
                float u = d.x * ws0;
                if (NOUT > 1) u = fmaf(d.y, ws1, u);
                if (NOUT > 2) u = fmaf(d.z, ws2, u);
                if (NOUT > 3) u = fmaf(d.w, ws3, u);
                z[j] = u * fmaf(-h, h, 1.0f);
                sb += z[j];
            }
            if (flast >= 0) {
                accb[L - 1] += sb; accWo0 += sw0; accWo1 += sw1;
                if (W4) { accWo2 += sw2; accWo3 += sw3; }
                unsigned char* pz = sm + ly.last;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint4 vh, vl;
                    ft_split2(z[8 * c], z[8 * c + 1], vh.x, vl.x); ft_split2(z[8 * c + 2], z[8 * c + 3], vh.y, vl.y);
                    ft_split2(z[8 * c + 4], z[8 * c + 5], vh.z, vl.z); ft_split2(z[8 * c + 6], z[8 * c + 7], vh.w, vl.w);
                    const uint32_t off = ft_row_off(flast, m0 + 8 * c);
                    *reinterpret_cast<uint4*>(pz + off) = vh;
                    *reinterpret_cast<uint4*>(pz + wd[L - 1] * 128 + off) = vl;
                }
            }
        }
        ++n_rec;
        if (it + 1 < nt) {                                       // x images of the next tile (its record arrived long ago)
            tc_wait(barL + (rslot ^ 1u), (n_rec >> 1) & 1u);
            build_x(rslot ^ 1u);
        }
        // NOTE: the Hs reads of the output-layer phase ended before the barrier after the head, and the delta images above were
        // written after it, so the aliasing of the fp32 tile and the delta images is race free
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- backward: for l = L-1 .. 1: {dH_{l-1}, dW_l} on the tensor cores, then dZ_{l-1} --------------------------------------
#pragma unroll
        for (int l = L - 1; l >= 1; --l) {
            const uint32_t z_img = l == L - 1 ? ly.last : ly.h[l];
            if (issuer && tc_elect_one()) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue_bwd(l, z_img, it == 0);
                if (l == L - 1 && it + 1 < nt) issue_g0();
            }
            tc_wait(barM, n_mma & 1u); ++n_mma;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float dz[16], gd[16];
            ft_ld16(my + FTG_COL_D + m0, dz);
            ft_ld16(my + FTG_COL_G + (l - 1) * 64 + m0, gd);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float sb = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) { dz[j] *= gd[j]; sb += dz[j]; }
            if (fl[l - 1] >= 0) accb[l - 1] += sb;
            // the dW_l GEMM reads H_{l-1} (and the delta image of layer l): it must be done before the buffers are reused
            tc_wait(barW, n_w & 1u); ++n_w;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (l - 1 >= 1) {
                if (fl[l - 1] >= 0) {
                    unsigned char* pz = sm + ly.h[l - 1];
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint4 vh, vl;
                        ft_split2(dz[8 * c], dz[8 * c + 1], vh.x, vl.x); ft_split2(dz[8 * c + 2], dz[8 * c + 3], vh.y, vl.y);
                        ft_split2(dz[8 * c + 4], dz[8 * c + 5], vh.z, vl.z); ft_split2(dz[8 * c + 6], dz[8 * c + 7], vh.w, vl.w);
                        const uint32_t off = ft_row_off(fl[l - 1], m0 + 8 * c);
                        *reinterpret_cast<uint4*>(pz + off) = vh;
                        *reinterpret_cast<uint4*>(pz + wd[l - 1] * 128 + off) = vl;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncthreads();
            } else {
                // layer 0: dW_0[d][f] += sum_m dZ_0[f][m] x[m][d]
                if (fl[0] >= 0) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float* x = rec + (m0 + j) * Dp;
#pragma unroll
                        for (int d4 = 0; d4 < FTG_MAX_OBS + 1; d4 += 4) {
                            if (d4 < Dp) {
                                const float4 xv = *reinterpret_cast<const float4*>(x + d4);
                                accW0[d4] = fmaf(dz[j], xv.x, accW0[d4]); accW0[d4 + 1] = fmaf(dz[j], xv.y, accW0[d4 + 1]);
                                accW0[d4 + 2] = fmaf(dz[j], xv.z, accW0[d4 + 2]); accW0[d4 + 3] = fmaf(dz[j], xv.w, accW0[d4 + 3]);
                            }
                        }
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncthreads();                                 // records, image buffers and D are free for the next tile
            }
        }
    }
    // ---- end of the pass: dW_l from TMEM, thin sums over the four sample quarters -> this CTA's partial plane -----------------------
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float kap[L];                                                 // delta scale of layer l: S * C2^(L-1-l)
    kap[L - 1] = invS;
#pragma unroll
    for (int l = L - 2; l >= 0; --l) kap[l] = kap[l + 1] * (1.0f / FT_C2);
#pragma unroll
    for (int l = 1; l < L; ++l) {
        const LayerDesc& Ll = pd.L[net][l];
        const int N = wd[l], per = N >> 2;                        // this warp's columns: sg * per .. + per
        if (nt > 0) {
            for (int c0 = 0; c0 < per; c0 += 16) {
                float v[16];
                ft_ld16(my + FTG_COL_DW + (l - 1) * 128 + sg * per + c0, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (fl[l - 1] >= 0) {
                    float* g = gp + Ll.pw_off + fl[l - 1] * N + sg * per + c0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                        *reinterpret_cast<float4*>(g + j) = make_float4(v[j] * kap[l], v[j + 1] * kap[l], v[j + 2] * kap[l], v[j + 3] * kap[l]);
                }
            }
        } else if (fl[l - 1] >= 0) {
            float* g = gp + Ll.pw_off + fl[l - 1] * N + sg * per;
            for (int j = 0; j < per; ++j) g[j] = 0.f;
        }
    }
    // thin sums: per layer bias, layer-0 weights, output-layer weights: sum over the four sample quarters through shared memory
    const int lane_f = 32 * q + lane;                             // scratch column of this thread
    auto quarter_sum = [&](float v, int slot) { sThin[(sg * 8 + slot) * 128 + lane_f] = v; };
    auto reduce_write = [&](int slot, int width, int layer_of_map, auto&& dst) {
        __syncthreads();
        for (int i = tid; i < 128; i += FTG_THREADS) {
            const float s = (sThin[(0 * 8 + slot) * 128 + i] + sThin[(1 * 8 + slot) * 128 + i]) + (sThin[(2 * 8 + slot) * 128 + i] + sThin[(3 * 8 + slot) * 128 + i]);
            // scratch column i belongs to feature: width 128 -> i, width 64 -> lanes 0..15 of quadrant i / 32
            const int ql = i >> 5, ll = i & 31;
            const int f = width == 128 ? i : (ll < 16 ? 16 * ql + ll : -1);
            if (f >= 0) dst(f, s);
        }
        __syncthreads();
        (void)layer_of_map;
    };
    // (a) biases of the hidden layers
#pragma unroll
    for (int l = 0; l < L; ++l) {
        quarter_sum(accb[l] * kap[l], 0);
        const LayerDesc& Ll = pd.L[net][l];
        reduce_write(0, wd[l], l, [&](int f, float s) { gp[Ll.pb_off + f] = s; });
    }
    // (b) layer-0 weights
    {
        const LayerDesc& L0 = pd.L[net][0];
#pragma unroll
        for (int d = 0; d < FTG_MAX_OBS + 1; ++d) {
            if (d < D) {
                quarter_sum(accW0[d] * kap[0], 0);
                reduce_write(0, wd[0], 0, [&](int f, float s) { gp[L0.pw_off + d * L0.Np + f] = s; });
            }
        }
    }
    // (c) output layer weights (unscaled), bias, log_std
    quarter_sum(accWo0, 0);
    reduce_write(0, wd[L - 1], L - 1, [&](int f, float s) { gp[Lout.pw_off + f * Lout.Np] = s; });
    if (NOUT > 1) {
        quarter_sum(accWo1, 0);
        reduce_write(0, wd[L - 1], L - 1, [&](int f, float s) { gp[Lout.pw_off + f * Lout.Np + 1] = s; });
    }
    if (NOUT > 2) {
        quarter_sum(accWo2, 0);
        reduce_write(0, wd[L - 1], L - 1, [&](int f, float s) { gp[Lout.pw_off + f * Lout.Np + 2] = s; });
    }
    if (NOUT > 3) {
        quarter_sum(accWo3, 0);
        reduce_write(0, wd[L - 1], L - 1, [&](int f, float s) { gp[Lout.pw_off + f * Lout.Np + 3] = s; });
    }
    if (tid < 64) {
        float hv[4] = {accbo0, accbo1, W4 ? accbo2 : accls0, W4 ? accbo3 : accls1};   // W4: discrete head, no log_std
#pragma unroll
        for (int i = 0; i < 4; ++i) hv[i] = warp_sum(hv[i]);
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) sMisc[8 + warp * 4 + i] = hv[i];
        }
    }
    __syncthreads();
    if (tid < 4) {
        const float s = sMisc[8 + tid] + sMisc[12 + tid];
        if (W4) { if (tid < NOUT) gp[Lout.pb_off + tid] = s; }
        else if (tid < 2) { if (tid < NOUT) gp[Lout.pb_off + tid] = s; }
        else if (HEAD == 1 && tid - 2 < NOUT) gp[pd.pack_fwd + (tid - 2)] = s;
    }
    __syncthreads();
}

template <int L, int CONT, int NOUT>
__global__ void __launch_bounds__(FTG_THREADS, 1) ppo_loss_grad_ftg_kernel(const __grid_constant__ LossArgs a, const __grid_constant__ TailArgs tl,
                                                                           const __grid_constant__ FtgArgs fa) {
    extern __shared__ __align__(1024) unsigned char ftg_smem_raw[];
    __shared__ __align__(8) uint64_t bars[8];
    __shared__ uint32_t tmem_base_s;
    __shared__ double scratch[32];
    __shared__ float s_f2[2];
    if (*a.stop_flag) return;
    const PolicyDesc& pd = a.pd;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const uint32_t raw = tc_smem_u32(ftg_smem_raw);
    const uint32_t sm_base = (raw + 1023u) & ~1023u;
    unsigned char* sm = ftg_smem_raw + (sm_base - raw);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(FTG_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&bars[i])));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);
    float adv_mean = 0.f, adv_den = 1.f;
    if (a.hp.normalize_advantage) {
        const double n = a.mb.global_count;
        const double mean = a.mbstats[0] / n;
        double var = (a.mbstats[1] - n * mean * mean) / (n - 1.0);
        if (var < 0.0) var = 0.0;
        adv_mean = (float)mean;
        adv_den = (float)sqrt(var) + 1e-8f;
    }
    const float invB = (float)(1.0 / a.mb.global_count);
    float stats[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float* gp = a.gpart + (size_t)blockIdx.x * pd.gpack;
    uint32_t n_rec = 0, n_g0 = 0, n_mma = 0, n_w = 0;  // completed phases of the record / G0 / GEMM / dW barriers (parities)
    ftg_pass<L, CONT ? 1 : 0, NOUT>(a, fa, sm, sm_base, tb, bars, n_rec, n_g0, n_mma, n_w, adv_mean, adv_den, invB, stats, gp);
    ftg_pass<L, 2, 1>(a, fa, sm, sm_base, tb, bars, n_rec, n_g0, n_mma, n_w, adv_mean, adv_den, invB, stats, gp);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double s = block_sum((double)stats[i], scratch);
        if (tid == 0) gp[pd.pack_fwd + pd.act_n + i] = (float)s;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(FTG_TMEM_COLS));
    if (tl.mode) tc_fused_tail(a, tl, reinterpret_cast<float*>(sm + fa.lay.part), scratch, s_f2);
}

// ---------------------------------------------------------------------------------------------------------------------
// Batched critic for the general rollout (rollout.cuh, RO_DEFER_CRITIC): V of all T*N buffer observations, of the N final
// observations (bootstrap of trajectories cut by the rollout end, trajectory.jl:65-70) and of the terminal observations of
// truncated steps (trajectory.jl:57-61), all already normalised as the policy saw them.  Forward half of ftg_pass for the
// critic net: 64 observations per tile, G0 -> tanh -> G1 -> tanh [-> G2 -> tanh] on tcgen05, output layer on CUDA cores.
// ---------------------------------------------------------------------------------------------------------------------
template <int L>
__global__ void __launch_bounds__(FTG_THREADS, 1) critic_values_ftg_kernel(const __grid_constant__ PolicyDesc pd, const float* __restrict__ pack,
                                                                           const BufDev buf, const DeferredCritic dc,
                                                                           const __grid_constant__ FtgLayout ly) {
    extern __shared__ __align__(1024) unsigned char ftg_smem_raw[];
    __shared__ __align__(8) uint64_t barM;
    __shared__ uint32_t tmem_base_s;
    constexpr int net = 1;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int lane = tid & 31, q = warp & 3, sg = warp >> 2;
    const int m0 = 16 * sg, ms = tid & 63, slice = tid >> 6;
    const bool issuer = warp == 0;
    const uint32_t raw = tc_smem_u32(ftg_smem_raw);
    const uint32_t sm_base = (raw + 1023u) & ~1023u;
    unsigned char* sm = ftg_smem_raw + (sm_base - raw);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(64));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&barM)));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    int wd[L], fl[L];
#pragma unroll
    for (int l = 0; l < L; ++l) {
        wd[l] = pd.L[net][l].N;
        fl[l] = wd[l] == 128 ? 32 * q + lane : (lane < 16 ? 16 * q + lane : -1);
    }
    const int D = pd.obs_dim;
    float* sSmall = reinterpret_cast<float*>(sm + ly.small);
    float2* sWout = reinterpret_cast<float2*>(sSmall);
    float* sMisc = sSmall + 256;
    float* Hs = reinterpret_cast<float*>(sm + ly.last);
    float4* sPart = reinterpret_cast<float4*>(sm + ly.part);
    __half* sXimg = reinterpret_cast<__half*>(sm + ly.ximg);
    const LayerDesc& Lout = pd.L[net][L];
    // ---- the critic's weights: images of C2 * W_l (l >= 1), of C2 * [W_0; b_0]^T, output layer in fp32 -------------------------
#pragma unroll
    for (int l = 1; l < L; ++l) {
        const LayerDesc& Ll = pd.L[net][l];
        const int K = wd[l - 1], N = wd[l], KB = K >> 3;
        __half* hi = reinterpret_cast<__half*>(sm + ly.w[l - 1]);
        __half* lo = hi + N * K;
        for (int i0 = tid * 4; i0 < K * N; i0 += FTG_THREADS * 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(pack + Ll.pw_off + i0);
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
        __half* lo = hi + wd[0] * 16;
        for (int i = tid; i < wd[0] * 16; i += FTG_THREADS) {
            const int k = i >> 4, d = i & 15;
            float w = d < D ? pack[L0.pw_off + d * L0.Np + k] : (d == D ? pack[L0.pb_off + k] : 0.f);
            w = fminf(fmaxf(w * FT_C2, -65504.f), 65504.f);
            const __half h = __float2half_rn(w);
            const int idx = ((k >> 3) * 2 + (d >> 3)) * 64 + (k & 7) * 8 + (d & 7);
            hi[idx] = h;
            lo[idx] = __float2half_rn(w - __half2float(h));
        }
    }
    for (int i = tid; i < wd[L - 1]; i += FTG_THREADS) sWout[i] = make_float2(pack[Lout.pw_off + i * Lout.Np], 0.f);
    if (tid == 0) sMisc[0] = pack[Lout.pb_off];
    for (int i = tid; i < 2 * 1024; i += FTG_THREADS) {
        const int e = i & 1023, d = ((e >> 9) << 3) + ((e >> 3) & 7);
        sXimg[i] = __float2half_rn((i < 1024 && d == D) ? 1.0f : 0.f);
    }
    float bsc[L];
#pragma unroll
    for (int l = 1; l < L; ++l) bsc[l] = fl[l] >= 0 ? pack[pd.L[net][l].pb_off + fl[l]] * FT_C2 : 0.f;
    bsc[0] = 0.f;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);
    const uint32_t my = tb + ((uint32_t)(q * 32) << 16);
    const long long TN = buf.T * buf.N;
    const unsigned int ntr = min(*dc.trunc_count, dc.cap);
    const long long total = TN + buf.N + (long long)ntr;
    const long long n_tiles = (total + 63) / 64;
    uint32_t n_mma = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // ---- x of the tile's 64 observations -> fp16 hi / lo rows of the x images ---------------------------------------------
        for (int i = tid; i < 64 * D; i += FTG_THREADS) {
            const int m = i & 63, d = i >> 6;
            const long long v = tile * 64 + m;
            float x = 0.f;
            if (v < TN) x = buf.obs[v * D + d];
            else if (v < TN + buf.N) x = dc.last_obs[(v - TN) * D + d];
            else if (v < total) x = dc.trunc_obs[(v - TN - buf.N) * D + d];
            x = fminf(fmaxf(x, -65504.f), 65504.f);
            const __half h = __float2half_rn(x);
            const int idx = ((d >> 3) * 8 + (m >> 3)) * 64 + (d & 7) * 8 + (m & 7);
            sXimg[idx] = h;
            sXimg[1024 + idx] = __float2half_rn(x - __half2float(h));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
#pragma unroll
        for (int l = 0; l < L; ++l) {
            if (issuer && tc_elect_one()) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (l == 0) {
                    const uint32_t id = ft_idesc(wd[0], 64, 0, 1);
#pragma unroll
                    for (int ps = 0; ps < 3; ++ps)
                        ft_mma(tb, tc_desc(sm_base + ly.w0a + (ps == 1 ? wd[0] * 32 : 0), 128, 256, 0),
                               tc_desc(sm_base + ly.ximg + (ps == 2 ? 2048 : 0), 1024, 128, 0), id, ps ? 1u : 0u);
                } else {
                    const int K = wd[l - 1], N = wd[l];
                    const uint32_t id = ft_idesc(N, 64, 0, 1);
#pragma unroll
                    for (int ps = 0; ps < 3; ++ps) {
                        const uint32_t ai = sm_base + ly.w[l - 1] + (ps == 1 ? N * K * 2 : 0), bi = sm_base + ly.h[l - 1] + (ps == 2 ? K * 128 : 0);
                        for (int kk = 0; kk < (K >> 4); ++kk)
                            ft_mma(tb, tc_desc(ai + kk * 256, 128, (K >> 3) * 128, 0), tc_desc(bi + kk * 2048, 1024, 128, 0), id, (ps || kk) ? 1u : 0u);
                    }
                }
                tc_commit(&barM);
            }
            tc_wait(&barM, n_mma & 1u); ++n_mma;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float v[16];
            ft_ld16(my + m0, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = ft_tanh_scaled(v[j] + bsc[l]);
            if (l + 1 < L) {
                if (fl[l] >= 0) {
                    unsigned char* ph = sm + ly.h[l];
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint4 vh, vl;
                        ft_split2(v[8 * c], v[8 * c + 1], vh.x, vl.x); ft_split2(v[8 * c + 2], v[8 * c + 3], vh.y, vl.y);
                        ft_split2(v[8 * c + 4], v[8 * c + 5], vh.z, vl.z); ft_split2(v[8 * c + 6], v[8 * c + 7], vh.w, vl.w);
                        const uint32_t off = ft_row_off(fl[l], m0 + 8 * c);
                        *reinterpret_cast<uint4*>(ph + off) = vh;
                        *reinterpret_cast<uint4*>(ph + wd[l] * 128 + off) = vl;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            } else if (fl[l] >= 0) {
                float* hr = Hs + fl[l] * FT_HS_LD + m0;
#pragma unroll
                for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(hr + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
        }
        {
            const int per = wd[L - 1] >> 3;
            float p0 = 0.f;
            const float* hp = Hs + (slice * per) * FT_HS_LD + ms;
            for (int n = 0; n < per; ++n) p0 = fmaf(hp[n * FT_HS_LD], sWout[slice * per + n].x, p0);
            sPart[slice * 64 + ms] = make_float4(p0, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        if (tid < 64) {
            float val = sMisc[0];
#pragma unroll
            for (int sl = 0; sl < 8; ++sl) val += sPart[sl * 64 + ms].x;
            const long long v = tile * 64 + ms;
            if (v < TN) buf.values[v] = val;
            else if (v < TN + buf.N) buf.last_values[v - TN] = val;
            else if (v < total) buf.boot[dc.trunc_idx[v - TN - buf.N]] = val;
        }
        __syncthreads();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(64));
}
