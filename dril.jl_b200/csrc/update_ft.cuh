// Features-on-lanes ("transposed") tensor-core variant of the fused PPO loss forward/backward for the reference's
// default network shape (two tanh MLPs, hidden_dims = [64, 64], obs_dim <= 4, Discrete(n <= 2); loss functor
// algorithms/ppo.jl:365-407, evaluate_actions layers/layer_methods.jl:46-55, Zygote reverse pass).
//
// Why transposed.  update_tc.cuh puts SAMPLES on TMEM lanes (D[m][n]); every sum over samples (db, dW of the thin
// layers) then needs cross-lane reductions and every MN-major image a transposing write, and actor and critic are two
// passes.  Here FEATURES sit on the lanes and samples on the columns:
//   G1  H1pre[n][m] = sum_k W1[k][n] H0[k][m]      A = W1 image [n][k] (K-major),   B = H0 image [k][m] (MN-major)
//   G2  dH0[k][m]   = sum_n W1[k][n] dZ1[n][m]     A = the same W1 image (MN-major), B = dZ1 image [n][m] (MN-major)
//   G3  dW1[k][n]   = sum_m H0[k][m] dZ1[n][m]     A = the same H0 image (K-major),  B = the same dZ1 image (K-major)
// so that thread <-> (net, feature) and its registers run over samples: all bias / thin-layer gradient sums are private
// register accumulations, the per-feature weights (W0 column, biases, W2 row) live in registers, and in the no-swizzle
// core layout of 16-bit operands ONE image per matrix serves both orientations (tools/ft_probe.cu, profiles/r02_ft_probe.txt).
// The only per-sample phase is the output layer + loss head (H1 through a shared-memory fp32 tile).
//
// Precision: fp16 hi/lo split on kind::f16 (x = hi + lo, hi = fp16(x), lo = fp16(x - hi); products hi*hi + lo*hi +
// hi*lo, fp32 accumulation): 22 significant bits like 3xTF32 at half the instructions and half the operand bytes.
// H0/H1 are tanh outputs and W1 is a weight matrix (bounded); the deltas dZ1 are not, so every group scales them by a
// power of two S chosen from a tile's max |dL/dout| and the net's max |W2| row sum such that |S dZ1|
// is below 2^4 on the tile that fixes it (the first tile of a group with a non-zero gradient).  dW1 stays in TMEM over all
// tiles of a group and everything is unscaled exactly at the end.  A later tile whose scaled bound would pass fp16's
// 65504 lowers S to sit where the first tile sat, and the group's dW1 columns and scaled sums are multiplied by the
// exact ratio; tiles inside that headroom compute what a fixed S computes.
//
// M = 64 accumulators use 16 lanes of every TMEM lane quadrant; the actor's sit at lane offset 0 and the critic's at
// lane offset 16 of the same columns, so warp q, lane l is feature 16 q + l % 16 of net l / 16 and both nets run in ONE
// pass over the minibatch.  Two groups of 8 warps work on alternate 64-sample tiles with private images and TMEM
// columns (no hand-over between the groups); within a group warps w and w + 4 share a lane quadrant and split the
// tile's samples.  Tiles arrive as contiguous 2304-byte records written for ALL epochs of the update by one launch of
// ft_permute_epochs_kernel (the DataLoader shuffle of ppo.jl:188-195, plus the minibatch advantage moments) and are
// prefetched with cp.async.bulk + mbarrier one tile ahead.
// A minibatch step ends with the cooperative tail of update_tc.cuh (reduction, peer exchange, clip, KL stop, Adam); in
// persistent mode (FtArgs::n_steps > 0) the kernel then crosses a grid barrier and runs the next step of the update.
#pragma once
#include <cuda_fp16.h>
#include "update_tc.cuh"

#define FT_TS 64
#define FT_THREADS 512
#define FT_COL_D 0            // G1 output -> H1 stash -> G2 output
#define FT_COL_D3 64          // G3 output (dW1 of this tile)
#define FT_COL_G0 128         // stash of 1 - H0^2
#define FT_COL_D0 192         // G0 output: H0pre of the group's NEXT tile
#define FT_COL_GROUP 256
#define FT_TMEM_COLS 512
#define FT_TILE_FLOATS 576
#define FT_TILE_BYTES (FT_TILE_FLOATS * 4)
#define FT_IMG 8192                                  // one 64 x 64 fp16 image
#define FT_OFF_W 0                                   // [net][hi, lo] images of C2 * W1, element (n, k) <-> row n, column k
#define FT_OFF_GROUP (4 * FT_IMG)
#define FT_G_P 0                                     // [net][hi, lo] H0 images, element (k, m)
#define FT_G_Q (4 * FT_IMG)                          // H1 fp32 [128 rows][68] for the output layer, then [net][hi, lo] dZ1 images (n, m)
#define FT_HS_LD 68
#define FT_G_IN (FT_G_Q + 128 * FT_HS_LD * 4)        // two tile records
#define FT_G_PART (FT_G_IN + 2 * FT_TILE_BYTES)      // [4 feature quarters][64 samples] float4 partial outputs
#define FT_G_DOUT (FT_G_PART + 4 * 64 * 16)          // [net][64 samples] float2 dL/dout
#define FT_G_MAX (FT_G_DOUT + 2 * 64 * 8)            // [net][sample half] max |dL/dout|
#define FT_G_XIMG (((FT_G_MAX + 64) + 127) / 128 * 128)   // [hi, lo] images of [x; 1; 0..] (16 rows x 64 samples) of the NEXT tile
#define FT_XIMG 2048
#define FT_GROUP_BYTES (80 * 1024)
#define FT_OFF_SMALL (FT_OFF_GROUP + 2 * FT_GROUP_BYTES)
#define FT_SMALL_BYTES 1024
#define FT_OFF_W0A (FT_OFF_SMALL + FT_SMALL_BYTES)   // [net][hi, lo] images of C2 * [W0; b0; 0..]^T (64 rows x 16)
#define FT_SMEM_BYTES (FT_OFF_W0A + 4 * FT_XIMG + 1024)
static_assert(FT_G_XIMG + 2 * FT_XIMG <= FT_GROUP_BYTES, "group region too small");
#define FT_C2 2.8853900817779268f                    // 2 log2(e): tanh(x) = 1 - 2 / (1 + 2^(C2 x)); folded into W0, b0, W1, b1

// tile record (floats): x [64][4] | advantage [64] | old log-prob [64] | action index [64] (int) | return [64] | old value [64]
#define FT_R_ADV 256
#define FT_R_OLP 320
#define FT_R_ACT 384
#define FT_R_RET 448
#define FT_R_OVAL 512

// -DTC_TRACE: phase timestamps of CTA 0 (thread 0 of each group): g_tc_trace[group][tile slot][point]
#ifdef TC_TRACE
#define FT_MARK(pt) do { if (t == 0 && blockIdx.x == 0) g_tc_trace[g][it & 31][pt] = clock64(); } while (0)
#else
#define FT_MARK(pt) do { } while (0)
#endif

struct FtArgs {
    const unsigned char* tiles;    // records of this epoch, [minibatch][tiles_per_mb]
    long long tile0;               // first record of this minibatch
    // persistent mode (n_steps > 0, cooperative launch with the fused tail): ONE launch runs the minibatch steps 0 .. n_steps-1 of
    // an update — step s is minibatch s % n_mb of staged epoch s / n_mb — separated by grid barriers; tile0 / LossArgs::mb /
    // LossArgs::mbstats then describe nothing and are derived per step from the fields below
    int n_steps, n_mb, tpm, nranks;
    long long batch, n_total, epoch_tiles;
    const double* mbstats0;        // advantage moments [epoch][minibatch][2]
};

// Sample records: the update gathers minibatches in shuffled order, and a gather from the time-major field arrays costs one
// 32-byte sector per 4-byte field (nine sectors per sample).  Once per iteration the fields of every sample are therefore
// packed into one contiguous record [obs (Dp) | action (A) | advantage | old log-prob | return | old value | pad] (stride a
// multiple of 4 floats) by a streaming kernel; the permute kernels then read two sectors per sample.
__host__ __device__ inline int ft_rec_stride(int obs_dim, int act_elems) { return ((((obs_dim + 3) & ~3) + act_elems + 4) + 3) & ~3; }
__global__ void __launch_bounds__(256) ft_pack_records_kernel(const BufDev buf, long long n_total, int stride, float* __restrict__ recs) {
    const int D = buf.obs_dim, Dp = (D + 3) & ~3, A = buf.act_dim;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_total; i += (long long)gridDim.x * blockDim.x) {
        auto val = [&](int k) -> float {
            if (k < Dp) return k < D ? buf.obs[i * D + k] : 0.f;
            k -= Dp;
            if (k < A) return reinterpret_cast<const float*>(buf.actions)[i * A + k];      // int32 bits for discrete actions
            k -= A;
            return k == 0 ? buf.advantages[i] : (k == 1 ? buf.logprobs[i] : (k == 2 ? buf.returns[i] : (k == 3 ? buf.values[i] : 0.f)));
        };
        float4* r = reinterpret_cast<float4*>(recs + i * stride);
        for (int k = 0; k < stride; k += 4) r[k >> 2] = make_float4(val(k), val(k + 1), val(k + 2), val(k + 3));
    }
}

// slot r of minibatch mb of an epoch -> its place in the tile records (padding slots are zero); returns the sample's advantage
__device__ __forceinline__ float ft_permute_slot(const float* __restrict__ recs, int stride, const FeistelKey& fk, long long n_total,
                                                 long long batch_size, long long per, long long mb, long long r, int identity, int act_start,
                                                 int nout, unsigned char* __restrict__ out, bool& valid) {
    const long long pos = mb * batch_size + r, s = mb * per + r;
    valid = r < batch_size && pos < n_total;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f), u = x, w = x;
    if (valid) {
        const long long sidx = identity ? pos : feistel_permute(pos, n_total, fk);
        const float4* rp = reinterpret_cast<const float4*>(recs + sidx * stride);      // obs (4) | action, adv, logp, ret | val
        x = rp[0]; u = rp[1]; w = rp[2];
    }
    int ai = valid ? __float_as_int(u.x) - act_start : 0;
    ai = ai < 0 ? 0 : (ai >= nout ? nout - 1 : ai);
    float* blk = reinterpret_cast<float*>(out + (s >> 6) * FT_TILE_BYTES);
    const int j = (int)(s & 63);
    reinterpret_cast<float4*>(blk)[j] = x;
    blk[FT_R_ADV + j] = u.y; blk[FT_R_OLP + j] = u.z; reinterpret_cast<int*>(blk)[FT_R_ACT + j] = ai;
    blk[FT_R_RET + j] = u.w; blk[FT_R_OVAL + j] = w.x;
    return u.y;
}
// One epoch's samples in shuffled order as contiguous tile records (fallback when all epochs exceed the staging budget, and the
// single-minibatch parity entry).
__global__ void __launch_bounds__(256) ft_permute_kernel(const float* __restrict__ recs, int stride, const FeistelKey fk, long long n_total,
                                                         long long batch_size, int n_mb, int tiles_per_mb, int identity, int act_start, int nout,
                                                         unsigned char* __restrict__ out) {
    const long long per = (long long)tiles_per_mb * FT_TS;
    const long long slots = per * n_mb;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += (long long)gridDim.x * blockDim.x) {
        const long long mb = s / per;
        bool valid;
        ft_permute_slot(recs, stride, fk, n_total, batch_size, per, mb, s - mb * per, identity, act_start, nout, out, valid);
    }
}
// ALL epochs of an update in one launch, grid (blocks per minibatch, minibatches, epochs): epoch e's records start at tile
// e * epoch_tiles; the same pass accumulates the minibatch's advantage moments (what adv_stats_kernel computes for the other
// loss/grad kernels, same partial layout: fixed-order sums => deterministic)
__global__ void __launch_bounds__(256) ft_permute_epochs_kernel(const float* __restrict__ recs, int stride, const __grid_constant__ FeistelKeys fks,
                                                                long long n_total, long long batch_size, int tiles_per_mb, int act_start,
                                                                int nout, unsigned char* __restrict__ out, long long epoch_tiles,
                                                                double* __restrict__ partial) {
    __shared__ double scratch[32];
    const FeistelKey& fk = fks.k[blockIdx.z];
    const long long per = (long long)tiles_per_mb * FT_TS, mb = blockIdx.y;
    unsigned char* o = out + (size_t)blockIdx.z * epoch_tiles * FT_TILE_BYTES;
    double sm = 0, sq = 0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < per; r += (long long)gridDim.x * blockDim.x) {
        bool valid;
        const float adv = ft_permute_slot(recs, stride, fk, n_total, batch_size, per, mb, r, 0, act_start, nout, o, valid);
        if (valid) { sm += (double)adv; sq += (double)adv * (double)adv; }
    }
    sm = block_sum(sm, scratch); sq = block_sum(sq, scratch);
    if (threadIdx.x == 0) {
        double* pp = partial + (((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 2;
        pp[0] = sm; pp[1] = sq;
    }
}

__device__ __forceinline__ uint32_t ft_idesc(int M, int N, int a_mn, int b_mn) {      // kind::f16: F16 x F16 -> F32
    return (1u << 4) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void ft_mma(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d),
                 "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
// x = hi + lo of two values, packed as half2 pairs; |x| > 65504 saturates instead of becoming inf
__device__ __forceinline__ void ft_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    uint32_t h;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));      // upper half <- first source, lower half <- second
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h));
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = h;
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void ft_st32(uint32_t taddr, const float* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,"
        "%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])), "r"(__float_as_uint(r[2])), "r"(__float_as_uint(r[3])), "r"(__float_as_uint(r[4])),
        "r"(__float_as_uint(r[5])), "r"(__float_as_uint(r[6])), "r"(__float_as_uint(r[7])), "r"(__float_as_uint(r[8])), "r"(__float_as_uint(r[9])),
        "r"(__float_as_uint(r[10])), "r"(__float_as_uint(r[11])), "r"(__float_as_uint(r[12])), "r"(__float_as_uint(r[13])), "r"(__float_as_uint(r[14])),
        "r"(__float_as_uint(r[15])), "r"(__float_as_uint(r[16])), "r"(__float_as_uint(r[17])), "r"(__float_as_uint(r[18])), "r"(__float_as_uint(r[19])),
        "r"(__float_as_uint(r[20])), "r"(__float_as_uint(r[21])), "r"(__float_as_uint(r[22])), "r"(__float_as_uint(r[23])), "r"(__float_as_uint(r[24])),
        "r"(__float_as_uint(r[25])), "r"(__float_as_uint(r[26])), "r"(__float_as_uint(r[27])), "r"(__float_as_uint(r[28])), "r"(__float_as_uint(r[29])),
        "r"(__float_as_uint(r[30])), "r"(__float_as_uint(r[31])) : "memory");
}
__device__ __forceinline__ void ft_ld16(uint32_t taddr, float* r) {
    uint32_t u[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]), "=r"(u[9]),
                   "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr));
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = __uint_as_float(u[j]);
}
// TMEM columns taddr .. taddr + n - 1 (n a multiple of 16) of this warp's lanes multiplied by r1 r2 (powers of two), after the
// MMAs that wrote them completed; out of line: it runs only when a tile lowers the delta scale
__device__ __noinline__ void ft_rescale_tmem(uint32_t taddr, int n, float r1, float r2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
    for (int c = 0; c < n; c += 16) {
        float v[16];
        ft_ld16(taddr + c, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = (v[j] * r1) * r2;
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr + c),
                     "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                     "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
                     "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
                     "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])) : "memory");
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ float ft_tanh_scaled(float xs) {       // tanh(x) from xs = C2 * x
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(xs));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}
// 16-byte row (8 consecutive columns starting at c, c % 8 == 0) of row r of a 64 x 64 fp16 image in the no-swizzle core layout
__device__ __forceinline__ uint32_t ft_row_off(int r, int c) { return (uint32_t)((((r >> 3) * 8 + (c >> 3)) << 7) + ((r & 7) << 4)); }

template <int NOUT>
__global__ void __launch_bounds__(FT_THREADS, 1) ppo_loss_grad_ft_kernel(const __grid_constant__ LossArgs a, const __grid_constant__ TailArgs tl,
                                                                         const __grid_constant__ FtArgs fa) {
    extern __shared__ __align__(1024) unsigned char ft_smem_raw[];
    __shared__ __align__(8) uint64_t bars[2][6];       // per group: tile record 0 / 1, G1, G2, G3, G0
    __shared__ __align__(8) uint64_t bar_stagger;       // group 1 starts when group 0 issues its first G2 / G3
    __shared__ uint32_t tmem_base_s;
    __shared__ double scratch[32];
    __shared__ float s_f2[2];
    __shared__ float s_head[8][8];                     // [(group, sample half, q)][bias sums 0..1, statistic sums 0..5] of the head warps
    if (*a.stop_flag) return;
    const PolicyDesc& pd = a.pd;
    const int tid = threadIdx.x;
#ifdef TC_TRACE
    const int trace_slot = tl.mode ? (int)(*tl.adam.step & 15) : 0;
    if (tid == 0 && blockIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        g_tc_trace[0][28][trace_slot] = (long long)gt;
        g_tc_trace[0][30][0] = clock64();
    }
#endif
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);          // warp-uniform for the compiler
    const int lane = tid & 31;
    const int g = warp >> 3, q = warp & 3, sh = (warp >> 2) & 1, t = tid & 255;
    const int net = lane >> 4, f = 16 * q + (lane & 15);             // feature role: TMEM lane 32 q + lane
    const int m0 = 32 * sh;                                          // this thread's samples of the tile: m0 .. m0 + 31
    const int ms = m0 + lane;                                        // sample role (output layer, loss head)
    const bool issuer = (warp & 7) == 0;                             // one elected lane of this warp issues the group's MMAs
    const uint32_t raw = tc_smem_u32(ft_smem_raw);
    const uint32_t sm_base = (raw + 1023u) & ~1023u;
    unsigned char* sm = ft_smem_raw + (sm_base - raw);
    unsigned char* smg = sm + FT_OFF_GROUP + g * FT_GROUP_BYTES;
    const uint32_t smg_base = sm_base + FT_OFF_GROUP + g * FT_GROUP_BYTES;
    float* sSmall = reinterpret_cast<float*>(sm + FT_OFF_SMALL);
    float2* sW2a = reinterpret_cast<float2*>(sSmall);             // [64] actor output weights
    float* sW2c = sSmall + 128;                                    // [64] critic output weights
    float* sb2 = sSmall + 192;                                     // [4]: actor b2[0..1], critic b2
    float* sWb = sSmall + 200;                                     // [2]: max row sum of |W2| per net
    float* sWmax = sSmall + 208;                                   // [4 warps][2 nets]
    float* Hs = reinterpret_cast<float*>(smg + FT_G_Q);
    float4* sPart = reinterpret_cast<float4*>(smg + FT_G_PART);
    float* sDout = reinterpret_cast<float*>(smg + FT_G_DOUT);     // [net][64 samples]: the sample's dL/dout scalar (see the loss head)
    float* sMax = reinterpret_cast<float*>(smg + FT_G_MAX);
    uint64_t* barL = &bars[g][0];
    uint64_t* bar1 = &bars[g][2];
    uint64_t* bar2 = &bars[g][3];
    uint64_t* bar3 = &bars[g][4];
    uint64_t* bar0 = &bars[g][5];
    __half* sXimg = reinterpret_cast<__half*>(smg + FT_G_XIMG);
    const LayerDesc& L0 = pd.L[net][0];
    const LayerDesc& L1 = pd.L[net][1];
    const LayerDesc& L2 = pd.L[net][2];

    // ---- prologue: TMEM, barriers, W1 images (scaled by C2), this thread's slices of the thin layers -------------------
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_s)), "r"(FT_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    const int n_steps = fa.n_steps > 0 ? fa.n_steps : 1;
    uint32_t tb = 0;
    for (int step = 0; step < n_steps; ++step) {
    // this step's minibatch
    long long mb_count = a.mb.count, tile0 = fa.tile0;
    double gcount = a.mb.global_count;
    const double* mbst = a.mbstats;
    if (fa.n_steps > 0) {
        const int e = step / fa.n_mb, i = step - e * fa.n_mb;
        mb_count = min(fa.batch, fa.n_total - (long long)i * fa.batch);
        tile0 = (long long)e * fa.epoch_tiles + (long long)i * fa.tpm;
        gcount = (double)mb_count * fa.nranks;
        mbst = fa.mbstats0 + 2 * ((size_t)e * fa.n_mb + i);
    }
    if (tid == 0) {
        // (every phase of the previous step's barriers has completed: its last MMAs were waited for before the end-of-pass)
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            if (step > 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(tc_smem_u32(&bars[0][0] + i)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&bars[0][0] + i)));
        }
        if (step > 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(tc_smem_u32(&bar_stagger)));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&bar_stagger)));
        asm volatile("fence.mbarrier_init.release.cluster;");
        // first tile record of both groups: in flight while the weight images are (re)built (records do not depend on the parameters)
        const long long n_tiles0 = (mb_count + FT_TS - 1) / FT_TS;
        const int nt0 = (long long)blockIdx.x < n_tiles0 ? (int)((n_tiles0 - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
#pragma unroll
        for (int gg = 0; gg < 2; ++gg) {
            if ((gg ? nt0 / 2 : (nt0 + 1) / 2) > 0) {
                const long long tile = (long long)blockIdx.x + (long long)gg * gridDim.x;
                const uint32_t dst = sm_base + FT_OFF_GROUP + (uint32_t)gg * FT_GROUP_BYTES + FT_G_IN;
                const uint32_t bar = tc_smem_u32(&bars[gg][0]);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(FT_TILE_BYTES) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                             "l"(fa.tiles + ((size_t)tile0 + (size_t)tile) * FT_TILE_BYTES), "r"(FT_TILE_BYTES), "r"(bar) : "memory");
            }
        }
    }
    {
        // 16 elements per thread, loads issued together (one L2 round trip)
        float wv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int i = tid + j * FT_THREADS, wn = i >> 12, kn = i & 4095;
            wv[j] = a.pack[pd.L[wn][1].pw_off + kn];
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int i = tid + j * FT_THREADS, wn = i >> 12, k = (i >> 6) & 63, n = i & 63;
            float w = wv[j] * FT_C2;
            w = fminf(fmaxf(w, -65504.f), 65504.f);
            const __half hi = __float2half_rn(w);
            const __half lo = __float2half_rn(w - __half2float(hi));
            const int idx = ((n >> 3) * 8 + (k >> 3)) * 64 + (n & 7) * 8 + (k & 7);
            reinterpret_cast<__half*>(sm + FT_OFF_W + (wn * 2) * FT_IMG)[idx] = hi;
            reinterpret_cast<__half*>(sm + FT_OFF_W + (wn * 2 + 1) * FT_IMG)[idx] = lo;
        }
    }
    if (tid < 64) {
        sW2a[tid] = make_float2(a.pack[pd.L[0][2].pw_off + tid * 4], NOUT > 1 ? a.pack[pd.L[0][2].pw_off + tid * 4 + 1] : 0.f);
        sW2c[tid] = a.pack[pd.L[1][2].pw_off + tid * 4];
    }
    if (tid < 4) sb2[tid] = tid < 2 ? (tid < NOUT ? a.pack[pd.L[0][2].pb_off + tid] : 0.f) : (tid == 2 ? a.pack[pd.L[1][2].pb_off] : 0.f);
    // layer 0 runs on the tensor cores as well: A = C2 * [W0; b0; 0]^T (64 x 16), B = [x; 1; 0] (16 x 64 samples)
    for (int i = tid; i < 2 * 64 * 16; i += FT_THREADS) {
        const int wn = i >> 10, k = (i >> 4) & 63, d = i & 15;
        const LayerDesc& W0 = pd.L[wn][0];
        float w = d < 4 ? a.pack[W0.pw_off + d * 64 + k] : (d == 4 ? a.pack[W0.pb_off + k] : 0.f);
        w = fminf(fmaxf(w * FT_C2, -65504.f), 65504.f);
        const __half hi = __float2half_rn(w);
        const __half lo = __float2half_rn(w - __half2float(hi));
        const int idx = ((k >> 3) * 2 + (d >> 3)) * 64 + (k & 7) * 8 + (d & 7);
        reinterpret_cast<__half*>(sm + FT_OFF_W0A + (wn * 2) * FT_XIMG)[idx] = hi;
        reinterpret_cast<__half*>(sm + FT_OFF_W0A + (wn * 2 + 1) * FT_XIMG)[idx] = lo;
    }
    for (int i = t; i < 2 * 1024; i += 256) {                        // x images: rows 5..15 stay zero, row 4 of the hi image is 1 (bias)
        const int r = (i & 1023) >> 3 & 7, hl = i >> 10;            // element index within an image: [d / 8][m / 8][d % 8][m % 8]
        sXimg[i] = __float2half_rn((hl == 0 && r == 4 && (i & 1023) < 512) ? 1.0f : 0.f);
    }
    const float b1s = a.pack[L1.pb_off + f] * FT_C2;
    const float w2_0 = a.pack[L2.pw_off + f * 4];
    const float w2_1 = (net == 0 && NOUT > 1) ? a.pack[L2.pw_off + f * 4 + 1] : 0.f;
    {
        float wb = fabsf(w2_0) + fabsf(w2_1);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) wb = fmaxf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
        if (warp < 4 && (lane & 15) == 0) sWmax[warp * 2 + net] = wb;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tb = __shfl_sync(0xffffffffu, tmem_base_s, 0);
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][1] = clock64();
#endif
    const float w2bound = fmaxf(fmaxf(sWmax[net], sWmax[2 + net]), fmaxf(sWmax[4 + net], sWmax[6 + net]));
    const uint32_t gcol = tb + (uint32_t)g * FT_COL_GROUP;
    const uint32_t my = gcol + ((uint32_t)(q * 32) << 16);            // this warp's lane quadrant, this group's columns

    float adv_mean = 0.f, adv_den = 1.f;
    if (a.hp.normalize_advantage) {
        const double n = gcount;
        const double mean = mbst[0] / n;
        double var = (mbst[1] - n * mean * mean) / (n - 1.0);
        if (var < 0.0) var = 0.0;
        adv_mean = (float)mean;
        adv_den = (float)sqrt(var) + 1e-8f;
    }
    const float invB = (float)(1.0 / gcount);
    float stats[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float accb2_0 = 0.f, accb2_1 = 0.f;                               // head threads: sums of dL/dout (output-layer bias gradients)
    // delta scale of this thread's net in this group: a power of two fixed at the group's first tile with a non-zero gradient
    // and lowered only when a later tile would leave fp16's range, so that dW1 can stay in TMEM over all the group's tiles;
    // the scaled sums below are unscaled once at the end
    float S = 1.0f, invS = 1.0f;
    bool s_fixed = false;
    float accb1 = 0.f, accW2_0 = 0.f, accb0 = 0.f, accW0_0 = 0.f, accW0_1 = 0.f, accW0_2 = 0.f, accW0_3 = 0.f;

    // tiles of this CTA: blockIdx.x + j * gridDim.x, j = 0 .. nt-1; group g takes j = g, g + 2, ...
    const long long n_tiles = (mb_count + FT_TS - 1) / FT_TS;
    const int nt = (long long)blockIdx.x < n_tiles ? (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
    const int n_own = g ? nt / 2 : (nt + 1) / 2;
    const unsigned char* rec0 = fa.tiles + (size_t)tile0 * FT_TILE_BYTES;
    auto load_tile = [&](int it) {                                    // one thread: bulk copy of tile `it` of this group into record buffer it & 1
        const long long tile = (long long)blockIdx.x + (long long)(2 * it + g) * gridDim.x;
        const uint32_t dst = smg_base + FT_G_IN + (uint32_t)(it & 1) * FT_TILE_BYTES;
        const uint32_t bar = tc_smem_u32(barL + (it & 1));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(FT_TILE_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(rec0 + (size_t)tile * FT_TILE_BYTES), "r"(FT_TILE_BYTES), "r"(bar) : "memory");
    };
    // (tile 0 of both groups was requested by thread 0 right after the barrier initialisation)

    const uint32_t idesc_g1 = ft_idesc(64, 64, 0, 1), idesc_g2 = ft_idesc(64, 64, 1, 1), idesc_g3 = ft_idesc(64, 64, 0, 0);
    const uint32_t imgP = smg_base + FT_G_P, imgQ = smg_base + FT_G_Q, imgW = sm_base + FT_OFF_W;
    const uint32_t imgX = smg_base + FT_G_XIMG, imgW0 = sm_base + FT_OFF_W0A;
    // x of tile `it` of this group -> fp16 hi / lo rows 0..3 of the x images (thread <-> (sample, component))
    auto build_x = [&](int it) {
        const float* r = reinterpret_cast<const float*>(smg + FT_G_IN + (it & 1) * FT_TILE_BYTES);
        const int m = t & 63, d = t >> 6;
        const float x = fminf(fmaxf(r[m * 4 + d], -65504.f), 65504.f);
        const __half hi = __float2half_rn(x);
        const int idx = (m >> 3) * 64 + d * 8 + (m & 7);
        sXimg[idx] = hi;
        sXimg[1024 + idx] = __float2half_rn(x - __half2float(hi));
    };
    // G0: H0pre = C2 (W0^T x + b0) of the tile whose x images were just built (one K = 16 step, 3 products, both nets)
    auto issue_g0 = [&]() {
#pragma unroll
        for (int wn = 0; wn < 2; ++wn)
#pragma unroll
            for (int ps = 0; ps < 3; ++ps)
                ft_mma(gcol + FT_COL_D0 + ((uint32_t)wn << 20), tc_desc(imgW0 + (wn * 2 + (ps == 1 ? 1 : 0)) * FT_XIMG, 128, 256, 0),
                       tc_desc(imgX + (ps == 2 ? 1 : 0) * FT_XIMG, 1024, 128, 0), idesc_g1, ps ? 1u : 0u);
        tc_commit(bar0);
    };
    if (n_own > 0) {
        tc_wait(barL, 0u);
        build_x(0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        tc_group_sync(g);
        if (issuer && tc_elect_one()) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            issue_g0();
        }
    }
    unsigned char* pP = smg + FT_G_P + (net * 2) * FT_IMG;           // this thread's net: hi image, lo image = + FT_IMG
    unsigned char* pQ = smg + FT_G_Q + (net * 2) * FT_IMG;

    // the groups would otherwise run in lock-step (same phases at the same time, tensor pipe and issue slots idle in turn)
    if (g == 1 && n_own > 0) tc_wait(&bar_stagger, 0u);
    for (int it = 0; it < n_own; ++it) {
        const uint32_t ph = (uint32_t)it & 1u;
        const float* rec = reinterpret_cast<const float*>(smg + FT_G_IN + (it & 1) * FT_TILE_BYTES);
        const float4* Xs = reinterpret_cast<const float4*>(rec);
        FT_MARK(0);
        if (t == 0 && it + 1 < n_own) load_tile(it + 1);              // the other record buffer was released by the barrier that ended tile it - 1
        tc_wait(bar0, ph);                                            // H0pre of this tile (issued during the previous tile / before the loop)
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        FT_MARK(1);
        // ---- A: H0 = tanh(H0pre) for (net, f) over 32 samples -> H0 images; 1 - H0^2 -> TMEM stash ----------------------------
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            float pre[16];
            ft_ld16(my + FT_COL_D0 + m0 + 16 * hh, pre);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                float h[8], gd[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    h[j] = ft_tanh_scaled(pre[8 * c + j]);
                    gd[j] = fmaf(-h[j], h[j], 1.0f);
                }
                uint4 vh, vl;
                ft_split2(h[0], h[1], vh.x, vl.x); ft_split2(h[2], h[3], vh.y, vl.y);
                ft_split2(h[4], h[5], vh.z, vl.z); ft_split2(h[6], h[7], vh.w, vl.w);
                const uint32_t off = ft_row_off(f, m0 + 16 * hh + 8 * c);
                *reinterpret_cast<uint4*>(pP + off) = vh;
                *reinterpret_cast<uint4*>(pP + FT_IMG + off) = vl;
                tc_st8(my + FT_COL_G0 + m0 + 16 * hh + 8 * c, gd);
            }
        }
        FT_MARK(2);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        tc_group_sync(g);
        // ---- G1: H1pre = W1^T H0, both nets (the critic's accumulator at lane offset 16) -------------------------------------
        if (issuer && tc_elect_one()) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int wn = 0; wn < 2; ++wn)
#pragma unroll
                for (int ps = 0; ps < 3; ++ps) {
                    const uint32_t ai = imgW + (wn * 2 + (ps == 1 ? 1 : 0)) * FT_IMG;
                    const uint32_t bi = imgP + (wn * 2 + (ps == 2 ? 1 : 0)) * FT_IMG;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        ft_mma(gcol + FT_COL_D + ((uint32_t)wn << 20), tc_desc(ai + kk * 256, 128, 1024, 0), tc_desc(bi + kk * 2048, 1024, 128, 0),
                               idesc_g1, (ps | kk) ? 1u : 0u);
                }
            tc_commit(bar1);
        }
        FT_MARK(3);
        tc_wait(bar1, ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        FT_MARK(4);
        // ---- B1: H1 = tanh(H1pre + b1) -> fp32 tile for the output layer + TMEM stash -------------------------------------
        {
            float h1[32];
            tc_ld32(my + FT_COL_D + m0, h1);
#pragma unroll
            for (int j = 0; j < 32; ++j) h1[j] = ft_tanh_scaled(h1[j] + b1s);
            float* hr = Hs + (net * 64 + f) * FT_HS_LD + m0;
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(hr + j) = make_float4(h1[j], h1[j + 1], h1[j + 2], h1[j + 3]);
            ft_st32(my + FT_COL_D + m0, h1);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        FT_MARK(5);
        tc_group_sync(g);
        FT_MARK(6);
        // ---- output layer partials: thread <-> (sample ms, feature quarter q) ---------------------------------------------------
        {
            float pa0 = 0.f, pa1 = 0.f, pc = 0.f;
            const float* ha = Hs + (16 * q) * FT_HS_LD + ms;
            const float* hc = Hs + (64 + 16 * q) * FT_HS_LD + ms;
#pragma unroll
            for (int n = 0; n < 16; ++n) {
                const float2 wa = sW2a[16 * q + n];
                const float hv = ha[n * FT_HS_LD];
                pa0 = fmaf(hv, wa.x, pa0);
                if (NOUT > 1) pa1 = fmaf(hv, wa.y, pa1);
                pc = fmaf(hc[n * FT_HS_LD], sW2c[16 * q + n], pc);
            }
            sPart[q * 64 + ms] = make_float4(pa0, pa1, pc, 0.f);
        }
        FT_MARK(7);
        tc_group_sync(g);
        FT_MARK(8);
        // ---- loss head: warps with q == 0 the actor's, q == 1 the critic's, one thread per sample --------------------------------
        if (q < 2) {
            const float4 p0 = sPart[ms], p1 = sPart[64 + ms], p2 = sPart[128 + ms], p3 = sPart[192 + ms];
            const long long tile = (long long)blockIdx.x + (long long)(2 * it + g) * gridDim.x;
            const bool valid = tile * FT_TS + ms < mb_count;
            float dmax;
            if (q == 0) {
                float out[NOUT], dout[NOUT];
                out[0] = sb2[0] + ((p0.x + p1.x) + (p2.x + p3.x));
                if (NOUT > 1) out[NOUT > 1 ? 1 : 0] = sb2[1] + ((p0.y + p1.y) + (p2.y + p3.y));
                float adv = rec[FT_R_ADV + ms];
                if (valid && a.hp.normalize_advantage) adv = (adv - adv_mean) / adv_den;
                const float olp = rec[FT_R_OLP + ms];
                const int aidx = reinterpret_cast<const int*>(rec)[FT_R_ACT + ms];
                // softmax -> log -> entropy exactly as categorical.jl:29-52 (log of the softmax); the exponential of the maximal
                // logit is exp(0) = 1 and log p[a] is one of the log p[j], so NOUT - 1 expf and NOUT logf are evaluated
                int jmax = 0;
                float mx = out[0];
#pragma unroll
                for (int j = 1; j < NOUT; ++j) if (out[j] > mx) { mx = out[j]; jmax = j; }
                float ex[NOUT], s = 0.f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) { ex[j] = j == jmax ? 1.0f : expf(out[j] - mx); s += ex[j]; }
                float pj[NOUT], lpj[NOUT], hsum = 0.f, logp = 0.f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) {
                    pj[j] = ex[j] / s; lpj[j] = logf(pj[j]); hsum += pj[j] * lpj[j];
                    if (j == aidx) logp = lpj[j];
                }
                const float ent = -hsum;
                const float log_ratio = logp - olp;
                const float ratio = expf(log_ratio);
                const float rc = fminf(fmaxf(ratio, 1.0f - a.hp.clip_range), 1.0f + a.hp.clip_range);
                const float s1 = ratio * adv, s2 = rc * adv;
                const float g_logp = (!valid || s2 < s1) ? 0.f : -invB * adv * ratio;
                const float g_ent = valid ? -a.hp.ent_coef * invB : 0.f;
#pragma unroll
                for (int j = 0; j < NOUT; ++j) dout[j] = g_logp * ((j == aidx ? 1.0f : 0.0f) - pj[j]) + g_ent * (-pj[j] * (lpj[j] + ent));
                if (valid) {
                    stats[0] += -fminf(s1, s2);
                    stats[2] += ent;
                    stats[3] += (ratio != rc) ? 1.0f : 0.0f;
                    stats[4] += ratio - 1.0f - log_ratio;
                    stats[5] += ratio;
                }
                accb2_0 += dout[0];
                if (NOUT > 1) accb2_1 += dout[NOUT > 1 ? 1 : 0];
                // two logits: the softmax gradient sums to zero (dL/dout_1 = -dL/dout_0 up to rounding), so ONE scalar per sample
                // goes to the feature threads (half the broadcast loads of the delta phase); their mean cancels the rounding
                sDout[ms] = NOUT > 1 ? 0.5f * (dout[0] - dout[NOUT > 1 ? 1 : 0]) : dout[0];
                dmax = fabsf(dout[0]);
                if (NOUT > 1) dmax = fmaxf(dmax, fabsf(dout[NOUT > 1 ? 1 : 0]));
            } else {
                const float v_raw = sb2[2] + ((p0.z + p1.z) + (p2.z + p3.z));
                const float ret = rec[FT_R_RET + ms], ov = rec[FT_R_OVAL + ms];
                float v = v_raw;
                bool v_pass = true;
                if (a.hp.clip_range_vf >= 0.f) {
                    const float dlt = v_raw - ov;
                    v_pass = dlt >= -a.hp.clip_range_vf && dlt <= a.hp.clip_range_vf;
                    v = ov + fminf(fmaxf(dlt, -a.hp.clip_range_vf), a.hp.clip_range_vf);
                }
                const float verr = v - ret;
                const float dc = (valid && v_pass) ? a.hp.vf_coef * 2.0f * verr * invB : 0.f;
                if (valid) stats[1] += verr * verr;
                accb2_0 += dc;
                sDout[64 + ms] = dc;
                dmax = fabsf(dc);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
            if (lane == 0) sMax[q * 2 + sh] = dmax;
        }
        FT_MARK(9);
        tc_group_sync(g);
        FT_MARK(10);
        // ---- B2: dZ1 = (W2 dout) .* (1 - H1^2), scaled by the tile's power of two -> dZ1 images; db1, dW2 sums -------------------
        {
            // the scale is fixed at the first tile with a non-zero gradient; a later tile whose bound would pass fp16's 65504
            // moves it down to sit where the first tile sat, and the group's dW1 in TMEM and the scaled register sums
            // are multiplied by the exact ratio of the two powers of two (dW1: the previous tile's G3 completed at bar3, this
            // tile's is issued after the group barrier below)
            const float bound = fmaxf(sMax[net * 2], sMax[net * 2 + 1]) * w2bound;
            const bool fix = bound > 0.f && bound < 3.0e38f && (!s_fixed || bound * S > 65504.0f);
            int E = ((__float_as_int(bound) >> 23) & 255) - 127;                  // bound < 2^(E + 1)
            E = E < -100 ? -100 : (E > 100 ? 100 : E);
            if (__any_sync(0xffffffffu, fix && s_fixed)) {                        // warp-uniform: both nets share the warp
                const int sE = 130 - (__float_as_int(S) >> 23);                   // S = 2^(3 - sE)
                const int d = (fix && s_fixed) ? sE - E : 0;                      // S_new / S_old = 2^d, -200 <= d <= 0
                const float r1 = __int_as_float((d / 2 + 127) << 23), r2 = __int_as_float((d - d / 2 + 127) << 23);
                ft_rescale_tmem(my + FT_COL_D3 + m0, 32, r1, r2);
                accb1 = (accb1 * r1) * r2; accb0 = (accb0 * r1) * r2;
                accW0_0 = (accW0_0 * r1) * r2; accW0_1 = (accW0_1 * r1) * r2; accW0_2 = (accW0_2 * r1) * r2; accW0_3 = (accW0_3 * r1) * r2;
            }
            if (fix) {
                S = __int_as_float((3 - E + 127) << 23);                          // |S dZ1| < 2^4 on this tile
                invS = __int_as_float((E - 3 + 127) << 23);
                s_fixed = true;
            }
            const float wsd = (w2_0 - w2_1) * S;                                  // actor, two logits: W2[f][0] - W2[f][1]; else W2[f][0] (w2_1 = 0)
            float z[32];
            tc_ld32(my + FT_COL_D + m0, z);                                       // H1
            const float* dd = sDout + net * 64 + m0;
            float sb = 0.f, sw0 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float d = dd[j];
                const float h = z[j];
                sw0 = fmaf(h, d, sw0);
                z[j] = (d * wsd) * fmaf(-h, h, 1.0f);
                sb += z[j];
            }
            accb1 += sb;
            accW2_0 += sw0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint4 vh, vl;
                ft_split2(z[8 * c], z[8 * c + 1], vh.x, vl.x); ft_split2(z[8 * c + 2], z[8 * c + 3], vh.y, vl.y);
                ft_split2(z[8 * c + 4], z[8 * c + 5], vh.z, vl.z); ft_split2(z[8 * c + 6], z[8 * c + 7], vh.w, vl.w);
                const uint32_t off = ft_row_off(f, m0 + 8 * c);
                *reinterpret_cast<uint4*>(pQ + off) = vh;
                *reinterpret_cast<uint4*>(pQ + FT_IMG + off) = vl;
            }
        }
        if (it + 1 < n_own) {                                         // x images of the next tile (its record arrived long ago)
            tc_wait(barL + ((it + 1) & 1), ((uint32_t)(it + 1) >> 1) & 1u);
            build_x(it + 1);
        }
        FT_MARK(11);
        if (g == 0 && it == 0 && t == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(&bar_stagger)) : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        tc_group_sync(g);
        // ---- G2: dH0 = W1 dZ1 (over the H1 stash), G3: dW1 = H0 dZ1^T, G0 of the next tile ---------------------------------------
        if (issuer && tc_elect_one()) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int wn = 0; wn < 2; ++wn)
#pragma unroll
                for (int ps = 0; ps < 3; ++ps) {
                    const uint32_t ai = imgW + (wn * 2 + (ps == 1 ? 1 : 0)) * FT_IMG;
                    const uint32_t bi = imgQ + (wn * 2 + (ps == 2 ? 1 : 0)) * FT_IMG;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        ft_mma(gcol + FT_COL_D + ((uint32_t)wn << 20), tc_desc(ai + kk * 2048, 1024, 128, 0), tc_desc(bi + kk * 2048, 1024, 128, 0),
                               idesc_g2, (ps | kk) ? 1u : 0u);
                }
            tc_commit(bar2);
#pragma unroll
            for (int wn = 0; wn < 2; ++wn)
#pragma unroll
                for (int ps = 0; ps < 3; ++ps) {
                    const uint32_t ai = imgP + (wn * 2 + (ps == 1 ? 1 : 0)) * FT_IMG;
                    const uint32_t bi = imgQ + (wn * 2 + (ps == 2 ? 1 : 0)) * FT_IMG;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        ft_mma(gcol + FT_COL_D3 + ((uint32_t)wn << 20), tc_desc(ai + kk * 256, 128, 1024, 0), tc_desc(bi + kk * 256, 128, 1024, 0),
                               idesc_g3, (it | ps | kk) ? 1u : 0u);          // accumulates over all tiles of the group
                }
            tc_commit(bar3);
            if (it + 1 < n_own) issue_g0();
        }
        FT_MARK(12);
        tc_wait(bar2, ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        FT_MARK(13);
        // ---- C: dZ0 = dH0 .* (1 - H0^2); db0 and dW0 sums over this thread's 32 samples ----------------------------------------
        {
            float sb = 0.f, s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                float dh[16], gd[16];
                ft_ld16(my + FT_COL_D + m0 + 16 * hh, dh);
                ft_ld16(my + FT_COL_G0 + m0 + 16 * hh, gd);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float zz = dh[j] * gd[j];
                    const float4 x = Xs[m0 + 16 * hh + j];
                    sb += zz;
                    s0 = fmaf(zz, x.x, s0); s1 = fmaf(zz, x.y, s1); s2 = fmaf(zz, x.z, s2); s3 = fmaf(zz, x.w, s3);
                }
            }
            accb0 += sb;
            accW0_0 += s0; accW0_1 += s1; accW0_2 += s2; accW0_3 += s3;
        }
        // ---- G3 reads the H0 / dZ1 images: it must be done before the next tile overwrites them ----------------------------------
        FT_MARK(14);
        tc_wait(bar3, ph);
        FT_MARK(15);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        tc_group_sync(g);
    }
    // unscale the sums that were accumulated from scaled deltas; this group's dW1 from TMEM
    accb1 *= invS;
    {
        const float cz = invS * (1.0f / FT_C2);
        accb0 *= cz; accW0_0 *= cz; accW0_1 *= cz; accW0_2 *= cz; accW0_3 *= cz;
    }
    float accW1[32];                                                  // dW1[f][m0 .. m0 + 31] of this thread's net
    if (n_own > 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tc_ld32(my + FT_COL_D3 + m0, accW1);
#pragma unroll
        for (int j = 0; j < 32; ++j) accW1[j] *= invS;
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) accW1[j] = 0.f;
    }

    // ---- end of the minibatch: combine sample halves and groups, write this CTA's partial plane -------------------------------
#ifdef TC_TRACE
    if ((tid & 255) == 0 && blockIdx.x == 0) g_tc_trace[0][30][4 + g] = clock64();
#endif
    __syncthreads();
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][2] = clock64();
#endif
    float* gp = a.gpart + (size_t)blockIdx.x * pd.gpack;
    float* sDW = reinterpret_cast<float*>(sm + FT_OFF_GROUP + FT_G_P);              // [net][64][64] (group 0's image region)
    float* sRed = reinterpret_cast<float*>(sm + FT_OFF_GROUP + FT_G_Q);             // [4 slots][8 sums][128]
    if (g == 1) {
        float* d = sDW + (net * 64 + f) * 64 + m0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(d + j) = make_float4(accW1[j], accW1[j + 1], accW1[j + 2], accW1[j + 3]);
    }
    {
        float* r = sRed + ((g * 2 + sh) * 8) * 128 + net * 64 + f;
        r[0] = accW0_0; r[128] = accW0_1; r[256] = accW0_2; r[384] = accW0_3; r[512] = accb0; r[640] = accb1; r[768] = accW2_0; r[896] = -accW2_0;     // dW2[f][1] = -dW2[f][0] (two logits)
    }
    if (q < 2) {
        // head warps: output-layer bias gradients and the six statistic sums (warp sums, then 8 warp slots in fixed order)
        float hv[8] = {accb2_0, accb2_1, stats[0], stats[1], stats[2], stats[3], stats[4], stats[5]};
#pragma unroll
        for (int i = 0; i < 8; ++i) hv[i] = warp_sum(hv[i]);
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) s_head[(g * 2 + sh) * 2 + q][i] = hv[i];
        }
    }
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][7] = clock64();
#endif
    __syncthreads();
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][8] = clock64();
#endif
    if (g == 0) {
        const float* d = sDW + (net * 64 + f) * 64 + m0;
        float* gw = gp + L1.pw_off + f * 64 + m0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 o = *reinterpret_cast<const float4*>(d + j);
            *reinterpret_cast<float4*>(gw + j) = make_float4(accW1[j] + o.x, accW1[j + 1] + o.y, accW1[j + 2] + o.z, accW1[j + 3] + o.w);
        }
    }
    for (int i = tid; i < 8 * 128; i += FT_THREADS) {
        const int qn = i >> 7, r = i & 127, rn = r >> 6, rf = r & 63;
        const float s = (sRed[(0 * 8 + qn) * 128 + r] + sRed[(1 * 8 + qn) * 128 + r]) + (sRed[(2 * 8 + qn) * 128 + r] + sRed[(3 * 8 + qn) * 128 + r]);
        const LayerDesc& R0 = pd.L[rn][0];
        const LayerDesc& R1 = pd.L[rn][1];
        const LayerDesc& R2 = pd.L[rn][2];
        if (qn < 4) gp[R0.pw_off + qn * 64 + rf] = s;
        else if (qn == 4) gp[R0.pb_off + rf] = s;
        else if (qn == 5) gp[R1.pb_off + rf] = s;
        else if (qn == 6 || (rn == 0 && NOUT > 1)) gp[R2.pw_off + rf * 4 + (qn - 6)] = s;
    }
    if (tid < 16) {
        // slot = (group, sample half, q): q = 0 actor head warps, q = 1 critic head warps
        const int i = tid & 7, hq = tid >> 3;
        double s = 0.0;
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) s += (double)s_head[sl * 2 + hq][i];
        if (hq == 0) {
            if (i < 2) { if (i < NOUT) gp[pd.L[0][2].pb_off + i] = (float)s; }
            else if (i != 3) gp[pd.pack_fwd + pd.act_n + (i - 2)] = (float)s;          // policy loss, entropy, clip fraction, kl, ratio
        } else {
            if (i == 0) gp[pd.L[1][2].pb_off] = (float)s;
            else if (i == 3) gp[pd.pack_fwd + pd.act_n + 1] = (float)s;                 // value loss
        }
    }
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][9] = clock64();
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][10] = clock64();
#endif
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) g_tc_trace[0][30][3] = clock64();
#endif
    bool stop = false;
    if (tl.mode) stop = tc_fused_tail(a, tl, reinterpret_cast<float*>(sm + FT_OFF_GROUP + FT_G_P), scratch, s_f2, gcount);
    if (stop) break;                                                  // target-KL stop: identical in every CTA (ppo.jl:235-238)
    if (step + 1 < n_steps) {
        // the next step builds its weight images from the parameters every CTA's Adam slice just wrote
        __threadfence();
        cooperative_groups::this_grid().sync();
    }
    }   // minibatch steps
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(FT_TMEM_COLS));
#ifdef TC_TRACE
    if (tid == 0 && blockIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        g_tc_trace[0][29][trace_slot] = (long long)gt;
        g_tc_trace[0][30][6] = clock64();
    }
#endif
}
