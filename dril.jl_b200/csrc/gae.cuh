// GAE as a per-env reverse scan over the time-major buffer.
// Replaces compute_advantages! (buffers/trajectory.jl:80-102) applied to every trajectory and
// `returns = advantages + values` (buffers/rollout_buffer.jl:83-87).  The carry
// (A_next, V_next) is reset wherever a trajectory closes (terminated | truncated | last step):
//   terminated           -> delta = r - V
//   truncated            -> delta = r + gamma * V(terminal_obs) - V      (boot[t][n])
//   rollout end, running -> delta = r + gamma * V(new_obs)      - V      (last_values[n])
// Latency-bound: every env is a dependent chain of T steps, thread per env, fully coalesced rows.  The t-loop runs in
// blocks of 8 rows, and the loads of the next block are in flight while the current one is computed.  Blocks of
// GAE_THREADS envs, so that the scans of a few thousand envs spread over the SMs.
//
// With sample records (GaeRecords::recs, iterations whose update runs a tcgen05 loss/grad kernel) the same launch also
// writes the per-sample records that ft_pack_records_kernel (update_ft.cuh) packs for other callers, same layout:
//   [obs (Dp = D rounded up to 4, zero padded) | action (A) | advantage | old log-prob | return | old value | zeros] (stride)
// The scan blocks write the part from the advantage on, which they hold in registers; blocks
// scan_ctas .. gridDim.x - 1 copy the obs | action part, a streaming copy that overlaps the scans.
#pragma once
#include "common.cuh"

#define GAE_UNROLL 8
#define GAE_THREADS 64

struct GaeRecords {
    const float* obs;           // [T * N][D]
    const float* actions;       // [T * N][A] (int32 bits for discrete actions)
    const float* logprobs;      // [T * N]
    float* recs;                // [T * N][stride], or null: no records
    int D, A, stride;
};

__global__ void __launch_bounds__(GAE_THREADS) gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                                          const unsigned char* __restrict__ flags,
                                                          const float* __restrict__ boot, const float* __restrict__ last_values,
                                                          float* __restrict__ adv, float* __restrict__ ret, long long T,
                                                          long long N, float gamma, float lambda, double* ev_acc4,
                                                          const GaeRecords rec, int scan_ctas) {
    __shared__ double scratch[32];
    const int Dp = (rec.D + 3) & ~3;
    if ((int)blockIdx.x >= scan_ctas) {
        const int D = rec.D, A = rec.A;
        const long long n_total = T * N, step = (long long)(gridDim.x - scan_ctas) * blockDim.x;
        for (long long i = (long long)(blockIdx.x - scan_ctas) * blockDim.x + threadIdx.x; i < n_total; i += step) {
            auto ob = [&](int k) { return k < D ? rec.obs[i * D + k] : 0.f; };
            float* r = rec.recs + i * rec.stride;
            for (int k = 0; k < Dp; k += 4) *reinterpret_cast<float4*>(r + k) = make_float4(ob(k), ob(k + 1), ob(k + 2), ob(k + 3));
            for (int k = 0; k < A; ++k) r[Dp + k] = rec.actions[i * A + k];
        }
        return;
    }
    long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = n < N;
    if (!live) n = N - 1;          // keep the thread for the block sums of the fused explained-variance moments (no stores)
    const bool wr = rec.recs != nullptr;
    const int back = Dp + rec.A;   // first float of a record's advantage | old log-prob | return | old value
    double sd = 0, sdd = 0, sr = 0, srr = 0;
    const float gl = __fmul_rn(gamma, lambda);
    float a_next = 0.f, v_next = 0.f;
    long long t = T - 1;
    auto step = [&](long long tt, float r, float v, unsigned char f, float lp) {
        const bool term = f & 1, trunc = f & 2;
        const bool last = term || trunc || (tt == T - 1);
        float a;
        if (last) {
            if (term) a = __fsub_rn(r, v);
            else {
                float b = trunc ? boot[tt * N + n] : last_values[n];
                a = __fsub_rn(__fadd_rn(r, __fmul_rn(gamma, b)), v);
            }
        } else {
            float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(gamma, v_next)), v);
            a = __fadd_rn(delta, __fmul_rn(gl, a_next));
        }
        const float rt = __fadd_rn(a, v);
        if (live) {
            adv[tt * N + n] = a;
            ret[tt * N + n] = rt;
            if (wr) {
                float* rp = rec.recs + (tt * N + n) * rec.stride + back;
                rp[0] = a; rp[1] = lp; rp[2] = rt; rp[3] = v;
                for (int k = back + 4; k < rec.stride; ++k) rp[k - back] = 0.f;
            }
            const double dv = (double)v - (double)rt, dr = (double)rt;
            sd += dv; sdd += dv * dv; sr += dr; srr += dr * dr;
        }
        a_next = a; v_next = v;
    };
    auto load = [&](long long tb, float* r, float* v, unsigned char* f, float* lp) {
#pragma unroll
        for (int i = 0; i < GAE_UNROLL; ++i) {
            const long long idx = (tb - i) * N + n;
            r[i] = rewards[idx]; v[i] = values[idx]; f[i] = flags[idx];
            lp[i] = wr ? rec.logprobs[idx] : 0.f;
        }
    };
    float r0[GAE_UNROLL], v0[GAE_UNROLL], l0[GAE_UNROLL];
    unsigned char f0[GAE_UNROLL];
    if (t >= GAE_UNROLL - 1) load(t, r0, v0, f0, l0);
    while (t >= GAE_UNROLL - 1) {
        float r1[GAE_UNROLL], v1[GAE_UNROLL], l1[GAE_UNROLL];
        unsigned char f1[GAE_UNROLL];
        const bool more = t >= 2 * GAE_UNROLL - 1;
        if (more) load(t - GAE_UNROLL, r1, v1, f1, l1);
#pragma unroll
        for (int i = 0; i < GAE_UNROLL; ++i) step(t - i, r0[i], v0[i], f0[i], l0[i]);
        t -= GAE_UNROLL;
        if (more) {
#pragma unroll
            for (int i = 0; i < GAE_UNROLL; ++i) { r0[i] = r1[i]; v0[i] = v1[i]; f0[i] = f1[i]; l0[i] = l1[i]; }
        }
    }
    // the remaining T % 8 rows
    for (; t >= 0; --t) step(t, rewards[t * N + n], values[t * N + n], flags[t * N + n], wr ? rec.logprobs[t * N + n] : 0.f);
    // explained_variance moments of the same rollout (algorithms/ppo.jl:256) without a second pass over the buffer
    if (ev_acc4) {
        sd = block_sum(sd, scratch); sdd = block_sum(sdd, scratch);
        sr = block_sum(sr, scratch); srr = block_sum(srr, scratch);
        if (threadIdx.x == 0) {
            atomicAdd(&ev_acc4[0], sd); atomicAdd(&ev_acc4[1], sdd); atomicAdd(&ev_acc4[2], sr); atomicAdd(&ev_acc4[3], srr);
        }
    }
}

// explained_variance = 1 - var(values - returns) / var(returns) (algorithms/ppo.jl:256):
// four double sums over the whole buffer; finalised on the host side of the ABI.
__global__ void __launch_bounds__(256) explained_variance_kernel(const float* __restrict__ values,
                                                                 const float* __restrict__ returns, long long n_total,
                                                                 double* acc4) {
    __shared__ double scratch[32];
    double sd = 0, sdd = 0, sr = 0, srr = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_total; i += (long long)gridDim.x * blockDim.x) {
        double v = values[i], r = returns[i], d = v - r;
        sd += d; sdd += d * d; sr += r; srr += r * r;
    }
    sd = block_sum(sd, scratch); sdd = block_sum(sdd, scratch);
    sr = block_sum(sr, scratch); srr = block_sum(srr, scratch);
    if (threadIdx.x == 0) {
        atomicAdd(&acc4[0], sd); atomicAdd(&acc4[1], sdd); atomicAdd(&acc4[2], sr); atomicAdd(&acc4[3], srr);
    }
}

// MonitorWrapperEnv ring buffers (monitorWrapperEnv.jl:1-7,52-53): push this rollout's finished
// episodes in the reference's order (step ascending, env ascending) into the `window`-deep ring.
// Only rows t >= t0 can still be inside the window at the end: t0 is the last row from which on the rows hold at least
// `window` episodes (0 when the rollout holds fewer).  With P(t) the exclusive prefix sum of done_count, the episode of
// row t >= t0, env n goes to ring position  head + P(t) - P(t0) + (episodes of row t before env n),  and the head
// advances by the total of those rows.  A position more than `window` below the new head would be overwritten by a later
// one of the same rollout, so it is not written; the remaining positions fall on distinct slots, and every row is
// compacted on its own: CTA b takes the rows t = b mod gridDim.x.  The last CTA to finish advances the head.
struct MonitorRing {
    float* ret;        // [window]
    int* len;          // [window]
    long long* head;   // [0] total pushes so far
    unsigned* ticket;  // [0] CTAs of the running monitor_finalize_kernel that have finished (0 between launches)
    int window;
};

#define MON_THREADS 256
// exclusive block scan of x over MON_THREADS threads; *total = the block's sum.  Contains two __syncthreads.
__device__ __forceinline__ long long mon_scan(long long x, long long* warp_tot, long long* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    long long inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    __syncthreads();
    if (lane == 31) warp_tot[w] = inc;
    __syncthreads();
    long long off = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < MON_THREADS / 32; ++i) { off += i < w ? warp_tot[i] : 0; tot += warp_tot[i]; }
    *total = tot;
    return off + inc - x;
}

__global__ void __launch_bounds__(MON_THREADS) monitor_finalize_kernel(MonitorRing ring, const unsigned char* __restrict__ flags,
                                                                       const float* __restrict__ ep_r, const int* __restrict__ ep_l,
                                                                       const int* __restrict__ done_count, long long T, long long N) {
    __shared__ long long warp_tot[MON_THREADS / 32];
    __shared__ long long s_pre[MON_THREADS];      // P(t) of the current chunk of rows
    __shared__ int s_dc[MON_THREADS];             // done_count of the current chunk of rows
    __shared__ long long s_head, s_t0, s_p0;
    const int tid = threadIdx.x;
    const long long W = ring.window, G = gridDim.x;
    long long tot;
    {
        long long s = 0;
        for (long long t = tid; t < T; t += MON_THREADS) s += done_count[t];
        mon_scan(s, warp_tot, &tot);
    }
    if (tid == 0) {
        s_head = *ring.head;
        s_t0 = tot < W ? 0 : T;      // T: not found yet
        s_p0 = 0;
    }
    long long carry = 0;
    const long long per = (N + MON_THREADS - 1) / MON_THREADS, n0 = tid * per, n1 = min(N, n0 + per);
    for (long long c = 0; c < T; c += MON_THREADS) {
        const long long t = c + tid;
        const int d = t < T ? done_count[t] : 0;
        long long ctot;
        const long long p = carry + mon_scan(d, warp_tot, &ctot);     // (its first __syncthreads publishes s_t0 / s_head)
        if (t < T && tot - p >= W && tot - p - d < W) { s_t0 = t; s_p0 = p; }
        s_pre[tid] = p; s_dc[tid] = d;
        carry += ctot;
        __syncthreads();
        const long long c1 = min(c + MON_THREADS, T);
        for (long long row = c + ((blockIdx.x - c % G) % G + G) % G; row < c1; row += G) {
            if (row < s_t0 || s_dc[row - c] == 0) continue;       // uniform over the block
            const unsigned char* fr = flags + row * N;
            int cnt = 0;
            for (long long n = n0; n < n1; ++n) cnt += (fr[n] & 3) ? 1 : 0;
            long long rtot;
            long long pos = s_head + (s_pre[row - c] - s_p0) + mon_scan(cnt, warp_tot, &rtot);
            const long long lo = s_head + (tot - s_p0) - W;
            for (long long n = n0; n < n1; ++n) {
                if (!(fr[n] & 3)) continue;
                if (pos >= lo) {
                    const int slot = (int)(pos % W);
                    ring.ret[slot] = ep_r[row * N + n];
                    ring.len[slot] = ep_l[row * N + n];
                }
                ++pos;
            }
        }
        __syncthreads();
    }
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(ring.ticket, 1u) == gridDim.x - 1) {      // every CTA has read the head
            *ring.head = s_head + (tot - s_p0);
            *ring.ticket = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Everything dril_iteration_result reports, gathered into one record at the end of an iteration so that the host
// needs a single pinned device->host copy per iteration and may enqueue the next iteration before reading it.
// ---------------------------------------------------------------------------------------------------------
struct IterRecord {
    double acc[16];             // iter_acc (update.cuh ITER_ACC_N)
    double ev[4];               // explained-variance moments (already summed over ranks)
    double roll_sums[2];
    unsigned long long roll_eps;
    long long ring_count;       // min(pushes, window)
    float ring_rew_mean, ring_len_mean;   // mean(::CircularBuffer{Float32}) order: sequential over the ring slots
    int stop, p2p_err;
};
struct IterRecordSrc {
    const double* acc; const double* ev; const double* roll_sums; const unsigned long long* roll_eps;
    const int* stop; const int* p2p_err; MonitorRing ring; int has_ring;
};
__global__ void iter_record_kernel(IterRecordSrc s, IterRecord* out) {
    const int t = threadIdx.x;
    if (t < 16) out->acc[t] = s.acc[t];
    if (t < 4) out->ev[t] = s.ev[t];
    if (t < 2) out->roll_sums[t] = s.roll_sums ? s.roll_sums[t] : 0.0;
    if (t == 0) {
        out->roll_eps = s.roll_eps ? *s.roll_eps : 0ull;
        out->stop = *s.stop;
        out->p2p_err = s.p2p_err ? *s.p2p_err : 0;
    }
    {   // window means: lane-strided partial sums, then a fixed-order butterfly (deterministic)
        long long cnt = 0;
        float sr = 0.f;
        double sl = 0.0;
        if (s.has_ring) {
            const long long head = *s.ring.head;
            cnt = head < s.ring.window ? head : s.ring.window;
            for (long long i = t; i < cnt; i += 32) { sr += s.ring.ret[i]; sl += (double)s.ring.len[i]; }
        }
        sr = warp_sum(sr); sl = warp_sum(sl);
        if (t == 31) {
            out->ring_count = cnt;
            out->ring_rew_mean = cnt ? sr / (float)cnt : nanf("");
            out->ring_len_mean = cnt ? (float)(sl / (double)cnt) : nanf("");
        }
    }
}
