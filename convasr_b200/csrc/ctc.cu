// CTC loss (alpha / beta / gradient), forced alignment, log_softmax(+argmax), top-K ids,
// greedy CTC collapse and the entropy reductions -- the latency/HBM-bound tail of the path.
//
// Replaces (reference file:line): F.ctc_loss call models.py:323 (arithmetic = ATen LossCTC);
// ctc.alignment ctc.py:6-75; F.log_softmax models.py:316; GreedyDecoder.decode
// decoders.py:5-16; GreedyCTCGenerator.generate transcript_generators.py:27-83;
// models.entropy / weighted_mean_entropy models.py:645-673.
//
// The recursions are T sequential steps, so each utterance gets one CTA with the extended
// target states across threads and the previous time step in shared memory -- or, for losses and
// alignments of targets too long for one CTA, one thread-block cluster (ctc_loss_cluster_kernel,
// ctc_align_cluster_kernel).
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>
#include <float.h>
#include <cuda_fp16.h>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

constexpr int kCtcMaxPer = 4;  // extended states per thread (S <= 4 * 1024)

__device__ __forceinline__ float lse3(float a, float b, float c) {
    const float m = fmaxf(a, fmaxf(b, c));
    if (m == -INFINITY) return -INFINITY;
    return logf(expf(a - m) + expf(b - m) + expf(c - m)) + m;
}
__device__ __forceinline__ float lse2(float a, float b) {
    const float m = fmaxf(a, b);
    if (m == -INFINITY) return -INFINITY;
    return logf(expf(a - m) + expf(b - m)) + m;
}

// ------------------------------------------------------------------------------------------
// CTC alpha / beta recursion.  grid = B * n_roles, block = threads (multiple of 32).
// beta is alpha on the time- and state-reversed problem (beta[t][s] = alpha'[il-1-t][S-1-s]),
// so one body serves both directions; with both roles in one grid the two latency-bound
// recursions of an utterance run concurrently on different SMs.
//
// Emissions are staged through shared memory with cp.async, G time steps per group and two
// groups in flight: s_e[group & 1][u][s] = lp[t0 + u, ext(s)].  The copy loop is laid out so that
// a warp reads 32 consecutive elements along the contiguous dimension of log_probs (time for the
// model's [B, C, T] layout), i.e. coalesced 128-byte lines instead of one sector per state and
// step; the sequential critical path only touches shared memory.
//
// Every kCtcRecentre steps the block maximum is subtracted from the live values and accumulated
// in fp64 (off_ws): stored alpha/beta stay O(10) instead of O(nll), which keeps fp32 rounding
// out of alpha + beta - nll for long utterances.
// ------------------------------------------------------------------------------------------
constexpr int kCtcPrefetch = 8;  // re-centring interval (also the offset-table granularity)

__device__ __forceinline__ float lse3_fast(float a, float b, float c) {
    const float m = fmaxf(a, fmaxf(b, c));
    if (m == -INFINITY) return -INFINITY;
    return __logf(__expf(a - m) + __expf(b - m) + __expf(c - m)) + m;
}
__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int PER>
__global__ void ctc_recursion_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc,
                                     const int64_t* __restrict__ targets, const int64_t* __restrict__ in_len,
                                     const int64_t* __restrict__ tgt_len, int B, int T, int L_max, int blank,
                                     int first_role, int G, float* __restrict__ alpha_ws,
                                     float* __restrict__ beta_ws, double* __restrict__ off_ws, int G_cap,
                                     float* __restrict__ nll) {
    extern __shared__ float sh[];
    const int b = blockIdx.x % B;
    const bool rev = (first_role + blockIdx.x / B) != 0;  // role 0 = alpha, role 1 = beta
    const int S_max = 2 * L_max + 1;
    const int S_pad = S_max | 1;  // odd row pitch: conflict-free transposed staging
    const int tl = (int)tgt_len[b];
    const int il = (int)in_len[b];
    const int S = 2 * tl + 1;
    float* buf0 = sh;  // index s+2 (two guard cells at the front)
    float* buf1 = sh + (S_max + 2);
    float* s_red = buf1 + (S_max + 2);                     // [32]
    int* s_ext = reinterpret_cast<int*>(s_red + 32);       // [S_max] class of virtual state s
    float* s_e = reinterpret_cast<float*>(s_ext + S_max);  // [2][G][S_pad]
    const float* lpb = lp + (int64_t)b * sb;
    float* ws = (rev ? beta_ws : alpha_ws) + (size_t)b * T * S_max;
    double* off = off_ws + ((size_t)b * 2 + (rev ? 1 : 0)) * G_cap;
    double O = 0.0;

    if (il <= 0 || il > T || tl > L_max || tl < 0) {
        if (threadIdx.x == 0 && !rev) {
            if (nll) nll[b] = INFINITY;
            off[G_cap - 1] = -(double)INFINITY;
        }
        return;
    }
    if (threadIdx.x == 0) off[0] = 0.0;

    // per-thread states (virtual index s runs in recursion order; sr is the real state)
    int sr[PER];
    bool skip[PER], live[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int s = threadIdx.x + i * blockDim.x;
        live[i] = s < S;
        sr[i] = rev ? S - 1 - s : s;
        int e = blank;
        skip[i] = false;
        if (live[i] && (sr[i] & 1)) {
            e = (int)targets[(size_t)b * L_max + (sr[i] >> 1)];
            if (s >= 2) {  // the state two behind in recursion order
                const int s2 = rev ? sr[i] + 2 : sr[i] - 2;
                skip[i] = e != (int)targets[(size_t)b * L_max + (s2 >> 1)];
            }
        }
        if (live[i]) s_ext[s] = e;
    }
    if (threadIdx.x < 2) { buf0[threadIdx.x] = -INFINITY; buf1[threadIdx.x] = -INFINITY; }
    const int64_t st_v = rev ? -st : st;                               // stride of one virtual step
    const float* lp0 = lpb + (int64_t)(rev ? il - 1 : 0) * st;         // virtual step 0
    const int64_t ws_v = rev ? -(int64_t)S_max : (int64_t)S_max;
    float* wsp = ws + (size_t)(rev ? il - 1 : 0) * S_max;              // row of virtual step 0
    __syncthreads();  // s_ext visible

    // stage group g: virtual steps 1 + g*G + u, u in [0, G).  A warp copies, for one state at a
    // time, 32 consecutive steps (time-contiguous layouts) or, for one step at a time, 32
    // consecutive states (class-contiguous layouts): coalesced either way, no div/mod.
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const bool time_contig = (st == 1 || st == -1);
    auto issue = [&](int g) {
        const int tg0 = 1 + g * G;
        if (tg0 < il) {
            float* dst = s_e + (size_t)(g & 1) * G * S_pad;
            const int n_u = min(G, il - tg0);
            if (time_contig) {
                for (int s = warp; s < S; s += n_warps) {
                    const float* src = lp0 + (int64_t)s_ext[s] * sc + (int64_t)tg0 * st_v;
                    for (int u = lane; u < n_u; u += 32) cp_async_4(dst + u * S_pad + s, src + (int64_t)u * st_v);
                }
            } else {
                for (int u = warp; u < n_u; u += n_warps) {
                    const float* src = lp0 + (int64_t)(tg0 + u) * st_v;
                    for (int s = lane; s < S; s += 32) cp_async_4(dst + u * S_pad + s, src + (int64_t)s_ext[s] * sc);
                }
            }
        }
        cp_async_commit();
    };
    issue(0);
    issue(1);

    // step 0
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int s = threadIdx.x + i * blockDim.x;
        if (live[i]) {
            float a = -INFINITY;
            if (s < 2) a = lp0[(int64_t)s_ext[s] * sc];
            buf0[s + 2] = a;
            wsp[sr[i]] = a;
        }
    }
    float* prev = buf0;
    float* cur = buf1;
    const int n_groups = (il - 1 + G - 1) / G;
    int t = 1;
    for (int g = 0; g < n_groups; ++g) {
        cp_async_wait<1>();  // this thread's copies of group g have landed
        __syncthreads();     // ... and everybody else's; also orders step 0 / previous group
        const float* se = s_e + (size_t)(g & 1) * G * S_pad + threadIdx.x;
        const int g_end = min(il, 1 + (g + 1) * G);
        while (t < g_end) {
            const int t0 = t;
            const int n_sub = min(kCtcPrefetch, g_end - t);
            float vlast[PER];
#pragma unroll
            for (int i = 0; i < PER; ++i) vlast[i] = -INFINITY;
            for (int u = 0; u < n_sub; ++u, ++t) {
                wsp += ws_v;
#pragma unroll
                for (int i = 0; i < PER; ++i) {
                    if (live[i]) {
                        const int s = threadIdx.x + i * blockDim.x;
                        const float e = se[i * blockDim.x];
                        const float a1 = prev[s + 2];
                        const float a2 = prev[s + 1];
                        const float a3 = skip[i] ? prev[s] : -INFINITY;
                        const float v = lse3_fast(a1, a2, a3) + e;
                        cur[s + 2] = v;
                        wsp[sr[i]] = v;
                        vlast[i] = v;
                    }
                }
                se += S_pad;
                __syncthreads();
                float* tmp = prev; prev = cur; cur = tmp;
            }
            // re-centre: subtract the block maximum from the live values (prev)
            float m = vlast[0];
#pragma unroll
            for (int i = 1; i < PER; ++i) m = fmaxf(m, vlast[i]);
            m = warp_max(m);
            if (lane == 0) s_red[warp] = m;
            __syncthreads();
            m = s_red[lane < n_warps ? lane : 0];
            m = warp_max(m);
            if (m > -INFINITY && m < INFINITY) {
#pragma unroll
                for (int i = 0; i < PER; ++i) {
                    const int s = threadIdx.x + i * blockDim.x;
                    if (live[i]) prev[s + 2] -= m;
                }
                O += (double)m;
            }
            if (threadIdx.x == 0) off[(t0 - 1) / kCtcPrefetch + 1] = O;
            __syncthreads();
        }
        issue(g + 2);  // refill the buffer everybody has just finished reading
    }
    cp_async_wait<0>();
    __syncthreads();
    if (threadIdx.x == 0 && !rev) {
        const float l1 = prev[S - 1 + 2];
        const float l2 = S > 1 ? prev[S - 2 + 2] : -INFINITY;
        const double ll = (double)lse2(l1, l2) + O;
        if (nll) nll[b] = (float)(-ll);
        off[G_cap - 1] = ll;
    }
}

// grad = exp(lp) * go for t < il, else 0.  Thread order follows the contiguous dim of grad.
__global__ void ctc_grad_init_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc,
                                     const int64_t* __restrict__ in_len, const float* __restrict__ go,
                                     int B, int T, int C, float* __restrict__ grad, int64_t gt, int64_t gb,
                                     int64_t gc) {
    if (gt == 1) {  // [B, C, T]-like (the model's layout): one (b, c) row of T frames at a time, no per-element division
        for (int row = blockIdx.x; row < B * C; row += gridDim.x) {
            const int b = row / C, c = row - b * C;
            const int il = (int)in_len[b];
            const float g0 = go[b];
            const float* src = lp + (int64_t)b * sb + (int64_t)c * sc;
            float* dst = grad + (int64_t)b * gb + (int64_t)c * gc;
            for (int t = threadIdx.x; t < T; t += blockDim.x) dst[t] = t < il ? expf(src[(int64_t)t * st]) * g0 : 0.f;
        }
        return;
    }
    if (gc == 1 && sc == 1) {  // class-contiguous rows (the large-vocabulary head's layout): one (b, t) row of C classes at a time
        for (int row = blockIdx.x; row < B * T; row += gridDim.x) {
            const int b = row / T, t = row - b * T;
            const bool on = t < (int)in_len[b];
            const float g0 = go[b];
            const float* src = lp + (int64_t)b * sb + (int64_t)t * st;
            float* dst = grad + (int64_t)b * gb + (int64_t)t * gt;
            if ((((uintptr_t)src | (uintptr_t)dst) & 15) == 0) {
                const int n4 = C >> 2;
                // 4 independent 16-byte loads in flight per thread (a 20 KB row is 5 trips of a 256-thread block otherwise)
                for (int i = threadIdx.x; i < n4; i += 4 * blockDim.x) {
                    float4 x[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (on && i + u * blockDim.x < n4) x[u] = reinterpret_cast<const float4*>(src)[i + u * blockDim.x];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (i + u * blockDim.x >= n4) break;
                        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (on) v = make_float4(__expf(x[u].x) * g0, __expf(x[u].y) * g0, __expf(x[u].z) * g0, __expf(x[u].w) * g0);
                        reinterpret_cast<float4*>(dst)[i + u * blockDim.x] = v;
                    }
                }
                for (int c = (n4 << 2) + threadIdx.x; c < C; c += blockDim.x) dst[c] = on ? expf(src[c]) * g0 : 0.f;
            } else {
                for (int c = threadIdx.x; c < C; c += blockDim.x) dst[c] = on ? expf(src[c]) * g0 : 0.f;
            }
        }
        return;
    }
    const int64_t n = (int64_t)B * T * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int b, c, t;
        {               // c fastest
            c = (int)(i % C); const int64_t r = i / C;
            if (gb < gt) { b = (int)(r % B); t = (int)(r / B); } else { t = (int)(r % T); b = (int)(r / T); }
        }
        float g = 0.f;
        if (t < (int)in_len[b]) g = expf(lp[(int64_t)t * st + (int64_t)b * sb + (int64_t)c * sc]) * go[b];
        grad[(int64_t)t * gt + (int64_t)b * gb + (int64_t)c * gc] = g;
    }
}

// grad[b, t, ext(s)] -= exp(alpha + beta + nll - lp) * go.  One warp per (b, t) row chunk.
__global__ void ctc_grad_scatter_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc,
                                        const int64_t* __restrict__ targets, const int64_t* __restrict__ in_len,
                                        const int64_t* __restrict__ tgt_len, int T, int L_max, int blank,
                                        const float* __restrict__ alpha_ws, const float* __restrict__ beta_ws,
                                        const double* __restrict__ off_ws, int G_cap, const float* __restrict__ go,
                                        float* __restrict__ grad, int64_t gt, int64_t gb, int64_t gc) {
    const int b = blockIdx.y;
    const int S_max = 2 * L_max + 1;
    const int tl = (int)tgt_len[b];
    const int il = (int)in_len[b];
    const int S = 2 * tl + 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * (blockDim.x >> 5) + warp;
    if (t >= il || tl > L_max) return;
    // alpha + beta - ll with the re-centring offsets folded in, in double: O(1) result
    const double* offa = off_ws + (size_t)b * 2 * G_cap;
    const double* offb = offa + G_cap;
    const int tb = il - 1 - t;  // step index of this frame in the reversed (beta) recursion
    const int ga = t == 0 ? 0 : (t - 1) / kCtcPrefetch, gbt = tb == 0 ? 0 : (tb - 1) / kCtcPrefetch;
    const float nl = (float)(offa[ga] + offb[gbt] - offa[G_cap - 1]);
    const float g = go[b];
    const float* lpt = lp + (int64_t)t * st + (int64_t)b * sb;
    float* gr = grad + (int64_t)t * gt + (int64_t)b * gb;
    const float lp_blank = lpt[(int64_t)blank * sc];
    const size_t row = ((size_t)b * T + t) * S_max;
    float blank_acc = 0.f;
    for (int s0 = 0; s0 < S; s0 += 32) {
        const int s = s0 + lane;
        if (s < S) {
            const float ab = alpha_ws[row + s] + beta_ws[row + s];
            if (s & 1) {
                const int c = (int)targets[(size_t)b * L_max + (s >> 1)];
                const float occ = expf(ab + nl - lpt[(int64_t)c * sc]);
                atomicAdd(gr + (int64_t)c * gc, -occ * g);
            } else {
                blank_acc += expf(ab + nl - lp_blank);
            }
        }
    }
    blank_acc = warp_sum(blank_acc);
    if (lane == 0) atomicAdd(gr + (int64_t)blank * gc, -blank_acc * g);
}

// ------------------------------------------------------------------------------------------
// ctc.alignment (ctc.py:6-75)
// ------------------------------------------------------------------------------------------
// HALF: the log-probs came from an fp16 tensor (exactly representable fp32 values here) and the reference ran its whole
// recursion in fp16 (ctc.py:29: "zero" = finfo(float16).min): torch.logsumexp on fp16 is the composite amax / sub / exp / sum /
// log / add with an fp16 result after EVERY operation (the 3-term sum accumulates in fp32 and rounds once), then the fp16
// add of the emission.  rh() reproduces those roundings; values stay fp16-representable in the fp32 buffers.
__device__ __forceinline__ float rh(float x) { return __half2float(__float2half_rn(x)); }
// exp / log of an fp16 value are functions on 65536 inputs: with tables (fp16 bit pattern -> fp16 bit pattern, e.g. taken from the
// host's torch) the recursion reproduces that implementation's fp16 results bit for bit; without, expf / logf rounded to fp16
// (two math libraries disagree on the fp16 rounding of ~1e-4 of the inputs, enough to flip an argmax tie in a long utterance).
__device__ __forceinline__ float half_fn(const uint16_t* __restrict__ table, float x_half_valued, float computed) {
    if (table == nullptr) return rh(computed);
    return __half2float(__ushort_as_half(__ldg(table + __half_as_ushort(__float2half_rn(x_half_valued)))));
}
// One state of one frame: alpha from the three predecessors p0 (stay), p1 (step), p2 (skip, already ZERO where the skip is
// not allowed) plus the emission e_t, and the back-pointer `arg` (first maximum wins: stay, then step, then skip, ctc.py:50).
// Shared by both alignment kernels, so they agree bit for bit wherever both run.
template <bool HALF>
__device__ __forceinline__ float ctc_align_state(float p0, float p1, float p2, float e_t, const uint16_t* __restrict__ tab_exp,
                                                 const uint16_t* __restrict__ tab_log, int& arg) {
    const float m = fmaxf(p0, fmaxf(p1, p2));
    arg = 0;
    if (p1 > p0) arg = 1;
    if (p2 > fmaxf(p0, p1)) arg = 2;
    const float ms = (fabsf(m) == INFINITY) ? 0.f : m;
    if (HALF) {
        const float d0 = rh(p0 - ms), d1 = rh(p1 - ms), d2 = rh(p2 - ms);
        const float e0 = half_fn(tab_exp, d0, expf(d0)), e1 = half_fn(tab_exp, d1, expf(d1)), e2 = half_fn(tab_exp, d2, expf(d2));
        const float ssum = rh((e0 + e1) + e2);
        const float lse = rh(half_fn(tab_log, ssum, logf(ssum)) + ms);
        return rh(e_t + lse);
    }
    const float lse = logf(expf(p0 - ms) + expf(p1 - ms) + expf(p2 - ms)) + ms;
    return e_t + lse;
}
template <bool HALF>
__global__ void ctc_align_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc,
                                 const int64_t* __restrict__ targets, const int64_t* __restrict__ in_len,
                                 const int64_t* __restrict__ tgt_len, int T, int L_max, int blank,
                                 uint8_t* __restrict__ bp_ws, int64_t* __restrict__ out,
                                 const uint16_t* __restrict__ tab_exp, const uint16_t* __restrict__ tab_log) {
    extern __shared__ float sh[];
    const float ZERO = HALF ? -65504.f : -FLT_MAX;  // torch.finfo(dtype).min, ctc.py:29
    const int b = blockIdx.x;
    const int S_max = 2 * L_max + 1;
    int tl = (int)tgt_len[b];
    if (tl > L_max) tl = L_max;
    const int il = (int)in_len[b];
    const int S = 2 * tl + 1;
    float* buf0 = sh;  // index s+2
    float* buf1 = sh + (S_max + 2);
    const float* lpb = lp + (int64_t)b * sb;
    uint8_t* bp = bp_ws + (size_t)b * T * S_max;

    for (int l = threadIdx.x; l < L_max; l += blockDim.x) out[(size_t)b * L_max + l] = 0;

    int ext[kCtcMaxPer];
    bool diff[kCtcMaxPer];
#pragma unroll
    for (int i = 0; i < kCtcMaxPer; ++i) {
        const int s = threadIdx.x + i * blockDim.x;
        ext[i] = blank;
        diff[i] = false;
        if (s < S) {
            if (s & 1) ext[i] = (int)targets[(size_t)b * L_max + (s >> 1)];
            if (s >= 2) {
                const int e2 = ((s - 2) & 1) ? (int)targets[(size_t)b * L_max + ((s - 2) >> 1)] : blank;
                diff[i] = ext[i] != e2;  // ctc.py:23-27 (blank vs blank -> False)
            }
        }
    }
    if (threadIdx.x < 2) { buf0[threadIdx.x] = ZERO; buf1[threadIdx.x] = ZERO; }
#pragma unroll
    for (int i = 0; i < kCtcMaxPer; ++i) {
        const int s = threadIdx.x + i * blockDim.x;
        if (s < S) buf0[s + 2] = (s < 2) ? lpb[(int64_t)ext[i] * sc] : ZERO;  // ctc.py:32-33
    }
    __syncthreads();
    float* prev = buf0;
    float* cur = buf1;
    // NB: the reference runs the recursion over ALL T frames of the padded batch (ctc.py:47)
    for (int t = 1; t < T; ++t) {
#pragma unroll
        for (int i = 0; i < kCtcMaxPer; ++i) {
            const int s = threadIdx.x + i * blockDim.x;
            if (s < S) {
                const float p0 = prev[s + 2];
                const float p1 = prev[s + 1];
                const float p2 = diff[i] ? prev[s] : ZERO;
                const float e_t = lpb[(int64_t)t * st + (int64_t)ext[i] * sc];
                int arg;
                cur[s + 2] = ctc_align_state<HALF>(p0, p1, p2, e_t, tab_exp, tab_log, arg);
                bp[(size_t)t * S_max + s] = (uint8_t)arg;
            }
        }
        __syncthreads();
        float* tmp = prev; prev = cur; cur = tmp;
    }
    if (threadIdx.x == 0 && il >= 1) {
        // terminal state from log_alpha after the FULL loop (global T-1), ctc.py:56-61
        const float l1 = prev[(2 * tl - 1) + 2];  // tl == 0 reads the guard cell (= ZERO)
        const float l2 = prev[(2 * tl) + 2];
        int s = 2 * tl - 1 + (l2 > l1 ? 1 : 0);
        if (s < 0) s = 0;
        int last_state = -1;
        for (int t = il - 1; t >= 0; --t) {
            if (s != last_state) {
                if (s & 1) out[(size_t)b * L_max + (s >> 1)] = t;  // last frame spent in label s
                last_state = s;
            }
            if (t > 0) {
                s -= (int)bp[(size_t)t * S_max + s];
                if (s < 0) s = 0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// ctc.alignment for long targets: one thread-block cluster per utterance.
// The extended states are cut into slices of W states (W % 4 == 0); slice k lives on CTA k % n of the cluster, in its
// local slot k / n (n = cluster size; one slot per CTA unless a caller forces small slices).  A slot holds two guard
// cells in front of its W states: the last two alpha values of slice k-1 at the previous frame, which the CTA owning
// slice k-1 stores there through distributed shared memory.  One cluster barrier per frame orders those stores
// (and the local double buffer) -- every CTA runs every frame, live states or not, so no barrier can be missed.
// A thread owns groups of 4 consecutive states: their four 2-bit back-pointers make one byte of the packed
// workspace [B, T, ceil(S_max / 4)] (code of state s in bits 2*(s%4)), so no two threads write the same byte.
// The recursion leaves the start state of the back-trace in out[b, 0]; ctc_align_backtrace_kernel takes it from there.
// ------------------------------------------------------------------------------------------
constexpr int kAlignClusterMax = 16;   // CTAs per utterance (non-portable cluster size)
constexpr int kAlignGroupsPer = 2;     // groups of 4 states per thread
constexpr int kAlignCtaStates = 4 * kAlignGroupsPer * 1024;  // states one CTA holds
constexpr int kAlignLongMaxL = (kAlignClusterMax * kAlignCtaStates - 1) / 2;  // 65535: S = 131071

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
// generic address of `p` (a shared-memory address of this CTA) in the shared memory of CTA `rank` of the cluster
__device__ __forceinline__ float* cluster_map(float* p, uint32_t rank) {
    uint64_t out;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"(reinterpret_cast<uint64_t>(p)), "r"(rank));
    return reinterpret_cast<float*>(out);
}

template <bool HALF>
__global__ void __launch_bounds__(1024, 1)
ctc_align_cluster_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc, const int64_t* __restrict__ targets,
                         const int64_t* __restrict__ in_len, const int64_t* __restrict__ tgt_len, int T, int L_max, int blank,
                         int W, int n_slots, int64_t pitch, uint8_t* __restrict__ bp_ws, int64_t* __restrict__ out,
                         const uint16_t* __restrict__ tab_exp, const uint16_t* __restrict__ tab_log) {
    extern __shared__ float sh[];
    const float ZERO = HALF ? -65504.f : -FLT_MAX;  // torch.finfo(dtype).min, ctc.py:29
    const int n = (int)cluster_nctarank(), c = (int)cluster_ctarank();
    const int b = blockIdx.x / n;
    int tl = (int)tgt_len[b];
    tl = tl < 0 ? 0 : (tl > L_max ? L_max : tl);
    const int S = 2 * tl + 1;
    const int slot_len = W + 2;
    const int buf_len = n_slots * slot_len;
    float* s_term = sh + 2 * buf_len;  // [2] alpha of states 2tl-1, 2tl at frame T-1 (on CTA 0)
    const int gps = W >> 2;            // groups per slice
    const int n_groups = n_slots * gps;
    const float* lpb = lp + (int64_t)b * sb;
    uint8_t* bp = bp_ws + (int64_t)b * T * pitch;

    for (int i = threadIdx.x; i < 2 * buf_len + 2; i += blockDim.x) sh[i] = ZERO;

    int loc[kAlignGroupsPer], s0[kAlignGroupsPer], lab1[kAlignGroupsPer], lab3[kAlignGroupsPer];
    bool live[kAlignGroupsPer], skip1[kAlignGroupsPer], skip3[kAlignGroupsPer];
    float* next_guard[kAlignGroupsPer];  // guard cells of slice k+1 in buffer 0 (buffer 1: + buf_len), or nullptr
#pragma unroll
    for (int i = 0; i < kAlignGroupsPer; ++i) {
        const int g = threadIdx.x + i * blockDim.x;
        const int j = g / gps, o = (g - j * gps) * 4, k = j * n + c;
        live[i] = g < n_groups && k * W + o < S;
        s0[i] = k * W + o;
        loc[i] = j * slot_len + 2 + o;
        lab1[i] = lab3[i] = blank;
        skip1[i] = skip3[i] = false;
        next_guard[i] = nullptr;
        if (!live[i]) continue;
        const int64_t* tg = targets + (int64_t)b * L_max;
        if (s0[i] + 1 < S) {  // odd states may skip from the label two behind when it differs (ctc.py:23-27)
            lab1[i] = (int)tg[(s0[i] + 1) >> 1];
            skip1[i] = s0[i] + 1 >= 3 && lab1[i] != (int)tg[((s0[i] + 1) >> 1) - 1];
        }
        if (s0[i] + 3 < S) {
            lab3[i] = (int)tg[(s0[i] + 3) >> 1];
            skip3[i] = lab3[i] != lab1[i];
        }
        const int k1 = k + 1;
        if (o == W - 4 && k1 < n * n_slots) {
            next_guard[i] = cluster_map(sh + (k1 / n) * slot_len, (uint32_t)(k1 % n));
        }
    }
    __syncthreads();  // ZERO fill before the frame-0 values
#pragma unroll
    for (int i = 0; i < kAlignGroupsPer; ++i)
        if (live[i] && s0[i] == 0) {  // ctc.py:32-33
            sh[loc[i]] = lpb[(int64_t)blank * sc];
            if (S > 1) sh[loc[i] + 1] = lpb[(int64_t)lab1[i] * sc];
        }

    // emissions of the next frame are loaded while the cluster barrier of this one is pending
    float eb[kAlignGroupsPer], e1[kAlignGroupsPer], e3[kAlignGroupsPer];
    auto load_e = [&](int t) {
#pragma unroll
        for (int i = 0; i < kAlignGroupsPer; ++i)
            if (live[i]) {
                const float* r = lpb + (int64_t)t * st;
                eb[i] = r[(int64_t)blank * sc];
                e1[i] = r[(int64_t)lab1[i] * sc];
                e3[i] = r[(int64_t)lab3[i] * sc];
            }
    };
    cluster_arrive();  // every CTA of the cluster has started and initialised its buffers
    if (T > 1) load_e(1);
    cluster_wait();

    // NB: the reference runs the recursion over ALL T frames of the padded batch (ctc.py:47)
    for (int t = 1; t < T; ++t) {
        const float* prev = sh + ((t - 1) & 1) * buf_len;
        float* cur = sh + (t & 1) * buf_len;
#pragma unroll
        for (int i = 0; i < kAlignGroupsPer; ++i) {
            if (!live[i]) continue;
            const float* p = prev + loc[i];
            const float am1 = p[-1], a0 = p[0], a1 = p[1], a2 = p[2], a3 = p[3];
            // all four states unconditionally (independent chains, no branches): states >= S of the last live group are
            // never read by a live state, the terminal read or the back-trace
            int arg0, arg1, arg2, arg3;
            const float v0 = ctc_align_state<HALF>(a0, am1, ZERO, eb[i], tab_exp, tab_log, arg0);  // even states: blanks, no skip
            const float v1 = ctc_align_state<HALF>(a1, a0, skip1[i] ? am1 : ZERO, e1[i], tab_exp, tab_log, arg1);
            const float v2 = ctc_align_state<HALF>(a2, a1, ZERO, eb[i], tab_exp, tab_log, arg2);
            const float v3 = ctc_align_state<HALF>(a3, a2, skip3[i] ? a1 : ZERO, e3[i], tab_exp, tab_log, arg3);
            cur[loc[i]] = v0;
            cur[loc[i] + 1] = v1;
            cur[loc[i] + 2] = v2;
            cur[loc[i] + 3] = v3;
            bp[(int64_t)t * pitch + (s0[i] >> 2)] = (uint8_t)(arg0 | (arg1 << 2) | (arg2 << 4) | (arg3 << 6));
            if (next_guard[i]) {
                float* gd = next_guard[i] + (t & 1) * buf_len;
                gd[0] = v2;
                gd[1] = v3;
            }
        }
        cluster_arrive();
        if (t + 1 < T) load_e(t + 1);
        cluster_wait();
    }

    // terminal state from log_alpha after the FULL loop (global T-1), ctc.py:56-61: both values meet on CTA 0
    if (threadIdx.x < 2) {
        const int x = 2 * tl - 1 + (int)threadIdx.x;  // tl == 0: state -1 keeps ZERO
        const int k = x / W;
        if (x >= 0 && k % n == c) *cluster_map(s_term + threadIdx.x, 0) = sh[((T - 1) & 1) * buf_len + (k / n) * slot_len + 2 + (x - k * W)];
    }
    cluster_arrive();
    cluster_wait();
    if (c == 0 && threadIdx.x == 0) {
        const int s = 2 * tl - 1 + (s_term[1] > s_term[0] ? 1 : 0);
        out[(int64_t)b * L_max] = s < 0 ? 0 : s;
    }
}

// Back-trace over the packed back-pointers, one warp per utterance.  s moves down by at most 2 per frame, so the codes of
// the next 32 frames lie within 17 bytes of each row: every lane fetches one row's window (all loads of a strip in
// flight at once), then lane 0 walks the strip from shared memory -- one memory round trip per 32 frames instead of one
// per frame.  Output: the last frame spent in each label, zeros past target_length, zeros everywhere when il < 1.
constexpr int kTraceWin = 17;
__global__ void __launch_bounds__(32)
ctc_align_backtrace_kernel(const uint8_t* __restrict__ bp_ws, int64_t pitch, const int64_t* __restrict__ in_len, int T, int L_max,
                           int64_t* __restrict__ out) {
    __shared__ uint8_t strip[32][kTraceWin + 3];
    const int b = blockIdx.x, lane = threadIdx.x;
    int64_t* ob = out + (int64_t)b * L_max;
    int s = (int)ob[0];  // start state left by ctc_align_cluster_kernel
    __syncwarp();
    for (int l = lane; l < L_max; l += 32) ob[l] = 0;
    int il = (int)in_len[b];
    if (il > T) il = T;
    if (il < 1) return;
    __syncwarp();
    const uint8_t* bpb = bp_ws + (int64_t)b * T * pitch;
    int last_state = -1;
    for (int t = il - 1; t >= 0; t -= 32) {
        const int wb = max(0, (s >> 2) - (kTraceWin - 1));
        const int r = t - lane;
        if (r > 0) {
            const uint8_t* row = bpb + (int64_t)r * pitch;
#pragma unroll
            for (int k = 0; k < kTraceWin; ++k)
                if (wb + k < pitch) strip[lane][k] = row[wb + k];
        }
        __syncwarp();
        if (lane == 0) {
            for (int u = 0; u < 32 && t - u >= 0; ++u) {
                const int tt = t - u;
                if (s != last_state) {
                    if (s & 1) ob[s >> 1] = tt;  // last frame spent in label s
                    last_state = s;
                }
                if (tt > 0) {
                    s -= (strip[u][(s >> 2) - wb] >> (2 * (s & 3))) & 3;
                    if (s < 0) s = 0;
                }
            }
        }
        s = __shfl_sync(0xffffffffu, s, 0);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// CTC loss for long targets: one thread-block cluster per utterance and direction, on the geometry of
// ctc_align_cluster_kernel (slices of W states, slice k in slot k / n of CTA k % n, two guard cells in front of each slot
// written by the owner of the previous slice through distributed shared memory, one cluster barrier per frame with the
// next frame's inputs loaded between arrive and wait).  Utterance b recurses over its own input_lengths[b] frames (all
// CTAs of a cluster share it, so none misses a barrier); "zero" is -inf.  Beta is alpha on the time- and state-reversed
// problem, as in ctc_recursion_kernel, whose arithmetic this is -- the same lse3_fast calls with the same argument order,
// re-centring by the maximum of the live values at the end of every kCtcPrefetch-frame sub-block counted from frame 1
// (and the final partial one), fp64 offsets in the same [B, 2, G_cap] table -- so the nll is bit-identical wherever both
// kernels run.  The maximum is taken over the cluster: at the end of a sub-block every CTA stores its block maximum into
// entry c of a 16-entry array on every CTA (two arrays, by sub-block parity) before it arrives; after the wait every CTA
// reduces the same values.  The shift is applied as the values are read at the next frame (v - m: the rounding of the
// one-CTA kernel's in-place subtraction), to the slice and its guard cells alike, so it needs no pass or barrier of its own.
// MODE 0: alpha, nll and offsets only.  MODE 1: also stores the re-centred alpha into ws [B, T, S_max].
// MODE 2: beta plus the gradient.  At every frame it reads that frame's stored alpha row (loaded a frame ahead, like the
// emissions) and subtracts exp(alpha + beta + (O_alpha + O_beta - ll) - lp) * go -- ctc_grad_scatter_kernel's formula --
// from grad (already exp(lp) * go from ctc_grad_init_kernel): atomics for label states; blank occupancies are summed per
// CTA in shared memory and added with one atomic per CTA and frame after the barrier.
// ------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(1024, 1)
ctc_loss_cluster_kernel(const float* __restrict__ lp, int64_t st, int64_t sb, int64_t sc, const int64_t* __restrict__ targets,
                        const int64_t* __restrict__ in_len, const int64_t* __restrict__ tgt_len, int T, int L_max, int blank,
                        int W, int n_slots, float* __restrict__ ws, double* __restrict__ off_ws, int G_cap,
                        float* __restrict__ nll, const float* __restrict__ go, float* __restrict__ grad, int64_t gt, int64_t gb,
                        int64_t gc) {
    constexpr bool rev = MODE == 2;
    extern __shared__ float sh[];
    const int n = (int)cluster_nctarank(), c = (int)cluster_ctarank();
    const int b = blockIdx.x / n;
    const int S_max = 2 * L_max + 1;
    const int tl = (int)tgt_len[b];
    const int il = (int)in_len[b];
    const int S = 2 * tl + 1;
    double* off = off_ws + ((int64_t)b * 2 + (rev ? 1 : 0)) * G_cap;
    if (il <= 0 || il > T || tl > L_max || tl < 0) {  // the same for every CTA of the cluster: all leave before any barrier
        if (!rev && c == 0 && threadIdx.x == 0) {
            nll[b] = INFINITY;
            off[G_cap - 1] = -(double)INFINITY;
        }
        return;
    }
    const int slot_len = W + 2;
    const int buf_len = n_slots * slot_len;
    float* s_max = sh + 2 * buf_len;                // [2][kAlignClusterMax] block maxima of the cluster, by sub-block parity
    float* s_red = s_max + 2 * kAlignClusterMax;    // [32] warp maxima
    float* s_misc = s_red + 32;                     // [2] alpha of states S-1, S-2 at the last frame (CTA 0) / blank sums by frame parity
    const int gps = W >> 2;                         // groups per slice
    const int n_groups = n_slots * gps;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int64_t* tg = targets + (int64_t)b * L_max;
    const float* lp0 = lp + (int64_t)b * sb + (int64_t)(rev ? il - 1 : 0) * st;  // virtual frame 0
    const int64_t st_v = rev ? -st : st;

    for (int i = threadIdx.x; i < 2 * buf_len; i += blockDim.x) sh[i] = -INFINITY;
    if (threadIdx.x < 2) s_misc[threadIdx.x] = rev ? 0.f : -INFINITY;
    if (c == 0 && threadIdx.x == 0) off[0] = 0.0;

    // virtual state s (recursion order) is real state rev ? S-1-s : s; S is odd, so even virtual states are blanks
    auto label = [&](int s) { return (int)tg[(rev ? S - 1 - s : s) >> 1]; };
    int loc[kAlignGroupsPer], s0[kAlignGroupsPer], lab1[kAlignGroupsPer], lab3[kAlignGroupsPer];
    bool live[kAlignGroupsPer], skip1[kAlignGroupsPer], skip3[kAlignGroupsPer];
    float* next_guard[kAlignGroupsPer];  // guard cells of slice k+1 in buffer 0 (buffer 1: + buf_len), or nullptr
#pragma unroll
    for (int i = 0; i < kAlignGroupsPer; ++i) {
        const int g = threadIdx.x + i * blockDim.x;
        const int j = g / gps, o = (g - j * gps) * 4, k = j * n + c;
        s0[i] = k * W + o;
        live[i] = g < n_groups && s0[i] < S;
        loc[i] = j * slot_len + 2 + o;
        lab1[i] = lab3[i] = blank;
        skip1[i] = skip3[i] = false;
        next_guard[i] = nullptr;
        if (!live[i]) continue;
        if (s0[i] + 1 < S) {  // a label state may skip from the one two behind when the labels differ
            lab1[i] = label(s0[i] + 1);
            skip1[i] = s0[i] >= 2 && lab1[i] != label(s0[i] - 1);
        }
        if (s0[i] + 3 < S) {
            lab3[i] = label(s0[i] + 3);
            skip3[i] = lab3[i] != lab1[i];
        }
        const int k1 = k + 1;
        if (o == W - 4 && k1 < n * n_slots) next_guard[i] = cluster_map(sh + (k1 / n) * slot_len, (uint32_t)(k1 % n));
    }

    float eb[kAlignGroupsPer], e1[kAlignGroupsPer], e3[kAlignGroupsPer];
    auto load_e = [&](int u) {
        const float* r = lp0 + (int64_t)u * st_v;
#pragma unroll
        for (int i = 0; i < kAlignGroupsPer; ++i)
            if (live[i]) {
                eb[i] = r[(int64_t)blank * sc];
                e1[i] = r[(int64_t)lab1[i] * sc];
                e3[i] = r[(int64_t)lab3[i] * sc];
            }
    };
    // MODE 2: the stored alpha of the frame (real states S-1-s0 .. S-4-s0) and its offset
    float al[kAlignGroupsPer][4];
    double oa = 0.0, ll = 0.0;
    float g_out = 0.f;
    const double* off_a = off_ws + (int64_t)b * 2 * G_cap;
    auto load_a = [&](int u) {
        const int t = il - 1 - u;
        const float* row = ws + ((int64_t)b * T + t) * S_max + (S - 1);
#pragma unroll
        for (int i = 0; i < kAlignGroupsPer; ++i)
            if (live[i]) {
#pragma unroll
                for (int q = 0; q < 4; ++q) al[i][q] = s0[i] + q < S ? row[-(s0[i] + q)] : 0.f;
            }
        oa = off_a[t == 0 ? 0 : (t - 1) / kCtcPrefetch];
    };
    if (rev) {
        ll = off_a[G_cap - 1];
        g_out = go[b];
    }

    cluster_arrive();  // every CTA of the cluster has started and initialised its buffers
    load_e(0);
    if (rev) load_a(0);
    cluster_wait();

    double O = 0.0;
    float shift = 0.f;  // re-centring still to be applied to the values of the previous frame
    for (int u = 0; u < il; ++u) {
        const float* prev = sh + ((u + 1) & 1) * buf_len;
        float* cur = sh + (u & 1) * buf_len;
        const int t = rev ? il - 1 - u : u;  // real frame
        const float nl = rev ? (float)(oa + O - ll) : 0.f;
        float* gr = rev ? grad + (int64_t)t * gt + (int64_t)b * gb : nullptr;
        float* wrow = MODE == 1 ? ws + ((int64_t)b * T + t) * S_max : nullptr;
        float mloc = -INFINITY, bacc = 0.f;
#pragma unroll
        for (int i = 0; i < kAlignGroupsPer; ++i) {
            if (!live[i]) continue;
            float v[4];
            if (u == 0) {
                v[0] = s0[i] == 0 ? eb[i] : -INFINITY;
                v[1] = s0[i] == 0 && S > 1 ? e1[i] : -INFINITY;
                v[2] = v[3] = -INFINITY;
            } else {
                const float* p = prev + loc[i];
                const float am1 = p[-1] - shift, a0 = p[0] - shift, a1 = p[1] - shift, a2 = p[2] - shift, a3 = p[3] - shift;
                // all four states unconditionally; states >= S of the last live group are never read by a live state
                v[0] = lse3_fast(a0, am1, -INFINITY) + eb[i];
                v[1] = lse3_fast(a1, a0, skip1[i] ? am1 : -INFINITY) + e1[i];
                v[2] = lse3_fast(a2, a1, -INFINITY) + eb[i];
                v[3] = lse3_fast(a3, a2, skip3[i] ? a1 : -INFINITY) + e3[i];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) cur[loc[i] + q] = v[q];
            if (next_guard[i]) {
                float* gd = next_guard[i] + (u & 1) * buf_len;
                gd[0] = v[2];
                gd[1] = v[3];
            }
            const int nv = S - s0[i];  // live states of the group (>= 1)
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (q < nv) {
                    mloc = fmaxf(mloc, v[q]);
                    if (MODE == 1) wrow[s0[i] + q] = v[q];
                    if (MODE == 2) {
                        const float e = (q & 1) ? (q == 1 ? e1[i] : e3[i]) : eb[i];
                        const float occ = expf((al[i][q] + v[q]) + nl - e);
                        if (q & 1) atomicAdd(gr + (int64_t)(q == 1 ? lab1[i] : lab3[i]) * gc, -occ * g_out);
                        else bacc += occ;
                    }
                }
        }
        if (rev) {
            bacc = warp_sum(bacc);
            if (lane == 0) atomicAdd(s_misc + (u & 1), bacc);
        }
        const bool block_end = u >= 1 && (u % kCtcPrefetch == 0 || u == il - 1);
        const int par = ((u - 1) / kCtcPrefetch) & 1;
        if (block_end) {
            mloc = warp_max(mloc);
            if (lane == 0) s_red[warp] = mloc;
            __syncthreads();
            if (warp == 0) {
                float m = s_red[lane < n_warps ? lane : 0];
                m = warp_max(m);
                if (lane < n) *cluster_map(s_max + par * kAlignClusterMax + c, (uint32_t)lane) = m;
            }
        }
        cluster_arrive();
        if (u + 1 < il) {
            load_e(u + 1);
            if (rev) load_a(u + 1);
        }
        cluster_wait();
        if (rev && threadIdx.x == 0) {
            const float s = s_misc[u & 1];
            s_misc[u & 1] = 0.f;
            atomicAdd(gr + (int64_t)blank * gc, -s * g_out);
        }
        shift = 0.f;
        if (block_end) {
            float m = s_max[par * kAlignClusterMax];
            for (int r = 1; r < n; ++r) m = fmaxf(m, s_max[par * kAlignClusterMax + r]);
            if (m > -INFINITY && m < INFINITY) {
                shift = m;
                O += (double)m;
            }
            if (c == 0 && threadIdx.x == 0) off[(u - 1) / kCtcPrefetch + 1] = O;
        }
    }
    if (rev) return;

    // log-likelihood from states S-1 and S-2 of the last frame, re-centred: both values meet on CTA 0
    if (threadIdx.x < 2) {
        const int x = S - 1 - (int)threadIdx.x;  // S == 1: state -1 keeps -inf
        const int k = x / W;
        if (x >= 0 && k % n == c)
            *cluster_map(s_misc + threadIdx.x, 0) = sh[((il - 1) & 1) * buf_len + (k / n) * slot_len + 2 + (x - k * W)] - shift;
    }
    cluster_arrive();
    cluster_wait();
    if (c == 0 && threadIdx.x == 0) {
        const double l = (double)lse2(s_misc[0], s_misc[1]) + O;
        nll[b] = (float)(-l);
        off[G_cap - 1] = l;
    }
}

// ------------------------------------------------------------------------------------------
// log_softmax + argmax over dim 1 of [B, C, T]; block = (32 t) x (8 class groups)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
log_softmax_argmax_kernel(const float* __restrict__ x, int B, int C, int T, float* __restrict__ out,
                          int* __restrict__ amax) {
    __shared__ float s_m[8][33], s_s[8][33];
    __shared__ int s_i[8][33];
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int t = blockIdx.x * 32 + lane;
    const bool ok = t < T;
    const float* xb = x + (size_t)b * C * T;
    float m = -INFINITY, s = 0.f;
    int im = 0x7fffffff;
    if (ok) {
        // 4 independent loads in flight per thread (a vocabulary of 5000 is 625 dependent updates otherwise)
        for (int c0 = grp; c0 < C; c0 += 32) {
            float v4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v4[u] = c0 + 8 * u < C ? xb[(size_t)(c0 + 8 * u) * T + t] : 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + 8 * u;
                if (c >= C) break;
                const float v = v4[u];
                if (v > m) { s = s * expf(m - v) + 1.f; m = v; im = c; }
                else if (v == -INFINITY && m == -INFINITY) { if (im == 0x7fffffff) im = c; }
                else s += expf(v - m);
            }
        }
    }
    s_m[grp][lane] = m; s_s[grp][lane] = s; s_i[grp][lane] = im;
    __syncthreads();
    float M = -INFINITY; int IM = 0x7fffffff;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const float mg = s_m[g][lane]; const int ig = s_i[g][lane];
        if (mg > M || (mg == M && ig < IM)) { M = mg; IM = ig; }
    }
    float Ssum = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const float mg = s_m[g][lane];
        if (mg != -INFINITY) Ssum += s_s[g][lane] * expf(mg - M);
    }
    const float lse = M + logf(Ssum);
    if (ok) {
        if (out != nullptr) {
            float* ob = out + (size_t)b * C * T;
            for (int c0 = grp; c0 < C; c0 += 32) {
                float v4[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v4[u] = c0 + 8 * u < C ? xb[(size_t)(c0 + 8 * u) * T + t] : 0.f;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (c0 + 8 * u < C) ob[(size_t)(c0 + 8 * u) * T + t] = v4[u] - lse;
            }
        }
        if (amax != nullptr && grp == 0) amax[(size_t)b * T + t] = IM == 0x7fffffff ? 0 : IM;
    }
}

// log_probs = logits - lse[row] over class-contiguous rows (second half of the fused large-vocabulary head)
__global__ void __launch_bounds__(256)
log_softmax_rows_kernel(const float* __restrict__ x, const float* __restrict__ lse, long long R, int C, int ld,
                        float* __restrict__ out) {
    const int n4 = C >> 2;  // ld % 4 == 0 and 16-byte aligned bases: float4 all the way, tail scalars
    for (long long r = blockIdx.x; r < R; r += gridDim.x) {
        const float l = __ldg(lse + r);
        const float4* src = reinterpret_cast<const float4*>(x + r * ld);
        float4* dst = reinterpret_cast<float4*>(out + r * ld);
        for (int i = threadIdx.x; i < n4; i += 4 * 256) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) if (i + u * 256 < n4) v[u] = src[i + u * 256];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * 256 < n4) dst[i + u * 256] = make_float4(v[u].x - l, v[u].y - l, v[u].z - l, v[u].w - l);
        }
        for (int c = (n4 << 2) + threadIdx.x; c < C; c += 256) out[r * ld + c] = x[r * ld + c] - l;
    }
}

__global__ void __launch_bounds__(256)
log_softmax_bwd_kernel(const float* __restrict__ lp, const float* __restrict__ go, int B, int C, int T,
                       float* __restrict__ gi) {
    __shared__ float s_s[8][33];
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int t = blockIdx.x * 32 + lane;
    const bool ok = t < T;
    const size_t base = (size_t)b * C * T;
    float s = 0.f;
    if (ok) for (int c = grp; c < C; c += 8) s += go[base + (size_t)c * T + t];
    s_s[grp][lane] = s;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) tot += s_s[g][lane];
    if (ok)
        for (int c = grp; c < C; c += 8) {
            const size_t o = base + (size_t)c * T + t;
            gi[o] = go[o] - expf(lp[o]) * tot;
        }
}

// ------------------------------------------------------------------------------------------
// top-K class ids per frame (K <= 8), ties -> lowest id first
// ------------------------------------------------------------------------------------------
constexpr int kTopKMax = 8;
__global__ void topk_ids_kernel(const float* __restrict__ x, int B, int C, int T, int K, int* __restrict__ out) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const float* xb = x + (size_t)b * C * T;
    float v[kTopKMax];
    int id[kTopKMax];
#pragma unroll
    for (int k = 0; k < kTopKMax; ++k) { v[k] = -INFINITY; id[k] = -1; }
    for (int c = 0; c < C; ++c) {
        float cv = xb[(size_t)c * T + t];
        int ci = c;
        // insert keeping (value desc, id asc); strict > keeps earlier ids first on ties
#pragma unroll
        for (int k = 0; k < kTopKMax; ++k) {
            if (k < K && (cv > v[k] || id[k] < 0)) {
                const float tv = v[k]; const int ti = id[k];
                v[k] = cv; id[k] = ci; cv = tv; ci = ti;
                if (ci < 0) break;
            }
        }
    }
    for (int k = 0; k < K; ++k) out[((size_t)b * K + k) * T + t] = id[k];
}

// two largest probabilities per frame, exp(top-2 log_probs) -- models.margin (models.py:676-677); out fp32 [B, 2, T]
__global__ void top2_probs_kernel(const float* __restrict__ x, int64_t sb, int64_t sc, int64_t st, int B, int C, int T,
                                  float* __restrict__ out) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const float* xb = x + (int64_t)b * sb + (int64_t)t * st;
    float v0 = -INFINITY, v1 = -INFINITY;
    for (int c = 0; c < C; ++c) {
        const float v = xb[(int64_t)c * sc];
        if (v > v0) { v1 = v0; v0 = v; }
        else if (v > v1) v1 = v;
    }
    out[((size_t)b * 2 + 0) * T + t] = expf(v0);
    out[((size_t)b * 2 + 1) * T + t] = expf(v1);
}

// ------------------------------------------------------------------------------------------
// greedy CTC collapse state machine (transcript_generators.py:32-83) as a segmented WARP scan, one utterance per warp.
//
// The serial machine carries (last token, allow_repeat, count_eps), but every decision is local: after ANY non-blank
// frame `last` equals that frame's id (it was either emitted or dropped because it equalled `last`) and allow_repeat is
// false, and a blank is either ignored (last == space) or counted.  So for a non-blank frame t with previous non-blank
// frame pt (id xp) and e = t - pt - 1 blanks in between:
//   emitted  <=>  first token, or  xp == space ? x != space : (e >= 1 || x != xp)
// and a blank frame t synthesises a space  <=>  t - pt == blank_to_space, xp != space and xp is not a word start.
// Each frame yields at most one output, in frame order: a ballot + popcount prefix gives the output slot.  32 frames per
// step, coalesced 128-byte reads; the carry between steps is (pt, xp).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
greedy_collapse_kernel(const int* __restrict__ ids, const int* __restrict__ lengths, int B,
                       int T, int C, int eps_id, int space_id,
                       const uint8_t* __restrict__ is_silence,
                       const uint8_t* __restrict__ is_word_start, int blank_to_space,
                       int* __restrict__ out_tok, int* __restrict__ out_frm, int T_cap,
                       int* __restrict__ out_cnt) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const int* row = ids + (size_t)b * T;
    int* tok = out_tok + (size_t)b * T_cap;
    int* frm = out_frm + (size_t)b * T_cap;
    int len = lengths ? lengths[b] : T;
    len = len < T ? len : T;
    // leading silence is skipped over the FULL row, not just `len` (transcript_generators.py:38-40)
    int t_start = T;
    for (int t0 = 0; t0 < T; t0 += 32) {
        const int t = t0 + lane;
        bool nonsil = false;
        if (t < T) {
            const int x = row[t];
            nonsil = !((x >= 0 && x < C) ? is_silence[x] != 0 : false);
        }
        const unsigned m = __ballot_sync(0xffffffffu, nonsil);
        if (m) { t_start = t0 + __ffs(m) - 1; break; }
    }
    if (t_start >= T) { if (lane == 0) out_cnt[b] = -1; return; }
    int n = 0;
    int pt = t_start - 1, xp = eps_id;  // previous non-blank frame and its id; the machine starts with tokens = [eps] (transcript_generators.py:42)
    for (int t0 = t_start & ~31; t0 < len; t0 += 32) {
        const int t = t0 + lane;
        const bool in = t >= t_start && t < len;
        const int x = in ? row[t] : eps_id;
        const bool is_tok = in && x != eps_id;
        const unsigned tokmask = __ballot_sync(0xffffffffu, is_tok);
        // previous non-blank frame of this lane: inside the step, else the carry
        const unsigned below = tokmask & ((1u << lane) - 1u);
        const int src = below ? 31 - __clz(below) : 0;
        const int x_in = __shfl_sync(0xffffffffu, x, src);
        const int my_pt = below ? t0 + src : pt;
        const int my_xp = below ? x_in : xp;
        bool out = false;
        int o_tok = x, o_frm = t;
        if (is_tok) {
            const int e = t - my_pt - 1;
            out = my_xp == space_id ? x != space_id : (e >= 1 || x != my_xp);
        } else if (in && t - my_pt == blank_to_space && my_xp != space_id) {
            const bool ws = (my_xp >= 0 && my_xp < C) ? is_word_start[my_xp] != 0 : false;
            if (!ws) { out = true; o_tok = space_id; o_frm = -(t + 1); }
        }
        const unsigned outmask = __ballot_sync(0xffffffffu, out);
        if (out) {
            const int pos = n + __popc(outmask & ((1u << lane) - 1u));
            if (pos < T_cap) { tok[pos] = o_tok; frm[pos] = o_frm; }
        }
        n += __popc(outmask);
        if (tokmask) {
            const int last = 31 - __clz(tokmask);
            pt = t0 + last;
            xp = __shfl_sync(0xffffffffu, x, last);
        }
    }
    if (lane == 0) out_cnt[b] = n < T_cap ? n : T_cap;
}

// ------------------------------------------------------------------------------------------
// entropy / weighted_mean_entropy (models.py:645-673), block per utterance
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
entropy_kernel(const float* __restrict__ lp, const int64_t* __restrict__ lengths, int B, int C, int T,
               int eps_id, float* __restrict__ out_e, float* __restrict__ out_w) {
    const int b = blockIdx.x;
    const float* xb = lp + (size_t)b * C * T;
    const int len = lengths ? (int)lengths[b] : T;
    const int eid = eps_id < 0 ? C + eps_id : eps_id;
    float se = 0.f, sew = 0.f, sw = 0.f;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        float e = 0.f;
        for (int c = 0; c < C; ++c) {
            const float l = xb[(size_t)c * T + t];
            e -= expf(l) * l;
        }
        float w = 1.f - expf(xb[(size_t)eid * T + t]);
        const bool in = t < len;
        if (lengths != nullptr) { if (!in) w = 0.f; }
        if (lengths == nullptr || in) se += e;
        sew += e * w;
        sw += w;
    }
    __shared__ float red[3][8];
    se = warp_sum(se); sew = warp_sum(sew); sw = warp_sum(sw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[0][warp] = se; red[1][warp] = sew; red[2][warp] = sw; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, bq = 0.f, c = 0.f;
        for (int i = 0; i < 8; ++i) { a += red[0][i]; bq += red[1][i]; c += red[2][i]; }
        if (out_e) out_e[b] = lengths ? a / (1e-9f + (float)len) : a / (float)T;
        if (out_w) out_w[b] = bq / (1e-9f + c);
    }
}

static int ctc_threads(int S_max) {
    // measured on B200 (S = 339, t = 753): 128 threads 609 us, 192: 422, 256: 375, 384: 267 --
    // the per-state lse chain is latency bound, so one state per thread wins while it fits
    int th = (S_max + 31) / 32 * 32;
    if (th > 1024) th = ((S_max + kCtcMaxPer - 1) / kCtcMaxPer + 31) / 32 * 32;
    if (th < 32) th = 32;
    return th;
}

// shared memory of ctc_recursion_kernel for a staging depth of G steps
constexpr size_t kCtcRecSmemBudget = 200 * 1024;
static size_t ctc_rec_bytes(int S_max, int G) {
    const int S_pad = S_max | 1;
    return sizeof(float) * (2 * (size_t)(S_max + 2) + 32 + (size_t)S_max + 2 * (size_t)G * S_pad);
}
// does ctc_recursion_kernel take targets of L_max labels (at least kCtcPrefetch staged frames in shared memory)?
static bool ctc_one_cta_covers(int L_max) {
    const int S_max = 2 * L_max + 1;
    return L_max >= 0 && S_max <= kCtcMaxPer * 1024 && ctc_rec_bytes(S_max, kCtcPrefetch) <= kCtcRecSmemBudget;
}

// picks the deepest staging that fits
static int ctc_rec_config(int S_max, int* G_out, size_t* smem_out) {
    for (int G = 32; G >= kCtcPrefetch; G >>= 1) {
        const size_t bytes = ctc_rec_bytes(S_max, G);
        if (bytes <= kCtcRecSmemBudget) {
            *G_out = G;
            *smem_out = bytes;
            static size_t attr_set = 0;
            if (bytes > attr_set) {
                if (cudaFuncSetAttribute(ctc_recursion_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return -1;
                if (cudaFuncSetAttribute(ctc_recursion_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return -1;
                if (cudaFuncSetAttribute(ctc_recursion_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return -1;
                attr_set = bytes;
            }
            return 0;
        }
    }
    return -1;
}

}  // namespace cab

using namespace cab;


#define CAB_LAUNCH_CTC_REC(grid, first_role, A, Bw, NLL)                                                        \
    do {                                                                                                        \
        const int per_ = (S_max + threads - 1) / threads;                                                       \
        if (per_ <= 1)                                                                                          \
            ctc_recursion_kernel<1><<<grid, threads, rec_smem, stream>>>(log_probs, stride_t, stride_b, stride_c, targets, input_lengths, target_lengths, B, T, L_max, blank, first_role, G, A, Bw, ws_offsets, G_cap, NLL); \
        else if (per_ <= 2)                                                                                     \
            ctc_recursion_kernel<2><<<grid, threads, rec_smem, stream>>>(log_probs, stride_t, stride_b, stride_c, targets, input_lengths, target_lengths, B, T, L_max, blank, first_role, G, A, Bw, ws_offsets, G_cap, NLL); \
        else                                                                                                    \
            ctc_recursion_kernel<4><<<grid, threads, rec_smem, stream>>>(log_probs, stride_t, stride_b, stride_c, targets, input_lengths, target_lengths, B, T, L_max, blank, first_role, G, A, Bw, ws_offsets, G_cap, NLL); \
    } while (0)

#define CTC_COMMON_CHECKS()                                                                       \
    CAB_CHECK_ARG(log_probs && targets && input_lengths && target_lengths, "null pointer argument"); \
    CAB_CHECK_ARG(B > 0 && T > 0 && C > 0 && L_max >= 0, "bad shape B=%d T=%d C=%d L=%d", B, T, C, L_max); \
    CAB_CHECK_ARG(blank >= 0 && blank < C, "blank=%d out of range", blank);                       \
    const int S_max = 2 * L_max + 1;                                                              \
    CAB_CHECK_ARG(S_max <= kCtcMaxPer * 1024, "target too long: L_max=%d", L_max);                \
    const int threads = ctc_threads(S_max);                                                       \
    const int G_cap = (T + kCtcPrefetch - 1) / kCtcPrefetch + 2;                                  \
    (void)G_cap;                                                                                  \
    const size_t smem = sizeof(float) * (2 * (S_max + 2) + 32);                                   \
    (void)smem;

extern "C" int cab_ctc_loss_fwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                const int64_t* targets, const int64_t* input_lengths,
                                const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                                float* ws_alpha, float* ws_beta, double* ws_offsets, float* nll,
                                cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTC_COMMON_CHECKS();
    CAB_CHECK_ARG(ws_alpha && ws_offsets && nll, "null workspace/output");
    // ws_beta given: run the beta recursion in the same grid (both are needed for the gradient)
    const int roles = ws_beta ? 2 : 1;
    int G = 0;
    size_t rec_smem = 0;
    CAB_CHECK_ARG(ctc_rec_config(S_max, &G, &rec_smem) == 0, "target too long for the staged recursion: L_max=%d", L_max);
    CAB_LAUNCH_CTC_REC(B * roles, 0, ws_alpha, ws_beta, nll);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_ctc_loss_bwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                const int64_t* targets, const int64_t* input_lengths,
                                const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                                const float* ws_alpha, float* ws_beta, int beta_ready, double* ws_offsets,
                                const float* grad_out, float* grad, int64_t gstride_t, int64_t gstride_b,
                                int64_t gstride_c, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTC_COMMON_CHECKS();
    CAB_CHECK_ARG(ws_alpha && ws_beta && ws_offsets && grad_out && grad, "null workspace/output");
    int n_launch = 2;
    if (!beta_ready) {
        int G = 0;
        size_t rec_smem = 0;
        CAB_CHECK_ARG(ctc_rec_config(S_max, &G, &rec_smem) == 0, "target too long for the staged recursion: L_max=%d", L_max);
        CAB_LAUNCH_CTC_REC(B, 1, (float*)nullptr, ws_beta, (float*)nullptr);
        CAB_CHECK_LAUNCH();
        ++n_launch;
    }
    {
        const int64_t n = (int64_t)B * T * C;
        int blocks = (int)((n + 255) / 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        ctc_grad_init_kernel<<<blocks, 256, 0, stream>>>(log_probs, stride_t, stride_b, stride_c, input_lengths,
                                                         grad_out, B, T, C, grad, gstride_t, gstride_b, gstride_c);
        CAB_CHECK_LAUNCH();
    }
    {
        dim3 grid((T + 7) / 8, B);
        ctc_grad_scatter_kernel<<<grid, 256, 0, stream>>>(log_probs, stride_t, stride_b, stride_c, targets,
                                                          input_lengths, target_lengths, T, L_max, blank, ws_alpha,
                                                          ws_beta, ws_offsets, G_cap, grad_out, grad, gstride_t,
                                                          gstride_b, gstride_c);
        CAB_CHECK_LAUNCH();
    }
    g_launch_count.fetch_add(n_launch, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_ctc_alignment(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                 const int64_t* targets, const int64_t* input_lengths,
                                 const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                                 uint8_t* ws_backptr, int64_t* out_alignment, int fp16_arithmetic, const uint16_t* fp16_exp_table,
                                 const uint16_t* fp16_log_table, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTC_COMMON_CHECKS();
    CAB_CHECK_ARG(ws_backptr && out_alignment, "null workspace/output");
    CAB_CHECK_ARG((fp16_exp_table == nullptr) == (fp16_log_table == nullptr), "give both fp16 tables or neither");
    if (fp16_arithmetic)
        ctc_align_kernel<true><<<B, threads, smem, stream>>>(log_probs, stride_t, stride_b, stride_c, targets, input_lengths, target_lengths, T, L_max, blank,
                                                             ws_backptr, out_alignment, fp16_exp_table, fp16_log_table);
    else
        ctc_align_kernel<false><<<B, threads, smem, stream>>>(log_probs, stride_t, stride_b, stride_c, targets, input_lengths, target_lengths, T, L_max, blank,
                                                              ws_backptr, out_alignment, nullptr, nullptr);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_ctc_alignment_long_workspace(int B, int T, int L_max, int64_t* bytes) {
    CAB_CHECK_ARG(bytes != nullptr, "null output");
    CAB_CHECK_ARG(B > 0 && T > 0 && L_max >= 0, "bad shape B=%d T=%d L=%d", B, T, L_max);
    CAB_CHECK_ARG(L_max <= kAlignLongMaxL, "target too long: L_max=%d (the cluster alignment handles L_max <= %d)", L_max, kAlignLongMaxL);
    *bytes = (int64_t)B * T * ((2 * (int64_t)L_max + 1 + 3) / 4);
    return 0;
}

// How the cluster kernels split S_max extended states: n CTAs, slices of W states (W % 4 == 0), n_slots slices per CTA.
// states_per_cta > 0 forces W, with slices round-robin over up to kAlignClusterMax CTAs; 0 gives one slice per CTA of
// at most ~2048 states.
static int ctc_cluster_geometry(int S_max, int states_per_cta, int* n_out, int* W_out, int* n_slots_out, int* threads_out) {
    int n, W, n_slots;
    if (states_per_cta > 0) {
        W = states_per_cta;
        const int n_slices = (S_max + W - 1) / W;
        n = n_slices < kAlignClusterMax ? n_slices : kAlignClusterMax;
        n_slots = (n_slices + n - 1) / n;
    } else {
        n = (S_max + 2047) / 2048;
        if (n > kAlignClusterMax) n = kAlignClusterMax;
        W = 4 * (((S_max + 3) / 4 + n - 1) / n);
        n_slots = 1;
    }
    CAB_CHECK_ARG((int64_t)n_slots * W <= kAlignCtaStates, "states_per_cta=%d puts %lld states on one CTA (at most %d)", states_per_cta,
                  (long long)n_slots * W, kAlignCtaStates);
    const int groups = n_slots * W / 4;
    const int per = groups > 1024 ? kAlignGroupsPer : 1;
    *n_out = n;
    *W_out = W;
    *n_slots_out = n_slots;
    *threads_out = ((groups + per - 1) / per + 31) / 32 * 32;
    return 0;
}

template <bool HALF>
static int launch_align_cluster(int n, int threads, size_t smem, cudaStream_t stream, int B, const float* log_probs, int64_t st,
                                int64_t sb, int64_t sc, const int64_t* targets, const int64_t* input_lengths,
                                const int64_t* target_lengths, int T, int L_max, int blank, int W, int n_slots, int64_t pitch,
                                uint8_t* ws, int64_t* out, const uint16_t* tab_exp, const uint16_t* tab_log) {
    auto kernel = ctc_align_cluster_kernel<HALF>;
    static size_t smem_set = 0;
    if (smem_set == 0) CAB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = n;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(B * n);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int clusters = 0;
    CAB_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg));
    CAB_CHECK_ARG(clusters > 0, "a cluster of %d CTAs x %d threads with %zu B of shared memory does not fit this device", n, threads, smem);
    CAB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, log_probs, st, sb, sc, targets, input_lengths, target_lengths, T, L_max, blank, W,
                                      n_slots, pitch, ws, out, tab_exp, tab_log));
    return 0;
}

extern "C" int cab_ctc_alignment_long(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                      const int64_t* targets, const int64_t* input_lengths, const int64_t* target_lengths, int B,
                                      int T, int C, int L_max, int blank, uint8_t* ws_backptr, int64_t* out_alignment,
                                      int fp16_arithmetic, const uint16_t* fp16_exp_table, const uint16_t* fp16_log_table,
                                      int states_per_cta, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(log_probs && targets && input_lengths && target_lengths, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && T > 0 && C > 0 && L_max >= 0, "bad shape B=%d T=%d C=%d L=%d", B, T, C, L_max);
    CAB_CHECK_ARG(blank >= 0 && blank < C, "blank=%d out of range", blank);
    CAB_CHECK_ARG(L_max <= kAlignLongMaxL, "target too long: L_max=%d (the cluster alignment handles L_max <= %d)", L_max, kAlignLongMaxL);
    CAB_CHECK_ARG(ws_backptr && out_alignment, "null workspace/output");
    CAB_CHECK_ARG((fp16_exp_table == nullptr) == (fp16_log_table == nullptr), "give both fp16 tables or neither");
    CAB_CHECK_ARG(states_per_cta >= 0 && states_per_cta % 4 == 0, "states_per_cta=%d must be 0 or a positive multiple of 4", states_per_cta);
    if (L_max == 0) return 0;  // out has no element
    const int S_max = 2 * L_max + 1;
    const int G4 = (S_max + 3) / 4;  // bytes per packed row
    int n, W, n_slots, threads;
    if (ctc_cluster_geometry(S_max, states_per_cta, &n, &W, &n_slots, &threads) != 0) return -1;
    const size_t smem = sizeof(float) * (2 * (size_t)n_slots * (W + 2) + 2);
    int rc = fp16_arithmetic
                 ? launch_align_cluster<true>(n, threads, smem, stream, B, log_probs, stride_t, stride_b, stride_c, targets, input_lengths,
                                              target_lengths, T, L_max, blank, W, n_slots, G4, ws_backptr, out_alignment, fp16_exp_table,
                                              fp16_log_table)
                 : launch_align_cluster<false>(n, threads, smem, stream, B, log_probs, stride_t, stride_b, stride_c, targets, input_lengths,
                                               target_lengths, T, L_max, blank, W, n_slots, G4, ws_backptr, out_alignment, nullptr, nullptr);
    if (rc != 0) return rc;
    ctc_align_backtrace_kernel<<<B, 32, 0, stream>>>(ws_backptr, G4, input_lengths, T, L_max, out_alignment);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(2, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_ctc_loss_one_cta_covers(int L_max) { return ctc_one_cta_covers(L_max) ? 1 : 0; }

extern "C" int cab_ctc_loss_long_workspace(int B, int T, int L_max, int64_t* bytes) {
    CAB_CHECK_ARG(bytes != nullptr, "null output");
    CAB_CHECK_ARG(B > 0 && T > 0 && L_max >= 0, "bad shape B=%d T=%d L=%d", B, T, L_max);
    CAB_CHECK_ARG(L_max <= kAlignLongMaxL, "target too long: L_max=%d (the cluster CTC loss handles L_max <= %d)", L_max, kAlignLongMaxL);
    *bytes = (int64_t)sizeof(float) * B * T * (2 * (int64_t)L_max + 1);
    return 0;
}

// one launch of ctc_loss_cluster_kernel<MODE>, B clusters of n CTAs
template <int MODE>
static int launch_loss_cluster(int states_per_cta, cudaStream_t stream, const float* log_probs, int64_t st, int64_t sb, int64_t sc,
                               const int64_t* targets, const int64_t* input_lengths, const int64_t* target_lengths, int B, int T,
                               int L_max, int blank, float* ws, double* ws_offsets, float* nll, const float* grad_out, float* grad,
                               int64_t gt, int64_t gb, int64_t gc) {
    int n, W, n_slots, threads;
    if (ctc_cluster_geometry(2 * L_max + 1, states_per_cta, &n, &W, &n_slots, &threads) != 0) return -1;
    // two frame buffers of n_slots * (W + 2) values, block maxima [2][16], warp maxima [32], two scalars
    const size_t smem = sizeof(float) * (2 * (size_t)n_slots * (W + 2) + 2 * kAlignClusterMax + 32 + 2);
    auto kernel = ctc_loss_cluster_kernel<MODE>;
    static size_t smem_set = 0;
    if (smem_set == 0) CAB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = n;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(B * n);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int clusters = 0;
    CAB_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg));
    CAB_CHECK_ARG(clusters > 0, "a cluster of %d CTAs x %d threads with %zu B of shared memory does not fit this device", n, threads, smem);
    const int G_cap = (T + kCtcPrefetch - 1) / kCtcPrefetch + 2;
    CAB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, log_probs, st, sb, sc, targets, input_lengths, target_lengths, T, L_max, blank, W,
                                      n_slots, ws, ws_offsets, G_cap, nll, grad_out, grad, gt, gb, gc));
    return 0;
}

#define CTC_LONG_CHECKS()                                                                                                  \
    CAB_CHECK_ARG(log_probs && targets && input_lengths && target_lengths, "null pointer argument");                      \
    CAB_CHECK_ARG(B > 0 && T > 0 && C > 0 && L_max >= 0, "bad shape B=%d T=%d C=%d L=%d", B, T, C, L_max);                \
    CAB_CHECK_ARG(blank >= 0 && blank < C, "blank=%d out of range", blank);                                                \
    CAB_CHECK_ARG(L_max <= kAlignLongMaxL, "target too long: L_max=%d (the cluster CTC loss handles L_max <= %d)", L_max, \
                  kAlignLongMaxL);                                                                                         \
    CAB_CHECK_ARG(states_per_cta >= 0 && states_per_cta % 4 == 0, "states_per_cta=%d must be 0 or a positive multiple of 4", \
                  states_per_cta);

extern "C" int cab_ctc_loss_long_fwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                     const int64_t* targets, const int64_t* input_lengths, const int64_t* target_lengths, int B,
                                     int T, int C, int L_max, int blank, float* ws_alpha, double* ws_offsets, float* nll,
                                     int states_per_cta, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTC_LONG_CHECKS();
    CAB_CHECK_ARG(ws_offsets && nll, "null workspace/output");
    const int rc = ws_alpha ? launch_loss_cluster<1>(states_per_cta, stream, log_probs, stride_t, stride_b, stride_c, targets, input_lengths,
                                                     target_lengths, B, T, L_max, blank, ws_alpha, ws_offsets, nll, nullptr, nullptr, 0, 0, 0)
                            : launch_loss_cluster<0>(states_per_cta, stream, log_probs, stride_t, stride_b, stride_c, targets, input_lengths,
                                                     target_lengths, B, T, L_max, blank, nullptr, ws_offsets, nll, nullptr, nullptr, 0, 0, 0);
    if (rc != 0) return rc;
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_ctc_loss_long_bwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                                     const int64_t* targets, const int64_t* input_lengths, const int64_t* target_lengths, int B,
                                     int T, int C, int L_max, int blank, const float* ws_alpha, double* ws_offsets,
                                     const float* grad_out, float* grad, int64_t gstride_t, int64_t gstride_b, int64_t gstride_c,
                                     int states_per_cta, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTC_LONG_CHECKS();
    CAB_CHECK_ARG(ws_alpha && ws_offsets && grad_out && grad, "null workspace/output");
    int n_, W_, n_slots_, threads_;  // a refused split launches nothing
    if (ctc_cluster_geometry(2 * L_max + 1, states_per_cta, &n_, &W_, &n_slots_, &threads_) != 0) return -1;
    {
        const int64_t n = (int64_t)B * T * C;
        int blocks = (int)((n + 255) / 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        ctc_grad_init_kernel<<<blocks, 256, 0, stream>>>(log_probs, stride_t, stride_b, stride_c, input_lengths, grad_out, B, T, C, grad,
                                                         gstride_t, gstride_b, gstride_c);
        CAB_CHECK_LAUNCH();
    }
    const int rc = launch_loss_cluster<2>(states_per_cta, stream, log_probs, stride_t, stride_b, stride_c, targets, input_lengths,
                                          target_lengths, B, T, L_max, blank, const_cast<float*>(ws_alpha), ws_offsets, nullptr, grad_out,
                                          grad, gstride_t, gstride_b, gstride_c);
    if (rc != 0) return rc;
    g_launch_count.fetch_add(2, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_log_softmax_argmax(const void* logits, int in_dtype, int B, int C, int T,
                                      float* out_log_probs, int32_t* out_argmax, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(logits != nullptr, "null logits");
    CAB_CHECK_ARG(in_dtype == 0, "only fp32 logits are supported (in_dtype=%d)", in_dtype);
    CAB_CHECK_ARG(B > 0 && C > 0 && T > 0, "bad shape");
    dim3 grid((T + 31) / 32, B);
    log_softmax_argmax_kernel<<<grid, 256, 0, stream>>>(static_cast<const float*>(logits), B, C, T,
                                                        out_log_probs, out_argmax);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_log_softmax_bwd(const float* log_probs, const float* grad_out, int B, int C, int T,
                                   float* grad_in, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(log_probs && grad_out && grad_in, "null pointer argument");
    dim3 grid((T + 31) / 32, B);
    log_softmax_bwd_kernel<<<grid, 256, 0, stream>>>(log_probs, grad_out, B, C, T, grad_in);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_topk_ids(const float* log_probs, int B, int C, int T, int K, int32_t* out_ids,
                            cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(log_probs && out_ids, "null pointer argument");
    CAB_CHECK_ARG(K >= 1 && K <= kTopKMax && K <= C, "K=%d out of [1,%d] (C=%d)", K, kTopKMax, C);
    dim3 grid((T + 127) / 128, B);
    topk_ids_kernel<<<grid, 128, 0, stream>>>(log_probs, B, C, T, K, out_ids);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_top2_probs(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t, int B, int C, int T,
                              float* out, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(log_probs && out && B > 0 && C >= 2 && T > 0, "bad arguments");
    dim3 grid((T + 127) / 128, B);
    top2_probs_kernel<<<grid, 128, 0, stream>>>(log_probs, stride_b, stride_c, stride_t, B, C, T, out);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_greedy_collapse(const int32_t* ids, const int32_t* lengths, int B, int T, int C, int eps_id,
                                   int space_id, const uint8_t* is_silence, const uint8_t* is_word_start,
                                   int blank_amount_to_space, int32_t* out_tokens, int32_t* out_frames, int T_cap,
                                   int32_t* out_counts, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(ids && is_silence && is_word_start && out_tokens && out_frames && out_counts, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && T > 0 && T_cap > 0, "bad shape");
    greedy_collapse_kernel<<<(B + 7) / 8, 256, 0, stream>>>(ids, lengths, B, T, C, eps_id, space_id, is_silence,
                                                             is_word_start, blank_amount_to_space, out_tokens,
                                                             out_frames, T_cap, out_counts);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_log_softmax_rows(const float* logits, const float* lse, int64_t R, int C, int ld, float* out_log_probs,
                                    cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(logits && lse && out_log_probs && R > 0 && C > 0, "bad arguments");
    CAB_CHECK_ARG(ld >= C && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 && (reinterpret_cast<uintptr_t>(out_log_probs) & 15) == 0, "rows must be 16-byte aligned (ld=%d)", ld);
    const long long blocks = R < 148LL * 16 ? R : 148LL * 16;
    log_softmax_rows_kernel<<<(int)blocks, 256, 0, stream>>>(logits, lse, (long long)R, C, ld, out_log_probs);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_entropy(const float* log_probs, const int64_t* lengths, int B, int C, int T, int eps_id,
                           float* out_entropy, float* out_weighted_entropy, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(log_probs != nullptr, "null log_probs");
    entropy_kernel<<<B, 256, 0, stream>>>(log_probs, lengths, B, C, T, eps_id, out_entropy, out_weighted_entropy);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}
