// Training-mode elementwise / reduction kernels around the conv GEMMs: BatchNorm batch statistics,
// BN-apply + activation + temporal mask (forward and backward), weight (un)packing, layout casts.
//
// Reference semantics (file:line): nn.BatchNorm1d(momentum=0.1, eps=1e-5) in training mode inside
// ConvBn1d.forward models.py:127-139 -- biased batch variance over ALL B*t positions (padded frames
// included, the mask is applied after the activation), running_var updated with the unbiased one;
// ResidualActivation.forward :357-371 (hardtanh passes gradient only for a < z < b; relu for z > 0;
// leaky_relu slope for z <= 0); temporal mask multiply :136-138 is part of the autograd graph.
// All of these are HBM bound: bf16 activations, 16-byte vector accesses, fp32 math.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

__device__ __forceinline__ float act_fwd(float z, int act, float a, float b) {
    switch (act) {
        case CAB_ACT_RELU: return fmaxf(z, 0.f);
        case CAB_ACT_HARDTANH: return fminf(fmaxf(z, a), b);
        case CAB_ACT_LEAKY_RELU: return z > 0.f ? z : z * a;
        default: return z;
    }
}
__device__ __forceinline__ float act_grad(float z, int act, float a, float b) {
    switch (act) {
        case CAB_ACT_RELU: return z > 0.f ? 1.f : 0.f;
        case CAB_ACT_HARDTANH: return (z > a && z < b) ? 1.f : 0.f;
        case CAB_ACT_LEAKY_RELU: return z > 0.f ? 1.f : a;
        default: return 1.f;
    }
}

// compile-time activation (the streamed kernels are instantiated per activation: a run-time switch per element cost ~28
// instructions of uniform branches per value and made the kernels issue bound at 50 % of the slots, ncu round 1)
template <int ACT>
__device__ __forceinline__ float act_fwd_t(float z, float a, float b) {
    if (ACT == CAB_ACT_RELU) return fmaxf(z, 0.f);
    if (ACT == CAB_ACT_HARDTANH) return fminf(fmaxf(z, a), b);
    if (ACT == CAB_ACT_LEAKY_RELU) return z > 0.f ? z : z * a;
    return z;
}
// g * act'(z): a select for the 0 / 1 gates
template <int ACT>
__device__ __forceinline__ float act_gate_t(float g, float z, float a, float b) {
    if (ACT == CAB_ACT_RELU) return z > 0.f ? g : 0.f;
    if (ACT == CAB_ACT_HARDTANH) return (z > a && z < b) ? g : 0.f;
    if (ACT == CAB_ACT_LEAKY_RELU) return z > 0.f ? g : g * a;
    return g;
}

// Dropout keep-decision: counter-based, recomputed identically in the backward pass (no mask is
// stored).  seed comes from DEVICE memory so that CUDA-graph replays draw fresh masks; the stream
// is this repo's own (F.dropout's Philox stream is not reproducible across implementations anyway,
// SURVEY.md 8a: parity runs use dropout = 0).
__device__ __forceinline__ bool dropout_keep(unsigned long long seed, unsigned long long idx, float p) {
    unsigned long long z = seed + idx * 0x9E3779B97F4A7C15ULL;  // splitmix64 finaliser
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return (float)(unsigned)(z >> 40) * (1.0f / 16777216.0f) >= p;  // 24 uniform bits
}

// ---------------------------------------------------------------------------------------
// Row-walker layout shared by the four activation-sized kernels: a thread owns ONE 16-byte channel
// vector (8 bf16 channels) and walks down the rows, so the per-channel coefficients live in
// registers and a warp touches 512 contiguous bytes per row.
//   block (32, 8): x = channel vector, y = row lane;  grid (ceil(ld/8/32), ceil(R/rows_per_block))
// rows_per_block is picked on the host so that every layer width fills the machine: narrow layers
// (256 channels = one block column) would otherwise launch fewer blocks than there are SMs x 2.
// ---------------------------------------------------------------------------------------
constexpr int kRowLanes = 8;
constexpr int kWalkerBlocksTarget = 148 * 8;

static inline int rows_per_block_for(int R, int ld) {
    const long long cols = (ld / 8 + 31) / 32;
    long long rpb = ((long long)R * cols + kWalkerBlocksTarget - 1) / kWalkerBlocksTarget;
    rpb = (rpb + 31) / 32 * 32;
    return (int)(rpb < 32 ? 32 : (rpb > 512 ? 512 : rpb));
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
        f[2 * j] = t.x;
        f[2 * j + 1] = t.y;
    }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

// reduce 2 x 8 per-thread partials over the row lanes, then one atomic per channel and statistic
// (mean, invstd given: the second statistic is centred first, q <- invstd * (q - mean * s))
template <typename OutT>
__device__ __forceinline__ void reduce_rows_and_add(float (&s)[8], float (&q)[8], int c0, int C, OutT* __restrict__ out,
                                                    const float* __restrict__ mean = nullptr, const float* __restrict__ invstd = nullptr) {
    __shared__ float sm[kRowLanes][32][17];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        sm[threadIdx.y][threadIdx.x][e] = s[e];
        sm[threadIdx.y][threadIdx.x][8 + e] = q[e];
    }
    __syncthreads();
    if (threadIdx.y == 0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float a = s[e], b = q[e];
            for (int y = 1; y < kRowLanes; ++y) {
                a += sm[y][threadIdx.x][e];
                b += sm[y][threadIdx.x][8 + e];
            }
            if (c0 + e < C) {
                if (mean != nullptr) b = invstd[c0 + e] * (b - mean[c0 + e] * a);
                atomicAdd(out + c0 + e, (OutT)a);
                atomicAdd(out + C + c0 + e, (OutT)b);
            }
        }
    }
}

// per-channel sum / sum of squares of a bf16 [R, ld] matrix (R = B*t rows)
__global__ void __launch_bounds__(256)
colstats_kernel(const __nv_bfloat16* __restrict__ x, int R, int C, int ld, double* __restrict__ out, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    float s[8], q[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; }
    if (c0 < ld) {
        const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
        // 4 independent 16-byte loads in flight per thread (the loop is latency bound otherwise)
        for (int r = r0 + threadIdx.y; r < r1; r += 4 * kRowLanes) {
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int rr = r + u * kRowLanes;
                v[u] = rr < r1 ? *reinterpret_cast<const uint4*>(x + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float f[8];
                unpack8(v[u], f);
#pragma unroll
                for (int e = 0; e < 8; ++e) { s[e] += f[e]; q[e] = fmaf(f[e], f[e], q[e]); }
            }
        }
    }
    reduce_rows_and_add(s, q, c0, C, out);
}

// mean / invstd / fused scale+shift, running statistics update (momentum, unbiased running_var)
__global__ void bn_finalize_kernel(const double* __restrict__ stats, int C, float n, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ out /* [4][C]: scale, shift, mean, invstd */, int sums_ld) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    // fp64 sums: E[x^2] - mean^2 without cancellation noise
    const double inv_nd = 1.0 / (double)n;
    const double mean_d = stats[c] * inv_nd;
    const float mean = (float)mean_d;
    const float var = (float)fmax(stats[sums_ld + c] * inv_nd - mean_d * mean_d, 0.0);
    const float invstd = rsqrtf(var + eps);
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    out[c] = g * invstd;
    out[C + c] = b - mean * g * invstd;
    out[2 * C + c] = mean;
    out[3 * C + c] = invstd;
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
    if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * (n / fmaxf(n - 1.f, 1.f));
}

// out = act(y * scale + shift) * (t < len_b)
__global__ void __launch_bounds__(256)
bn_act_mask_fwd_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ ss, int B, int T, int C, int ld,
                       int act, float a, float bb, const float* __restrict__ xlen, __nv_bfloat16* __restrict__ out,
                       float drop_p, const long long* __restrict__ seed_ptr, unsigned long long salt, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    if (c0 >= ld) return;
    float sc[8], sh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const bool ok = c0 + e < C;
        sc[e] = ok ? ss[c0 + e] : 0.f;
        sh[e] = ok ? ss[C + c0 + e] : 0.f;
    }
    const int R = B * T;
    const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
    for (int r = r0 + threadIdx.y; r < r1; r += 4 * kRowLanes) {
        uint4 v[4];
        bool keep[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int rr = r + u * kRowLanes;
            const int b = rr / T, t = rr - b * T;
            keep[u] = rr < r1 && (xlen == nullptr || t < frac_len(__ldg(xlen + b), T));
            v[u] = keep[u] ? *reinterpret_cast<const uint4*>(y + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int rr = r + u * kRowLanes;
            if (rr >= r1) break;
            float f[8];
            unpack8(v[u], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = (keep[u] && c0 + e < C) ? act_fwd(fmaf(f[e], sc[e], sh[e]), act, a, bb) : 0.f;
            if (drop_p > 0.f) {
                const unsigned long long seed = (unsigned long long)seed_ptr[0] + salt * 0xD1B54A32D192ED03ULL;
                const float inv_keep = 1.f / (1.f - drop_p);
#pragma unroll
                for (int e = 0; e < 8; ++e) f[e] = dropout_keep(seed, (unsigned long long)rr * ld + c0 + e, drop_p) ? f[e] * inv_keep : 0.f;
            }
            *reinterpret_cast<uint4*>(out + (size_t)rr * ld + c0) = pack8(f);
        }
    }
}

// backward pass 1: per-channel sum(dz), sum(dz * xhat), dz = g * act'(z) * mask.  The loop accumulates
// sum(dz * y); xhat = (y - mean) * invstd is linear in y, so the block's partial is corrected once
// at the end (sum(dz * xhat) = invstd * (sum(dz * y) - mean * sum(dz))) -- 16 fewer live registers.
__global__ void __launch_bounds__(256)
bn_act_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ g,
                         const float* __restrict__ ss, int B, int T, int C, int ld, int act, float a, float bb,
                         const float* __restrict__ xlen, float* __restrict__ out, float drop_p,
                         const long long* __restrict__ seed_ptr, unsigned long long salt, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    float s[8], q[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; }
    if (c0 < ld) {
        float sc[8], sh[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const bool ok = c0 + e < C;
            sc[e] = ok ? ss[c0 + e] : 0.f;
            sh[e] = ok ? ss[C + c0 + e] : 0.f;
        }
        const int R = B * T;
        const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
        constexpr int U = 4;  // 8 independent 16-byte loads in flight per thread
        for (int r = r0 + threadIdx.y; r < r1; r += U * kRowLanes) {
            uint4 yv[U], gv[U];
            bool on[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int rr = r + u * kRowLanes;
                const int b = rr / T, t = rr - b * T;
                on[u] = rr < r1 && (xlen == nullptr || t < frac_len(__ldg(xlen + b), T));
                yv[u] = on[u] ? *reinterpret_cast<const uint4*>(y + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
                gv[u] = on[u] ? *reinterpret_cast<const uint4*>(g + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!on[u]) continue;
                float yf[8], gf[8];
                unpack8(yv[u], yf);
                unpack8(gv[u], gf);
                if (drop_p > 0.f) {
                    const unsigned long long seed = (unsigned long long)seed_ptr[0] + salt * 0xD1B54A32D192ED03ULL;
                    const float inv_keep = 1.f / (1.f - drop_p);
                    const int rr = r + u * kRowLanes;
#pragma unroll
                    for (int e = 0; e < 8; ++e) gf[e] = dropout_keep(seed, (unsigned long long)rr * ld + c0 + e, drop_p) ? gf[e] * inv_keep : 0.f;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float dz = gf[e] * act_grad(fmaf(yf[e], sc[e], sh[e]), act, a, bb);
                    s[e] += dz;
                    q[e] = fmaf(dz, yf[e], q[e]);
                }
            }
        }
    }
    reduce_rows_and_add(s, q, c0, C, out, ss + 2 * C, ss + 3 * C);
}

// backward pass 2: dy = scale * (dz - sum_dz/n - xhat * sum_dzx/n) = scale*dz + k0 + k1*y
__global__ void __launch_bounds__(256)
bn_act_bwd_apply_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ g,
                        const float* __restrict__ ss, const float* __restrict__ sums, float inv_n, int B, int T, int C,
                        int ld, int act, float a, float bb, const float* __restrict__ xlen,
                        __nv_bfloat16* __restrict__ dy, float drop_p, const long long* __restrict__ seed_ptr,
                        unsigned long long salt, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    if (c0 >= ld) return;
    float sc[8], sh[8], k0[8], k1[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = c0 + e;
        const bool ok = c < C;
        sc[e] = ok ? ss[c] : 0.f;
        sh[e] = ok ? ss[C + c] : 0.f;
        const float mean = ok ? ss[2 * C + c] : 0.f, istd = ok ? ss[3 * C + c] : 0.f;
        const float m1 = ok ? sums[c] * inv_n : 0.f, m2 = ok ? sums[C + c] * inv_n : 0.f;
        k1[e] = -sc[e] * m2 * istd;          // coefficient of y
        k0[e] = -sc[e] * m1 - k1[e] * mean;  // constant term
    }
    const int R = B * T;
    const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
    for (int r = r0 + threadIdx.y; r < r1; r += 4 * kRowLanes) {
        uint4 yv[4], gv[4];
        bool keep[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int rr = r + u * kRowLanes;
            const int b = rr / T, t = rr - b * T;
            keep[u] = rr < r1 && (xlen == nullptr || t < frac_len(__ldg(xlen + b), T));
            yv[u] = rr < r1 ? *reinterpret_cast<const uint4*>(y + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
            gv[u] = keep[u] ? *reinterpret_cast<const uint4*>(g + (size_t)rr * ld + c0) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int rr = r + u * kRowLanes;
            if (rr >= r1) break;
            float yf[8], gf[8], o[8];
            unpack8(yv[u], yf);
            unpack8(gv[u], gf);
            if (drop_p > 0.f) {
                const unsigned long long seed = (unsigned long long)seed_ptr[0] + salt * 0xD1B54A32D192ED03ULL;
                const float inv_keep = 1.f / (1.f - drop_p);
#pragma unroll
                for (int e = 0; e < 8; ++e) gf[e] = dropout_keep(seed, (unsigned long long)rr * ld + c0 + e, drop_p) ? gf[e] * inv_keep : 0.f;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float dz = keep[u] ? gf[e] * act_grad(fmaf(yf[e], sc[e], sh[e]), act, a, bb) : 0.f;
                o[e] = fmaf(sc[e], dz, fmaf(k1[e], yf[e], k0[e]));
            }
            *reinterpret_cast<uint4*>(dy + (size_t)rr * ld + c0) = pack8(o);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Streamed versions of the three activation-sized kernels (the ones the training step uses).
// The row walkers above keep at most 48-64 KB of loads in flight per SM (registers bound the
// unroll), which measured 2.6-4.0 TB/s; HBM3e wants ~100 KB+ in flight per SM.  Here the loads
// are decoupled from registers: a persistent CTA streams its chunks of FULL rows (contiguous in
// the [R, ld] layout) through a ring of shared-memory stages with 1-D bulk async copies
// (cp.async.bulk ... mbarrier::complete_tx), one elected thread issuing, everybody consuming.
//   threads = vectors * lanes (vectors = ld/8 16-byte channel vectors per row); thread `tid` owns
//   channel vector tid % vectors for the whole kernel (coefficients in registers) and touches the
//   16-byte units tid, tid + threads, ... of every chunk: conflict-free smem reads, fully coalesced
//   global writes.  A chunk is 4 * lanes rows; 2 CTAs per SM; stages fill ~100 KB per CTA.
// ---------------------------------------------------------------------------------------
constexpr int kStreamUnits = 4;        // 16-byte units per thread per chunk
constexpr int kStreamMaxThreads = 512;
constexpr int kBnSumReplicas = 8;      // atomics of the reduction are spread over this many copies

__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct StreamArgs {
    const __nv_bfloat16* y;
    const __nv_bfloat16* g;    // grad w.r.t. the layer output (backward modes)
    __nv_bfloat16* out;        // forward: activations; apply: grad_y
    // split-bf16 ("fp32 tier"): every tensor is a (hi, lo) pair, value = hi + lo
    const __nv_bfloat16* y_lo;
    const __nv_bfloat16* g_lo;
    __nv_bfloat16* out_lo;
    const float* ss;           // [4][C] scale, shift, mean, invstd
    const float* xlen;
    double* partials;          // [kBnSumReplicas][2][C]: sum dz, sum dz * y (fp64: reproducible)
    float* sums;               // [2][C] totals (written by the apply pass)
    const long long* seed_ptr;
    unsigned long long salt;
    // forward with the BatchNorm finalize folded in (raw_sums != null): coefficients from the conv epilogue's raw sums
    const double* raw_sums;    // [2][sums_ld]
    const float* gamma;
    const float* beta;
    float* running_mean;
    float* running_var;
    float* ss_out;             // [4][C], written by CTA 0
    int sums_ld;
    float n_rows, eps, momentum;
    float a, bb, drop_p, inv_n;
    int B, T, C, ld, act;
    int vectors, rows_per_chunk, n_chunks, stages, stage_bytes;
    int reverse;
    double inv_n_rows;         // forward with folded finalize: 1 / n_rows
    int coef_off;              // byte offset of the [4][ld] coefficient table in dynamic shared memory
};

__device__ __forceinline__ void add8(float (&f)[8], const uint4& lo) {
    float l[8];
    unpack8(lo, l);
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] += l[e];
}
// lo half of a split-bf16 store: what the bf16 rounding of `hi` lost
__device__ __forceinline__ uint4 pack8_lo(const float (&f)[8], const uint4& hi) {
    float h[8], r[8];
    unpack8(hi, h);
#pragma unroll
    for (int e = 0; e < 8; ++e) r[e] = f[e] - h[e];
    return pack8(r);
}

template <int MODE, bool SPLIT, int ACT>  // MODE 0: forward, 1: backward reduce, 2: backward apply; ACT: the activation, compile time
__global__ void __launch_bounds__(kStreamMaxThreads)
bn_stream_kernel(const StreamArgs p) {
    constexpr int NT = MODE == 0 ? 1 : 2;          // tensors read (y [, g])
    constexpr int NIN = NT * (SPLIT ? 2 : 1);      // smem planes per stage: y, g, y_lo, g_lo
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)p.stages * NIN * p.stage_bytes);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int cv = tid % p.vectors, lane = tid / p.vectors, lanes = nthreads / p.vectors;
    const int c0 = cv * 8, C = p.C, ld = p.ld, R = p.B * p.T;
    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) mbar_init(&full[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    const int stride = gridDim.x;
    // p.reverse: walk the chunks from the last row to the first.  The producer of the tensor (a conv / dgrad GEMM, or the pass
    // before this one) finished with the high rows, so those are what is still resident in L2; an ascending walk over a tensor
    // larger than what L2 keeps would evict exactly the lines it is about to need.
    auto issue = [&](int ci, int s) {
        const int chunk = p.reverse ? p.n_chunks - 1 - ci : ci;
        const int row0 = chunk * p.rows_per_chunk;
        const uint32_t bytes = (uint32_t)(min(p.rows_per_chunk, R - row0) * ld) * 2u;
        unsigned char* dst = smem_raw + (size_t)s * NIN * p.stage_bytes;
        mbar_expect_tx(&full[s], bytes * NIN);
        bulk_load_1d(dst, p.y + (size_t)row0 * ld, bytes, &full[s]);
        if (NT == 2) bulk_load_1d(dst + p.stage_bytes, p.g + (size_t)row0 * ld, bytes, &full[s]);
        if (SPLIT) {
            bulk_load_1d(dst + (size_t)NT * p.stage_bytes, p.y_lo + (size_t)row0 * ld, bytes, &full[s]);
            if (NT == 2) bulk_load_1d(dst + (size_t)(NT + 1) * p.stage_bytes, p.g_lo + (size_t)row0 * ld, bytes, &full[s]);
        }
    };
    if (tid == 0)
        for (int s = 0; s < p.stages; ++s)
            if (blockIdx.x + s * stride < p.n_chunks) issue(blockIdx.x + s * stride, s);

    // Per-channel coefficients, computed ONCE per CTA (channel c by thread c % nthreads) into a shared-memory table and then
    // picked up by the `lanes` threads that own the channel.  Every thread used to derive its 8 channels itself: lanes x
    // redundant, and with the BatchNorm finalize folded in that meant 16 fp64 divisions per thread -- ~10 us of a 28 us launch
    // at 256 channels (tools/time_train_kernels.py: the kernels stream at 6.2-6.4 TB/s on top of a 17-25 us fixed cost).
    float* coef = reinterpret_cast<float*>(smem_raw + p.coef_off);  // [4][ld]: scale, shift, k0, k1
    {
        const double inv_nd = p.inv_n_rows;  // 1 / n_rows, from the host: no fp64 division on the device
        for (int c = tid; c < ld; c += nthreads) {
            float sc_ = 0.f, sh_ = 0.f, k0_ = 0.f, k1_ = 0.f;
            if (c < C) {
                if (MODE == 0 && p.raw_sums != nullptr) {
                    // same arithmetic as bn_finalize_kernel
                    const float n = p.n_rows;
                    const double mean_d = p.raw_sums[c] * inv_nd;
                    const float mean = (float)mean_d;
                    const float var = (float)fmax(p.raw_sums[p.sums_ld + c] * inv_nd - mean_d * mean_d, 0.0);
                    const float invstd = rsqrtf(var + p.eps);
                    const float g = p.gamma ? p.gamma[c] : 1.f, b = p.beta ? p.beta[c] : 0.f;
                    sc_ = g * invstd;
                    sh_ = b - mean * g * invstd;
                    if (blockIdx.x == 0) {
                        p.ss_out[c] = sc_;
                        p.ss_out[C + c] = sh_;
                        p.ss_out[2 * C + c] = mean;
                        p.ss_out[3 * C + c] = invstd;
                        if (p.running_mean) p.running_mean[c] = (1.f - p.momentum) * p.running_mean[c] + p.momentum * mean;
                        if (p.running_var) p.running_var[c] = (1.f - p.momentum) * p.running_var[c] + p.momentum * var * (n / fmaxf(n - 1.f, 1.f));
                    }
                } else {
                    sc_ = p.ss[c];
                    sh_ = p.ss[C + c];
                }
                if (MODE == 2) {
                    const float mean = p.ss[2 * C + c], istd = p.ss[3 * C + c];
                    double d1 = 0.0, d2 = 0.0;
#pragma unroll
                    for (int r = 0; r < kBnSumReplicas; ++r) {
                        d1 += p.partials[(size_t)r * 2 * C + c];
                        d2 += p.partials[(size_t)r * 2 * C + C + c];
                    }
                    // sum(dz * xhat) = invstd * (sum(dz * y) - mean * sum(dz)), centred in fp64
                    const float m1 = (float)d1;
                    const float m2 = (float)((double)istd * (d2 - (double)mean * d1));
                    if (blockIdx.x == 0) { p.sums[c] = m1; p.sums[C + c] = m2; }
                    k1_ = -sc_ * (m2 * p.inv_n) * istd;        // coefficient of y
                    k0_ = -sc_ * (m1 * p.inv_n) - k1_ * mean;  // constant term
                }
            }
            coef[c] = sc_;
            coef[ld + c] = sh_;
            coef[2 * ld + c] = k0_;
            coef[3 * ld + c] = k1_;
        }
    }
    __syncthreads();
    float sc[8], sh[8], k0[8], k1[8], acc_s[8], acc_q[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        sc[e] = coef[c0 + e];
        sh[e] = coef[ld + c0 + e];
        k0[e] = coef[2 * ld + c0 + e];
        k1[e] = coef[3 * ld + c0 + e];
        acc_s[e] = 0.f; acc_q[e] = 0.f;
    }
    const float act_a = p.a, act_b = p.bb;
    const bool dropping = p.drop_p > 0.f;
    const unsigned long long seed = dropping ? (unsigned long long)p.seed_ptr[0] + p.salt * 0xD1B54A32D192ED03ULL : 0ull;
    const float inv_keep = dropping ? 1.f / (1.f - p.drop_p) : 1.f;

    int it = 0;
    for (int ci = blockIdx.x; ci < p.n_chunks; ci += stride, ++it) {
        const int chunk = p.reverse ? p.n_chunks - 1 - ci : ci;
        const int s = it % p.stages;
        mbar_wait(&full[s], (uint32_t)(it / p.stages) & 1u);
        const unsigned char* src = smem_raw + (size_t)s * NIN * p.stage_bytes;
        const int row0 = chunk * p.rows_per_chunk;
        // one division per chunk; the 4 rows of this thread are `lanes` apart, (b, t) advance incrementally
        int b = (row0 + lane) / p.T, t = (row0 + lane) - b * p.T;
        int len = p.xlen == nullptr ? p.T : frac_len(__ldg(p.xlen + min(b, p.B - 1)), p.T);
#pragma unroll
        for (int u = 0; u < kStreamUnits; ++u) {
            const int rr = row0 + u * lanes + lane;
            if (rr >= R) break;
            if (u > 0) {
                t += lanes;
                while (t >= p.T) {
                    t -= p.T;
                    ++b;
                    len = p.xlen == nullptr ? p.T : frac_len(__ldg(p.xlen + b), p.T);
                }
            }
            const bool keep = t < len;
            const size_t unit = (size_t)u * nthreads + tid;
            if (MODE == 1 && !keep) continue;
            float yf[8], o[8];
            unpack8(*reinterpret_cast<const uint4*>(src + unit * 16), yf);
            if (SPLIT) add8(yf, *reinterpret_cast<const uint4*>(src + (size_t)NT * p.stage_bytes + unit * 16));
            if (MODE == 0) {
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = (keep && c0 + e < C) ? act_fwd_t<ACT>(fmaf(yf[e], sc[e], sh[e]), act_a, act_b) : 0.f;
                if (dropping) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = dropout_keep(seed, (unsigned long long)rr * ld + c0 + e, p.drop_p) ? o[e] * inv_keep : 0.f;
                }
            } else {
                float gf[8];
                unpack8(*reinterpret_cast<const uint4*>(src + p.stage_bytes + unit * 16), gf);
                if (SPLIT) add8(gf, *reinterpret_cast<const uint4*>(src + (size_t)(NT + 1) * p.stage_bytes + unit * 16));
                if (dropping) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) gf[e] = dropout_keep(seed, (unsigned long long)rr * ld + c0 + e, p.drop_p) ? gf[e] * inv_keep : 0.f;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    // padded rows may hold anything in g (nobody is required to write them): select, never multiply
                    const float dz = keep ? act_gate_t<ACT>(gf[e], fmaf(yf[e], sc[e], sh[e]), act_a, act_b) : 0.f;
                    if (MODE == 1) {
                        acc_s[e] += dz;
                        acc_q[e] = fmaf(dz, yf[e], acc_q[e]);
                    } else {
                        o[e] = fmaf(sc[e], dz, fmaf(k1[e], yf[e], k0[e]));
                    }
                }
            }
            if (MODE != 1) {
                const uint4 hi = pack8(o);
                *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(p.out) + ((size_t)row0 * ld * 2) + unit * 16) = hi;
                if (SPLIT) *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(p.out_lo) + ((size_t)row0 * ld * 2) + unit * 16) = pack8_lo(o, hi);
            }
        }
        __syncthreads();  // everybody is done reading stage s
        if (tid == 0 && ci + p.stages * stride < p.n_chunks) issue(ci + p.stages * stride, s);
    }
    if (MODE == 1) {
        // every issued chunk was consumed, so the stages are free: reduce the 16 partials over the row lanes
        float* red = reinterpret_cast<float*>(smem_raw);  // [lane][16][vectors]
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            red[((size_t)lane * 16 + e) * p.vectors + cv] = acc_s[e];
            red[((size_t)lane * 16 + 8 + e) * p.vectors + cv] = acc_q[e];
        }
        __syncthreads();
        if (lane == 0) {
            double* dst = p.partials + (size_t)(blockIdx.x % kBnSumReplicas) * 2 * C;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float a_ = 0.f, b_ = 0.f;
                for (int l = 0; l < lanes; ++l) {
                    a_ += red[((size_t)l * 16 + e) * p.vectors + cv];
                    b_ += red[((size_t)l * 16 + 8 + e) * p.vectors + cv];
                }
                const int c = c0 + e;
                if (c < C) {
                    atomicAdd(dst + c, (double)a_);
                    atomicAdd(dst + C + c, (double)b_);
                }
            }
        }
    }
}

// launch geometry of the streamed kernels; false = this row pitch is not covered (row walkers run)
static bool stream_geometry(int R, int ld, int n_inputs, StreamArgs& a, int& threads, int& grid, size_t& smem) {
    if (ld % 8 != 0 || R <= 0) return false;
    const int vectors = ld / 8;
    // CTA size and bytes of stages per CTA: the fastest backward of the 128-512 thread x 32-96 KB sweep over the BatchNorm layers
    // of the training step (profiles/r02b_bn_geometry.log)
    constexpr int target_threads = 256, stage_budget = 48 * 1024;
    int lanes = target_threads / vectors;  // ~256 threads: the kernels are register-heavy, more CTAs per SM beat bigger CTAs
    if (lanes < 1) lanes = 1;
    while ((vectors * lanes) % 32 != 0) ++lanes;
    threads = vectors * lanes;
    if (threads > kStreamMaxThreads) return false;
    a.vectors = vectors;
    a.rows_per_chunk = kStreamUnits * lanes;
    a.n_chunks = (R + a.rows_per_chunk - 1) / a.rows_per_chunk;
    a.stage_bytes = kStreamUnits * threads * 16;
    // ~48 KB of stages per CTA: 3-4 CTAs per SM (ncu: with 2 fat CTAs the SM idled on LDS / fixed-latency waits at
    // 52 % issue utilisation); bytes in flight per SM stay ~150-190 KB
    int stages = (int)((size_t)stage_budget / ((size_t)n_inputs * a.stage_bytes));
    a.stages = stages < 2 ? 2 : (stages > 8 ? 8 : stages);
    smem = (size_t)a.stages * n_inputs * a.stage_bytes + 8 * a.stages;
    smem = (smem + 15) & ~(size_t)15;
    a.coef_off = (int)smem;
    smem += (size_t)4 * ld * sizeof(float);
    if (smem < (size_t)threads * 64) smem = (size_t)threads * 64;  // the reduction scratch of the reduce pass
    if (smem > 220 * 1024) return false;
    grid = 0;  // sized by stream_launch from the occupancy of the instantiation
    return true;
}

static int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

template <int MODE, bool SPLIT, int ACT>
static cudaError_t stream_launch_act(const StreamArgs& a, int threads, int grid, size_t smem, cudaStream_t stream) {
    static size_t smem_set = 0;
    if (smem > smem_set) {
        cudaError_t e = cudaFuncSetAttribute(bn_stream_kernel<MODE, SPLIT, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        smem_set = smem;
    }
    // persistent grid = exactly one wave: resident CTAs per SM for this (threads, smem), cached
    static int cache_threads[8], cache_smem[8], cache_per_sm[8], n_cache = 0;
    int per_sm = 0;
    for (int i = 0; i < n_cache; ++i)
        if (cache_threads[i] == threads && cache_smem[i] == (int)smem) per_sm = cache_per_sm[i];
    if (per_sm == 0) {
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bn_stream_kernel<MODE, SPLIT, ACT>, threads, smem);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
        if (n_cache < 8) { cache_threads[n_cache] = threads; cache_smem[n_cache] = (int)smem; cache_per_sm[n_cache] = per_sm; ++n_cache; }
    }
    (void)grid;
    const int g = a.n_chunks < num_sms() * per_sm ? a.n_chunks : num_sms() * per_sm;
    bn_stream_kernel<MODE, SPLIT, ACT><<<g, threads, smem, stream>>>(a);
    return cudaGetLastError();
}
template <int MODE, bool SPLIT>
static cudaError_t stream_launch(const StreamArgs& a, int threads, int grid, size_t smem, cudaStream_t stream) {
    switch (a.act) {
        case CAB_ACT_RELU: return stream_launch_act<MODE, SPLIT, CAB_ACT_RELU>(a, threads, grid, smem, stream);
        case CAB_ACT_HARDTANH: return stream_launch_act<MODE, SPLIT, CAB_ACT_HARDTANH>(a, threads, grid, smem, stream);
        case CAB_ACT_LEAKY_RELU: return stream_launch_act<MODE, SPLIT, CAB_ACT_LEAKY_RELU>(a, threads, grid, smem, stream);
        default: return stream_launch_act<MODE, SPLIT, CAB_ACT_NONE>(a, threads, grid, smem, stream);
    }
}

// ---------------------------------------------------------------------------------------
// weight packing: fp32 [Co, Ci, K] -> bf16 tap-major [K, Co, ci_ld] (forward operand) and/or
// bf16 [K, Ci, co_ld] with flipped taps (dgrad operand); inverse for the gradient.
// ---------------------------------------------------------------------------------------
// block = (32, 8): a 32 (co) x 32 (ci) tile for all K taps; reads run along (ci, k) of one co row,
// writes run along ci (forward operand) or co (dgrad operand)
__global__ void __launch_bounds__(256)
pack_weight_kernel(const float* __restrict__ w, int Co, int Ci, int K, __nv_bfloat16* __restrict__ fwd,
                   int ci_ld, __nv_bfloat16* __restrict__ dgr, int co_ld) {
    extern __shared__ float tile[];  // [32 co][32 ci * K + 1]
    const int co0 = blockIdx.y * 32, ci0 = blockIdx.x * 32;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int run = 32 * K, pitch = run + 1;
    const int ci_n = min(32, Ci - ci0), co_n = min(32, Co - co0);
    for (int co = threadIdx.y; co < co_n; co += 8) {
        const float* src = w + ((size_t)(co0 + co) * Ci + ci0) * K;
        for (int i = threadIdx.x; i < ci_n * K; i += 32) tile[co * pitch + i] = src[i];
    }
    __syncthreads();
    for (int i = tid; i < 32 * 32 * K; i += 256) {
        // forward operand: ci fastest
        int ci = i % 32, co = (i / 32) % 32, k = i / 1024;
        if (fwd && ci < ci_n && co < co_n) fwd[((size_t)k * Co + co0 + co) * ci_ld + ci0 + ci] = __float2bfloat16_rn(tile[co * pitch + ci * K + k]);
        // dgrad operand: co fastest, taps flipped
        co = i % 32; ci = (i / 32) % 32;
        if (dgr && ci < ci_n && co < co_n) dgr[((size_t)(K - 1 - k) * Ci + ci0 + ci) * co_ld + co0 + co] = __float2bfloat16_rn(tile[co * pitch + ci * K + k]);
    }
}
// All layers in ONE launch: the per-layer grids above are 64-900 blocks of a 17-27 us kernel each (launch /
// ramp-up bound: 18 launches = 0.5 ms of a 23 ms step for 0.5 GB of traffic).  Tile = 16 co x 32 ci x K.
// mode 1 = stride-2 conv as a stride-1 conv over frame pairs (engine.pack_taps_stride2): tap kk of the original
// kernel lands at pair tap dp = floor((kk - pad) / 2) - dp_min, channel block q = (kk - pad) - 2 dp of a
// [taps2, Co, 2 * ci_alloc] operand (ci_ld = 2 * ci_alloc; unfilled slots stay as the caller zeroed them).
constexpr int kPackMaxItems = 32;
struct PackBatch {
    const float* w[kPackMaxItems];
    __nv_bfloat16* fwd[kPackMaxItems];
    __nv_bfloat16* dgr[kPackMaxItems];
    __nv_bfloat16* fwd_lo[kPackMaxItems];
    __nv_bfloat16* dgr_lo[kPackMaxItems];
    int Co[kPackMaxItems], Ci[kPackMaxItems], K[kPackMaxItems], ci_ld[kPackMaxItems], co_ld[kPackMaxItems];
    int mode[kPackMaxItems], pad[kPackMaxItems];
    int tile_start[kPackMaxItems + 1];
    int n;
};
__device__ __forceinline__ int floordiv2(int j) { return j >= 0 ? j / 2 : -((1 - j) / 2); }
__device__ __forceinline__ void store_split(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t idx, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[idx] = h;
    if (lo) lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__global__ void __launch_bounds__(256)
pack_weights_batched_kernel(const PackBatch pb) {
    extern __shared__ float tile[];  // [16 co][32 ci * K + 1]
    int item = 0;
    while (item + 1 < pb.n && (int)blockIdx.x >= pb.tile_start[item + 1]) ++item;
    const int Co = pb.Co[item], Ci = pb.Ci[item], K = pb.K[item], ci_ld = pb.ci_ld[item], co_ld = pb.co_ld[item];
    const int mode = pb.mode[item], pad = pb.pad[item];
    const float* __restrict__ w = pb.w[item];
    __nv_bfloat16* __restrict__ fwd = pb.fwd[item];
    __nv_bfloat16* __restrict__ dgr = pb.dgr[item];
    __nv_bfloat16* __restrict__ fwd_lo = pb.fwd_lo[item];
    __nv_bfloat16* __restrict__ dgr_lo = pb.dgr_lo[item];
    const int local = blockIdx.x - pb.tile_start[item];
    const int n_ci_tiles = (Ci + 31) / 32;
    const int co0 = (local / n_ci_tiles) * 16, ci0 = (local % n_ci_tiles) * 32;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int run = 32 * K, pitch = run + 1;
    const int ci_n = min(32, Ci - ci0), co_n = min(16, Co - co0);
    for (int co = threadIdx.y; co < co_n; co += 8) {
        const float* src = w + ((size_t)(co0 + co) * Ci + ci0) * K;
        for (int i = threadIdx.x; i < ci_n * K; i += 32) tile[co * pitch + i] = src[i];
    }
    __syncthreads();
    const int dp_min = floordiv2(-pad);
    for (int i = tid; i < 16 * 32 * K; i += 256) {
        const int k = i / 512, r = i - k * 512;
        int ci = r % 32, co = r / 32;  // forward operand: ci fastest
        if (fwd && ci < ci_n && co < co_n) {
            const float v = tile[co * pitch + ci * K + k];
            if (mode == 0) {
                store_split(fwd, fwd_lo, ((size_t)k * Co + co0 + co) * ci_ld + ci0 + ci, v);
            } else {
                const int j = k - pad, dp = floordiv2(j), q = j - 2 * dp;
                store_split(fwd, fwd_lo, ((size_t)(dp - dp_min) * Co + co0 + co) * ci_ld + q * (ci_ld / 2) + ci0 + ci, v);
            }
        }
        co = r % 16; ci = r / 16;      // dgrad operand: co fastest, taps flipped
        if (dgr && ci < ci_n && co < co_n) store_split(dgr, dgr_lo, ((size_t)(K - 1 - k) * Ci + ci0 + ci) * co_ld + co0 + co, tile[co * pitch + ci * K + k]);
    }
}

// packed gradient fp32 [K, M, ld] -> fp32 [Co, Ci, K]; transposed = packed is [K, Ci, Co]
// transposed = 2: packed is the stride-2 pair layout [taps2, Co, ld] of pack mode 1 (`pair_pad` = the conv's padding,
// channel block q starts at q * (pair_ci_alloc))
__global__ void unpack_wgrad_kernel(const float* __restrict__ packed, int K, int Co, int Ci, int ld, int transposed,
                                    float* __restrict__ grad, int accumulate, int pair_pad, int pair_ci_alloc) {
    const size_t n = (size_t)Co * Ci * K;
    const int dp_min = floordiv2(-pair_pad);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i % K);
        const int ci = (int)((i / K) % Ci);
        const int co = (int)(i / ((size_t)K * Ci));
        float v;
        if (transposed == 2) {
            const int j = k - pair_pad, dp = floordiv2(j), q = j - 2 * dp;
            v = packed[((size_t)(dp - dp_min) * Co + co) * ld + q * pair_ci_alloc + ci];
        } else {
            v = transposed ? packed[((size_t)k * Ci + ci) * ld + co] : packed[((size_t)k * Co + co) * ld + ci];
        }
        grad[i] = accumulate ? grad[i] + v : v;
    }
}

// All layers in ONE launch (19 per-layer launches were 0.46 ms of a 24 ms step, launch / latency bound).  thread = (co, ci):
// reads run along ci (coalesced in every packed layout), each thread writes its K taps -- a warp's writes form one contiguous
// span of the parameter-layout gradient.
constexpr int kUnpackMaxItems = 32;
struct UnpackBatch {
    const float* packed[kUnpackMaxItems];
    float* grad[kUnpackMaxItems];
    int K[kUnpackMaxItems], Co[kUnpackMaxItems], Ci[kUnpackMaxItems], ld[kUnpackMaxItems], mode[kUnpackMaxItems];
    int pair_pad[kUnpackMaxItems], pair_ci_alloc[kUnpackMaxItems];
    int block_start[kUnpackMaxItems + 1];
    int n;
};
__global__ void __launch_bounds__(256)
unpack_wgrad_batched_kernel(const UnpackBatch ub) {
    extern __shared__ float ut[];  // [256 (co, ci) pairs][K] in parameter order
    int item = 0;
    while (item + 1 < ub.n && (int)blockIdx.x >= ub.block_start[item + 1]) ++item;
    const int K = ub.K[item], Co = ub.Co[item], Ci = ub.Ci[item], ld = ub.ld[item], mode = ub.mode[item];
    const float* __restrict__ packed = ub.packed[item];
    float* __restrict__ grad = ub.grad[item];
    const long long base = (long long)(blockIdx.x - ub.block_start[item]) * 256;
    const long long total = (long long)Co * Ci;
    const long long idx = base + threadIdx.x;
    if (idx < total) {
        const int co = (int)(idx / Ci), ci = (int)(idx - (long long)co * Ci);
        float* dst = ut + threadIdx.x * K;  // stride K: K odd for every conv of the model zoo -> conflict free
        if (mode == 2) {
            const int pad = ub.pair_pad[item], ca = ub.pair_ci_alloc[item];
            const int dp_min = floordiv2(-pad);
            for (int k = 0; k < K; ++k) {
                const int j = k - pad, dp = floordiv2(j), q = j - 2 * dp;
                dst[k] = packed[((size_t)(dp - dp_min) * Co + co) * ld + q * ca + ci];
            }
        } else if (mode == 1) {
            for (int k = 0; k < K; ++k) dst[k] = packed[((size_t)k * Ci + ci) * ld + co];
        } else {
            for (int k = 0; k < K; ++k) dst[k] = packed[((size_t)k * Co + co) * ld + ci];
        }
    }
    __syncthreads();
    // the block's 256 * K outputs are one contiguous span of the parameter-layout gradient
    const long long n_out = (total - base < 256 ? total - base : 256) * K;
    float* out = grad + base * K;
    for (long long i = threadIdx.x; i < n_out; i += 256) out[i] = ut[i];
}

// fp32 [B, C, T] -> bf16 channels-last [B, T, ld] (zero padded channels) + per-class sums over (b, t)
__global__ void __launch_bounds__(256)
bct_to_btc_kernel(const float* __restrict__ x, int B, int C, int T, int ld, __nv_bfloat16* __restrict__ out,
                  __nv_bfloat16* __restrict__ out_lo, float* __restrict__ csum) {
    // block = (32-class tile, utterance) walking over the frames: the per-class sums stay in registers and cost 32 atomics per
    // block (one per (b, class)) instead of one per 32 frames (123 k same-address atomics made this 9 MB kernel take 73 us)
    __shared__ float tile[32][33];
    const int b = blockIdx.y, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    float acc[4] = {0.f, 0.f, 0.f, 0.f};  // rows ty, ty + 8, ty + 16, ty + 24 of the class tile
    for (int t0 = 0; t0 < T; t0 += 32) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = c0 + ty + 8 * r, t = t0 + tx;
            float v = 0.f;
            if (c < C && t < T) v = x[((size_t)b * C + c) * T + t];
            tile[ty + 8 * r][tx] = v;
            acc[r] += v;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int t = t0 + ty + 8 * r, c = c0 + tx;
            if (t < T && c < ld) store_split(out, out_lo, ((size_t)b * T + t) * ld + c, tile[tx][ty + 8 * r]);
        }
        __syncthreads();
    }
    if (csum != nullptr) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float s = warp_sum(acc[r]);
            const int c = c0 + ty + 8 * r;
            if (tx == 0 && c < C) atomicAdd(csum + c, s);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Residual topologies (models.py:129-133: on the last repeat of a block every residual source goes through its own
// 1x1 conv + BatchNorm and is ADDED before the activation; 'flat' residuals are added as they are):
//   forward : out = mask(dropout(act(sum_i (scale_i * y_i + shift_i))))       bn_multi_fwd_kernel
//   backward: dz = g * act'(.) * mask * dropout, gate taken from `out`         act_bwd_dz_kernel
//             then every BatchNorm branch is the plain single-input backward on (y_i, dz) with act = none
// Row walkers (a thread owns one 16-byte channel vector and walks rows): these run on the last repeat of a block only.
// ---------------------------------------------------------------------------------------
constexpr int kMaxBranches = CAB_MAX_BN_BRANCHES;
struct MultiArgs {
    const __nv_bfloat16* y[kMaxBranches];
    const __nv_bfloat16* y_lo[kMaxBranches];
    const float* ss[kMaxBranches];  // [4][C] or null (identity branch)
    int n;
};

template <bool SPLIT>
__global__ void __launch_bounds__(256)
bn_multi_fwd_kernel(const MultiArgs m, int B, int T, int C, int ld, int act, float a, float bb, const float* __restrict__ xlen,
                    __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo, float drop_p,
                    const long long* __restrict__ seed_ptr, unsigned long long salt, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    if (c0 >= ld) return;
    const int R = B * T;
    const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
    const unsigned long long seed = drop_p > 0.f ? (unsigned long long)seed_ptr[0] + salt * 0xD1B54A32D192ED03ULL : 0ull;
    const float inv_keep = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    for (int r = r0 + threadIdx.y; r < r1; r += kRowLanes) {
        const int b = r / T, t = r - b * T;
        const bool keep = xlen == nullptr || t < frac_len(__ldg(xlen + b), T);
        float z[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) z[e] = 0.f;
        if (keep) {
            for (int i = 0; i < m.n; ++i) {
                float f[8];
                unpack8(*reinterpret_cast<const uint4*>(m.y[i] + (size_t)r * ld + c0), f);
                if (SPLIT) add8(f, *reinterpret_cast<const uint4*>(m.y_lo[i] + (size_t)r * ld + c0));
                const float* ss = m.ss[i];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int c = c0 + e;
                    if (c < C) z[e] += ss ? fmaf(f[e], __ldg(ss + c), __ldg(ss + C + c)) : f[e];
                }
            }
        }
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = (keep && c0 + e < C) ? act_fwd(z[e], act, a, bb) : 0.f;
        if (drop_p > 0.f) {
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = dropout_keep(seed, (unsigned long long)r * ld + c0 + e, drop_p) ? o[e] * inv_keep : 0.f;
        }
        const uint4 hi = pack8(o);
        *reinterpret_cast<uint4*>(out + (size_t)r * ld + c0) = hi;
        if (SPLIT) *reinterpret_cast<uint4*>(out_lo + (size_t)r * ld + c0) = pack8_lo(o, hi);
    }
}

// dz = g * act'(z) * mask * dropout with the gate read off the stored output v = out * (1 - p) (a kept element is
// act(z) / (1 - p), rounded to bf16 -- or to hi + lo in the split tier -- and scaled back in fp32); dropped or masked
// elements get 0.  relu / leaky: z > 0 <=> v > 0 holds exactly (rounding and scaling keep the sign and zero).  hardtanh:
// the gate is a < v < b, which is NOT the same as a < z < b next to a clamp bound -- a z within one rounding of the stored
// value from a or b (bf16: z in [19.9375, 20) stores 20.0 for b = 20; split tier: ~2^-16 relative; wider with dropout,
// whose 1 / (1 - p) and (1 - p) round) reads as clamped and gets gate 0 where autograd's z-gate gives 1, or the reverse.
// Recomputing z would mean re-reading every branch; the tests pin this contract exactly.
template <bool SPLIT>
__global__ void __launch_bounds__(256)
act_bwd_dz_kernel(const __nv_bfloat16* __restrict__ out, const __nv_bfloat16* __restrict__ out_lo,
                  const __nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ g_lo, int B, int T, int C, int ld,
                  int act, float a, float bb, const float* __restrict__ xlen, __nv_bfloat16* __restrict__ dz,
                  __nv_bfloat16* __restrict__ dz_lo, float drop_p, const long long* __restrict__ seed_ptr,
                  unsigned long long salt, int kRowsPerBlock) {
    const int cv = blockIdx.x * 32 + threadIdx.x;
    const int c0 = cv * 8;
    if (c0 >= ld) return;
    const int R = B * T;
    const int r0 = blockIdx.y * kRowsPerBlock, r1 = min(R, r0 + kRowsPerBlock);
    const unsigned long long seed = drop_p > 0.f ? (unsigned long long)seed_ptr[0] + salt * 0xD1B54A32D192ED03ULL : 0ull;
    const float inv_keep = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f, keep_p = 1.f - drop_p;
    for (int r = r0 + threadIdx.y; r < r1; r += kRowLanes) {
        const int b = r / T, t = r - b * T;
        const bool keep = xlen == nullptr || t < frac_len(__ldg(xlen + b), T);
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = 0.f;
        if (keep) {
            float of[8], gf[8];
            unpack8(*reinterpret_cast<const uint4*>(out + (size_t)r * ld + c0), of);
            unpack8(*reinterpret_cast<const uint4*>(g + (size_t)r * ld + c0), gf);
            if (SPLIT) {
                add8(of, *reinterpret_cast<const uint4*>(out_lo + (size_t)r * ld + c0));
                add8(gf, *reinterpret_cast<const uint4*>(g_lo + (size_t)r * ld + c0));
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (c0 + e >= C) continue;
                float gate;
                const float v = of[e] * keep_p;
                if (act == CAB_ACT_RELU) gate = v > 0.f ? 1.f : 0.f;
                else if (act == CAB_ACT_HARDTANH) gate = (v > a && v < bb) ? 1.f : 0.f;
                else if (act == CAB_ACT_LEAKY_RELU) gate = v > 0.f ? 1.f : a;
                else gate = 1.f;
                float d = gf[e] * gate;
                if (drop_p > 0.f) d = dropout_keep(seed, (unsigned long long)r * ld + c0 + e, drop_p) ? d * inv_keep : 0.f;
                o[e] = d;
            }
        }
        const uint4 hi = pack8(o);
        *reinterpret_cast<uint4*>(dz + (size_t)r * ld + c0) = hi;
        if (SPLIT) *reinterpret_cast<uint4*>(dz_lo + (size_t)r * ld + c0) = pack8_lo(o, hi);
    }
}

}  // namespace cab

using namespace cab;

#define GRID_1D(n, per) (int)(((n) / (per) + 255) / 256 > (size_t)num_sms() * 8 ? (size_t)num_sms() * 8 : (((n) / (per) + 255) / 256 < 1 ? 1 : ((n) / (per) + 255) / 256))

extern "C" int cab_bn_batch_stats(const void* y, int B, int T, int C, int ld, const float* gamma, const float* beta, float eps,
                                  float momentum, float* running_mean, float* running_var, double* ws_sums /*[2][C]*/,
                                  float* out_ss /*[4][C]*/, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(y && ws_sums && out_ss, "null pointer argument");
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout C=%d ld=%d", C, ld);
    CAB_CHECK_CUDA(cudaMemsetAsync(ws_sums, 0, sizeof(double) * 2 * C, stream));
    const int R = B * T, rpb = rows_per_block_for(R, ld);
    dim3 grid((ld / 8 + 31) / 32, (R + rpb - 1) / rpb), block(32, kRowLanes);
    colstats_kernel<<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(y), R, C, ld, ws_sums, rpb);
    CAB_CHECK_LAUNCH();
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(ws_sums, C, (float)R, gamma, beta, eps, momentum, running_mean, running_var, out_ss, C);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(2, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_bn_finalize(const double* sums, int n_rows, int C, const float* gamma, const float* beta, float eps,
                               float momentum, float* running_mean, float* running_var, float* out_ss, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(sums && out_ss && n_rows > 0 && C > 0, "bad arguments");
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(sums, C, (float)n_rows, gamma, beta, eps, momentum, running_mean, running_var, out_ss, C);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_bn_act_mask_fwd(const void* y, const void* y_lo, const float* ss, int B, int T, int C, int ld, int act,
                                   float act_a, float act_b, const float* xlen_frac, void* out, void* out_lo, float dropout_p,
                                   const int64_t* seed, int64_t salt, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(y && ss && out, "null pointer argument");
    CAB_CHECK_ARG((y_lo == nullptr) == (out_lo == nullptr), "split-bf16 tier needs both y_lo and out_lo");
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout");
    CAB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || seed != nullptr), "bad dropout arguments");
    const bool split = y_lo != nullptr;
    StreamArgs sa{};
    int threads, grid_s;
    size_t smem;
    if (stream_geometry(B * T, ld, split ? 2 : 1, sa, threads, grid_s, smem)) {
        sa.y = static_cast<const __nv_bfloat16*>(y); sa.out = static_cast<__nv_bfloat16*>(out); sa.ss = ss; sa.xlen = xlen_frac;
        sa.y_lo = static_cast<const __nv_bfloat16*>(y_lo); sa.out_lo = static_cast<__nv_bfloat16*>(out_lo);
        sa.seed_ptr = reinterpret_cast<const long long*>(seed); sa.salt = (unsigned long long)salt;
        sa.a = act_a; sa.bb = act_b; sa.drop_p = dropout_p; sa.B = B; sa.T = T; sa.C = C; sa.ld = ld; sa.act = act;
        sa.reverse = 1;  // the conv that produced y finished with the high rows
        if (split) CAB_CHECK_CUDA((stream_launch<0, true>(sa, threads, grid_s, smem, stream)));
        else CAB_CHECK_CUDA((stream_launch<0, false>(sa, threads, grid_s, smem, stream)));
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
        return 0;
    }
    CAB_CHECK_ARG(!split, "split-bf16 BatchNorm forward: row pitch ld=%d not covered by the streamed kernel", ld);
    const int rpb = rows_per_block_for(B * T, ld);
    dim3 grid((ld / 8 + 31) / 32, (B * T + rpb - 1) / rpb), block(32, kRowLanes);
    bn_act_mask_fwd_kernel<<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(y), ss, B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(out), dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_bn_act_mask_fwd_stats(const void* y, const void* y_lo, const double* raw_sums, int sums_ld, int n_rows,
                                         const float* gamma, const float* beta, float eps, float momentum, float* running_mean,
                                         float* running_var, float* out_ss, int B, int T, int C, int ld, int act, float act_a,
                                         float act_b, const float* xlen_frac, void* out, void* out_lo, float dropout_p,
                                         const int64_t* seed, int64_t salt, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(y && raw_sums && out_ss && out && n_rows > 0 && sums_ld >= C, "bad arguments");
    CAB_CHECK_ARG((y_lo == nullptr) == (out_lo == nullptr), "split-bf16 tier needs both y_lo and out_lo");
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout");
    CAB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || seed != nullptr), "bad dropout arguments");
    const bool split = y_lo != nullptr;
    StreamArgs sa{};
    int threads, grid_s;
    size_t smem;
    if (!stream_geometry(B * T, ld, split ? 2 : 1, sa, threads, grid_s, smem)) {
        // row pitch not covered by the streamed kernel: finalize, then the row walker
        bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(raw_sums, C, (float)n_rows, gamma, beta, eps, momentum, running_mean, running_var, out_ss, sums_ld);
        CAB_CHECK_LAUNCH();
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
        return cab_bn_act_mask_fwd(y, y_lo, out_ss, B, T, C, ld, act, act_a, act_b, xlen_frac, out, out_lo, dropout_p, seed, salt, stream_);
    }
    sa.y = static_cast<const __nv_bfloat16*>(y); sa.out = static_cast<__nv_bfloat16*>(out); sa.ss = nullptr; sa.xlen = xlen_frac;
    sa.y_lo = static_cast<const __nv_bfloat16*>(y_lo); sa.out_lo = static_cast<__nv_bfloat16*>(out_lo);
    sa.seed_ptr = reinterpret_cast<const long long*>(seed); sa.salt = (unsigned long long)salt;
    sa.raw_sums = raw_sums; sa.sums_ld = sums_ld; sa.gamma = gamma; sa.beta = beta; sa.running_mean = running_mean; sa.running_var = running_var;
    sa.ss_out = out_ss; sa.n_rows = (float)n_rows; sa.inv_n_rows = 1.0 / (double)(float)n_rows; sa.eps = eps; sa.momentum = momentum;
    sa.a = act_a; sa.bb = act_b; sa.drop_p = dropout_p; sa.B = B; sa.T = T; sa.C = C; sa.ld = ld; sa.act = act;
    sa.reverse = 1;
    if (split) CAB_CHECK_CUDA((stream_launch<0, true>(sa, threads, grid_s, smem, stream)));
    else CAB_CHECK_CUDA((stream_launch<0, false>(sa, threads, grid_s, smem, stream)));
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

static int bn_bwd_impl(const void* y, const void* y_lo, const void* grad_out, const void* grad_out_lo, const float* ss,
                       int B, int T, int C, int ld, int act, float act_a, float act_b, const float* xlen_frac,
                       float* sums /*[2][C]: dbeta, dgamma*/, void* grad_y, void* grad_y_lo, float dropout_p,
                       const int64_t* seed, int64_t salt, int frozen, double* ws_partials, bool partials_ready, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(y && grad_out && ss && sums && grad_y, "null pointer argument");
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout");
    CAB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || seed != nullptr), "bad dropout arguments");
    const bool split = y_lo != nullptr;
    CAB_CHECK_ARG(split == (grad_out_lo != nullptr) && split == (grad_y_lo != nullptr), "split-bf16 tier needs y_lo, grad_out_lo and grad_y_lo together");
    {
        StreamArgs sa{};
        int threads, grid_s;
        size_t smem;
        if (ws_partials != nullptr && stream_geometry(B * T, ld, split ? 4 : 2, sa, threads, grid_s, smem)) {
            sa.y = static_cast<const __nv_bfloat16*>(y); sa.g = static_cast<const __nv_bfloat16*>(grad_out);
            sa.y_lo = static_cast<const __nv_bfloat16*>(y_lo); sa.g_lo = static_cast<const __nv_bfloat16*>(grad_out_lo);
            sa.out = static_cast<__nv_bfloat16*>(grad_y); sa.out_lo = static_cast<__nv_bfloat16*>(grad_y_lo);
            sa.ss = ss; sa.xlen = xlen_frac; sa.partials = ws_partials; sa.sums = sums;
            sa.seed_ptr = reinterpret_cast<const long long*>(seed); sa.salt = (unsigned long long)salt;
            sa.a = act_a; sa.bb = act_b; sa.drop_p = dropout_p; sa.inv_n = frozen ? 0.f : 1.f / (float)(B * T);  // frozen: grad_y = scale * dz
            sa.B = B; sa.T = T; sa.C = C; sa.ld = ld; sa.act = act;
            if (partials_ready) {
                // the dgrad GEMM that produced grad_out also accumulated the sums and finished with the high rows: descend
                sa.reverse = 1;
                if (split) CAB_CHECK_CUDA((stream_launch<2, true>(sa, threads, grid_s, smem, stream)));
                else CAB_CHECK_CUDA((stream_launch<2, false>(sa, threads, grid_s, smem, stream)));
                g_launch_count.fetch_add(1, std::memory_order_relaxed);
                return 0;
            }
            CAB_CHECK_CUDA(cudaMemsetAsync(ws_partials, 0, sizeof(double) * kBnSumReplicas * 2 * C, stream));
            // reduce pass: descending (the dgrad GEMM that produced grad_out finished with the high rows); apply pass: ascending
            // (the reduce pass finished with the low rows)
            StreamArgs sr = sa;
            sr.reverse = 1;
            sa.reverse = 0;
            if (split) {
                CAB_CHECK_CUDA((stream_launch<1, true>(sr, threads, grid_s, smem, stream)));
                CAB_CHECK_CUDA((stream_launch<2, true>(sa, threads, grid_s, smem, stream)));
            } else {
                CAB_CHECK_CUDA((stream_launch<1, false>(sr, threads, grid_s, smem, stream)));
                CAB_CHECK_CUDA((stream_launch<2, false>(sa, threads, grid_s, smem, stream)));
            }
            g_launch_count.fetch_add(2, std::memory_order_relaxed);
            return 0;
        }
    }
    CAB_CHECK_ARG(!partials_ready, "cab_bn_act_mask_bwd_apply: row pitch ld=%d is not covered by the streamed kernel", ld);
    CAB_CHECK_ARG(!split, "split-bf16 BatchNorm backward needs ws_partials and a row pitch the streamed kernel covers (ld=%d)", ld);
    CAB_CHECK_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * 2 * C, stream));
    const int R = B * T, rpb = rows_per_block_for(R, ld);
    dim3 grid((ld / 8 + 31) / 32, (R + rpb - 1) / rpb), block(32, kRowLanes);
    bn_act_bwd_reduce_kernel<<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(y), static_cast<const __nv_bfloat16*>(grad_out), ss, B, T, C, ld, act, act_a, act_b, xlen_frac, sums, dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    CAB_CHECK_LAUNCH();
    bn_act_bwd_apply_kernel<<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(y), static_cast<const __nv_bfloat16*>(grad_out), ss, sums, frozen ? 0.f : 1.f / (float)R, B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(grad_y), dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(2, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_bn_act_mask_bwd(const void* y, const void* y_lo, const void* grad_out, const void* grad_out_lo, const float* ss,
                                   int B, int T, int C, int ld, int act, float act_a, float act_b, const float* xlen_frac,
                                   float* sums, void* grad_y, void* grad_y_lo, float dropout_p, const int64_t* seed, int64_t salt,
                                   int frozen, double* ws_partials, cab_stream_t stream_) {
    return bn_bwd_impl(y, y_lo, grad_out, grad_out_lo, ss, B, T, C, ld, act, act_a, act_b, xlen_frac, sums, grad_y, grad_y_lo, dropout_p, seed, salt,
                       frozen, ws_partials, false, stream_);
}

extern "C" int cab_bn_act_mask_bwd_apply(const void* y, const void* y_lo, const void* grad_out, const void* grad_out_lo, const float* ss,
                                         int B, int T, int C, int ld, int act, float act_a, float act_b, const float* xlen_frac,
                                         float* sums, void* grad_y, void* grad_y_lo, float dropout_p, const int64_t* seed, int64_t salt,
                                         int frozen, const double* partials, cab_stream_t stream_) {
    CAB_CHECK_ARG(partials != nullptr, "partials is null");
    return bn_bwd_impl(y, y_lo, grad_out, grad_out_lo, ss, B, T, C, ld, act, act_a, act_b, xlen_frac, sums, grad_y, grad_y_lo, dropout_p, seed, salt,
                       frozen, const_cast<double*>(partials), true, stream_);
}

extern "C" int cab_bn_bwd_apply_covers(int R, int ld, int split) {
    StreamArgs sa{};
    int threads = 0, grid_s = 0;
    size_t smem = 0;
    return stream_geometry(R, ld, split ? 4 : 2, sa, threads, grid_s, smem) ? 1 : 0;
}

extern "C" int cab_bn_multi_act_mask_fwd(const cab_bn_branch_t* branches, int n_branches, int B, int T, int C, int ld, int act,
                                         float act_a, float act_b, const float* xlen_frac, void* out, void* out_lo,
                                         float dropout_p, const int64_t* seed, int64_t salt, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(branches && out && n_branches >= 1 && n_branches <= kMaxBranches, "n_branches=%d out of [1,%d]", n_branches, kMaxBranches);
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout");
    CAB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || seed != nullptr), "bad dropout arguments");
    const bool split = out_lo != nullptr;
    MultiArgs m{};
    m.n = n_branches;
    for (int i = 0; i < n_branches; ++i) {
        CAB_CHECK_ARG(branches[i].y != nullptr && (!split || branches[i].y_lo != nullptr), "branch %d: null pointer", i);
        m.y[i] = static_cast<const __nv_bfloat16*>(branches[i].y);
        m.y_lo[i] = static_cast<const __nv_bfloat16*>(branches[i].y_lo);
        m.ss[i] = branches[i].ss;
    }
    const int R = B * T, rpb = rows_per_block_for(R, ld);
    dim3 grid((ld / 8 + 31) / 32, (R + rpb - 1) / rpb), block(32, kRowLanes);
    if (split) bn_multi_fwd_kernel<true><<<grid, block, 0, stream>>>(m, B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(out), static_cast<__nv_bfloat16*>(out_lo), dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    else bn_multi_fwd_kernel<false><<<grid, block, 0, stream>>>(m, B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(out), nullptr, dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_act_mask_bwd_dz(const void* out, const void* out_lo, const void* grad_out, const void* grad_out_lo, int B, int T,
                                   int C, int ld, int act, float act_a, float act_b, const float* xlen_frac, void* dz, void* dz_lo,
                                   float dropout_p, const int64_t* seed, int64_t salt, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(out && grad_out && dz, "null pointer argument");
    CAB_CHECK_ARG(ld % 8 == 0 && ld >= C, "bad channel layout");
    CAB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f && (dropout_p == 0.f || seed != nullptr), "bad dropout arguments");
    const bool split = dz_lo != nullptr;
    CAB_CHECK_ARG(!split || (out_lo && grad_out_lo), "split-bf16 tier needs out_lo and grad_out_lo");
    const int R = B * T, rpb = rows_per_block_for(R, ld);
    dim3 grid((ld / 8 + 31) / 32, (R + rpb - 1) / rpb), block(32, kRowLanes);
    if (split) act_bwd_dz_kernel<true><<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(out), static_cast<const __nv_bfloat16*>(out_lo), static_cast<const __nv_bfloat16*>(grad_out), static_cast<const __nv_bfloat16*>(grad_out_lo), B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(dz), static_cast<__nv_bfloat16*>(dz_lo), dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    else act_bwd_dz_kernel<false><<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(out), nullptr, static_cast<const __nv_bfloat16*>(grad_out), nullptr, B, T, C, ld, act, act_a, act_b, xlen_frac, static_cast<__nv_bfloat16*>(dz), nullptr, dropout_p, reinterpret_cast<const long long*>(seed), (unsigned long long)salt, rpb);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_pack_weight(const float* w, int Co, int Ci, int K, void* fwd, int ci_ld, void* dgrad, int co_ld, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(w && (fwd || dgrad), "null pointer argument");
    CAB_CHECK_ARG((!fwd || ci_ld >= Ci) && (!dgrad || co_ld >= Co), "bad pitch");
    const size_t smem = sizeof(float) * 32 * (32 * K + 1);
    CAB_CHECK_ARG(smem <= 160 * 1024, "kernel size K=%d too large for the packing tile", K);
    static size_t smem_set = 0;
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(pack_weight_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    dim3 grid((Ci + 31) / 32, (Co + 31) / 32), block(32, 8);
    pack_weight_kernel<<<grid, block, smem, stream>>>(w, Co, Ci, K, static_cast<__nv_bfloat16*>(fwd), ci_ld, static_cast<__nv_bfloat16*>(dgrad), co_ld);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_pack_weights_batched(const cab_pack_item_t* items, int n, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(items && n >= 1 && n <= kPackMaxItems, "n=%d out of [1,%d]", n, kPackMaxItems);
    static thread_local PackBatch pb;
    int max_k = 1, tiles = 0;
    for (int i = 0; i < n; ++i) {
        const cab_pack_item_t& it = items[i];
        CAB_CHECK_ARG(it.w && (it.fwd || it.dgrad) && it.Co > 0 && it.Ci > 0 && it.K > 0, "item %d: bad arguments", i);
        CAB_CHECK_ARG((!it.fwd || it.ci_ld >= it.Ci) && (!it.dgrad || it.co_ld >= it.Co), "item %d: bad pitch", i);
        CAB_CHECK_ARG((!it.fwd_lo || it.fwd) && (!it.dgrad_lo || it.dgrad), "item %d: lo output without its hi output", i);
        pb.w[i] = it.w; pb.fwd[i] = static_cast<__nv_bfloat16*>(it.fwd); pb.dgr[i] = static_cast<__nv_bfloat16*>(it.dgrad);
        pb.fwd_lo[i] = static_cast<__nv_bfloat16*>(it.fwd_lo); pb.dgr_lo[i] = static_cast<__nv_bfloat16*>(it.dgrad_lo);
        pb.Co[i] = it.Co; pb.Ci[i] = it.Ci; pb.K[i] = it.K; pb.ci_ld[i] = it.ci_ld; pb.co_ld[i] = it.co_ld;
        pb.mode[i] = it.mode; pb.pad[i] = it.pad;
        CAB_CHECK_ARG(it.mode == 0 || (it.mode == 1 && it.dgrad == nullptr && it.ci_ld % 2 == 0 && it.ci_ld / 2 >= it.Ci), "item %d: bad stride-2 pair packing arguments", i);
        pb.tile_start[i] = tiles;
        tiles += ((it.Co + 15) / 16) * ((it.Ci + 31) / 32);
        max_k = it.K > max_k ? it.K : max_k;
    }
    pb.tile_start[n] = tiles;
    pb.n = n;
    const size_t smem = sizeof(float) * 16 * (32 * max_k + 1);
    CAB_CHECK_ARG(smem <= 160 * 1024, "kernel size K=%d too large for the packing tile", max_k);
    static size_t smem_set = 0;
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(pack_weights_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    pack_weights_batched_kernel<<<tiles, dim3(32, 8), smem, stream>>>(pb);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_unpack_wgrad(const float* packed, int K, int Co, int Ci, int ld, int transposed, float* grad, int accumulate,
                                int pair_pad, int pair_ci_alloc, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(packed && grad, "null pointer argument");
    CAB_CHECK_ARG(transposed >= 0 && transposed <= 2, "transposed=%d", transposed);
    const size_t n = (size_t)Co * Ci * K;
    unpack_wgrad_kernel<<<GRID_1D(n, 1), 256, 0, stream>>>(packed, K, Co, Ci, ld, transposed, grad, accumulate, pair_pad, pair_ci_alloc);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_unpack_wgrad_batched(const cab_unpack_item_t* items, int n, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(items && n >= 1 && n <= kUnpackMaxItems, "n=%d out of [1,%d]", n, kUnpackMaxItems);
    static thread_local UnpackBatch ub;
    int blocks = 0;
    for (int i = 0; i < n; ++i) {
        const cab_unpack_item_t& it = items[i];
        CAB_CHECK_ARG(it.packed && it.grad && it.K > 0 && it.Co > 0 && it.Ci > 0 && it.transposed >= 0 && it.transposed <= 2, "item %d: bad arguments", i);
        ub.packed[i] = it.packed; ub.grad[i] = it.grad; ub.K[i] = it.K; ub.Co[i] = it.Co; ub.Ci[i] = it.Ci; ub.ld[i] = it.ld; ub.mode[i] = it.transposed;
        ub.pair_pad[i] = it.pair_pad; ub.pair_ci_alloc[i] = it.pair_ci_alloc;
        ub.block_start[i] = blocks;
        blocks += (int)(((long long)it.Co * it.Ci + 255) / 256);
    }
    ub.block_start[n] = blocks;
    ub.n = n;
    int max_k = 1;
    for (int i = 0; i < n; ++i) max_k = items[i].K > max_k ? items[i].K : max_k;
    const size_t smem = sizeof(float) * 256 * max_k;
    CAB_CHECK_ARG(smem <= 96 * 1024, "kernel size K=%d too large for the unpack tile", max_k);
    static size_t smem_set = 0;
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(unpack_wgrad_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    unpack_wgrad_batched_kernel<<<blocks, 256, smem, stream>>>(ub);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_bct_to_btc(const float* x, int B, int C, int T, int ld, void* out, void* out_lo, float* class_sums, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(x && out, "null pointer argument");
    CAB_CHECK_ARG(ld >= C, "bad pitch");
    if (class_sums) CAB_CHECK_CUDA(cudaMemsetAsync(class_sums, 0, sizeof(float) * C, stream));
    dim3 grid((ld + 31) / 32, B);
    bct_to_btc_kernel<<<grid, 256, 0, stream>>>(x, B, C, T, ld, static_cast<__nv_bfloat16*>(out), static_cast<__nv_bfloat16*>(out_lo), class_sums);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}
