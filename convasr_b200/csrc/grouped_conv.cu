// Grouped Conv1d + bias + ReLU: the depthwise-like first stage of the separable ConvSamePadding
// (models.py:50-64; JasperNetSeparable: groups = 128, 2-7 channels per group, k = 11..25).
//
// Why SIMT and not tcgen05: with 2-7 input channels per group the contraction length per output is
// cin_g * K = 22..150.  Laid on a 64-wide tensor-core tile the block-diagonal weights waste 10-30x of
// the MMAs and the operand traffic per output tile (K taps x 24 KB) is L2 bound; on the fp32 pipe the
// layer is issue bound at its real FLOPs.  B200-specific pieces: packed FFMA2 (fma.rn.f32x2, two
// channels of the group per instruction, so the fma pipe runs at its full 128 lanes/clk/SM), weights
// resident in shared memory for the whole life of a persistent CTA, register-blocked sliding window
// over time (each weight pair feeds 8 outputs, each input pair up to K outputs).
//
//   CTA  = one block of 64 output channels x a persistent loop over (utterance, 32-frame) tiles
//   thread = (output channel, strip of 8 frames); accumulators: 8 x float2 (even / odd input channel)
//   x tile: the input channels those 64 outputs need (<= 104), 64 + K - 1 frames, raw bf16 in smem,
//           double buffered with cp.async (zero fill = conv padding): the next tile lands during
//           the current tile's math; bf16 -> fp32 is a shift at load time.
//   FP8 (inference tier): x and the output are E4M3 -- the tile holds raw bytes (16 channels per 16-byte vector), a channel
//           pair is dequantised with one cvt (x = q * in_scale, the scale applied once to the sum), and the output is
//           stored as satfinite(rn(v / s_out)).
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

constexpr int kGcCo = 64;       // output channels per CTA
constexpr int kGcStrips = 4;    // frame strips per tile
constexpr int kGcTT = 16;       // frames per strip (register blocking)
constexpr int kGcTile = kGcStrips * kGcTT;
constexpr int kGcThreads = kGcCo * kGcStrips;
constexpr int kGcMaxCols = 104;  // tile width in input channels (multiple of 8)
constexpr int kGcMaxVec = 5;    // 16-byte prefetch vectors per thread and tensor

__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}

struct GroupedArgs {
    const __nv_bfloat16* x;
    const __nv_bfloat16* x_lo;
    const float* w;     // [C_out][cin_g][K]
    const float* bias;  // [C_out] or null
    __nv_bfloat16* out;
    __nv_bfloat16* out_lo;
    int B, T, T_rows, C_in, ld_in, C_out, ld_out, out_T_rows, groups, pad;
    int tiles_per_utt, n_items, parts, cols_max;
    int relu;           // 1: + bias, ReLU (forward of the separable pair); 0: plain grouped conv (its input gradient)
    const __nv_bfloat16* dy;     // wgrad: gradient w.r.t. the grouped conv's output [B, T_rows_dy, ld_dy]
    const __nv_bfloat16* dy_lo;
    int ld_dy, dy_T_rows;
    float* dw;          // wgrad: fp32 [C_out][cin_g][K], zeroed by the host wrapper
    float* db;          // wgrad: fp32 [C_out] or null
    float in_scale, out_inv;  // FP8: x = q * in_scale; stored q = v * out_inv
};

__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc, bool valid) {
    const uint32_t n = valid ? 16u : 0u;  // src-size 0: the 16 bytes are zero-filled (conv padding, rows outside [0, T))
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// two adjacent bf16 channels -> float2; ALIGNED: the pair sits in one 32-bit word
template <bool ALIGNED>
__device__ __forceinline__ float2 load_pair(const unsigned char* p) {
    if (ALIGNED) {
        const uint32_t v = *reinterpret_cast<const uint32_t*>(p);
        return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
    }
    const uint32_t a = *reinterpret_cast<const unsigned short*>(p), b = *reinterpret_cast<const unsigned short*>(p + 2);
    return make_float2(__uint_as_float(a << 16), __uint_as_float(b << 16));
}

// two adjacent E4M3 channels -> float2 (exact)
template <bool ALIGNED>
__device__ __forceinline__ float2 load_pair_e4m3(const unsigned char* p) {
    if (ALIGNED) return unpack_e4m3x2(*reinterpret_cast<const uint16_t*>(p));
    return unpack_e4m3x2((uint16_t)(p[0] | (p[1] << 8)));
}

template <int K, bool HAS_LO, bool ALIGNED, bool FP8 = false>
__global__ void __launch_bounds__(kGcThreads, 2)
grouped_conv_ffma2_kernel(const GroupedArgs p) {
    constexpr int kRows = kGcTile + K - 1;   // frames in the x tile
    constexpr int kWin = kGcTT + K - 1;      // frames one thread slides over
    constexpr int NT = HAS_LO ? 2 : 1;       // tensors per tile (hi, lo)
    constexpr int E = FP8 ? 1 : 2;           // bytes per element
    constexpr int kVecCh = 16 / E;           // channels per 16-byte vector
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int cin_g = p.C_in / p.groups, cout_g = p.C_out / p.groups;
    const int n_jp = (cin_g + 1) / 2;
    float2* ws = reinterpret_cast<float2*>(smem_raw);                                  // [n_jp][K][kGcCo]
    unsigned char* xs = smem_raw + sizeof(float2) * n_jp * K * kGcCo;                  // [2 buffers][NT][kRows][cols] bf16
    constexpr int tile_bytes = kRows * kGcMaxCols * 2;

    const int tid = threadIdx.x;
    const int co_l = tid % kGcCo, strip = tid / kGcCo;
    const int cb = blockIdx.x, part = blockIdx.y;
    const int co = cb * kGcCo + co_l;
    const bool live = co < p.C_out;
    // input channel window of this channel block, 16-byte aligned on the left
    const int co_last = min(cb * kGcCo + kGcCo, p.C_out) - 1;
    const int ci_first = co_last >= cb * kGcCo ? (cb * kGcCo / cout_g) * cin_g : 0;
    const int ci_end = co_last >= cb * kGcCo ? (co_last / cout_g + 1) * cin_g + 1 : 8;  // +1: pad channel of an odd cin_g
    const int ci_lo = ci_first & ~(kVecCh - 1);
    const int cols = ((ci_end - ci_lo + kVecCh - 1) & ~(kVecCh - 1));
    const int n_vec = cols / kVecCh;
    constexpr int pitch = kGcMaxCols * 2;  // bytes, compile-time: the window loads below use immediate offsets

    // weights -> smem, paired over input channels: ws[jp][k][co] = (w[co][2jp][k], w[co][2jp+1][k] or 0)
    for (int i = tid; i < n_jp * K * kGcCo; i += kGcThreads) {
        const int c = i % kGcCo, k = (i / kGcCo) % K, jp = i / (kGcCo * K);
        const int cg = cb * kGcCo + c;
        float2 v = make_float2(0.f, 0.f);
        if (cg < p.C_out) {
            v.x = p.w[((size_t)cg * cin_g + 2 * jp) * K + k];
            if (2 * jp + 1 < cin_g) v.y = p.w[((size_t)cg * cin_g + 2 * jp + 1) * K + k];
        }
        ws[i] = v;
    }
    const float bv = (live && p.bias) ? p.bias[co] : 0.f;
    const int col0 = live ? (co / cout_g) * cin_g - ci_lo : 0;
    const unsigned char* const xg = reinterpret_cast<const unsigned char*>(p.x);

    const int total_vec = kRows * n_vec;
    auto issue = [&](int item, int buf) {
        const int b = item / p.tiles_per_utt, t0 = (item - b * p.tiles_per_utt) * kGcTile;
        const uint32_t base = smem_u32(xs) + buf * NT * tile_bytes;
#pragma unroll
        for (int v = 0; v < kGcMaxVec; ++v) {
            const int idx = tid + v * kGcThreads;
            if (idx >= total_vec) break;
            const int r = idx / n_vec, cvec = idx - r * n_vec;
            const int u = t0 - p.pad + r, ch = ci_lo + cvec * kVecCh;
            const bool ok = u >= 0 && u < p.T && ch < p.ld_in;
            const size_t off = ok ? ((size_t)b * p.T_rows + u) * p.ld_in + ch : 0;
            const uint32_t dst = base + r * pitch + cvec * 16;
            cp_async_16(dst, xg + off * E, ok);
            if (HAS_LO) cp_async_16(dst + tile_bytes, p.x_lo + off, ok);
        }
        cp_async_commit();
    };

    int item = part, buf = 0;
    if (item < p.n_items) issue(item, 0);
    for (; item < p.n_items; item += p.parts, buf ^= 1) {
        const bool more = item + p.parts < p.n_items;
        if (more) issue(item + p.parts, buf ^ 1);  // lands while this tile is being computed
        if (more) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncthreads();  // tile `buf` is complete for everybody (and, first pass, so are the weights)

        const int b = item / p.tiles_per_utt, t0 = (item - b * p.tiles_per_utt) * kGcTile;
        float2 acc[kGcTT];
#pragma unroll
        for (int i = 0; i < kGcTT; ++i) acc[i] = make_float2(FP8 ? 0.f : bv, 0.f);
        if (live) {
            const unsigned char* xt = xs + buf * NT * tile_bytes + (strip * kGcTT) * pitch + col0 * E;
            for (int jp = 0; jp < n_jp; ++jp) {
                const unsigned char* xr = xt + jp * 2 * E;
                float2 xw[kWin];
#pragma unroll
                for (int m = 0; m < kWin; ++m) {
                    if (FP8) xw[m] = load_pair_e4m3<ALIGNED>(xr + m * pitch);
                    else xw[m] = load_pair<ALIGNED>(xr + m * pitch);
                    if (HAS_LO) {  // split-bf16 ("fp32 tier"): value = hi + lo
                        const float2 l = load_pair<ALIGNED>(xr + tile_bytes + m * pitch);
                        xw[m].x += l.x;
                        xw[m].y += l.y;
                    }
                }
                const float2* wr = ws + (size_t)jp * K * kGcCo + co_l;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const float2 w2 = wr[k * kGcCo];
#pragma unroll
                    for (int i = 0; i < kGcTT; ++i) acc[i] = fma2(w2, xw[i + k], acc[i]);
                }
            }
        }
        if (FP8 && co < p.ld_out) {
            const int t_first = t0 + strip * kGcTT;
            unsigned char* o = reinterpret_cast<unsigned char*>(p.out) + ((size_t)b * p.out_T_rows + t_first) * p.ld_out + co;
            const int n_t = min(kGcTT, p.T - t_first);
#pragma unroll
            for (int i = 0; i < kGcTT; ++i) {
                if (i < n_t) {
                    const float v = live ? (p.relu ? fmaxf(fmaf(acc[i].x + acc[i].y, p.in_scale, bv), 0.f) : fmaf(acc[i].x + acc[i].y, p.in_scale, bv)) : 0.f;
                    o[(size_t)i * p.ld_out] = (unsigned char)(pack_e4m3x2(v * p.out_inv, 0.f) & 0xffu);
                }
            }
        } else if (co < p.ld_out) {
            const int t_first = t0 + strip * kGcTT;
            __nv_bfloat16* o_hi = p.out + ((size_t)b * p.out_T_rows + t_first) * p.ld_out + co;
            __nv_bfloat16* o_lo = HAS_LO && p.out_lo ? p.out_lo + ((size_t)b * p.out_T_rows + t_first) * p.ld_out + co : nullptr;
            const int n_t = min(kGcTT, p.T - t_first);
#pragma unroll
            for (int i = 0; i < kGcTT; ++i) {
                if (i < n_t) {
                    const float v = live ? (p.relu ? fmaxf(acc[i].x + acc[i].y, 0.f) : acc[i].x + acc[i].y) : 0.f;  // padding channels: zeros (the pointwise GEMM contracts over them)
                    const __nv_bfloat16 h = __float2bfloat16_rn(v);
                    o_hi[i * p.ld_out] = h;
                    if (HAS_LO && o_lo) o_lo[i * p.ld_out] = __float2bfloat16_rn(v - __bfloat162float(h));
                }
            }
        }
        __syncthreads();  // everybody is done with tile `buf` before the next iteration refills it
    }
}

static int gc_num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

static size_t grouped_smem_bytes(int cin_g, int K, int cols_max, bool has_lo) {  // (the tile's byte size is the same for E4M3)
    return sizeof(float2) * ((cin_g + 1) / 2) * K * kGcCo + (size_t)2 * (has_lo ? 2 : 1) * (kGcTile + K - 1) * kGcMaxCols * 2;
}

template <int K, bool HAS_LO, bool ALIGNED, bool FP8 = false>
static int launch_grouped_t(const GroupedArgs& a, int n_cb, cudaStream_t stream) {
    const size_t smem = grouped_smem_bytes(a.C_in / a.groups, K, a.cols_max, HAS_LO);
    static size_t smem_set = 0;
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(grouped_conv_ffma2_kernel<K, HAS_LO, ALIGNED, FP8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    grouped_conv_ffma2_kernel<K, HAS_LO, ALIGNED, FP8><<<dim3(n_cb, a.parts), kGcThreads, smem, stream>>>(a);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

template <int K>
static int launch_grouped(const GroupedArgs& a, int n_cb, cudaStream_t stream, bool fp8 = false) {
    const bool aligned = (a.C_in / a.groups) % 2 == 0;
    if (fp8) return aligned ? launch_grouped_t<K, false, true, true>(a, n_cb, stream) : launch_grouped_t<K, false, false, true>(a, n_cb, stream);
    if (a.x_lo) return aligned ? launch_grouped_t<K, true, true>(a, n_cb, stream) : launch_grouped_t<K, true, false>(a, n_cb, stream);
    return aligned ? launch_grouped_t<K, false, true>(a, n_cb, stream) : launch_grouped_t<K, false, false>(a, n_cb, stream);
}

// returns 1 when this shape is not covered (caller runs the generic kernel), 0 on launch, < 0 on error
// fp8: E4M3 act and out (act_lo / out_lo null), x = q * in_scale, stored q = v * out_inv
int grouped_conv_fast(const void* act, const void* act_lo, int B, int T, int T_rows, int C_in, int ld_in, const float* wgt,
                      const float* bias, int C_out, int groups, int k, int pad_left, void* out, void* out_lo,
                      int out_T_rows, int ld_out, int relu, cudaStream_t stream, bool fp8, float in_scale, float out_inv) {
    const int vec_ch = fp8 ? 16 : 8;  // channels per 16-byte vector
    if (ld_in % vec_ch != 0 || C_in % groups != 0 || C_out % groups != 0) return 1;
    const int cin_g = C_in / groups, cout_g = C_out / groups;
    const int n_cb = (ld_out + kGcCo - 1) / kGcCo;
    // widest input window over the channel blocks, and the prefetch budget
    int cols_max = 8;
    for (int cb = 0; cb < n_cb; ++cb) {
        const int co_last = (cb * kGcCo + kGcCo < C_out ? cb * kGcCo + kGcCo : C_out) - 1;
        if (co_last < cb * kGcCo) continue;
        const int ci_first = (cb * kGcCo / cout_g) * cin_g, ci_end = (co_last / cout_g + 1) * cin_g + 1;
        const int cols = ((ci_end - (ci_first & ~(vec_ch - 1))) + vec_ch - 1) & ~(vec_ch - 1);
        cols_max = cols > cols_max ? cols : cols_max;
    }
    if (cols_max * (fp8 ? 1 : 2) > kGcMaxCols * 2) return 1;  // tile row: kGcMaxCols * 2 bytes
    if ((kGcTile + k - 1) * (cols_max / vec_ch) > kGcMaxVec * kGcThreads) return 1;
    const size_t smem = grouped_smem_bytes(cin_g, k, cols_max, act_lo != nullptr);
    if (smem > 200 * 1024) return 1;
    const int ctas_per_sm = smem > 113 * 1024 ? 1 : 2;
    GroupedArgs a{};
    a.x = static_cast<const __nv_bfloat16*>(act); a.x_lo = static_cast<const __nv_bfloat16*>(act_lo); a.w = wgt; a.bias = bias;
    a.out = static_cast<__nv_bfloat16*>(out); a.out_lo = static_cast<__nv_bfloat16*>(out_lo);
    a.B = B; a.T = T; a.T_rows = T_rows; a.C_in = C_in; a.ld_in = ld_in; a.C_out = C_out; a.ld_out = ld_out; a.out_T_rows = out_T_rows;
    a.groups = groups; a.pad = pad_left; a.cols_max = cols_max; a.relu = relu; a.in_scale = in_scale; a.out_inv = out_inv;
    a.tiles_per_utt = (T + kGcTile - 1) / kGcTile;
    a.n_items = B * a.tiles_per_utt;
    // one wave: every CTA must be resident at once (2 per SM), a 297th CTA would run alone afterwards
    int parts = (gc_num_sms() * ctas_per_sm) / n_cb;
    parts = parts < 1 ? 1 : parts;
    a.parts = parts < a.n_items ? parts : a.n_items;
    switch (k) {
        case 3: return launch_grouped<3>(a, n_cb, stream, fp8);
        case 5: return launch_grouped<5>(a, n_cb, stream, fp8);
        case 7: return launch_grouped<7>(a, n_cb, stream, fp8);
        case 9: return launch_grouped<9>(a, n_cb, stream, fp8);
        case 11: return launch_grouped<11>(a, n_cb, stream, fp8);
        case 13: return launch_grouped<13>(a, n_cb, stream, fp8);
        case 15: return launch_grouped<15>(a, n_cb, stream, fp8);
        case 17: return launch_grouped<17>(a, n_cb, stream, fp8);
        case 19: return launch_grouped<19>(a, n_cb, stream, fp8);
        case 21: return launch_grouped<21>(a, n_cb, stream, fp8);
        case 23: return launch_grouped<23>(a, n_cb, stream, fp8);
        case 25: return launch_grouped<25>(a, n_cb, stream, fp8);
        case 27: return launch_grouped<27>(a, n_cb, stream, fp8);
        default: return 1;
    }
}


// ---------------------------------------------------------------------------------------
// Weight / bias gradient of the grouped conv (training of the separable blocks; in the reference this is autograd's
// grouped cudnn wgrad behind loss.backward(), train.py:770-774):
//   dW[co, j, k] = sum_{b,t} dy[b, t, co] * x[b, t + k - pad, g(co) * cin_g + j],   db[co] = sum_{b,t} dy[b, t, co]
// Same tiling as the forward kernel (CTA = 64 output channels x a persistent loop over (utterance, 64-frame) tiles, x tile
// and dy tile staged with cp.async, double buffered).  thread = (output channel, input-channel pair jp, frame-strip
// class): it keeps the K accumulators (float2: even / odd input channel) of its (co, jp) in registers for the whole
// life of the CTA, slides a register window of x over each 16-frame strip, and adds its partial sums to dW with fp32
// atomics once at the end (a few thousand per CTA, spread over all weights).
// ---------------------------------------------------------------------------------------
template <int K, bool HAS_LO>
__global__ void __launch_bounds__(kGcThreads, 1)
grouped_conv_wgrad_kernel(const GroupedArgs p) {
    constexpr int kRows = kGcTile + K - 1;
    constexpr int kWin = kGcTT + K - 1;
    constexpr int NT = HAS_LO ? 2 : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int tile_bytes = kRows * kGcMaxCols * 2;
    constexpr int dy_bytes = kGcTile * kGcCo * 2;
    constexpr int buf_bytes = NT * (tile_bytes + dy_bytes);
    constexpr int pitch = kGcMaxCols * 2;
    const int cin_g = p.C_in / p.groups, cout_g = p.C_out / p.groups;
    const int n_jp = (cin_g + 1) / 2;
    const int ways = n_jp >= 3 ? 1 : (n_jp == 2 ? 2 : 4);  // frame-strip classes per (co, jp) so that all 4 thread rows work
    const int tid = threadIdx.x;
    const int co_l = tid % kGcCo, q = tid / kGcCo;
    const int jp = q % n_jp, fs = q / n_jp;
    const bool worker = q < n_jp * ways && jp < n_jp;
    const int cb = blockIdx.x, part = blockIdx.y;
    const int co = cb * kGcCo + co_l;
    const bool live = co < p.C_out && worker;
    const int co_last = min(cb * kGcCo + kGcCo, p.C_out) - 1;
    const int ci_first = co_last >= cb * kGcCo ? (cb * kGcCo / cout_g) * cin_g : 0;
    const int ci_end = co_last >= cb * kGcCo ? (co_last / cout_g + 1) * cin_g + 1 : 8;
    const int ci_lo = ci_first & ~7;
    const int cols = ((ci_end - ci_lo + 7) & ~7);
    const int n_vec = cols / 8;
    const int col0 = co < p.C_out ? (co / cout_g) * cin_g - ci_lo : 0;
    const int total_vec = kRows * n_vec;
    constexpr int dy_vec = kGcTile * kGcCo / 8;  // 16-byte vectors of the dy tile

    auto issue = [&](int item, int buf) {
        const int b = item / p.tiles_per_utt, t0 = (item - b * p.tiles_per_utt) * kGcTile;
        const uint32_t base = smem_u32(smem_raw) + buf * buf_bytes;
#pragma unroll
        for (int v = 0; v < kGcMaxVec; ++v) {
            const int idx = tid + v * kGcThreads;
            if (idx >= total_vec) break;
            const int r = idx / n_vec, cvec = idx - r * n_vec;
            const int u = t0 - p.pad + r, ch = ci_lo + cvec * 8;
            const bool ok = u >= 0 && u < p.T && ch < p.ld_in;
            const size_t off = ok ? ((size_t)b * p.T_rows + u) * p.ld_in + ch : 0;
            const uint32_t dst = base + r * pitch + cvec * 16;
            cp_async_16(dst, p.x + off, ok);
            if (HAS_LO) cp_async_16(dst + tile_bytes, p.x_lo + off, ok);
        }
        const uint32_t dbase = base + NT * tile_bytes;
#pragma unroll
        for (int v = 0; v < dy_vec / kGcThreads; ++v) {
            const int idx = tid + v * kGcThreads;
            const int r = idx / (kGcCo / 8), cvec = idx - r * (kGcCo / 8);
            const int t = t0 + r, ch = cb * kGcCo + cvec * 8;
            const bool ok = t < p.T && ch < p.ld_dy;
            const size_t off = ok ? ((size_t)b * p.dy_T_rows + t) * p.ld_dy + ch : 0;
            const uint32_t dst = dbase + r * (kGcCo * 2) + cvec * 16;
            cp_async_16(dst, p.dy + off, ok);
            if (HAS_LO) cp_async_16(dst + dy_bytes, p.dy_lo + off, ok);
        }
        cp_async_commit();
    };

    float2 acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = make_float2(0.f, 0.f);
    float bsum = 0.f;

    int item = part, buf = 0;
    if (item < p.n_items) issue(item, 0);
    for (; item < p.n_items; item += p.parts, buf ^= 1) {
        const bool more = item + p.parts < p.n_items;
        if (more) issue(item + p.parts, buf ^ 1);
        if (more) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncthreads();
        if (live) {
            const unsigned char* xt = smem_raw + buf * buf_bytes + col0 * 2 + jp * 4;
            const unsigned char* dt = smem_raw + buf * buf_bytes + NT * tile_bytes + co_l * 2;
            for (int s = fs; s < kGcStrips; s += ways) {
                float d[kGcTT];
#pragma unroll
                for (int i = 0; i < kGcTT; ++i) {
                    const unsigned char* a = dt + (s * kGcTT + i) * (kGcCo * 2);
                    d[i] = __uint_as_float((uint32_t)*reinterpret_cast<const unsigned short*>(a) << 16);
                    if (HAS_LO) d[i] += __uint_as_float((uint32_t)*reinterpret_cast<const unsigned short*>(a + dy_bytes) << 16);
                    if (jp == 0) bsum += d[i];
                }
                float2 xw[kWin];
                const unsigned char* xr = xt + (s * kGcTT) * pitch;
#pragma unroll
                for (int m = 0; m < kWin; ++m) {
                    xw[m] = load_pair<false>(xr + m * pitch);
                    if (HAS_LO) {
                        const float2 l = load_pair<false>(xr + tile_bytes + m * pitch);
                        xw[m].x += l.x;
                        xw[m].y += l.y;
                    }
                }
#pragma unroll
                for (int k = 0; k < K; ++k) {
#pragma unroll
                    for (int i = 0; i < kGcTT; ++i) acc[k] = fma2(make_float2(d[i], d[i]), xw[i + k], acc[k]);
                }
            }
        }
        __syncthreads();
    }
    if (live) {
        float* w0 = p.dw + ((size_t)co * cin_g + 2 * jp) * K;
        const bool odd_ok = 2 * jp + 1 < cin_g;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            atomicAdd(w0 + k, acc[k].x);
            if (odd_ok) atomicAdd(w0 + K + k, acc[k].y);
        }
        if (jp == 0 && p.db != nullptr) atomicAdd(p.db + co, bsum);
    }
}

template <int K>
static int launch_grouped_wgrad(const GroupedArgs& a, int n_cb, cudaStream_t stream) {
    const bool lo = a.x_lo != nullptr;
    const size_t smem = (size_t)2 * (lo ? 2 : 1) * ((kGcTile + K - 1) * kGcMaxCols * 2 + kGcTile * kGcCo * 2);
    static size_t smem_set[2] = {0, 0};
    if (smem > smem_set[lo]) {
        if (lo) CAB_CHECK_CUDA(cudaFuncSetAttribute(grouped_conv_wgrad_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else CAB_CHECK_CUDA(cudaFuncSetAttribute(grouped_conv_wgrad_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set[lo] = smem;
    }
    if (lo) grouped_conv_wgrad_kernel<K, true><<<dim3(n_cb, a.parts), kGcThreads, smem, stream>>>(a);
    else grouped_conv_wgrad_kernel<K, false><<<dim3(n_cb, a.parts), kGcThreads, smem, stream>>>(a);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

}  // namespace cab

using namespace cab;

extern "C" int cab_grouped_conv1d_wgrad(const void* dy, const void* dy_lo, int dy_T_rows, int ld_dy, const void* x, const void* x_lo,
                                        int B, int T, int T_rows, int C_in, int ld_in, int C_out, int groups, int k, int pad_left,
                                        float* dw, float* db, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(dy && x && dw, "null pointer argument");
    CAB_CHECK_ARG((dy_lo == nullptr) == (x_lo == nullptr), "split-bf16 tier needs both dy_lo and x_lo");
    CAB_CHECK_ARG(groups > 0 && C_in % groups == 0 && C_out % groups == 0 && ld_in % 8 == 0 && ld_dy % 8 == 0 && ld_dy >= C_out, "bad grouped conv layout");
    CAB_CHECK_ARG(k % 2 == 1 && pad_left == k / 2, "grouped conv wgrad: odd kernel sizes with 'same' padding only (k=%d pad=%d)", k, pad_left);
    const int cin_g = C_in / groups, cout_g = C_out / groups;
    CAB_CHECK_ARG((cin_g + 1) / 2 <= kGcStrips, "grouped conv wgrad: at most %d input channels per group (got %d)", 2 * kGcStrips, cin_g);
    const int n_cb = (C_out + kGcCo - 1) / kGcCo;
    int cols_max = 8;
    for (int cb = 0; cb < n_cb; ++cb) {
        const int co_last = (cb * kGcCo + kGcCo < C_out ? cb * kGcCo + kGcCo : C_out) - 1;
        const int ci_first = (cb * kGcCo / cout_g) * cin_g, ci_end = (co_last / cout_g + 1) * cin_g + 1;
        const int cols = ((ci_end - (ci_first & ~7)) + 7) & ~7;
        cols_max = cols > cols_max ? cols : cols_max;
    }
    CAB_CHECK_ARG(cols_max <= kGcMaxCols && (kGcTile + k - 1) * (cols_max / 8) <= kGcMaxVec * kGcThreads, "grouped conv wgrad: input window of %d channels per 64 outputs is not covered", cols_max);
    GroupedArgs a{};
    a.x = static_cast<const __nv_bfloat16*>(x); a.x_lo = static_cast<const __nv_bfloat16*>(x_lo);
    a.dy = static_cast<const __nv_bfloat16*>(dy); a.dy_lo = static_cast<const __nv_bfloat16*>(dy_lo); a.ld_dy = ld_dy; a.dy_T_rows = dy_T_rows;
    a.dw = dw; a.db = db;
    a.B = B; a.T = T; a.T_rows = T_rows; a.C_in = C_in; a.ld_in = ld_in; a.C_out = C_out; a.groups = groups; a.pad = pad_left; a.cols_max = cols_max;
    a.tiles_per_utt = (T + kGcTile - 1) / kGcTile;
    a.n_items = B * a.tiles_per_utt;
    int parts = gc_num_sms() / n_cb;  // one CTA per SM (register-heavy), one wave
    parts = parts < 1 ? 1 : parts;
    a.parts = parts < a.n_items ? parts : a.n_items;
    CAB_CHECK_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)C_out * cin_g * k, stream));
    if (db) CAB_CHECK_CUDA(cudaMemsetAsync(db, 0, sizeof(float) * C_out, stream));
    switch (k) {
        case 3: return launch_grouped_wgrad<3>(a, n_cb, stream);
        case 5: return launch_grouped_wgrad<5>(a, n_cb, stream);
        case 7: return launch_grouped_wgrad<7>(a, n_cb, stream);
        case 9: return launch_grouped_wgrad<9>(a, n_cb, stream);
        case 11: return launch_grouped_wgrad<11>(a, n_cb, stream);
        case 13: return launch_grouped_wgrad<13>(a, n_cb, stream);
        case 15: return launch_grouped_wgrad<15>(a, n_cb, stream);
        case 17: return launch_grouped_wgrad<17>(a, n_cb, stream);
        case 19: return launch_grouped_wgrad<19>(a, n_cb, stream);
        case 21: return launch_grouped_wgrad<21>(a, n_cb, stream);
        case 23: return launch_grouped_wgrad<23>(a, n_cb, stream);
        case 25: return launch_grouped_wgrad<25>(a, n_cb, stream);
        case 27: return launch_grouped_wgrad<27>(a, n_cb, stream);
        default: CAB_CHECK_ARG(false, "grouped conv wgrad: kernel size %d has no instantiation (odd 3..27)", k);
    }
    return 0;
}
