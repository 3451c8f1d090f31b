// Log-mel frontend + masked instance norm for sm_100a.
//
// Replaces (reference file:line): normalize_signal models.py:684-686; LogFilterBankFrontend
// .forward models.py:565-597 (pre-emphasis :572, mask :575, reflect/zero pad :577-582, STFT
// :590, power :592-594, mel+eps+log :595); MaskedInstanceNorm1d.forward models.py:694-719 as
// called from JasperNet.forward :298-301.
//
// These stages are HBM/latency bound (SURVEY.md 8d: 57.6 KB per audio second), so there is no
// GEMM here: each warp runs one radix-2 DIF FFT of nfft complex points holding TWO real frames
// (frame A in the real lane, frame B in the imaginary lane), split afterwards with the
// conjugate-symmetry identity.  The mel projection walks only the non-zero band of each
// triangular filter.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

// ------------------------------------------------------------------------------------------
// K1: per-utterance max |x|  (models.py:685)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void absmax_kernel(const T* __restrict__ x, int Tn, float* __restrict__ out) {
    const int b = blockIdx.y;
    const T* row = x + size_t(b) * Tn;
    const int base = blockIdx.x * (256 * 16);
    float m = 0.f;
    constexpr int PER = 16 / sizeof(T);  // elements per 16-byte load
    if ((reinterpret_cast<uintptr_t>(row) & 15) == 0 && base + 256 * 16 <= Tn) {
        // aligned interior block: 16-byte loads, all in flight at once
        const uint4* src = reinterpret_cast<const uint4*>(row + base);
        uint4 v[16 / PER];
#pragma unroll
        for (int k = 0; k < 16 / PER; ++k) v[k] = src[k * 256 + threadIdx.x];
#pragma unroll
        for (int k = 0; k < 16 / PER; ++k) {
            const T* e = reinterpret_cast<const T*>(&v[k]);
#pragma unroll
            for (int j = 0; j < PER; ++j) m = fmaxf(m, fabsf((float)e[j]));
        }
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int i = base + k * 256 + threadIdx.x;
            if (i < Tn) m = fmaxf(m, fabsf((float)row[i]));
        }
    }
    m = warp_max(m);
    __shared__ float sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 8) {
        m = sm[threadIdx.x];
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffu, m, o));
        // non-negative floats order like their bit patterns
        if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(out + b), __float_as_uint(m));
    }
}

// ------------------------------------------------------------------------------------------
// K2-K4: framing + window + FFT + power + mel + log
// ------------------------------------------------------------------------------------------
constexpr int kFrontendWarps = 8;
constexpr int kFramesPerCta = 32;

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

template <int LOG2N>
__device__ __forceinline__ int bitrev(int v) {
    return (int)(__brev((unsigned)v) >> (32 - LOG2N));
}

// In-warp DIF FFT.  Element n = j*32 + lane lives in z[j] of lane `lane`.
// Result: position p holds X[bitrev(p)].
template <int LOG2N>
__device__ __forceinline__ void warp_fft(float2 (&z)[(1 << LOG2N) / 32], const float2* __restrict__ tw,
                                         int lane) {
    constexpr int N = 1 << LOG2N;
    constexpr int PER = N / 32;
    // in-lane stages: spans N/2 ... 32  (j distance h/32)
#pragma unroll
    for (int h = N / 2; h >= 32; h >>= 1) {
        const int jd = h / 32;
        const int tw_mul = (N / 2) / h;  // W_{2h}^r = W_N^{r * N/(2h)}
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            if ((j & jd) == 0) {
                const int r = ((j * 32) & (h - 1)) + lane;  // n mod h, with n = j*32+lane, h >= 32
                float2 a = z[j], b = z[j + jd];
                z[j] = make_float2(a.x + b.x, a.y + b.y);
                float2 d = make_float2(a.x - b.x, a.y - b.y);
                z[j + jd] = cmul(d, tw[r * tw_mul]);
            }
        }
    }
    // cross-lane stages: spans 16 ... 1
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1) {
        const int tw_mul = (N / 2) / h;
        const bool upper = (lane & h) != 0;
        const float2 w = tw[(lane & (h - 1)) * tw_mul];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            float2 mine = z[j];
            float2 other;
            other.x = __shfl_xor_sync(0xffffffffu, mine.x, h);
            other.y = __shfl_xor_sync(0xffffffffu, mine.y, h);
            if (upper) {
                float2 d = make_float2(other.x - mine.x, other.y - mine.y);
                z[j] = cmul(d, w);
            } else {
                z[j] = make_float2(mine.x + other.x, mine.y + other.y);
            }
        }
    }
}

struct FrontendParams {
    const void* signal;
    const float* xlen;
    const float* absmax;
    const float* window;
    const float* mel_fb;
    const int* mel_band;  // [n_mels, 2]: first / one-past-last non-zero bin
    const float2* twiddle;
    float* out;
    int is_int16, B, T, F, win, hop, nfft, n_mels, n_freq;
    int first_off;  // sample index of frame 0, window tap 0:  -(nfft/2) + (nfft-win)/2
    float preemph, log_eps, denom_mult;
    int normalize;
};

// logmel16_kernel modes.  kComputedStats is the one-shot path with per-utterance abs-max and instance-norm statistics;
// kFixedStats multiplies the signal by the caller's scale and emits no statistics; kStream is kFixedStats over per-stream
// staged samples: row b holds samples [base, base + n_staged) of its stream and the CTA tiles start at frame f_first.
enum { kComputedStats = 0, kFixedStats = 1, kStream = 2 };
enum { kRowFirstFrame = 0, kRowFrames, kRowBase, kRowStaged, kRowReflect, kStreamRowInts };

template <int LOG2N>
__global__ void __launch_bounds__(kFrontendWarps * 32)
logmel_kernel(const FrontendParams p) {
    constexpr int N = 1 << LOG2N;
    constexpr int PER = N / 32;
    extern __shared__ float smem_f[];
    const int n_samples = (kFramesPerCta - 1) * p.hop + p.win;
    float* s_e = smem_f;                                  // [n_samples] pre-emphasised signal
    float* s_win = s_e + ((n_samples + 3) & ~3);          // [win]
    float2* s_tw = reinterpret_cast<float2*>(s_win + ((p.win + 3) & ~3));  // [N/2]
    float2* s_z = s_tw + N / 2;                           // [warps][N]
    float* s_pw = reinterpret_cast<float*>(s_z + kFrontendWarps * N);  // [warps][2][n_freq_pad]
    const int nfp = (p.n_freq + 3) & ~3;
    float* s_out = s_pw + kFrontendWarps * 2 * nfp;       // [n_mels][kFramesPerCta+1]

    const int b = blockIdx.y;
    const int f0 = blockIdx.x * kFramesPerCta;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    for (int i = tid; i < p.win; i += blockDim.x) s_win[i] = p.window[i];
    for (int i = tid; i < N / 2; i += blockDim.x) s_tw[i] = p.twiddle[i];

    // ---- stage the pre-emphasised, masked, reflect-padded signal
    int n_valid = p.T;
    if (p.xlen != nullptr) n_valid = min(p.T, frac_len(p.xlen[b], p.T));
    float denom = 1.f;
    if (p.normalize) denom = __fmul_rn(__fadd_rn(p.absmax[b], 1e-5f), p.denom_mult);
    const bool reflect = (p.nfft / 2) < p.T;  // models.py:578: 'constant' pad if pad >= T
    const int start = f0 * p.hop + p.first_off;
    const float* xf = static_cast<const float*>(p.signal) + size_t(b) * p.T;
    const short* xs = static_cast<const short*>(p.signal) + size_t(b) * p.T;
    for (int i = tid; i < n_samples; i += blockDim.x) {
        int n = start + i;
        float e = 0.f;
        bool ok = true;
        if (n < 0) { if (reflect) n = -n; else ok = false; }
        if (ok && n < n_valid) {
            float x1 = p.is_int16 ? (float)xs[n] : xf[n];
            if (p.normalize) x1 = __fdiv_rn(x1, denom);
            if (n > 0 && p.preemph > 0.f) {
                float x0 = p.is_int16 ? (float)xs[n - 1] : xf[n - 1];
                if (p.normalize) x0 = __fdiv_rn(x0, denom);
                e = __fsub_rn(x1, __fmul_rn(p.preemph, x0));
            } else {
                e = x1;
            }
        }
        s_e[i] = e;
    }
    __syncthreads();

    float2* zbuf = s_z + warp * N;
    float* pwA = s_pw + warp * 2 * nfp;
    float* pwB = pwA + nfp;

    for (int pair = warp; pair < kFramesPerCta / 2; pair += kFrontendWarps) {
        const int fa = 2 * pair, fb = 2 * pair + 1;  // local frame indices
        float2 z[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int n = j * 32 + lane;
            float2 v = make_float2(0.f, 0.f);
            if (n < p.win) {
                const float w = s_win[n];
                v.x = w * s_e[fa * p.hop + n];
                v.y = w * s_e[fb * p.hop + n];
            }
            z[j] = v;
        }
        warp_fft<LOG2N>(z, s_tw, lane);
#pragma unroll
        for (int j = 0; j < PER; ++j) zbuf[bitrev<LOG2N>(j * 32 + lane)] = z[j];
        __syncwarp();
        // split the two real spectra: A[k] = (Z[k] + conj Z[N-k]) / 2, B[k] = (Z[k] - conj Z[N-k]) / 2i
        for (int k = lane; k < p.n_freq; k += 32) {
            const float2 zk = zbuf[k];
            const float2 zn = zbuf[(N - k) & (N - 1)];
            const float ar = 0.5f * (zk.x + zn.x), ai = 0.5f * (zk.y - zn.y);
            const float br = 0.5f * (zk.y + zn.y), bi = 0.5f * (zn.x - zk.x);
            pwA[k] = ar * ar + ai * ai;
            pwB[k] = br * br + bi * bi;
        }
        __syncwarp();
        for (int m = lane; m < p.n_mels; m += 32) {
            const int lo = p.mel_band[2 * m], hi = p.mel_band[2 * m + 1];
            const float* mrow = p.mel_fb + size_t(m) * p.n_freq;
            float accA = 0.f, accB = 0.f;
            for (int k = lo; k < hi; ++k) {
                const float w = __ldg(mrow + k);
                accA = fmaf(w, pwA[k], accA);
                accB = fmaf(w, pwB[k], accB);
            }
            s_out[m * (kFramesPerCta + 1) + fa] = logf(accA + p.log_eps);
            s_out[m * (kFramesPerCta + 1) + fb] = logf(accB + p.log_eps);
        }
        __syncwarp();
    }
    __syncthreads();
    // coalesced store: each warp writes rows of kFramesPerCta consecutive frames
    for (int m = warp; m < p.n_mels; m += kFrontendWarps) {
        const int f = f0 + lane;
        if (f < p.F) p.out[(size_t(b) * p.n_mels + m) * p.F + f] = s_out[m * (kFramesPerCta + 1) + lane];
    }
}

// ------------------------------------------------------------------------------------------
// Round 2 frontend (nfft = 256): radix-16 x radix-16 FFT with 16 complex points per lane.
//
// The radix-2 kernel above spends its time in 5 shuffle stages x 8 elements and shared-memory round trips per frame pair
// (ncu r01: issue slots 57 %, DRAM 1.4 %; 157 us for 120 k frames).  Here a HALF-warp transforms one 256-point complex
// sequence (two real frames, one in the real and one in the imaginary lane): lane n2 holds z[16 n1 + n2], runs a 16-point
// FFT over n1 in registers, applies W_256^(n2 k1), the 16 x 16 tile is transposed through padded shared memory (conflict
// free), and lane k1 runs the second 16-point FFT over n2 -- two register FFTs and one transpose per 2 frames, 4 frames
// per warp.  The conjugate-symmetric split needs Z[256 - k]: that lives in lane 16 - k1 at the mirrored position, one
// shuffle per bin.  CTA = 64 frames of one utterance; the raw samples are staged with ONE 1-D bulk async copy
// (cp.async.bulk, mbarrier completion) when the row is 16-byte aligned, and read once.  The log-mel tile leaves through
// shared memory in 256-byte rows, and the masked instance-norm statistics of the tile (count, mean, M2 per mel channel;
// exact two-pass inside the tile) are written as partials that instnorm_pack_partials_kernel combines (Chan) in a fixed order.
// ------------------------------------------------------------------------------------------
constexpr int kPackFrames = 32;
constexpr int kF16Frames = 64;   // frames per CTA
constexpr int kF16Warps = 8;     // 4 frames per warp and pass -> 2 passes

template <int J>  // multiply by W_16^J = exp(-2 pi i J / 16), J in [0, 8)
__device__ __forceinline__ float2 mul_w16(float2 a) {
    constexpr float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, r = 0.70710678118654752f;
    if (J == 0) return a;
    if (J == 4) return make_float2(a.y, -a.x);
    if (J == 2) return make_float2(r * (a.x + a.y), r * (a.y - a.x));
    if (J == 6) return make_float2(r * (a.y - a.x), -r * (a.x + a.y));
    if (J == 1) return make_float2(c1 * a.x + s1 * a.y, c1 * a.y - s1 * a.x);
    if (J == 3) return make_float2(s1 * a.x + c1 * a.y, s1 * a.y - c1 * a.x);
    if (J == 5) return make_float2(-s1 * a.x + c1 * a.y, -s1 * a.y - c1 * a.x);
    return make_float2(-c1 * a.x + s1 * a.y, -c1 * a.y - s1 * a.x);  // J == 7
}
template <int I, int HALF>
__device__ __forceinline__ void bfly16(float2 (&v)[16]) {
    constexpr int j = (I % HALF) * (8 / HALF);  // W_{2 HALF}^(I mod HALF) = W_16^j
    const float2 a = v[I], b = v[I + HALF];
    v[I] = make_float2(a.x + b.x, a.y + b.y);
    v[I + HALF] = mul_w16<j>(make_float2(a.x - b.x, a.y - b.y));
}
// 16-point DIF FFT in registers: natural-order input, position p holds X[bitrev4(p)]
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
    bfly16<0, 8>(v); bfly16<1, 8>(v); bfly16<2, 8>(v); bfly16<3, 8>(v); bfly16<4, 8>(v); bfly16<5, 8>(v); bfly16<6, 8>(v); bfly16<7, 8>(v);
    bfly16<0, 4>(v); bfly16<1, 4>(v); bfly16<2, 4>(v); bfly16<3, 4>(v); bfly16<8, 4>(v); bfly16<9, 4>(v); bfly16<10, 4>(v); bfly16<11, 4>(v);
    bfly16<0, 2>(v); bfly16<1, 2>(v); bfly16<4, 2>(v); bfly16<5, 2>(v); bfly16<8, 2>(v); bfly16<9, 2>(v); bfly16<12, 2>(v); bfly16<13, 2>(v);
    bfly16<0, 1>(v); bfly16<2, 1>(v); bfly16<4, 1>(v); bfly16<6, 1>(v); bfly16<8, 1>(v); bfly16<10, 1>(v); bfly16<12, 1>(v); bfly16<14, 1>(v);
}
__host__ __device__ constexpr int brev4(int p) { return ((p & 1) << 3) | ((p & 2) << 1) | ((p & 4) >> 1) | ((p & 8) >> 3); }

template <int MODE>
__global__ void __launch_bounds__(kF16Warps * 32)
logmel16_kernel(const FrontendParams p, float* __restrict__ partials /* [B][tiles][n_mels][2] mean, M2, or null */, int stats_masked,
                float* __restrict__ stats /* [B][n_mels][2] mean, sd */, unsigned int* __restrict__ done /* [B] zeroed */, float norm_eps,
                const float* __restrict__ scale /* kFixedStats / kStream: the caller's signal scale [B] */,
                const int32_t* __restrict__ stream_rows /* kStream: [B][kStreamRowInts] (cab_frontend_stream) */) {
    constexpr int N = 256;
    extern __shared__ __align__(16) unsigned char smem16[];
    const int n_samples = (kF16Frames - 1) * p.hop + p.win;      // pre-emphasised samples this CTA needs
    const int nfp = 132;                                         // power-spectrum row pitch (129 bins)
    float* s_e = reinterpret_cast<float*>(smem16);                                   // [n_samples]
    float2* s_tw = reinterpret_cast<float2*>(s_e + ((n_samples + 3) & ~3));          // [128]  W_256^r
    float2* s_tr = s_tw + 128;                                                        // [warps][2][16][17] transpose tiles
    float* s_pw = reinterpret_cast<float*>(s_tr + kF16Warps * 2 * 16 * 17);          // [warps][4][nfp]
    float* s_out = s_pw + kF16Warps * 4 * nfp;                                        // [n_mels][kF16Frames + 1]
    unsigned char* s_raw = reinterpret_cast<unsigned char*>(s_out + p.n_mels * (kF16Frames + 1));  // raw samples (bulk copy target), 16-byte aligned
    s_raw = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(s_raw) + 15) & ~uintptr_t(15));
    __shared__ uint64_t bar;

    const int b = blockIdx.y;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int esz = p.is_int16 ? 2 : 4;
    // kStream: sample indices below are relative to the row's first staged sample (base); frames with a negative start
    // are only emitted while base == 0, so the reflected head is addressed exactly as in the one-shot row
    const int32_t* srow = MODE == kStream ? stream_rows + b * kStreamRowInts : nullptr;
    const int f0 = blockIdx.x * kF16Frames + (MODE == kStream ? srow[kRowFirstFrame] : 0);
    const int start = f0 * p.hop + p.first_off - (MODE == kStream ? srow[kRowBase] : 0);  // sample index of s_e[0] (may be negative: reflect)
    // raw window [r0, r1): everything s_e needs, incl. the sample before (pre-emphasis) and the reflected head
    const bool reflect = MODE == kStream ? srow[kRowReflect] != 0 : (p.nfft / 2) < p.T;
    int r0 = start - 1, r1 = start + n_samples;
    if (start < 0) { r0 = 0; r1 = max(r1, -start + 1); }
    r0 = max(r0, 0); r1 = min(r1, p.T);
    const unsigned char* rowp = static_cast<const unsigned char*>(p.signal) + (size_t)b * p.T * esz;
    // bulk-copy path: 16-byte aligned source and size (round the window outwards inside the row)
    const uintptr_t row_addr = reinterpret_cast<uintptr_t>(rowp);
    const int a0 = (int)(((row_addr + (size_t)r0 * esz) & ~uintptr_t(15)) - row_addr) / esz;  // may be < r0 (never < 0 when the row is aligned)
    const bool row_aligned = (row_addr & 15) == 0 && ((size_t)p.T * esz) % 16 == 0;
    int c0 = r0, c1 = r1;
    if (row_aligned) {
        c0 = a0;
        const int per16 = 16 / esz;
        c1 = min(p.T, (r1 + per16 - 1) / per16 * per16);
    }
    const int n_copy = max(c1 - c0, 0);
    const bool bulk = row_aligned && n_copy > 0 && ((size_t)n_copy * esz) % 16 == 0 && n_copy <= n_samples + 24;  // the staging buffer holds n_samples + 32 elements
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (bulk && tid == 0) {
        mbar_expect_tx(&bar, (uint32_t)(n_copy * esz));
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(s_raw)), "l"(rowp + (size_t)c0 * esz), "r"((uint32_t)(n_copy * esz)), "r"(smem_u32(&bar)) : "memory");
    }
    for (int i = tid; i < 128; i += blockDim.x) s_tw[i] = p.twiddle[i];
    // this lane's window taps: n = 16 n1 + n2
    const int n2 = lane & 15, half = lane >> 4;
    float wv[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
        const int n = 16 * n1 + n2;
        wv[n1] = n < p.win ? __ldg(p.window + n) : 0.f;
    }
    __syncthreads();  // s_tw
    // this lane's inter-stage twiddles W_256^(n2 * k1), k1 = brev4(q): registers for the whole CTA
    float2 tw[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int r = n2 * brev4(q);  // <= 225: W^r = -W^(r - 128) beyond the table
        float2 w = s_tw[r & 127];
        if (r & 128) { w.x = -w.x; w.y = -w.y; }
        tw[q] = w;
    }
    int n_valid = p.T;
    if (MODE == kStream) n_valid = srow[kRowStaged];
    else if (p.xlen != nullptr) n_valid = min(p.T, frac_len(p.xlen[b], p.T));
    float denom = 1.f;
    if (MODE == kComputedStats && p.normalize) denom = __fmul_rn(__fadd_rn(p.absmax[b], 1e-5f), p.denom_mult);
    if (bulk) mbar_wait(&bar, 0);
    auto raw = [&](int n) -> float {  // sample n of this row, n in [0, T)
        if (bulk) return p.is_int16 ? (float)reinterpret_cast<const short*>(s_raw)[n - c0] : reinterpret_cast<const float*>(s_raw)[n - c0];
        return p.is_int16 ? (float)reinterpret_cast<const short*>(rowp)[n] : reinterpret_cast<const float*>(rowp)[n];
    };
    // pre-emphasised, masked, reflect-padded signal: e[n] = s[n] - preemph * s[n-1], s = x / denom (models.py:570-575).  The
    // division is a multiplication by the reciprocal here (<= 1 ulp from the reference's quotient, far inside the 2e-4
    // log-mel bar; two IEEE divisions per sample were a quarter of this kernel's instructions)
    const float inv_denom = MODE != kComputedStats ? scale[b] : p.normalize ? __frcp_rn(denom) : 1.f;
    // fast path (int16, bulk-staged, interior tile): 8 consecutive samples per thread from one 16-byte shared-memory load
    // plus the sample before; the group is aligned because start - c0 is a multiple of 8 there
    const bool fast = bulk && p.is_int16 && start >= 8 && ((start - c0) & 7) == 0 && p.preemph > 0.f;
    const int n_fast = fast ? (max(0, min(n_samples, n_valid - start)) & ~7) : 0;  // whole groups inside the valid signal
    for (int i0 = tid * 8; i0 < n_fast; i0 += blockDim.x * 8) {
        const short* src = reinterpret_cast<const short*>(s_raw) + (start + i0 - c0);
        const uint4 v = *reinterpret_cast<const uint4*>(src);
        const short* e8 = reinterpret_cast<const short*>(&v);
        float prev = (float)src[-1] * inv_denom;
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float x = (float)e8[j] * inv_denom;
            o[j] = __fsub_rn(x, __fmul_rn(p.preemph, prev));
            prev = x;
        }
        *reinterpret_cast<float4*>(s_e + i0) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(s_e + i0 + 4) = make_float4(o[4], o[5], o[6], o[7]);
    }
    for (int i = n_fast + tid; i < n_samples; i += blockDim.x) {
        int n = start + i;
        float e = 0.f;
        bool ok = true;
        if (n < 0) { if (reflect) n = -n; else ok = false; }
        if (ok && n < n_valid) {
            const float x1 = raw(n) * inv_denom;
            e = (n > 0 && p.preemph > 0.f) ? __fsub_rn(x1, __fmul_rn(p.preemph, raw(n - 1) * inv_denom)) : x1;
        }
        s_e[i] = e;
    }
    __syncthreads();

    float2* tr = s_tr + (warp * 2 + half) * 16 * 17;
    float* pw = s_pw + warp * 4 * nfp;
    const int partner = (half << 4) | ((16 - n2) & 15);
    for (int pass = 0; pass < kF16Frames / (4 * kF16Warps); ++pass) {
        const int fa = pass * 4 * kF16Warps + warp * 4 + half * 2;  // local frame of the real lane; fa + 1 rides in the imaginary lane
        float2 v[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const int n = 16 * n1 + n2;
            float2 z = make_float2(0.f, 0.f);
            if (n < p.win) {
                z.x = wv[n1] * s_e[fa * p.hop + n];
                z.y = wv[n1] * s_e[(fa + 1) * p.hop + n];
            }
            v[n1] = z;
        }
        fft16(v);  // over n1: position q holds Y[k1 = brev4(q)][n2]
#pragma unroll
        for (int q = 0; q < 16; ++q) tr[brev4(q) * 17 + n2] = cmul(v[q], tw[q]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = tr[n2 * 17 + j];  // this lane is now k1 = n2: all 16 n2' of its row
        __syncwarp();
        fft16(v);  // over n2: position q holds Z[k1 + 16 * brev4(q)]
        // bins k = k1 + 16 k2 <= 128: k2 = 0..7 (even positions), and k = 128 for k1 == 0 (position 1)
        const int k1 = n2;
#pragma unroll
        for (int k2 = 0; k2 <= 8; ++k2) {
            const int q = brev4(k2);
            // Z[256 - k]: lane 16 - k1 at position 15 - q; for k1 == 0 this lane at position brev4((16 - k2) % 16)
            const float2 mirror = v[15 - q];
            float2 zp;
            zp.x = __shfl_sync(0xffffffffu, mirror.x, partner);
            zp.y = __shfl_sync(0xffffffffu, mirror.y, partner);
            if (k1 == 0) zp = v[brev4((16 - k2) & 15)];
            if (k2 == 8 && k1 != 0) continue;
            const float2 zk = v[q];
            const float ar = 0.5f * (zk.x + zp.x), ai = 0.5f * (zk.y - zp.y);
            const float br = 0.5f * (zk.y + zp.y), bi = 0.5f * (zp.x - zk.x);
            const int k = k1 + 16 * k2;
            pw[(half * 2) * nfp + k] = ar * ar + ai * ai;
            pw[(half * 2 + 1) * nfp + k] = br * br + bi * bi;
        }
        __syncwarp();
        // mel projection over the non-zero band of each filter, 4 frames per warp
        const int fw = pass * 4 * kF16Warps + warp * 4;
        for (int m = lane; m < p.n_mels; m += 32) {
            const int lo = p.mel_band[2 * m], hi = p.mel_band[2 * m + 1];
            const float* mrow = p.mel_fb + size_t(m) * p.n_freq;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int k = lo; k < hi; ++k) {
                const float w = __ldg(mrow + k);
#pragma unroll
                for (int f = 0; f < 4; ++f) acc[f] = fmaf(w, pw[f * nfp + k], acc[f]);
            }
#pragma unroll
            for (int f = 0; f < 4; ++f) s_out[m * (kF16Frames + 1) + fw + f] = __logf(acc[f] + p.log_eps);  // lg2.approx * ln 2: abs error ~1e-6 in the log
        }
        __syncwarp();
    }
    __syncthreads();
    // coalesced store of the tile + instance-norm partials (valid frames only; exact two-pass inside the tile)
    int F_valid = p.F;
    if (p.xlen != nullptr && stats_masked) F_valid = min(p.F, frac_len(p.xlen[b], p.F));
    const int n_here = max(0, min(kF16Frames, F_valid - f0));
    // stores: a half-warp writes the 64 frames of one mel row (256 contiguous bytes); kStream rows start at their first new frame
    {
        const int fo = MODE == kStream ? blockIdx.x * kF16Frames : f0;
        float* outb = p.out + size_t(b) * p.n_mels * p.F + fo;
        const int c4 = (tid & 15) * 4, r0_ = tid >> 4;
        for (int m = r0_; m < p.n_mels; m += (kF16Warps * 32) >> 4) {
            const float* rowv = s_out + m * (kF16Frames + 1) + c4;
            float* dst = outb + size_t(m) * p.F + c4;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (fo + c4 + j < p.F) dst[j] = rowv[j];
        }
    }
    if constexpr (MODE != kComputedStats) return;
    // statistics: one thread per mel channel walks its row twice (exact two-pass mean / centred second moment)
    for (int mch = tid; partials != nullptr && mch < p.n_mels; mch += blockDim.x) {
        const float* rowv = s_out + mch * (kF16Frames + 1);
        float sum = 0.f;
        for (int i = 0; i < n_here; ++i) sum += rowv[i];
        const float mean = n_here > 0 ? sum / (float)n_here : 0.f;
        float q = 0.f;
        for (int i = 0; i < n_here; ++i) {
            const float d = rowv[i] - mean;
            q = fmaf(d, d, q);
        }
        float* dst = partials + ((size_t(b) * gridDim.x + blockIdx.x) * p.n_mels + mch) * 2;
        dst[0] = mean;
        dst[1] = q;
    }
    if (partials == nullptr) return;
    // the LAST CTA of this utterance to finish combines the per-tile partials (count, mean, M2) in TILE order (Chan et al.):
    // the result does not depend on which CTA does it -- deterministic, and as accurate as the reference's
    // mean -> centred second moment (models.py:715-718)
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(done + b, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int n_tiles = gridDim.x;
    for (int c = tid; c < p.n_mels; c += blockDim.x) {
        float cnt = 0.f, mean = 0.f, m2 = 0.f;
        for (int t = 0; t < n_tiles; ++t) {
            const float nb = (float)max(0, min(kF16Frames, F_valid - t * kF16Frames));
            if (nb <= 0.f) break;
            const volatile float* src = partials + ((size_t(b) * n_tiles + t) * p.n_mels + c) * 2;
            const float mb = src[0], qb = src[1];
            const float tot = cnt + nb, delta = mb - mean;
            mean += delta * (nb / tot);
            m2 += qb + delta * delta * (cnt * nb / tot);
            cnt = tot;
        }
        stats[2 * (b * p.n_mels + c)] = mean;
        stats[2 * (b * p.n_mels + c) + 1] = sqrtf(m2 / fmaxf(cnt, 1.f) + norm_eps);
    }
}

// ------------------------------------------------------------------------------------------
// K5: masked instance norm statistics + normalise/transpose/pack
// ------------------------------------------------------------------------------------------
// one warp per (b, c): two passes over the (L2-resident) row, exactly the reference's
// mean -> centred sum of squares order (models.py:715-718 / :704-709).
__global__ void instnorm_stats_kernel(const float* __restrict__ feat, const float* __restrict__ xlen,
                                      int B, int C, int F, float eps, float* __restrict__ stats) {
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= B * C) return;
    const int b = gw / C;
    int n = F;
    if (xlen != nullptr) n = min(F, frac_len(xlen[b], F));
    const float* row = feat + size_t(gw) * F;
    float s = 0.f;
    for (int i = lane; i < n; i += 32) s += row[i];
    s = warp_sum(s);
    const float mean = s / (float)n;
    float q = 0.f;
    for (int i = lane; i < n; i += 32) {
        const float d = row[i] - mean;
        q = fmaf(d, d, q);
    }
    q = warp_sum(q);
    const float sd = sqrtf(q / (float)n + eps);
    if (lane == 0) {
        stats[2 * gw] = mean;
        stats[2 * gw + 1] = sd;
    }
}

// FIXED: stats holds the caller's (mean, invstd) per (b, c) and the kernel multiplies by invstd; otherwise (mean, sd) as
// computed by the statistics kernels, divided by
template <bool FIXED>
__global__ void __launch_bounds__(256)
instnorm_pack_kernel(const float* __restrict__ feat, const float* __restrict__ xlen,
                     const float* __restrict__ stats, int B, int C, int F, int F_pad, int C_pad,
                     __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo,
                     float* __restrict__ out_f32, int normalize) {
    extern __shared__ float tile[];  // [kPackFrames][C_pad + 1]
    const int b = blockIdx.y;
    const int f0 = blockIdx.x * kPackFrames;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int n = F;
    if (xlen != nullptr) n = min(F, frac_len(xlen[b], F));
    const int ldt = C_pad + 1;
    for (int c = warp; c < C_pad; c += 8) {
        const int f = f0 + lane;
        float v = 0.f;
        if (c < C && f < n) {
            v = feat[(size_t(b) * C + c) * F + f];
            if (normalize) {
                const float mean = stats[2 * (b * C + c)], sd = stats[2 * (b * C + c) + 1];
                if constexpr (FIXED) v = __fmul_rn(v - mean, sd);
                else v = __fdiv_rn(v - mean, sd);
            }
        }
        if (out_f32 != nullptr && c < C && f < F) out_f32[(size_t(b) * C + c) * F + f] = v;
        tile[lane * ldt + c] = v;
    }
    __syncthreads();
    if (C_pad % 8 == 0) {  // 16-byte stores: 8 channels per thread
        const int vecs = C_pad / 8;
        for (int i = threadIdx.x; i < kPackFrames * vecs; i += blockDim.x) {
            const int fl = i / vecs, cv = i - fl * vecs;
            const int f = f0 + fl;
            if (f >= F_pad) continue;
            float x[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) x[e] = tile[fl * ldt + cv * 8 + e];
            const uint4 hi = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
            const size_t o = (size_t(b) * F_pad + f) * C_pad + cv * 8;
            if (out_hi != nullptr) *reinterpret_cast<uint4*>(out_hi + o) = hi;
            if (out_lo != nullptr) {
                const uint32_t hw[4] = {hi.x, hi.y, hi.z, hi.w};
                uint32_t lw[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 h = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hw[e]));
                    lw[e] = pack_bf16x2(x[2 * e] - h.x, x[2 * e + 1] - h.y);
                }
                *reinterpret_cast<uint4*>(out_lo + o) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
        }
        return;
    }
    for (int i = threadIdx.x; i < kPackFrames * C_pad; i += blockDim.x) {
        const int fl = i / C_pad, c = i - fl * C_pad;
        const int f = f0 + fl;
        if (f < F_pad) {
            const float v = tile[fl * ldt + c];
            const __nv_bfloat16 h = __float2bfloat16_rn(v);
            const size_t o = (size_t(b) * F_pad + f) * C_pad + c;
            if (out_hi != nullptr) out_hi[o] = h;
            if (out_lo != nullptr) out_lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
        }
    }
}

// which STFT kernel: the radix-16 x radix-16 kernel covers nfft = 256 with windows of at most 256 samples; every other
// nfft or longer window runs the radix-2 logmel_kernel
static bool use_fft16(int nfft, int win, int hop) {
    return nfft == 256 && win <= 256 && hop > 0;
}

static size_t fft16_smem_bytes(int win, int hop, int n_mels) {
    const int n_samples = (kF16Frames - 1) * hop + win;
    return sizeof(float) * (size_t)((n_samples + 3) & ~3) + sizeof(float2) * 128 + sizeof(float2) * kF16Warps * 2 * 16 * 17 + sizeof(float) * kF16Warps * 4 * 132 +
           sizeof(float) * (size_t)n_mels * (kF16Frames + 1) + 16 + sizeof(float) * (size_t)(n_samples + 32);
}

template <int MODE = kComputedStats>
static int launch_logmel16(const FrontendParams& p, float* partials, int stats_masked, float* stats, unsigned int* done, float norm_eps, cudaStream_t stream,
                           const float* scale = nullptr, const int32_t* stream_rows = nullptr) {
    const size_t smem = fft16_smem_bytes(p.win, p.hop, p.n_mels);
    CAB_CHECK_ARG(smem <= 200 * 1024, "frontend tile does not fit shared memory (win=%d hop=%d)", p.win, p.hop);
    static size_t smem_set = 0;  // one per mode
    if (smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(logmel16_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    dim3 grid((p.F + kF16Frames - 1) / kF16Frames, p.B);
    logmel16_kernel<MODE><<<grid, kF16Warps * 32, smem, stream>>>(p, partials, stats_masked, stats, done, norm_eps, scale, stream_rows);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

}  // namespace cab

using namespace cab;

extern "C" int cab_frontend_logmel(const void* signal, int signal_is_int16, const float* xlen_frac,
                                   int B, int T, int win_length, int hop, int nfft, int n_mels,
                                   const float* window, const float* mel_fb, const int32_t* mel_band,
                                   const float* twiddle, float preemphasis, float log_eps,
                                   int normalize_signal, float denom_multiplier, float* out_logmel,
                                   float* ws_absmax, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(signal && window && mel_fb && mel_band && twiddle && out_logmel, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && T > 0, "bad shape B=%d T=%d", B, T);
    CAB_CHECK_ARG(nfft == 256 || nfft == 512 || nfft == 1024, "nfft=%d unsupported (256/512/1024)", nfft);
    CAB_CHECK_ARG(win_length > 0 && win_length <= nfft && hop > 0, "bad window %d / hop %d", win_length, hop);
    CAB_CHECK_ARG(!normalize_signal || ws_absmax, "ws_absmax required when normalize_signal");
    const int F = T / hop + 1;

    if (normalize_signal) {
        CAB_CHECK_CUDA(cudaMemsetAsync(ws_absmax, 0, sizeof(float) * B, stream));
        dim3 grid((T + 256 * 16 - 1) / (256 * 16), B);
        if (signal_is_int16)
            absmax_kernel<short><<<grid, 256, 0, stream>>>(static_cast<const short*>(signal), T, ws_absmax);
        else
            absmax_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(signal), T, ws_absmax);
        CAB_CHECK_LAUNCH();
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
    }

    FrontendParams p;
    p.signal = signal; p.xlen = xlen_frac; p.absmax = ws_absmax; p.window = window;
    p.mel_fb = mel_fb; p.mel_band = mel_band; p.twiddle = reinterpret_cast<const float2*>(twiddle);
    p.out = out_logmel; p.is_int16 = signal_is_int16; p.B = B; p.T = T; p.F = F;
    p.win = win_length; p.hop = hop; p.nfft = nfft; p.n_mels = n_mels; p.n_freq = nfft / 2 + 1;
    p.first_off = -(nfft / 2) + (nfft - win_length) / 2;
    p.preemph = preemphasis; p.log_eps = log_eps; p.denom_mult = denom_multiplier;
    p.normalize = normalize_signal;

    if (use_fft16(nfft, win_length, hop)) return launch_logmel16(p, nullptr, 0, nullptr, nullptr, 0.f, stream);
    const int n_samples = (kFramesPerCta - 1) * hop + win_length;
    const int nfp = (p.n_freq + 3) & ~3;
    size_t smem = sizeof(float) * (((n_samples + 3) & ~3) + ((win_length + 3) & ~3)) +
                  sizeof(float2) * (nfft / 2 + kFrontendWarps * nfft) +
                  sizeof(float) * (kFrontendWarps * 2 * nfp + n_mels * (kFramesPerCta + 1));
    dim3 grid((F + kFramesPerCta - 1) / kFramesPerCta, B);
    auto launch = [&](auto kern) -> int {
        static size_t smem_set = 0;  // one static per kernel instantiation (generic lambda)
        if (smem > smem_set) {
            CAB_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            smem_set = smem;
        }
        kern<<<grid, kFrontendWarps * 32, smem, stream>>>(p);
        CAB_CHECK_LAUNCH();
        return 0;
    };
    int rc = nfft == 256 ? launch(logmel_kernel<8>) : nfft == 512 ? launch(logmel_kernel<9>) : launch(logmel_kernel<10>);
    if (rc) return rc;
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// frontend + masked instance norm + layout change as three launches that touch every byte once or twice:
//   absmax (16-byte loads) -> logmel16 (bulk-staged samples, register FFTs, log-mel tile + per-tile statistics) ->
//   pack (statistics combined from the partials, normalise, transpose, bf16 hi [+ lo] channels-last)
extern "C" int cab_frontend_features(const void* signal, int signal_is_int16, const float* xlen_frac, int B, int T, int win_length,
                                     int hop, int nfft, int n_mels, const float* window, const float* mel_fb, const int32_t* mel_band,
                                     const float* twiddle, float preemphasis, float log_eps, int normalize_signal, float denom_multiplier,
                                     int normalize_features, int norm_masked, float norm_eps, float* ws_logmel, int F_pad, int C_pad,
                                     void* out_hi, void* out_lo, float* out_f32, float* ws_absmax, float* ws_partials,
                                     cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(signal && window && mel_fb && mel_band && twiddle && ws_logmel, "null pointer argument");
    CAB_CHECK_ARG(out_hi || out_f32, "no output requested");
    CAB_CHECK_ARG(B > 0 && T > 0, "bad shape B=%d T=%d", B, T);
    const int F = T / hop + 1;
    CAB_CHECK_ARG(F_pad >= F && C_pad >= n_mels && C_pad % 8 == 0, "bad output layout F_pad=%d C_pad=%d", F_pad, C_pad);
    if (!use_fft16(nfft, win_length, hop)) {
        // round-1 path (also other FFT sizes): log-mel, then statistics + pack
        int rc = cab_frontend_logmel(signal, signal_is_int16, xlen_frac, B, T, win_length, hop, nfft, n_mels, window, mel_fb, mel_band, twiddle,
                                     preemphasis, log_eps, normalize_signal, denom_multiplier, ws_logmel, ws_absmax, stream_);
        if (rc) return rc;
        CAB_CHECK_ARG(ws_partials != nullptr, "ws_partials (>= B * n_mels * 2 floats) required");
        return cab_instnorm_pack(ws_logmel, norm_masked ? xlen_frac : nullptr, B, n_mels, F, norm_eps, normalize_features, F_pad, C_pad, out_hi, out_lo, out_f32, ws_partials, stream_);
    }
    CAB_CHECK_ARG(ws_absmax != nullptr, "ws_absmax (2 * B floats) required");
    CAB_CHECK_ARG(!normalize_features || ws_partials, "ws_partials required when normalize_features");
    // ws_absmax: [B] abs-max, then [B] per-utterance completion counters of the statistics combine
    CAB_CHECK_CUDA(cudaMemsetAsync(ws_absmax, 0, sizeof(float) * 2 * B, stream));
    if (normalize_signal) {
        dim3 grid((T + 256 * 16 - 1) / (256 * 16), B);
        if (signal_is_int16) absmax_kernel<short><<<grid, 256, 0, stream>>>(static_cast<const short*>(signal), T, ws_absmax);
        else absmax_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(signal), T, ws_absmax);
        CAB_CHECK_LAUNCH();
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
    }
    FrontendParams p;
    p.signal = signal; p.xlen = xlen_frac; p.absmax = ws_absmax; p.window = window;
    p.mel_fb = mel_fb; p.mel_band = mel_band; p.twiddle = reinterpret_cast<const float2*>(twiddle);
    p.out = ws_logmel; p.is_int16 = signal_is_int16; p.B = B; p.T = T; p.F = F;
    p.win = win_length; p.hop = hop; p.nfft = nfft; p.n_mels = n_mels; p.n_freq = nfft / 2 + 1;
    p.first_off = -(nfft / 2) + (nfft - win_length) / 2;
    p.preemph = preemphasis; p.log_eps = log_eps; p.denom_mult = denom_multiplier;
    p.normalize = normalize_signal;
    const int n_tiles = (F + kF16Frames - 1) / kF16Frames;
    // ws_partials: [B][n_tiles][n_mels][2] per-tile partials, then [B][n_mels][2] combined (mean, sd)
    float* stats = normalize_features ? ws_partials + (size_t)B * n_tiles * n_mels * 2 : nullptr;
    if (int rc = launch_logmel16(p, normalize_features ? ws_partials : nullptr, norm_masked, stats, reinterpret_cast<unsigned int*>(ws_absmax + B), norm_eps, stream)) return rc;
    dim3 grid((F_pad + kPackFrames - 1) / kPackFrames, B);
    const size_t smem = sizeof(float) * kPackFrames * (C_pad + 1);
    CAB_CHECK_ARG(smem <= 48 * 1024, "C_pad=%d too large for the pack tile", C_pad);
    instnorm_pack_kernel<false><<<grid, 256, smem, stream>>>(ws_logmel, (normalize_features && norm_masked) ? xlen_frac : nullptr, stats, B, n_mels, F, F_pad, C_pad, static_cast<__nv_bfloat16*>(out_hi),
                                                      static_cast<__nv_bfloat16*>(out_lo), out_f32, normalize_features);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// frontend + instance norm under fixed normalisation (cab_frontend_features_fixed): the same STFT / mel / log kernel with
// the caller's signal scale, then the pack with the caller's (mean, invstd).  Two launches, no statistics.
static int frontend_fixed_params(FrontendParams& p, int B, int T, int F, int win_length, int hop, int nfft, int n_mels, const float* window,
                                 const float* mel_fb, const int32_t* mel_band, const float* twiddle, float preemphasis, float log_eps,
                                 float* ws_logmel) {
    CAB_CHECK_ARG(window && mel_fb && mel_band && twiddle && ws_logmel, "null pointer argument");
    CAB_CHECK_ARG(use_fft16(nfft, win_length, hop), "fixed normalisation and streaming cover the nfft = 256 frontend only (nfft=%d win=%d hop=%d)", nfft, win_length, hop);
    p = FrontendParams{};
    p.window = window; p.mel_fb = mel_fb; p.mel_band = mel_band; p.twiddle = reinterpret_cast<const float2*>(twiddle);
    p.out = ws_logmel; p.B = B; p.T = T; p.F = F;
    p.win = win_length; p.hop = hop; p.nfft = nfft; p.n_mels = n_mels; p.n_freq = nfft / 2 + 1;
    p.first_off = -(nfft / 2) + (nfft - win_length) / 2;
    p.preemph = preemphasis; p.log_eps = log_eps; p.denom_mult = 1.f;
    return 0;
}

static int launch_pack_fixed(const float* logmel, const float* xlen_frac, const float* norm_stats, int B, int C, int F, int F_pad, int C_pad,
                             void* out_hi, void* out_lo, cudaStream_t stream) {
    dim3 grid((F_pad + kPackFrames - 1) / kPackFrames, B);
    const size_t smem = sizeof(float) * kPackFrames * (C_pad + 1);
    CAB_CHECK_ARG(smem <= 48 * 1024, "C_pad=%d too large for the pack tile", C_pad);
    instnorm_pack_kernel<true><<<grid, 256, smem, stream>>>(logmel, xlen_frac, norm_stats, B, C, F, F_pad, C_pad, static_cast<__nv_bfloat16*>(out_hi),
                                                            static_cast<__nv_bfloat16*>(out_lo), nullptr, 1);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_frontend_features_fixed(const void* signal, int signal_is_int16, const float* xlen_frac, int B, int T, int win_length, int hop,
                                           int nfft, int n_mels, const float* window, const float* mel_fb, const int32_t* mel_band,
                                           const float* twiddle, float preemphasis, float log_eps, const float* signal_scale,
                                           const float* norm_stats, int norm_masked, float* ws_logmel, int F_pad, int C_pad, void* out_hi,
                                           void* out_lo, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(signal && signal_scale && norm_stats && out_hi, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && T > 0, "bad shape B=%d T=%d", B, T);
    CAB_CHECK_ARG(hop > 0, "bad hop %d", hop);
    const int F = T / hop + 1;
    CAB_CHECK_ARG(F_pad >= F && C_pad >= n_mels && C_pad % 8 == 0, "bad output layout F_pad=%d C_pad=%d", F_pad, C_pad);
    FrontendParams p;
    if (int rc = frontend_fixed_params(p, B, T, F, win_length, hop, nfft, n_mels, window, mel_fb, mel_band, twiddle, preemphasis, log_eps, ws_logmel)) return rc;
    p.signal = signal; p.xlen = xlen_frac; p.is_int16 = signal_is_int16;
    if (int rc = launch_logmel16<kFixedStats>(p, nullptr, 0, nullptr, nullptr, 0.f, stream, signal_scale)) return rc;
    return launch_pack_fixed(ws_logmel, norm_masked ? xlen_frac : nullptr, norm_stats, B, n_mels, F, F_pad, C_pad, out_hi, out_lo, stream);
}

extern "C" int cab_frontend_stream(const float* staged, int pitch, const int32_t* rows, int B, int F, int win_length, int hop, int nfft,
                                   int n_mels, const float* window, const float* mel_fb, const int32_t* mel_band, const float* twiddle,
                                   float preemphasis, float log_eps, const float* signal_scale, const float* norm_stats, float* ws_logmel,
                                   int C_pad, void* out_hi, void* out_lo, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(staged && rows && signal_scale && norm_stats && out_hi, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && F > 0 && pitch > 0 && pitch % 4 == 0, "bad shape B=%d F=%d pitch=%d (a multiple of 4 samples)", B, F, pitch);
    CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(staged) & 15) == 0, "staged samples must be 16-byte aligned");
    CAB_CHECK_ARG(C_pad >= n_mels && C_pad % 8 == 0, "bad output layout C_pad=%d", C_pad);
    FrontendParams p;
    if (int rc = frontend_fixed_params(p, B, pitch, F, win_length, hop, nfft, n_mels, window, mel_fb, mel_band, twiddle, preemphasis, log_eps, ws_logmel)) return rc;
    p.signal = staged; p.is_int16 = 0;
    if (int rc = launch_logmel16<kStream>(p, nullptr, 0, nullptr, nullptr, 0.f, stream, signal_scale, rows)) return rc;
    return launch_pack_fixed(ws_logmel, nullptr, norm_stats, B, n_mels, F, F, C_pad, out_hi, out_lo, stream);
}

extern "C" int cab_instnorm_pack(const float* feat, const float* xlen_frac, int B, int C, int F,
                                 float eps, int normalize, int F_pad, int C_pad, void* out_hi,
                                 void* out_lo, float* out_f32, float* ws_stats, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(feat && ws_stats, "null pointer argument");
    CAB_CHECK_ARG(out_hi || out_f32, "no output requested");
    CAB_CHECK_ARG(B > 0 && C > 0 && F > 0 && F_pad >= F && C_pad >= C, "bad shape B=%d C=%d F=%d F_pad=%d C_pad=%d", B, C, F, F_pad, C_pad);
    if (normalize) {
        const int warps = B * C;
        const int blocks = (warps * 32 + 255) / 256;
        instnorm_stats_kernel<<<blocks, 256, 0, stream>>>(feat, xlen_frac, B, C, F, eps, ws_stats);
        CAB_CHECK_LAUNCH();
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
    }
    {
        dim3 grid((F_pad + kPackFrames - 1) / kPackFrames, B);
        size_t smem = sizeof(float) * kPackFrames * (C_pad + 1);
        CAB_CHECK_ARG(smem <= 48 * 1024, "C_pad=%d too large for the pack tile", C_pad);
        instnorm_pack_kernel<false><<<grid, 256, smem, stream>>>(feat, xlen_frac, ws_stats, B, C, F, F_pad, C_pad,
                                                          static_cast<__nv_bfloat16*>(out_hi),
                                                          static_cast<__nv_bfloat16*>(out_lo), out_f32, normalize);
        CAB_CHECK_LAUNCH();
        g_launch_count.fetch_add(1, std::memory_order_relaxed);
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// FP8 inference tier: calibration abs-max of a bf16 activation, and the E4M3 quantisation of the packed features
// ------------------------------------------------------------------------------------------
namespace cab {
// 16 elements per thread: two 16-byte bf16 loads -> one 16-byte E4M3 store; q = satfinite(rn(x * scale_inv))
__global__ void quantize_e4m3_kernel(const uint4* __restrict__ x, int64_t n16, float scale_inv, uint4* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 a = x[2 * i], b = x[2 * i + 1];
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t q[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[2 * k]));
            const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[2 * k + 1]));
            q[k] = (uint32_t)pack_e4m3x2(lo.x * scale_inv, lo.y * scale_inv) | ((uint32_t)pack_e4m3x2(hi.x * scale_inv, hi.y * scale_inv) << 16);
        }
        out[i] = make_uint4(q[0], q[1], q[2], q[3]);
    }
}
}  // namespace cab

extern "C" int cab_absmax_bf16(const void* x, int64_t n, float* out, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(x != nullptr && out != nullptr, "null pointer argument");
    CAB_CHECK_ARG(n >= 0 && n <= INT32_MAX, "n=%lld out of [0, 2^31)", (long long)n);
    CAB_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float), stream));
    if (n == 0) return 0;
    const dim3 grid((unsigned)((n + 256 * 16 - 1) / (256 * 16)), 1);
    absmax_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), (int)n, out);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_quantize_e4m3(const void* x, int64_t n, float scale_inv, void* out, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(x != nullptr && out != nullptr, "null pointer argument");
    CAB_CHECK_ARG(n >= 0 && n % 16 == 0, "n=%lld must be a multiple of 16", (long long)n);
    CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "x and out must be 16-byte aligned");
    if (n == 0) return 0;
    const int64_t n16 = n / 16;
    const int64_t blocks = (n16 + 255) / 256;
    quantize_e4m3_kernel<<<(unsigned)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, stream>>>(static_cast<const uint4*>(x), n16, scale_inv,
                                                                                             static_cast<uint4*>(out));
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}
