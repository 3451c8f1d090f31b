// Conv1d (+folded BN) + residual 1x1 convs + activation + temporal mask as one persistent,
// warp-specialised tcgen05/TMEM implicit GEMM for sm_100a.
//
// Replaces (reference file:line): ConvBn1d.forward models.py:127-139 in fuse_conv_bn_eval form
// (:141-151), ConvSamePadding :47-77, ResidualActivation.forward :357-371, temporal mask
// :136-138/:611-619, Decoder :23-44 + log_softmax :316 + argmax transcript_generators.py:27.
//
// Mapping
//   M = 128 consecutive output frames of ONE utterance (tiles never straddle utterances)
//   N = block_n output channels (<= 256, runtime), K = sum over sources/taps of C_in
//   A tile  = x[b, t0 + tap*dil - pad : +128, ci0 : ci0+64]  -- a 3-D TMA box; rows outside
//             [0, T_in) are zero-filled by the TMA unit, which IS the conv zero padding.
//   B tile  = W[tap, n0 : n0+block_n, ci0 : ci0+64]          -- 3-D TMA box, K-major.
//   Both land in shared memory with the 128-byte swizzle and are consumed by
//   tcgen05.mma.cta_group::1.kind::f16 (M=128, N=block_n, K=16) accumulating fp32 in TMEM.
//   TMEM holds two 256-column accumulators so the epilogue of tile i overlaps the MMAs of
//   tile i+1.
//   E4M3 operand mode (conv1d_umma_kernel<true>, cab_conv1d_fused_fp8): the same tiles with 1-byte
//   elements -- a 128-byte swizzle row holds 128 channels, so a stage carries K = 128 and the same four
//   MMAs per row are tcgen05.mma.kind::f8f6f4 with K = 32; the epilogue scales the accumulator by a
//   per-column alpha[n] before the bias, and the activation epilogue stores E4M3 (x 1/s_out, saturating).
// Warp roles (256 threads): warp0 = TMA producer, warp1 = MMA issuer, warp2 = TMEM allocator,
//   warps4-7 = epilogue (TMEM lane quarter = warp_idx % 4).
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <mutex>
#include <atomic>

namespace cab {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // bf16 elements = 128 bytes = one swizzle row
constexpr int kStages = 4;
constexpr int kMaxBlockN = 256;
constexpr int kATileBytes = kBlockM * kBlockK * 2;     // 16 KB
constexpr int kBTileBytes = kMaxBlockN * kBlockK * 2;  // 32 KB
constexpr int kStageBytes = kATileBytes + kBTileBytes;
constexpr int kAccStages = 2;
constexpr int kTmemCols = 512;
constexpr int kNumThreads = 256;
// epilogue staging: bf16 [128 rows][32 cols] tiles (64-byte rows, 64B swizzle) for TMA stores,
// double buffered, one pair for the hi tensor and one for the lo tensor; plus the tile's bias
constexpr int kEpiCols = 32;
constexpr int kEpiTileBytes = kBlockM * kEpiCols * 2;  // 8 KB
constexpr int kOffStageOut = kStages * kStageBytes;    // 4 staging tiles
constexpr int kOffBias = kOffStageOut + 4 * kEpiTileBytes;
constexpr int kOffBars = kOffBias + kMaxBlockN * 4;
constexpr int kSmemBytes = kOffBars + 1024 /*align slack*/ + 256 /*barriers*/;
static_assert(kSmemBytes <= 232448, "exceeds the 227 KB dynamic shared memory limit");

struct SrcDev {
    int a_ch_off, w_ch_off, n_chunks, taps, dil, pad_left;
};

struct alignas(64) ConvParams {
    CUtensorMap amap[CAB_MAX_CONV_SOURCES];
    CUtensorMap wmap[CAB_MAX_CONV_SOURCES];
    CUtensorMap omap_hi, omap_lo;  // bf16 outputs, box {32 ch, 128 rows, 1}, 64B swizzle
    SrcDev src[CAB_MAX_CONV_SOURCES];
    int n_src;
    int B, T_out, C_out, block_n;
    int mtiles_per_b, n_ntiles, n_tiles;
    int epilogue, act;
    float act_a, act_b;
    const float* bias;
    const float* xlen;
    __nv_bfloat16* out_hi;
    __nv_bfloat16* out_lo;
    int out_T_rows, out_ld;
    float* logits;
    float* log_probs;
    int* argmax;
    double* stats;  // [2][C_out] per-channel sum / sum of squares of the stored outputs, or null.  fp64 accumulators: the order of
                    // the atomics then only touches bits far below the fp32 result -- batch statistics are reproducible run to run
    // CAB_EPI_LOGITS_ROWS: fp32 logits in class-contiguous memory [B, T_out, logits_ld] through omap_hi (box {32 fp32, 128 rows}),
    // per-row log-sum-exp and argmax from an online softmax across the N tiles of an M tile (M-tile-major schedule)
    float* lse;
    int mtile_major;
    // rows t >= ceil(skip_frac[b] * skip_T) + skip_margin of utterance b are structural zeros (padding of a
    // ragged batch): M tiles that lie entirely there are not computed, the epilogue stores zeros
    const float* skip_frac;
    int skip_T, skip_margin;
    // BatchNorm-backward reduction folded into a dgrad launch (bf16 tier): this launch produces g = dL/d(out) of a layer whose
    // pre-BatchNorm conv output is `y` (same [B, T_out, out_ld] geometry as the output, read through ymap: box {32 ch, 128 rows},
    // 64B swizzle -- the mirror image of the output store).  After a 32-column chunk of g is staged (bf16-rounded, exactly what
    // the BatchNorm backward will read), the epilogue accumulates sum(dz) and sum(dz * y) per channel, dz = g * act'(y*scale +
    // shift) * (t < len_b), into fp64 partials [CAB_BN_SUM_REPLICAS][2][bnr_C]: the separate reduce pass over (y, g) -- two of the
    // five activation-sized passes of the BatchNorm backward -- disappears.
    CUtensorMap ymap;
    const float* bnr_ss;     // [4][bnr_C]: scale, shift, (mean, invstd)
    const float* bnr_xlen;   // temporal mask of the layer (or null)
    double* bnr_partials;    // null = no fold
    int bnr_C, bnr_act;
    float bnr_a, bnr_b;
    // E4M3 mode: per-column multiplier of the accumulator [C_out], and 1/scale of the stored E4M3 activation
    const float* alpha;
    float out_inv;
};

// Tile schedule.  Only M tiles that hold at least one live row are enumerated ("compacted" index am), so
// the static round-robin over CTAs stays balanced on ragged batches; every role walks the same
// sequence with its own cursor (utterance b owns compacted indices [base, end)).
__device__ __forceinline__ int live_mtiles(const ConvParams& p, int b) {
    if (p.skip_frac == nullptr) return p.mtiles_per_b;
    const int rows = min(p.T_out, frac_len(__ldg(p.skip_frac + b), p.skip_T) + p.skip_margin);
    return rows <= 0 ? 0 : (rows + 127) / 128;
}
// Unit sequence of one CTA.  A unit is a tile (N tile fastest: neighbouring units share the A tile in L2), or -- mtile_major --
// one compacted M tile whose N tiles the CTA then walks in order (the online softmax of the large-vocabulary head needs every
// class of a row in one CTA).  Unit j of this CTA is blockIdx.x + j * gridDim.x; every role walks this sequence on its own
// and derives (am, nt) and its TileCursor position from it.  An atomic-claim schedule, where late CTAs take fewer units, was
// measured 1 % slower on the training step on one B200 and 3 % slower on eight (profiles/r02_tile_schedule_ab.md).
// next (am, nt) of a role's walk; `u` (starts at blockIdx.x - gridDim.x) and `nt_next` (starts at 0) are the role's private state
#define CAB_NEXT_UNIT()                                                        \
    int am, nt;                                                                \
    if (p.mtile_major) {                                                       \
        if (nt_next == 0) u += gridDim.x;                                      \
        am = u;                                                                \
        nt = nt_next;                                                          \
        nt_next = nt_next + 1 == p.n_ntiles ? 0 : nt_next + 1;                 \
    } else {                                                                   \
        u += gridDim.x;                                                        \
        nt = u % p.n_ntiles;                                                   \
        am = u / p.n_ntiles;                                                   \
    }
struct TileCursor {
    int b, base, end;
    __device__ __forceinline__ void init(const ConvParams& p) { b = 0; base = 0; end = live_mtiles(p, 0); }
    __device__ __forceinline__ bool seek(const ConvParams& p, int am) {  // false: past the last utterance
        while (am >= end) {
            if (++b >= p.B) return false;
            base = end;
            end += live_mtiles(p, b);
        }
        return true;
    }
};

__device__ __forceinline__ float apply_act(float x, int act, float a, float b) {
    switch (act) {
        case CAB_ACT_RELU: return fmaxf(x, 0.f);
        case CAB_ACT_HARDTANH: return fminf(fmaxf(x, a), b);
        case CAB_ACT_LEAKY_RELU: return x > 0.f ? x : x * a;
        default: return x;
    }
}

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_bar(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

template <int ACT>
__device__ __forceinline__ float act_t(float x, float a, float b) {
    if (ACT == CAB_ACT_RELU) return fmaxf(x, 0.f);
    if (ACT == CAB_ACT_HARDTANH) return fminf(fmaxf(x, a), b);
    if (ACT == CAB_ACT_LEAKY_RELU) return x > 0.f ? x : x * a;
    return x;
}

// One 32-column chunk of the bf16 epilogue: bias + activation + mask, pack to bf16 (hi, lo),
// write the thread's 64-byte row into the 64B-swizzled staging tile(s).
template <int ACT, bool LO>
__device__ __forceinline__ void epi_chunk(const uint32_t (&v)[32], const float* __restrict__ sb, float a, float b,
                                          bool keep, int row, uint8_t* st_hi, uint8_t* st_lo) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
        float x0 = act_t<ACT>(__uint_as_float(v[j]) + sb[j], a, b);
        float x1 = act_t<ACT>(__uint_as_float(v[j + 1]) + sb[j + 1], a, b);
        if (!keep) { x0 = 0.f; x1 = 0.f; }
        __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
        hi[j >> 1] = *reinterpret_cast<uint32_t*>(&h);
        if (LO) {
            float2 hf = __bfloat1622float2(h);
            lo[j >> 1] = pack_bf16x2(x0 - hf.x, x1 - hf.y);
        }
    }
    // 64-byte rows, 16-byte chunk index XOR ((row >> 1) & 3)  == CU_TENSOR_MAP_SWIZZLE_64B
    const int sw = (row >> 1) & 3;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int off = row * 64 + ((q ^ sw) << 4);
        *reinterpret_cast<uint4*>(st_hi + off) = make_uint4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
        if (LO) *reinterpret_cast<uint4*>(st_lo + off) = make_uint4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
    }
}

// E4M3 twin of epi_chunk: acc * alpha + bias -> activation -> mask -> x 1/s_out -> E4M3 (saturating), the thread's
// 32-byte row into an unswizzled [128 rows][32 B] staging tile.
template <int ACT>
__device__ __forceinline__ void epi_chunk_e4m3(const uint32_t (&v)[32], const float* __restrict__ sb, const float* __restrict__ sa,
                                               float a, float b, bool keep, float inv, int row, uint8_t* st) {
    uint32_t q[8];
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        float x[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            x[i] = act_t<ACT>(fmaf(__uint_as_float(v[j + i]), sa[j + i], sb[j + i]), a, b);
            x[i] = keep ? x[i] * inv : 0.f;
        }
        q[j >> 2] = (uint32_t)pack_e4m3x2(x[0], x[1]) | ((uint32_t)pack_e4m3x2(x[2], x[3]) << 16);
    }
    *reinterpret_cast<uint4*>(st + row * 32) = make_uint4(q[0], q[1], q[2], q[3]);
    *reinterpret_cast<uint4*>(st + row * 32 + 16) = make_uint4(q[4], q[5], q[6], q[7]);
}

// Folded BatchNorm-backward reduction over one staged chunk: g and y are bf16 [128 rows][32 cols] tiles in the 64B-swizzled
// staging layout.  Thread = (column et % 32, row group et / 32): the per-channel coefficients are two scalars, the 32 lanes of
// a warp read the 64 contiguous (swizzled) bytes of one row -- conflict free -- and no cross-lane reduction is needed; the
// four row groups meet in the fp64 atomics.  Same arithmetic per element as bn_stream_kernel<1> (train.cu).
template <int ACT>
__device__ __forceinline__ void bnr_column_pass(const uint8_t* __restrict__ st_g, const uint8_t* __restrict__ st_y, int et, int nrows,
                                                float sc, float sh, float a, float b, float& s_out, float& q_out) {
    const int c = et & 31, rg = et >> 5;
    const int r_end = min(rg * 32 + 32, nrows);
    const int cq = c >> 3, cb = (c & 7) << 1;
    float s = 0.f, q = 0.f;
#pragma unroll 8
    for (int r = rg * 32; r < r_end; ++r) {
        const int off = r * 64 + ((cq ^ ((r >> 1) & 3)) << 4) + cb;
        const float g = __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(st_g + off)) << 16);
        const float y = __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(st_y + off)) << 16);
        const float z = fmaf(y, sc, sh);
        float dz;
        if (ACT == CAB_ACT_RELU) dz = z > 0.f ? g : 0.f;
        else if (ACT == CAB_ACT_HARDTANH) dz = (z > a && z < b) ? g : 0.f;
        else if (ACT == CAB_ACT_LEAKY_RELU) dz = z > 0.f ? g : g * a;
        else dz = g;
        s += dz;
        q = fmaf(dz, y, q);
    }
    s_out = s;
    q_out = q;
}

// Forward batch statistics over one staged chunk, same thread mapping as bnr_column_pass: per-channel sum / sum of squares of
// the stored values (hi [+ lo]) over the tile's rows < nrows.
template <bool LO>
__device__ __forceinline__ void stats_column_pass(const uint8_t* __restrict__ st_h, const uint8_t* __restrict__ st_l, int et, int nrows,
                                                  float& s_out, float& q_out) {
    const int c = et & 31, rg = et >> 5;
    const int r_end = min(rg * 32 + 32, nrows);
    const int cq = c >> 3, cb = (c & 7) << 1;
    float s = 0.f, q = 0.f;
#pragma unroll 8
    for (int r = rg * 32; r < r_end; ++r) {
        const int off = r * 64 + ((cq ^ ((r >> 1) & 3)) << 4) + cb;
        float x = __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(st_h + off)) << 16);
        if (LO) x += __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(st_l + off)) << 16);
        s += x;
        q = fmaf(x, x, q);
    }
    s_out = s;
    q_out = q;
}

// FP8: E4M3 operands (kind::f8f6f4); the stage layout and byte counts are those of the bf16 mode.
template <bool FP8>
__global__ void __launch_bounds__(kNumThreads, 1)
conv1d_umma_kernel(const __grid_constant__ ConvParams p) {
    constexpr int kChunk = FP8 ? 2 * kBlockK : kBlockK;  // channels per 128-byte swizzle row
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment required by the 128B swizzle atoms
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                               ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kOffBars);
    float* s_bias = reinterpret_cast<float*>(smem + kOffBias);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + kAccStages;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + kAccStages);  // 4 bytes in an 8-byte slot
    uint64_t* ybar = tmem_empty + kAccStages + 1;  // [2]: y tiles of the folded BatchNorm-backward reduction

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.n_src; ++s) {
            tma_prefetch_desc(&p.amap[s]);
            tma_prefetch_desc(&p.wmap[s]);
        }
        if (p.epilogue == CAB_EPI_LOGITS_ROWS) tma_prefetch_desc(&p.omap_hi);
        if (p.epilogue == CAB_EPI_ACT_BF16) {
            tma_prefetch_desc(&p.omap_hi);
            if (p.out_lo != nullptr) tma_prefetch_desc(&p.omap_lo);
            if (p.bnr_partials != nullptr) tma_prefetch_desc(&p.ymap);
        }
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < kAccStages; ++i) {
            mbar_init(&tmem_full[i], 1);
            mbar_init(&tmem_empty[i], 4);  // one arrive per epilogue warp
        }
        mbar_init(&ybar[0], 1);
        mbar_init(&ybar[1], 1);
        mbar_fence_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr, kTmemCols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int block_n = p.block_n;
    const uint32_t stage_tx_bytes = kATileBytes + block_n * kBlockK * 2;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            TileCursor cur;
            cur.init(p);
            int u = (int)blockIdx.x - (int)gridDim.x, nt_next = 0;
            for (;;) {
                CAB_NEXT_UNIT()
                if (!cur.seek(p, am)) break;
                const int b = cur.b;
                const int t0 = (am - cur.base) * kBlockM;
                const int n0 = nt * block_n;
                for (int s = 0; s < p.n_src; ++s) {
                    const SrcDev sd = p.src[s];
                    for (int tap = 0; tap < sd.taps; ++tap) {
                        const int trow = t0 + tap * sd.dil - sd.pad_left;
                        for (int ch = 0; ch < sd.n_chunks; ++ch) {
                            mbar_wait(&empty_bar[stage], phase ^ 1);
                            uint8_t* a_dst = smem + stage * kStageBytes;
                            uint8_t* b_dst = a_dst + kATileBytes;
                            mbar_expect_tx(&full_bar[stage], stage_tx_bytes);
                            tma_load_3d(a_dst, &p.amap[s], &full_bar[stage],
                                        sd.a_ch_off + ch * kChunk, trow, b);
                            tma_load_3d(b_dst, &p.wmap[s], &full_bar[stage],
                                        sd.w_ch_off + ch * kChunk, n0, tap);
                            if (++stage == kStages) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc = FP8 ? umma_idesc_e4m3(kBlockM, block_n) : umma_idesc_bf16(kBlockM, block_n);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            TileCursor cur;
            cur.init(p);
            int u = (int)blockIdx.x - (int)gridDim.x, nt_next = 0;
            for (;;) {
                CAB_NEXT_UNIT()
                (void)nt;
                if (!cur.seek(p, am)) break;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kMaxBlockN;
                uint32_t accumulate = 0;
                for (int s = 0; s < p.n_src; ++s) {
                    const int ksteps = p.src[s].taps * p.src[s].n_chunks;
                    for (int ks = 0; ks < ksteps; ++ks) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
                        const uint32_t b_addr = a_addr + kATileBytes;
                        const uint64_t a_desc = umma_desc_sw128(a_addr);
                        const uint64_t b_desc = umma_desc_sw128(b_addr);
#pragma unroll
                        for (int k = 0; k < kBlockK / 16; ++k) {
                            // +32 bytes per K=16 (bf16) / K=32 (E4M3) slice inside the 128B swizzle row (>>4 => +2)
                            if (FP8) umma_e4m3(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, accumulate);
                            else umma_bf16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, accumulate);
                            accumulate = 1;
                        }
                        umma_commit(&empty_bar[stage]);  // frees the smem slot when MMAs retire
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                }
                umma_commit(&tmem_full[acc]);  // accumulator ready for the epilogue
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int q = warp & 3;  // TMEM lane quarter this warp may read
        const int row = q * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        uint32_t epi_chunks = 0;
        TileCursor cur;
        cur.init(p);
        float run_m = -INFINITY, run_s = 0.f;  // CAB_EPI_LOGITS_ROWS: online softmax of this thread's row across N tiles
        int run_i = 0;
        uint32_t yphase = 0;  // bit i = parity ybar[i] completes next
        const bool fold = p.bnr_partials != nullptr;  // (host: ACT_BF16 epilogue, no lo output, no stats)
        int u = (int)blockIdx.x - (int)gridDim.x, nt_next = 0;
        for (;;) {
            CAB_NEXT_UNIT()
            if (!cur.seek(p, am)) break;
            const int b = cur.b;
            const int t0 = (am - cur.base) * kBlockM;
            const int n0 = nt * block_n;
            const int t = t0 + row;
            const bool row_ok = t < p.T_out;

            const uint32_t taddr = tmem_base + acc * kMaxBlockN + (uint32_t(q * 32) << 16);
            if (p.epilogue != CAB_EPI_ACT_BF16) {
                mbar_wait(&tmem_full[acc], acc_phase);
                tc_fence_after();
            }  // (CAB_EPI_LOGITS_ROWS stages its bias after this wait: one barrier pair per tile, negligible next to 8 TMA stores)

            if (p.epilogue == CAB_EPI_ACT_BF16) {
                int len = p.T_out;
                if (p.xlen != nullptr) len = frac_len(__ldg(p.xlen + b), p.T_out);
                const bool keep = t < len;
                const int et = threadIdx.x - 128;  // 0..127 within the epilogue warps
                const bool has_lo = p.out_lo != nullptr;
                uint8_t* const ystage = smem + kOffStageOut + 2 * kEpiTileBytes;  // the lo staging pair is free in the bf16 tier
                int bnr_rows = 0;
                if (fold) {
                    // y tile of this tile's first chunk: buffer (epi_chunks & 1) was last read two chunks ago, and every thread
                    // finished that read before the epi_bar(2) of the chunk after it, which this thread has passed
                    if (et == 0) {
                        const int ybuf = epi_chunks & 1;
                        mbar_expect_tx(&ybar[ybuf], kEpiTileBytes);
                        tma_load_3d(ystage + ybuf * kEpiTileBytes, &p.ymap, &ybar[ybuf], n0, t0, b);
                    }
                    int blen = p.T_out;
                    if (p.bnr_xlen != nullptr) blen = min(blen, frac_len(__ldg(p.bnr_xlen + b), p.T_out));
                    bnr_rows = min(max(blen - t0, 0), kBlockM);
                }
                // stage this tile's bias (zeros past C_out / without bias)
                epi_bar(1);  // previous tile's readers are done with s_bias
                // E4M3 mode: alpha goes where the lo staging pair would be (no lo output, no folded reduction there)
                float* const s_alpha = reinterpret_cast<float*>(smem + kOffStageOut + 2 * kEpiTileBytes);
                for (int i = et; i < block_n; i += 128) {
                    const int n = n0 + i;
                    s_bias[i] = (p.bias != nullptr && n < p.C_out) ? __ldg(p.bias + n) : 0.f;
                    if (FP8) s_alpha[i] = n < p.C_out ? __ldg(p.alpha + n) : 0.f;
                }
                epi_bar(1);
                mbar_wait(&tmem_full[acc], acc_phase);  // bias staging above overlaps the MMAs
                tc_fence_after();
                uint8_t* stage = smem + kOffStageOut;
                for (int c0 = 0; c0 < block_n; c0 += kEpiCols) {
                    if (n0 + c0 >= p.C_out) break;  // uniform
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + c0, v);
                    tmem_ld_wait();
                    if (c0 + kEpiCols >= block_n || n0 + c0 + kEpiCols >= p.C_out) {
                        // accumulator fully read: hand the TMEM stage back to the MMA warp early
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
                    }
                    const int buf = epi_chunks & 1;
                    uint8_t* st_hi = stage + buf * kEpiTileBytes;
                    uint8_t* st_lo = stage + (2 + buf) * kEpiTileBytes;
                    // the TMA store that last read this buffer was committed two chunks ago
                    if (et == 0) bulk_wait_read<1>();
                    float bnr_sc = 0.f, bnr_sh = 0.f;
                    const int bnr_col = n0 + c0 + (et & 31);
                    if (fold && bnr_col < p.bnr_C) {
                        bnr_sc = __ldg(p.bnr_ss + bnr_col);
                        bnr_sh = __ldg(p.bnr_ss + p.bnr_C + bnr_col);
                    }
                    epi_bar(2);
                    if (fold && et == 0 && c0 + kEpiCols < block_n && n0 + c0 + kEpiCols < p.C_out) {
                        // y tile of the NEXT chunk of this tile into the other buffer: its last readers (the column pass of the
                        // previous chunk) all arrived at the barrier above
                        const int ynext = (epi_chunks + 1) & 1;
                        mbar_expect_tx(&ybar[ynext], kEpiTileBytes);
                        tma_load_3d(ystage + ynext * kEpiTileBytes, &p.ymap, &ybar[ynext], n0 + c0 + kEpiCols, t0, b);
                    }
                    const float* sb = s_bias + c0;
#define CAB_EPI_CALL(ACT)                                                                          \
    if (FP8) epi_chunk_e4m3<ACT>(v, sb, s_alpha + c0, p.act_a, p.act_b, keep, p.out_inv, row, st_hi); \
    else if (has_lo) epi_chunk<ACT, true>(v, sb, p.act_a, p.act_b, keep, row, st_hi, st_lo);       \
    else epi_chunk<ACT, false>(v, sb, p.act_a, p.act_b, keep, row, st_hi, st_lo);
                    switch (p.act) {
                        case CAB_ACT_RELU: CAB_EPI_CALL(CAB_ACT_RELU) break;
                        case CAB_ACT_HARDTANH: CAB_EPI_CALL(CAB_ACT_HARDTANH) break;
                        case CAB_ACT_LEAKY_RELU: CAB_EPI_CALL(CAB_ACT_LEAKY_RELU) break;
                        default: CAB_EPI_CALL(CAB_ACT_NONE) break;
                    }
#undef CAB_EPI_CALL
                    fence_async_smem();  // generic-proxy smem writes -> visible to the TMA engine
                    epi_bar(3);
                    if (et == 0) {
                        tma_store_3d(&p.omap_hi, st_hi, n0 + c0, t0, b);  // rows >= T_out are clipped
                        if (has_lo) tma_store_3d(&p.omap_lo, st_lo, n0 + c0, t0, b);
                        bulk_commit();
                    }
                    if (p.stats != nullptr) {
                        // BatchNorm batch statistics of what was just stored (bf16-rounded; hi + lo in the split tier), valid rows
                        // only, column-parallel over the staged tile (every thread's row is there: barrier 3 above; the
                        // buffer is rewritten two chunks from now, behind that chunk's barrier 2)
                        float cs, cq;
                        const int srows = min(max(p.T_out - t0, 0), kBlockM);
                        if (has_lo) stats_column_pass<true>(st_hi, st_lo, et, srows, cs, cq);
                        else stats_column_pass<false>(st_hi, st_lo, et, srows, cs, cq);
                        const int col = n0 + c0 + (et & 31);
                        if (col < p.C_out && srows > (et >> 5) * 32) {
                            atomicAdd(p.stats + col, (double)cs);
                            atomicAdd(p.stats + p.C_out + col, (double)cq);
                        }
                    }
                    if (fold) {
                        // every thread's row of g is staged (barrier 3 above); the y tile was requested a chunk ago
                        mbar_wait(&ybar[buf], (yphase >> buf) & 1u);
                        yphase ^= 1u << buf;
                        const uint8_t* st_y = ystage + buf * kEpiTileBytes;
                        float cs, cq;
                        switch (p.bnr_act) {
                            case CAB_ACT_RELU: bnr_column_pass<CAB_ACT_RELU>(st_hi, st_y, et, bnr_rows, bnr_sc, bnr_sh, p.bnr_a, p.bnr_b, cs, cq); break;
                            case CAB_ACT_HARDTANH: bnr_column_pass<CAB_ACT_HARDTANH>(st_hi, st_y, et, bnr_rows, bnr_sc, bnr_sh, p.bnr_a, p.bnr_b, cs, cq); break;
                            case CAB_ACT_LEAKY_RELU: bnr_column_pass<CAB_ACT_LEAKY_RELU>(st_hi, st_y, et, bnr_rows, bnr_sc, bnr_sh, p.bnr_a, p.bnr_b, cs, cq); break;
                            default: bnr_column_pass<CAB_ACT_NONE>(st_hi, st_y, et, bnr_rows, bnr_sc, bnr_sh, p.bnr_a, p.bnr_b, cs, cq); break;
                        }
                        if (bnr_col < p.bnr_C && bnr_rows > (et >> 5) * 32) {
                            double* dst = p.bnr_partials + (size_t)(blockIdx.x % CAB_BN_SUM_REPLICAS) * 2 * p.bnr_C;
                            atomicAdd(dst + bnr_col, (double)cs);
                            atomicAdd(dst + p.bnr_C + bnr_col, (double)cq);
                        }
                    }
                    ++epi_chunks;
                }
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
                continue;
            } else if (p.epilogue == CAB_EPI_LOGITS_ROWS) {
                // fp32 logits, class-contiguous rows: 32-column chunks staged in smem (128-byte rows, 128B swizzle) and written
                // with TMA stores; running (max, sum exp, argmax) per row across the N tiles of this M tile
                const int et = threadIdx.x - 128;
                const int C = p.C_out;
                epi_bar(1);
                for (int i = et; i < block_n; i += 128) {
                    const int n = n0 + i;
                    s_bias[i] = (p.bias != nullptr && n < C) ? __ldg(p.bias + n) : 0.f;
                }
                epi_bar(1);
                if (nt == 0) { run_m = -INFINITY; run_s = 0.f; run_i = 0; }
                uint8_t* stage = smem + kOffStageOut;  // two 16 KB buffers
                for (int c0 = 0; c0 < block_n; c0 += 32) {
                    if (n0 + c0 >= C) break;  // uniform
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + c0, v);
                    tmem_ld_wait();
                    if (c0 + 32 >= block_n || n0 + c0 + 32 >= C) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
                    }
                    float x[32];
                    float cm = -INFINITY;
                    int ci = 0;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const bool in = n0 + c0 + j < C;
                        if (FP8) x[j] = fmaf(__uint_as_float(v[j]), in ? __ldg(p.alpha + n0 + c0 + j) : 0.f, s_bias[c0 + j]);
                        else x[j] = __uint_as_float(v[j]) + s_bias[c0 + j];
                        if (in && x[j] > cm) { cm = x[j]; ci = n0 + c0 + j; }
                    }
                    if (cm > run_m) {  // strict: ties keep the lowest class id (classes are visited in increasing order)
                        run_s *= __expf(run_m - cm);
                        run_m = cm;
                        run_i = ci;
                    }
                    float cs = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) cs += (n0 + c0 + j < C) ? __expf(x[j] - run_m) : 0.f;
                    run_s += cs;
                    const int buf = epi_chunks & 1;
                    uint8_t* st = stage + buf * (2 * kEpiTileBytes);
                    if (et == 0) bulk_wait_read<1>();
                    epi_bar(2);
                    // 128-byte rows, 16-byte chunk index XOR (row & 7) == CU_TENSOR_MAP_SWIZZLE_128B
#pragma unroll
                    for (int q4 = 0; q4 < 8; ++q4)
                        *reinterpret_cast<float4*>(st + row * 128 + ((q4 ^ (row & 7)) << 4)) = make_float4(x[4 * q4], x[4 * q4 + 1], x[4 * q4 + 2], x[4 * q4 + 3]);
                    fence_async_smem();
                    epi_bar(3);
                    if (et == 0) {
                        tma_store_3d(&p.omap_hi, st, n0 + c0, t0, b);  // rows >= T_out and columns >= C are clipped
                        bulk_commit();
                    }
                    ++epi_chunks;
                }
                if (nt == p.n_ntiles - 1 && row_ok) {
                    if (p.lse) p.lse[size_t(b) * p.T_out + t] = run_m + logf(run_s);
                    if (p.argmax) p.argmax[size_t(b) * p.T_out + t] = run_i;
                }
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
                continue;
            } else if (p.epilogue == CAB_EPI_LOGSOFTMAX) {
                // Single N tile holds all classes.  Three passes over TMEM (cheap) keep the
                // register footprint small: max/argmax, sum of exp, then write.
                const int C = p.C_out;
                float vmax = -INFINITY;
                int imax = 0;
                for (int c0 = 0; c0 < C; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld_32x16(taddr + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int c = c0 + j;
                        if (c < C) {
                            float x = (FP8 ? __uint_as_float(v[j]) * __ldg(p.alpha + c) : __uint_as_float(v[j])) + (p.bias ? __ldg(p.bias + c) : 0.f);
                            if (x > vmax) { vmax = x; imax = c; }
                        }
                    }
                }
                float ssum = 0.f;
                for (int c0 = 0; c0 < C; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld_32x16(taddr + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int c = c0 + j;
                        if (c < C) {
                            float x = (FP8 ? __uint_as_float(v[j]) * __ldg(p.alpha + c) : __uint_as_float(v[j])) + (p.bias ? __ldg(p.bias + c) : 0.f);
                            ssum += expf(x - vmax);
                        }
                    }
                }
                const float lse = vmax + logf(ssum);
                for (int c0 = 0; c0 < C; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld_32x16(taddr + c0, v);
                    tmem_ld_wait();
                    if (row_ok) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int c = c0 + j;
                            if (c < C) {
                                float x = (FP8 ? __uint_as_float(v[j]) * __ldg(p.alpha + c) : __uint_as_float(v[j])) + (p.bias ? __ldg(p.bias + c) : 0.f);
                                const size_t o = (size_t(b) * C + c) * p.T_out + t;  // lanes -> consecutive t
                                if (p.logits) p.logits[o] = x;
                                if (p.log_probs) p.log_probs[o] = x - lse;
                            }
                        }
                    }
                }
                if (row_ok && p.argmax) p.argmax[size_t(b) * p.T_out + t] = imax;
            } else {  // CAB_EPI_LOGITS_F32
                const int C = p.C_out;
                for (int c0 = 0; c0 < block_n; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld_32x16(taddr + c0, v);
                    tmem_ld_wait();
                    if (row_ok) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int c = n0 + c0 + j;
                            if (c < C) {
                                float x = (FP8 ? __uint_as_float(v[j]) * __ldg(p.alpha + c) : __uint_as_float(v[j])) + (p.bias ? __ldg(p.bias + c) : 0.f);
                                p.logits[(size_t(b) * C + c) * p.T_out + t] = apply_act(x, p.act, p.act_a, p.act_b);
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        }
        if (p.skip_frac != nullptr && p.epilogue == CAB_EPI_ACT_BF16) {
            // M tiles that are pure padding: nobody computed them, store zeros (same staging buffers / TMA
            // stores as above).  Cursor over the compacted index of SKIPPED tiles.
            const int et = threadIdx.x - 128;
            const bool has_lo = p.out_lo != nullptr;
            uint8_t* stage = smem + kOffStageOut;
            int b = 0, base = 0, end = p.mtiles_per_b - live_mtiles(p, 0);
            for (int z = blockIdx.x;; z += gridDim.x) {
                const int nt = z % p.n_ntiles;
                const int sm = z / p.n_ntiles;
                bool done = false;
                while (sm >= end) {
                    if (++b >= p.B) { done = true; break; }
                    base = end;
                    end += p.mtiles_per_b - live_mtiles(p, b);
                }
                if (done) break;
                const int t0 = (live_mtiles(p, b) + (sm - base)) * kBlockM;
                const int n0 = nt * block_n;
                for (int c0 = 0; c0 < block_n; c0 += kEpiCols) {
                    if (n0 + c0 >= p.C_out) break;  // uniform
                    const int buf = epi_chunks & 1;
                    uint8_t* st_hi = stage + buf * kEpiTileBytes;
                    uint8_t* st_lo = stage + (2 + buf) * kEpiTileBytes;
                    if (et == 0) bulk_wait_read<1>();
                    epi_bar(2);
                    uint4* zh = reinterpret_cast<uint4*>(st_hi + row * (FP8 ? 32 : 64));
                    uint4* zl = reinterpret_cast<uint4*>(st_lo + row * 64);
#pragma unroll
                    for (int qd = 0; qd < (FP8 ? 2 : 4); ++qd) {
                        zh[qd] = make_uint4(0, 0, 0, 0);
                        if (has_lo) zl[qd] = make_uint4(0, 0, 0, 0);
                    }
                    fence_async_smem();
                    epi_bar(3);
                    if (et == 0) {
                        tma_store_3d(&p.omap_hi, st_hi, n0 + c0, t0, b);
                        if (has_lo) tma_store_3d(&p.omap_lo, st_lo, n0 + c0, t0, b);
                        bulk_commit();
                    }
                    ++epi_chunks;
                }
            }
        }
        if (threadIdx.x == 128) bulk_wait_all();  // all TMA stores of this CTA have completed
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) ==
                cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    });
    return fn;
}

// 3-D bf16 (elem_bytes 2) or E4M3 (elem_bytes 1, mapped as bytes) map: dims (innermost first) {d0, d1, d2}, row pitch /
// slab pitch in elements.
static int encode_map_3d(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                         uint64_t pitch1_elems, uint64_t pitch2_elems, uint32_t box0,
                         uint32_t box1, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, int elem_bytes = 2) {
    EncodeTiledFn enc = get_encode_fn();
    CAB_CHECK_ARG(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {pitch1_elems * elem_bytes, pitch2_elems * elem_bytes};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims,
                     strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CAB_CHECK_ARG(r == CUDA_SUCCESS,
                  "cuTensorMapEncodeTiled failed (%d): base=%p dims=%llu,%llu,%llu pitch=%llu,%llu "
                  "box=%u,%u",
                  (int)r, base, (unsigned long long)d0, (unsigned long long)d1,
                  (unsigned long long)d2, (unsigned long long)pitch1_elems,
                  (unsigned long long)pitch2_elems, box0, box1);
    return 0;
}

static int pick_block_n(int C_out, int epilogue, long long m_tiles, int num_sms) {
    if (epilogue == CAB_EPI_LOGSOFTMAX) return ((C_out + 15) / 16) * 16;
    // N tile (multiple of 32: the epilogue works in 32-column TMEM loads).  A k-step costs ~(block_n + 96)
    // (MMA time grows with block_n, the A-tile load and the per-step latencies do not) and the persistent
    // grid needs ceil(tiles / #SMs) rounds: large batches end up with the fewest, widest tiles (256 -> 1x256,
    // 640 -> 3x224, 896 -> 4x224), small batches (B = 8: 32 M tiles for 148 SMs) split N further so that
    // every SM gets a tile.
    int best_bn = 0;
    double best_cost = 0.0;
    const int min_tiles = (C_out + kMaxBlockN - 1) / kMaxBlockN;
    for (int n_tiles = min_tiles; n_tiles <= min_tiles * 8; ++n_tiles) {
        int bn = (C_out + n_tiles - 1) / n_tiles;
        bn = ((bn + 31) / 32) * 32;
        if (bn < 64 && n_tiles > min_tiles) break;
        const long long tiles = m_tiles * ((C_out + bn - 1) / bn);
        const double cost = (double)((tiles + num_sms - 1) / num_sms) * (bn + 96);
        if (best_bn == 0 || cost < best_cost * 0.98) { best_bn = bn; best_cost = cost; }
    }
    return best_bn;
}

extern std::atomic<int64_t> g_launch_count;

}  // namespace cab

using namespace cab;

// FP8: E4M3 sources and (ACT_BF16 epilogue) E4M3 output; alpha [C_out] scales the accumulator, out_inv the stored value
template <bool FP8>
static int conv1d_launch(const cab_conv_source_t* srcs, int n_src, const cab_conv_epilogue_t* ep, const float* alpha,
                         float out_inv, cudaStream_t stream) {
    constexpr int kChunk = FP8 ? 2 * kBlockK : kBlockK;
    constexpr int kElem = FP8 ? 1 : 2;
    CAB_CHECK_ARG(srcs && ep, "null sources/epilogue");
    CAB_CHECK_ARG(n_src >= 1 && n_src <= CAB_MAX_CONV_SOURCES, "n_sources=%d out of [1,%d]", n_src,
                  CAB_MAX_CONV_SOURCES);
    CAB_CHECK_ARG(ep->B > 0 && ep->T_out > 0 && ep->C_out > 0, "bad output shape B=%d T=%d C=%d",
                  ep->B, ep->T_out, ep->C_out);

    static thread_local ConvParams p;  // too big for the stack of small threads; reused
    p.n_src = n_src;
    p.B = ep->B;
    p.T_out = ep->T_out;
    p.C_out = ep->C_out;
    static int sms_for_tiling = 0;
    if (sms_for_tiling == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms_for_tiling, cudaDevAttrMultiProcessorCount, dev);
        if (sms_for_tiling <= 0) sms_for_tiling = 148;
    }
    int bn = ep->block_n > 0 ? ep->block_n : pick_block_n(ep->C_out, ep->epilogue, (long long)ep->B * ((ep->T_out + kBlockM - 1) / kBlockM), sms_for_tiling);
    CAB_CHECK_ARG(bn % 16 == 0 && bn >= 16 && bn <= kMaxBlockN, "block_n=%d must be a multiple of 16 in [16,256]", bn);
    if (ep->epilogue == CAB_EPI_ACT_BF16) {
        CAB_CHECK_ARG(bn % 32 == 0, "block_n=%d must be a multiple of 32 for the bf16 epilogue", bn);
        CAB_CHECK_ARG(ep->C_out % 32 == 0, "C_out=%d must be a multiple of 32 (pad on the host)", ep->C_out);
        CAB_CHECK_ARG(ep->out_hi != nullptr, "out_hi is null");
        CAB_CHECK_ARG(ep->out_ld_ch >= ep->C_out && ep->out_ld_ch % 8 == 0, "bad out_ld_ch=%d", ep->out_ld_ch);
        CAB_CHECK_ARG(ep->out_T_rows >= ep->T_out, "out_T_rows=%d < T_out=%d", ep->out_T_rows, ep->T_out);
        CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(ep->out_hi) & 15) == 0, "out_hi must be 16-byte aligned");
    } else if (ep->epilogue == CAB_EPI_LOGSOFTMAX) {
        CAB_CHECK_ARG(ep->C_out <= kMaxBlockN, "log_softmax epilogue supports at most %d classes (got %d)", kMaxBlockN, ep->C_out);
        CAB_CHECK_ARG(bn >= ep->C_out, "block_n=%d must cover all %d classes", bn, ep->C_out);
    } else if (ep->epilogue == CAB_EPI_LOGITS_F32) {
        CAB_CHECK_ARG(ep->logits != nullptr, "logits is null");
    } else if (ep->epilogue == CAB_EPI_LOGITS_ROWS) {
        CAB_CHECK_ARG(ep->logits != nullptr, "logits is null");
        CAB_CHECK_ARG(bn % 32 == 0, "block_n=%d must be a multiple of 32 for the row-major logits epilogue", bn);
        CAB_CHECK_ARG(ep->out_ld_ch >= ep->C_out && ep->out_ld_ch % 4 == 0 && (reinterpret_cast<uintptr_t>(ep->logits) & 15) == 0, "row-major logits need a 16-byte aligned base and a row pitch that is a multiple of 4 floats (got %d)", ep->out_ld_ch);
        CAB_CHECK_ARG(ep->act == CAB_ACT_NONE, "the row-major logits epilogue applies no activation");
    } else {
        CAB_CHECK_ARG(false, "unknown epilogue %d", ep->epilogue);
    }
    p.block_n = bn;
    p.mtiles_per_b = (ep->T_out + kBlockM - 1) / kBlockM;
    p.n_ntiles = (ep->C_out + bn - 1) / bn;
    p.n_tiles = p.B * p.mtiles_per_b * p.n_ntiles;
    p.epilogue = ep->epilogue;
    p.act = ep->act;
    p.act_a = ep->act_a;
    p.act_b = ep->act_b;
    p.bias = ep->bias;
    p.xlen = ep->xlen_frac;
    p.out_hi = static_cast<__nv_bfloat16*>(ep->out_hi);
    p.out_lo = static_cast<__nv_bfloat16*>(ep->out_lo);
    p.out_T_rows = ep->out_T_rows;
    p.out_ld = ep->out_ld_ch;
    p.logits = ep->logits;
    p.log_probs = ep->log_probs;
    p.argmax = ep->argmax;
    p.stats = ep->epilogue == CAB_EPI_ACT_BF16 ? ep->stats : nullptr;
    p.lse = ep->epilogue == CAB_EPI_LOGITS_ROWS ? ep->log_probs : nullptr;  // the log_probs slot carries the [B, T_out] log-sum-exp output
    p.mtile_major = ep->epilogue == CAB_EPI_LOGITS_ROWS ? 1 : 0;
    p.alpha = alpha;
    p.out_inv = out_inv;
    if (FP8) {
        CAB_CHECK_ARG(alpha != nullptr, "alpha is null");
        CAB_CHECK_ARG(ep->out_lo == nullptr && ep->stats == nullptr && ep->bnr_partials == nullptr && ep->skip_frac == nullptr,
                      "the E4M3 mode has no lo output, no statistics, no folded reduction and no explicit skip rows");
        if (ep->epilogue == CAB_EPI_ACT_BF16)
            CAB_CHECK_ARG(ep->out_ld_ch % 16 == 0, "E4M3 output: out_ld_ch=%d must be a multiple of 16", ep->out_ld_ch);
    }
    if (ep->epilogue == CAB_EPI_LOGITS_ROWS) {
        EncodeTiledFn enc = get_encode_fn();
        CAB_CHECK_ARG(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
        cuuint64_t dims[3] = {(cuuint64_t)ep->C_out, (cuuint64_t)ep->T_out, (cuuint64_t)ep->B};
        cuuint64_t strides[2] = {(cuuint64_t)ep->out_ld_ch * 4, (cuuint64_t)ep->T_out * ep->out_ld_ch * 4};
        cuuint32_t box[3] = {32, kBlockM, 1};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&p.omap_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ep->logits, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        CAB_CHECK_ARG(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) for the row-major logits", (int)r);
    }
    // structural-zero rows: given explicitly (training: zero input rows / don't-care gradient rows), or implied
    // by the temporal mask this launch applies itself
    p.skip_frac = nullptr; p.skip_T = 0; p.skip_margin = 0;
    if (ep->epilogue == CAB_EPI_ACT_BF16) {
        if (ep->skip_frac != nullptr) {
            CAB_CHECK_ARG(ep->skip_T > 0 && ep->skip_margin >= 0, "bad skip_T=%d / skip_margin=%d", ep->skip_T, ep->skip_margin);
            p.skip_frac = ep->skip_frac; p.skip_T = ep->skip_T; p.skip_margin = ep->skip_margin;
        } else if (ep->xlen_frac != nullptr) {
            p.skip_frac = ep->xlen_frac; p.skip_T = ep->T_out;
        }
    }
    if (p.stats != nullptr) CAB_CHECK_CUDA(cudaMemsetAsync(p.stats, 0, sizeof(double) * 2 * ep->C_out, stream));
    // folded BatchNorm-backward reduction (see ConvParams)
    p.bnr_partials = nullptr; p.bnr_ss = nullptr; p.bnr_xlen = nullptr; p.bnr_C = 0; p.bnr_act = CAB_ACT_NONE; p.bnr_a = 0.f; p.bnr_b = 0.f;
    if (ep->bnr_partials != nullptr) {
        CAB_CHECK_ARG(ep->epilogue == CAB_EPI_ACT_BF16 && ep->out_lo == nullptr && ep->stats == nullptr, "the folded BatchNorm-backward reduction needs the bf16 activation epilogue without a lo output and without forward statistics");
        CAB_CHECK_ARG(ep->bnr_y != nullptr && ep->bnr_ss != nullptr && ep->bnr_C > 0 && ep->bnr_C <= ep->C_out, "folded BatchNorm-backward reduction: bad y / ss / C=%d", ep->bnr_C);
        CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(ep->bnr_y) & 15) == 0, "bnr_y must be 16-byte aligned");
        p.bnr_partials = ep->bnr_partials; p.bnr_ss = ep->bnr_ss; p.bnr_xlen = ep->bnr_xlen_frac; p.bnr_C = ep->bnr_C;
        p.bnr_act = ep->bnr_act; p.bnr_a = ep->bnr_act_a; p.bnr_b = ep->bnr_act_b;
        int rc = encode_map_3d(&p.ymap, ep->bnr_y, (uint64_t)ep->out_ld_ch, (uint64_t)ep->T_out, (uint64_t)ep->B,
                               (uint64_t)ep->out_ld_ch, (uint64_t)ep->out_T_rows * ep->out_ld_ch, kEpiCols, kBlockM,
                               CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc) return rc;
        CAB_CHECK_CUDA(cudaMemsetAsync(p.bnr_partials, 0, sizeof(double) * CAB_BN_SUM_REPLICAS * 2 * ep->bnr_C, stream));
    }
    if (ep->epilogue == CAB_EPI_ACT_BF16) {
        CAB_CHECK_ARG(ep->out_lo == nullptr || (reinterpret_cast<uintptr_t>(ep->out_lo) & 15) == 0, "out_lo must be 16-byte aligned");
        // E4M3: 32-byte staging rows, unswizzled
        int rc = encode_map_3d(&p.omap_hi, ep->out_hi, (uint64_t)ep->out_ld_ch, (uint64_t)ep->T_out, (uint64_t)ep->B,
                               (uint64_t)ep->out_ld_ch, (uint64_t)ep->out_T_rows * ep->out_ld_ch, kEpiCols, kBlockM,
                               FP8 ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_64B, kElem);
        if (rc) return rc;
        if (ep->out_lo != nullptr) {
            rc = encode_map_3d(&p.omap_lo, ep->out_lo, (uint64_t)ep->out_ld_ch, (uint64_t)ep->T_out, (uint64_t)ep->B,
                               (uint64_t)ep->out_ld_ch, (uint64_t)ep->out_T_rows * ep->out_ld_ch, kEpiCols, kBlockM,
                               CU_TENSOR_MAP_SWIZZLE_64B);
            if (rc) return rc;
        }
    }

    for (int s = 0; s < n_src; ++s) {
        const cab_conv_source_t& c = srcs[s];
        CAB_CHECK_ARG(c.act && c.wgt, "source %d: null pointer", s);
        CAB_CHECK_ARG(c.C_in > 0 && c.C_in % kChunk == 0, "source %d: C_in=%d must be a multiple of %d", s, c.C_in, kChunk);
        CAB_CHECK_ARG(c.ch_off >= 0 && c.ch_off + c.C_in <= c.ld_ch && c.ld_ch % (16 / kElem) == 0, "source %d: bad channel window off=%d C_in=%d ld=%d", s, c.ch_off, c.C_in, c.ld_ch);
        CAB_CHECK_ARG(c.w_ch_off >= 0 && c.w_ch_off + c.C_in <= c.w_ld_ch && c.w_ld_ch % (16 / kElem) == 0, "source %d: bad weight channel window", s);
        CAB_CHECK_ARG(c.taps >= 1 && c.dilation >= 1, "source %d: taps=%d dilation=%d", s, c.taps, c.dilation);
        CAB_CHECK_ARG(c.T_in >= 1 && c.T_rows >= c.T_in, "source %d: T_in=%d T_rows=%d", s, c.T_in, c.T_rows);
        CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(c.act) & 15) == 0 && (reinterpret_cast<uintptr_t>(c.wgt) & 15) == 0, "source %d: pointers must be 16-byte aligned", s);
        int rc = encode_map_3d(&p.amap[s], c.act, (uint64_t)c.ld_ch, (uint64_t)c.T_in, (uint64_t)ep->B,
                               (uint64_t)c.ld_ch, (uint64_t)c.T_rows * c.ld_ch, kChunk, kBlockM, CU_TENSOR_MAP_SWIZZLE_128B, kElem);
        if (rc) return rc;
        rc = encode_map_3d(&p.wmap[s], c.wgt, (uint64_t)c.w_ld_ch, (uint64_t)c.w_rows, (uint64_t)c.taps,
                           (uint64_t)c.w_ld_ch, (uint64_t)c.w_rows * c.w_ld_ch, kChunk, (uint32_t)bn, CU_TENSOR_MAP_SWIZZLE_128B, kElem);
        if (rc) return rc;
        p.src[s].a_ch_off = c.ch_off;
        p.src[s].w_ch_off = c.w_ch_off;
        p.src[s].n_chunks = c.C_in / kChunk;
        p.src[s].taps = c.taps;
        p.src[s].dil = c.dilation;
        p.src[s].pad_left = c.pad_left;
    }

    static int num_sms = 0;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [] {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        attr_err = cudaFuncSetAttribute(conv1d_umma_kernel<FP8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    });
    CAB_CHECK_ARG(attr_err == cudaSuccess, "cudaFuncSetAttribute(smem=%d) failed: %s", kSmemBytes, cudaGetErrorString(attr_err));
    CAB_CHECK_ARG(num_sms > 0, "no CUDA device");
    int grid = p.n_tiles < num_sms ? p.n_tiles : num_sms;
    if (p.mtile_major) grid = p.B * p.mtiles_per_b < num_sms ? p.B * p.mtiles_per_b : num_sms;
    conv1d_umma_kernel<FP8><<<grid, kNumThreads, kSmemBytes, stream>>>(p);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_conv1d_fused(const cab_conv_source_t* srcs, int n_src,
                                const cab_conv_epilogue_t* ep, cab_stream_t stream) {
    return conv1d_launch<false>(srcs, n_src, ep, nullptr, 1.f, static_cast<cudaStream_t>(stream));
}

extern "C" int cab_conv1d_fused_fp8(const cab_conv_source_t* srcs, int n_src, const cab_conv_epilogue_t* ep,
                                    const float* alpha, float out_scale_inv, cab_stream_t stream) {
    return conv1d_launch<true>(srcs, n_src, ep, alpha, out_scale_inv, static_cast<cudaStream_t>(stream));
}
