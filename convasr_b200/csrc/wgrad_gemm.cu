// Conv1d weight gradient as a persistent tcgen05/TMEM GEMM for sm_100a.
//
//   dW[tap][m][n] = sum_{b, t} A[b, t, m] * Bx[b, t + tap*dil - pad, n]
//
// with A = gradient w.r.t. the conv output and Bx = the conv input (or the other way round, the
// host picks which tensor sits on the 128-row M side), both bf16 channels-last [B, T, C]: the
// contraction runs over TIME, so both operands are "MN-major" for the tensor core (the channel
// dimension is contiguous in shared memory).  Training counterpart of conv1d_umma_kernel; in the
// reference this arithmetic is autograd's cudnn wgrad behind `loss.backward()` (train.py:770-774).
//
// Tiling: M = 128 channels of A (two 64-wide swizzle atoms), N = block_n <= 256 channels of Bx
// (block_n/64 atoms), K = 64 frames per pipeline stage (4 MMAs of K=16).  Each TMA box is
// {64 channels, 64 frames} = 8 KB with the 128-byte swizzle; frames outside [0, T) are zero-filled
// by the TMA unit, which implements both the conv zero padding and the ragged tile tail.
// Work item = (tap, m-tile, n-tile, batch split), CTA i takes items i, i + gridDim.x, ... (the static
// schedule of conv1d_umma_kernel); partial sums of different splits are combined
// with fp32 reductions in L2 (red.global.add), so dW must be zero-initialised by the caller when
// n_splits > 1 (the host wrapper does it).
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>
#include <mutex>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

namespace wg {
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // frames per stage
constexpr int kAtom = 64;    // channels per TMA box / swizzle atom
constexpr int kSubTile = kBlockK * kAtom * 2;  // 8 KB
constexpr int kMaxBlockN = 256;
constexpr int kATileBytes = 2 * kSubTile;                      // 16 KB
constexpr int kBTileBytes = (kMaxBlockN / kAtom) * kSubTile;   // 32 KB
constexpr int kStageBytes = kATileBytes + kBTileBytes;
constexpr int kStages = 4;
constexpr int kAccStages = 2;
constexpr int kTmemCols = 512;
constexpr int kNumThreads = 256;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;

struct alignas(64) Params {
    CUtensorMap amap, bmap;
    int B, T_a;             // frames of the A tensor (= conv output frames)
    int taps, dil, pad_left;
    int M_total, N_total;   // real channel counts
    int block_n, n_mtiles, n_ntiles, n_splits, n_items;
    int chunks_per_b;       // ceil(T_a / 64)
    float* out;             // fp32 [taps][M_total][out_ld]
    int out_ld;
    int accumulate;         // use reductions instead of stores
    const float* skip_frac; // frames >= ceil(skip_frac[b] * skip_T) + skip_margin contribute zeros: not contracted
    int skip_T, skip_margin;
};

// 64-frame K chunks of utterance b that can hold non-zero products
__device__ __forceinline__ int live_chunks(const Params& p, int b) {
    if (p.skip_frac == nullptr) return p.chunks_per_b;
    const int rows = min(p.T_a, frac_len(__ldg(p.skip_frac + b), p.skip_T) + p.skip_margin);
    const int n = (rows + 63) / 64;
    return n < 1 ? 1 : n;
}

// MN-major, 128B-swizzled operand: 64-channel atoms LBO bytes apart, 8-frame groups SBO bytes apart
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__global__ void __launch_bounds__(kNumThreads, 1) wgrad_umma_kernel(const __grid_constant__ Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + kAccStages;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + kAccStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.amap);
        tma_prefetch_desc(&p.bmap);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < kAccStages; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
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
    const int n_batoms = (block_n + kAtom - 1) / kAtom;  // 64-channel TMA boxes covering the N tile
    const uint32_t stage_tx = kATileBytes + n_batoms * kSubTile;

    // item -> (split, mt, nt, tap), tap fastest and the batch split SLOWEST: the ~148 items in flight
    // then all stream the same slab of utterances in the same order (it stays L2 resident; with the
    // split as the fastest index every CTA walked a different slab and the operands -- 184 MB for a
    // 768-channel layer -- were re-fetched from HBM: 2.5 GB of DRAM reads per launch, ncu r01)
    auto decode = [&](int item, int& tap, int& mt, int& nt, int& b0, int& b1) {
        const int tiles = p.taps * p.n_mtiles * p.n_ntiles;
        const int split = item / tiles;
        int r = item - split * tiles;
        tap = r % p.taps; r /= p.taps;
        nt = r % p.n_ntiles;
        mt = r / p.n_ntiles;
        b0 = (int)((long long)p.B * split / p.n_splits);
        b1 = (int)((long long)p.B * (split + 1) / p.n_splits);
    };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
                int tap, mt, nt, b0, b1;
                decode(item, tap, mt, nt, b0, b1);
                const int m0 = mt * kBlockM, n0 = nt * block_n;
                const int shift = tap * p.dil - p.pad_left;
                for (int b = b0; b < b1; ++b) {
                    const int n_chunks = live_chunks(p, b);
                    for (int j = 0; j < n_chunks; ++j) {
                        const int t0 = j * kBlockK;
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        uint8_t* a_dst = smem + stage * kStageBytes;
                        uint8_t* b_dst = a_dst + kATileBytes;
                        mbar_expect_tx(&full_bar[stage], stage_tx);
                        // one 4-D box per operand: {64 ch, 64 frames, atoms, 1} lands as [atom][frame][64 ch]
                        tma_load_4d(a_dst, &p.amap, &full_bar[stage], 0, t0, m0 / kAtom, b);
                        tma_load_4d(b_dst, &p.bmap, &full_bar[stage], 0, t0 + shift, n0 / kAtom, b);
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // M=128, N=block_n, bf16 x bf16 -> fp32, both operands MN-major (bits 15, 16)
            const uint32_t idesc = umma_idesc_bf16(kBlockM, block_n) | (1u << 15) | (1u << 16);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
                int tap, mt, nt, b0, b1;
                decode(item, tap, mt, nt, b0, b1);
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kMaxBlockN;
                uint32_t accumulate = 0;
                int ksteps = 0;
                for (int b = b0; b < b1; ++b) ksteps += live_chunks(p, b);
                for (int ks = 0; ks < ksteps; ++ks) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
                    const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k) {
                        // 16 frames = two 8-frame groups = 2 KB further into every atom
                        const uint64_t a_desc = desc_mn_sw128(a_addr + k * 2048, kSubTile, 1024);
                        const uint64_t b_desc = desc_mn_sw128(b_addr + k * 2048, kSubTile, 1024);
                        umma_bf16(d_tmem, a_desc, b_desc, idesc, accumulate);
                        accumulate = 1;
                    }
                    umma_commit(&empty_bar[stage]);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full[acc]);
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int row = q * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int tap, mt, nt, b0, b1;
            decode(item, tap, mt, nt, b0, b1);
            const int m = mt * kBlockM + row;
            const int n0 = nt * block_n;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * kMaxBlockN + (uint32_t(q * 32) << 16);
            float* orow = p.out + ((size_t)tap * p.M_total + m) * p.out_ld + n0;
            for (int c0 = 0; c0 < block_n; c0 += 32) {
                uint32_t v[32];
                tmem_ld_32x32(taddr + c0, v);
                tmem_ld_wait();
                if (m < p.M_total && b1 > b0) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int n = n0 + c0 + j;
                        if (n + 3 < p.N_total) {
                            if (p.accumulate)
                                red_add_v4(orow + c0 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                            else
                                *reinterpret_cast<float4*>(orow + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                        } else {
                            for (int e = 0; e < 4; ++e)
                                if (n + e < p.N_total) {
                                    if (p.accumulate) atomicAdd(orow + c0 + j + e, __uint_as_float(v[j + e]));
                                    else orow[c0 + j + e] = __uint_as_float(v[j + e]);
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
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    });
    return fn;
}
// channels-last [B, T_rows, ld] viewed as 4-D {64 ch, T frames, ld/64 atoms, B}: a box of `atoms`
// 64-channel atoms lands in shared memory atom-major, i.e. as the 8 KB sub-tiles UMMA wants
static int encode_cl(CUtensorMap* map, const void* base, int ld, int T, int T_rows, int B, int atoms) {
    EncodeTiledFn enc = encode_fn();
    CAB_CHECK_ARG(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
    CAB_CHECK_ARG(ld % kAtom == 0, "wgrad operands need a channel pitch that is a multiple of 64 (got %d)", ld);
    cuuint64_t dims[4] = {(cuuint64_t)kAtom, (cuuint64_t)T, (cuuint64_t)(ld / kAtom), (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)kAtom * 2, (cuuint64_t)T_rows * ld * 2};
    cuuint32_t box[4] = {kAtom, kBlockK, (cuuint32_t)atoms, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CAB_CHECK_ARG(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) for wgrad operand ld=%d T=%d B=%d", (int)r, ld, T, B);
    return 0;
}
}  // namespace wg
}  // namespace cab

using namespace cab;

extern "C" int cab_conv1d_wgrad(const void* a, int a_T, int a_T_rows, int a_ld, int M_total, const void* bx, int b_T,
                                int b_T_rows, int b_ld, int N_total, int B, int taps, int dilation, int pad_left,
                                float* out, int out_ld, int n_splits, const float* skip_frac, int skip_T, int skip_margin,
                                int accumulate_into, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(a && bx && out, "null pointer argument");
    CAB_CHECK_ARG(B > 0 && a_T > 0 && b_T > 0 && taps > 0 && dilation != 0, "bad shape");
    CAB_CHECK_ARG(a_ld % 64 == 0 && b_ld % 64 == 0 && a_ld >= M_total && b_ld >= N_total, "bad channel pitch (multiples of 64 required)");
    CAB_CHECK_ARG(out_ld % 4 == 0 && out_ld >= N_total, "out_ld=%d must be a multiple of 4 and >= N_total", out_ld);
    CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(bx) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "pointers must be 16-byte aligned");
    static thread_local wg::Params p;
    p.B = B; p.T_a = a_T; p.taps = taps; p.dil = dilation; p.pad_left = pad_left;
    p.M_total = M_total; p.N_total = N_total;
    const int n_nt = (N_total + wg::kMaxBlockN - 1) / wg::kMaxBlockN;
    int bn = (N_total + n_nt - 1) / n_nt;
    bn = (bn + wg::kAtom - 1) / wg::kAtom * wg::kAtom;  // whole 64-channel atoms (one TMA box per operand)
    p.block_n = bn;
    int rc = wg::encode_cl(&p.amap, a, a_ld, a_T, a_T_rows, B, 2);
    if (rc) return rc;
    rc = wg::encode_cl(&p.bmap, bx, b_ld, b_T, b_T_rows, B, bn / wg::kAtom);
    if (rc) return rc;
    p.n_mtiles = (M_total + wg::kBlockM - 1) / wg::kBlockM;
    p.n_ntiles = (N_total + bn - 1) / bn;
    static int num_sms = 0;
    static cudaError_t attr_err = cudaSuccess;
    static std::once_flag once;
    std::call_once(once, [] {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        attr_err = cudaFuncSetAttribute(wg::wgrad_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wg::kSmemBytes);
    });
    CAB_CHECK_ARG(attr_err == cudaSuccess && num_sms > 0, "wgrad kernel setup failed: %s", cudaGetErrorString(attr_err));
    const int tiles = taps * p.n_mtiles * p.n_ntiles;
    if (n_splits <= 0) {
        // All items cost the same and every persistent CTA takes ceil(items / #SMs) of them, so pick
        // the batch split that wastes the least of the last wave (ties: fewer splits = less L2
        // reduction traffic); never more splits than utterances, at least ~2 waves when possible.
        double best = -1.0;
        n_splits = 1;
        const int max_splits = B < 24 ? B : 24;
        for (int sp = 1; sp <= max_splits; ++sp) {
            const long long items = (long long)tiles * sp;
            const long long waves = (items + num_sms - 1) / num_sms;
            double eff = (double)items / (double)(waves * num_sms);
            if (items < 2LL * num_sms) eff *= 0.9;  // too few items to hide the pipeline fill
            if (eff > best + 0.02) { best = eff; n_splits = sp; }
        }
    }
    CAB_CHECK_ARG(n_splits <= B, "n_splits=%d > B=%d", n_splits, B);
    p.n_splits = n_splits;
    p.n_items = tiles * n_splits;
    p.chunks_per_b = (a_T + wg::kBlockK - 1) / wg::kBlockK;
    p.out = out; p.out_ld = out_ld;
    CAB_CHECK_ARG(skip_frac == nullptr || (skip_T > 0 && skip_margin >= 0), "bad skip_T=%d / skip_margin=%d", skip_T, skip_margin);
    p.skip_frac = skip_frac; p.skip_T = skip_T; p.skip_margin = skip_margin;
    // accumulate_into: add to what `out` already holds (the hi*lo + lo*hi partial products of the split-bf16 tier)
    p.accumulate = (n_splits > 1 || accumulate_into) ? 1 : 0;
    if (p.accumulate && !accumulate_into) CAB_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)taps * M_total * out_ld, stream));
    const int grid = p.n_items < num_sms ? p.n_items : num_sms;
    wg::wgrad_umma_kernel<<<grid, wg::kNumThreads, wg::kSmemBytes, stream>>>(p);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}
