// C-ABI plumbing shared by all entry points: error string, launch counter, and the small
// grouped-conv kernel of the separable blocks.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>
#include <cstdarg>
#include <cstdio>

namespace cab {

std::atomic<int64_t> g_launch_count{0};
static thread_local char g_err[512] = "";

void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// Grouped Conv1d + bias + ReLU (models.py:50-64, first two stages of the separable
// ConvSamePadding): GENERIC kernel for shapes grouped_conv.cu's FFMA2 kernel does not cover
// (kernel sizes outside its instantiations, very wide groups).  Block = one frame strip x all
// output channels; weights stay in L1.
int grouped_conv_fast(const void* act, const void* act_lo, int B, int T, int T_rows, int C_in, int ld_in, const float* wgt,
                      const float* bias, int C_out, int groups, int k, int pad_left, void* out, void* out_lo,
                      int out_T_rows, int ld_out, int relu, cudaStream_t stream, bool fp8, float in_scale, float out_inv);
constexpr int kGcFrames = 8;
__global__ void __launch_bounds__(256)
grouped_conv_relu_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ x_lo, int T,
                         int T_rows, int C_in, int ld_in, const float* __restrict__ w,
                         const float* __restrict__ bias, int C_out, int groups, int K, int pad,
                         __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo, int out_T_rows,
                         int ld_out, int relu) {
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * kGcFrames;
    const int cin_g = C_in / groups, cout_g = C_out / groups;
    const __nv_bfloat16* xb = x + (size_t)b * T_rows * ld_in;
    const __nv_bfloat16* xlb = x_lo ? x_lo + (size_t)b * T_rows * ld_in : nullptr;
    for (int co = threadIdx.x; co < ld_out; co += blockDim.x) {
        if (co >= C_out) {  // zero the padding channels: the pointwise GEMM contracts over them
            for (int i = 0; i < kGcFrames; ++i)
                if (t0 + i < T) {
                    const size_t o = ((size_t)b * out_T_rows + t0 + i) * ld_out + co;
                    out[o] = __float2bfloat16_rn(0.f);
                    if (out_lo) out_lo[o] = __float2bfloat16_rn(0.f);
                }
            continue;
        }
        const int g = co / cout_g;
        const float* wc = w + (size_t)co * cin_g * K;
        const float bv = bias ? bias[co] : 0.f;
        float acc[kGcFrames];
#pragma unroll
        for (int i = 0; i < kGcFrames; ++i) acc[i] = bv;
        for (int j = 0; j < cin_g; ++j) {
            const int ci = g * cin_g + j;
            // slide over the input strip once: input frame u feeds outputs t = u - k + pad
            for (int u = t0 - pad; u < t0 + kGcFrames - 1 - pad + K; ++u) {
                if (u < 0 || u >= T) continue;
                float xv = __bfloat162float(xb[(size_t)u * ld_in + ci]);
                if (xlb) xv += __bfloat162float(xlb[(size_t)u * ld_in + ci]);
#pragma unroll
                for (int i = 0; i < kGcFrames; ++i) {
                    const int k = u - (t0 + i) + pad;
                    if (k >= 0 && k < K) acc[i] = fmaf(__ldg(wc + j * K + k), xv, acc[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < kGcFrames; ++i) {
            const int t = t0 + i;
            if (t < T) {
                const size_t o = ((size_t)b * out_T_rows + t) * ld_out + co;
                const float v = relu ? fmaxf(acc[i], 0.f) : acc[i];
                const __nv_bfloat16 h = __float2bfloat16_rn(v);
                out[o] = h;
                if (out_lo) out_lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
            }
        }
    }
}

}  // namespace cab

using namespace cab;

extern "C" int cab_abi_version(void) { return CAB_ABI_VERSION; }
extern "C" const char* cab_last_error(void) { return g_err; }
extern "C" int64_t cab_launch_count(void) { return g_launch_count.load(); }

extern "C" int cab_grouped_conv1d(const void* act, const void* act_lo, int B, int T, int T_rows, int C_in,
                                  int ld_in, const float* wgt, const float* bias, int C_out, int groups,
                                  int k, int pad_left, void* out, void* out_lo, int out_T_rows, int ld_out, int relu,
                                  cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(act && wgt && out, "null pointer argument");
    CAB_CHECK_ARG(groups > 0 && C_in % groups == 0 && C_out % groups == 0, "channels not divisible by groups");
    CAB_CHECK_ARG(T_rows >= T && out_T_rows >= T, "row allocation smaller than T");
    CAB_CHECK_ARG(ld_in >= C_in && ld_out >= C_out, "row pitch smaller than channel count");
    {
        const int rc = grouped_conv_fast(act, act_lo, B, T, T_rows, C_in, ld_in, wgt, bias, C_out, groups, k, pad_left, out, out_lo, out_T_rows, ld_out, relu, stream, false, 1.f, 1.f);
        if (rc <= 0) return rc;  // launched (0) or failed (< 0); 1 = shape not covered by the FFMA2 kernel
    }
    dim3 grid((T + kGcFrames - 1) / kGcFrames, B);
    grouped_conv_relu_kernel<<<grid, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(act), static_cast<const __nv_bfloat16*>(act_lo), T, T_rows, C_in, ld_in, wgt,
        bias, C_out, groups, k, pad_left, static_cast<__nv_bfloat16*>(out), static_cast<__nv_bfloat16*>(out_lo),
        out_T_rows, ld_out, relu);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int cab_grouped_conv1d_fp8(const void* act, int B, int T, int T_rows, int C_in, int ld_in, float in_scale,
                                      const float* wgt, const float* bias, int C_out, int groups, int k, int pad_left,
                                      void* out, int out_T_rows, int ld_out, float out_scale_inv, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(act && wgt && out, "null pointer argument");
    CAB_CHECK_ARG(groups > 0 && C_in % groups == 0 && C_out % groups == 0, "channels not divisible by groups");
    CAB_CHECK_ARG(T_rows >= T && out_T_rows >= T, "row allocation smaller than T");
    CAB_CHECK_ARG(ld_in >= C_in && ld_out >= C_out, "row pitch smaller than channel count");
    CAB_CHECK_ARG((reinterpret_cast<uintptr_t>(act) & 15) == 0, "act must be 16-byte aligned");
    const int rc = grouped_conv_fast(act, nullptr, B, T, T_rows, C_in, ld_in, wgt, bias, C_out, groups, k, pad_left, out, nullptr,
                                     out_T_rows, ld_out, 1, stream, true, in_scale, out_scale_inv);
    CAB_CHECK_ARG(rc != 1, "E4M3 grouped conv: shape not covered (k=%d odd in 3..27, ld_in=%d a multiple of 16, input window of "
                           "at most 208 channels per 64 outputs)", k, ld_in);
    return rc;
}
