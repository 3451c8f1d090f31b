// Multi-tensor optimizer step: gradient-norm clipping + SGD(momentum, weight decay, nesterov) or
// NovoGrad, for ALL parameters in three launches (section 8f "next" #3).
//
// Replaces (reference file:line): torch.nn.utils.clip_grad_norm_ at train.py:776-779,
// optimizers.NovoGrad.step optimizers.py:72-90 (a Python loop with ~8 launches per tensor), and
// torch.optim.SGD as configured at train.py:657-662.  HBM bound: every element of p, g, m is read
// and p, m written exactly once (5 x 4 B per parameter per step); 128-bit accesses where the tensors are 16-byte aligned.
//
// Tensors are described by device tables (pointers, sizes) and a flat chunk list for load balance.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

constexpr int kOptThreads = 256;

// sum of squares of one chunk of a gradient -> out[chunk] (no atomics: the per-tensor and total norms are then summed in a
// fixed order, so data-parallel replicas derive bit-identical clip coefficients from bit-identical gradients)
__global__ void __launch_bounds__(kOptThreads)
mt_sumsq_kernel(const long long* __restrict__ grad_ptrs, const long long* __restrict__ numels,
                const int* __restrict__ chunk_tensor, const long long* __restrict__ chunk_off, int chunk_elems,
                float* __restrict__ out) {
    const int ti = chunk_tensor[blockIdx.x];
    const long long off = chunk_off[blockIdx.x];
    const float* g = reinterpret_cast<const float*>(grad_ptrs[ti]) + off;
    const long long n = min((long long)chunk_elems, numels[ti] - off);
    float acc = 0.f;
    // 128-bit loads only from a 16-byte aligned base (chunk offsets are multiples of 4): a gradient may be a view at any
    // float offset of a larger buffer
    const long long n4 = (reinterpret_cast<uintptr_t>(g) & 15) == 0 ? n >> 2 : 0;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (long long i = threadIdx.x; i < n4; i += kOptThreads) {
        const float4 v = g4[i];
        acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += kOptThreads) acc += g[i] * g[i];
    acc = warp_sum(acc);
    __shared__ float sm[kOptThreads / 32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < kOptThreads / 32) {
        acc = sm[threadIdx.x];
#pragma unroll
        for (int o = kOptThreads / 64; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffu, acc, o);
        if (threadIdx.x == 0) out[blockIdx.x] = acc;
    }
}

// per-tensor scalars: clip coefficient, NovoGrad second-moment EMA -> scale[i]; step counter / first flag
// state: [0] = step count (as float bits are avoided: int), kept in an int64 device cell
__global__ void mt_prepare_kernel(float* __restrict__ sumsq, const float* __restrict__ chunk_sumsq, const int* __restrict__ chunk_tensor,
                                  int n_chunks, int n, int mode, float max_norm, float beta2, float eps,
                                  float* __restrict__ ema, float* __restrict__ scale, long long* __restrict__ step_cell,
                                  int* __restrict__ first_flag, float* __restrict__ total_norm_out,
                                  const float* __restrict__ ext_total_norm) {
    __shared__ float s_total;
    // per-tensor sums from the chunk partials, in chunk order (chunks of a tensor are consecutive: binary search for the first)
    if (chunk_sumsq != nullptr) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            int lo = 0, hi = n_chunks;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (chunk_tensor[mid] < i) lo = mid + 1; else hi = mid;
            }
            float a = 0.f;
            for (int c = lo; c < n_chunks && chunk_tensor[c] == i; ++c) a += chunk_sumsq[c];
            sumsq[i] = a;
        }
        __syncthreads();
    }
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += sumsq[i];
    acc = warp_sum(acc);
    __shared__ float sm[32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
        // ext_total_norm: the gradient norm over ALL parameter groups (clip_grad_norm_ is global, train.py:776-779)
        s_total = ext_total_norm ? ext_total_norm[0] : sqrtf(t);
        if (total_norm_out) total_norm_out[0] = s_total;
    }
    __syncthreads();
    if (mode == 2) return;  // norm only
    const bool first = step_cell[0] == 0;
    // torch.nn.utils.clip_grad_norm_: coef = clamp(max_norm / (total + 1e-6), max = 1)
    const float c = max_norm > 0.f ? fminf(max_norm / (s_total + 1e-6f), 1.f) : 1.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (mode == 1) {  // NovoGrad: EMA of the squared norm of the (clipped) gradient, optimizers.py:77-79
            const float g2 = c * c * sumsq[i];
            // a tensor that joins later (its first gradient) starts its EMA like a first step does: ema == 0 marks it
            const float e = (first || ema[i] == 0.f) ? g2 : ema[i] * beta2 + g2 * (1.f - beta2);
            ema[i] = e;
            scale[i] = c / sqrtf(e + eps);
        } else {
            scale[i] = c;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        first_flag[0] = first ? 1 : 0;
        step_cell[0] += 1;
    }
}

__global__ void __launch_bounds__(kOptThreads)
mt_update_kernel(const long long* __restrict__ param_ptrs, const long long* __restrict__ grad_ptrs,
                 const long long* __restrict__ mom_ptrs, const long long* __restrict__ numels,
                 const int* __restrict__ chunk_tensor, const long long* __restrict__ chunk_off, int chunk_elems,
                 const float* __restrict__ scale, const int* __restrict__ first_flag, const float* __restrict__ lr_ptr,
                 int mode, float momentum, float weight_decay, float dampening, int nesterov) {
    const int ti = chunk_tensor[blockIdx.x];
    const long long off = chunk_off[blockIdx.x];
    float* p = reinterpret_cast<float*>(param_ptrs[ti]) + off;
    const float* g = reinterpret_cast<const float*>(grad_ptrs[ti]) + off;
    float* m = reinterpret_cast<float*>(mom_ptrs[ti]) + off;
    const long long n = min((long long)chunk_elems, numels[ti] - off);
    const float sc = scale[ti], lr = lr_ptr[0];
    const bool first = first_flag[0] != 0;
    auto upd = [&](float pv, float gv, float mv, float& p_out, float& m_out) {
        float gp = gv * sc;                 // clip (+ NovoGrad normalisation)
        gp = fmaf(weight_decay, pv, gp);    // L2 weight decay on the (normalised) gradient
        float buf;
        if (mode == 1) {                    // NovoGrad, optimizers.py:81-90
            if (dampening != 0.f) gp *= (1.f - momentum);
            buf = first ? gp : fmaf(mv, momentum, gp);
            p_out = fmaf(-lr, buf, pv);
        } else {                            // torch.optim.SGD
            buf = first ? gp : fmaf(mv, momentum, (1.f - dampening) * gp);
            const float step = nesterov ? fmaf(momentum, buf, gp) : buf;
            p_out = fmaf(-lr, step, pv);
        }
        m_out = buf;
    };
    // the float4 path needs all three bases 16-byte aligned; a tensor with any other offset takes the scalar loop
    const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m)) & 15) == 0;
    const long long n4 = vec ? n >> 2 : 0;
    float4* p4 = reinterpret_cast<float4*>(p);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    for (long long i = threadIdx.x; i < n4; i += kOptThreads) {
        float4 pv = p4[i], gv = g4[i], mv = m4[i], po, mo;
        upd(pv.x, gv.x, mv.x, po.x, mo.x);
        upd(pv.y, gv.y, mv.y, po.y, mo.y);
        upd(pv.z, gv.z, mv.z, po.z, mo.z);
        upd(pv.w, gv.w, mv.w, po.w, mo.w);
        p4[i] = po;
        m4[i] = mo;
    }
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += kOptThreads) upd(p[i], g[i], m[i], p[i], m[i]);
}

}  // namespace cab

using namespace cab;

extern "C" int cab_optimizer_step(int mode, int n_tensors, const int64_t* param_ptrs, const int64_t* grad_ptrs,
                                  const int64_t* mom_ptrs, const int64_t* numels, int n_chunks,
                                  const int32_t* chunk_tensor, const int64_t* chunk_off, int chunk_elems,
                                  float* ws_sumsq, float* ema, float* ws_scale, int64_t* step_cell, int32_t* ws_first,
                                  const float* lr_dev, float momentum, float beta2, float eps, float weight_decay,
                                  float dampening, int nesterov, float max_grad_norm, float* total_norm_out,
                                  const float* ext_total_norm, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(mode >= 0 && mode <= 2, "mode must be 0 (SGD), 1 (NovoGrad) or 2 (gradient norm only)");
    CAB_CHECK_ARG(n_tensors > 0 && n_chunks > 0 && chunk_elems > 0 && chunk_elems % 4 == 0, "bad table sizes");
    CAB_CHECK_ARG(grad_ptrs && numels && chunk_tensor && chunk_off && ws_sumsq, "null pointer argument");
    CAB_CHECK_ARG(mode == 2 ? total_norm_out != nullptr : (param_ptrs && mom_ptrs && ws_scale && step_cell && ws_first && lr_dev), "null pointer argument");
    CAB_CHECK_ARG(mode != 1 || ema != nullptr, "NovoGrad needs the ema state");
    int launches = 1;
    const bool need_norm = mode >= 1 || (max_grad_norm > 0.f && ext_total_norm == nullptr) || total_norm_out != nullptr;
    // ws_sumsq: [n_tensors] per-tensor sums followed by [n_chunks] per-chunk partials
    if (need_norm) {
        mt_sumsq_kernel<<<n_chunks, kOptThreads, 0, stream>>>(reinterpret_cast<const long long*>(grad_ptrs), reinterpret_cast<const long long*>(numels), chunk_tensor, reinterpret_cast<const long long*>(chunk_off), chunk_elems, ws_sumsq + n_tensors);
        CAB_CHECK_LAUNCH();
        ++launches;
    } else {
        CAB_CHECK_CUDA(cudaMemsetAsync(ws_sumsq, 0, sizeof(float) * n_tensors, stream));
    }
    mt_prepare_kernel<<<1, 256, 0, stream>>>(ws_sumsq, need_norm ? ws_sumsq + n_tensors : nullptr, chunk_tensor, n_chunks, n_tensors, mode, (need_norm || ext_total_norm) ? max_grad_norm : 0.f, beta2, eps, ema, ws_scale, reinterpret_cast<long long*>(step_cell), ws_first, total_norm_out, ext_total_norm);
    CAB_CHECK_LAUNCH();
    if (mode == 2) {
        g_launch_count.fetch_add(launches, std::memory_order_relaxed);
        return 0;
    }
    mt_update_kernel<<<n_chunks, kOptThreads, 0, stream>>>(reinterpret_cast<const long long*>(param_ptrs), reinterpret_cast<const long long*>(grad_ptrs), reinterpret_cast<const long long*>(mom_ptrs), reinterpret_cast<const long long*>(numels), chunk_tensor, reinterpret_cast<const long long*>(chunk_off), chunk_elems, ws_scale, ws_first, lr_dev, mode, momentum, weight_decay, dampening, nesterov);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(launches + 1, std::memory_order_relaxed);
    return 0;
}
