/*
 * convasr_b200 -- C ABI of the B200-native (sm_100a) acoustic-model hot path of convasr.
 *
 * The reference (vadimkantorov/convasr) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md section 8b); the boundary it exposes is the Python module surface
 * `models / ctc / decoders / transcript_generators`.  This header is the C layer that the
 * drop-in Python modules in `convasr_b200/` bind with ctypes.  Every entry point names the
 * reference call site (file:line under the reference tree) whose arithmetic it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller owns all buffers (including workspaces) and passes the CUDA stream;
 *   - kernels never allocate, never synchronise;
 *   - return value: 0 = ok, negative = error, message via cab_last_error() (thread local);
 *   - "frac" lengths are the reference's fp32 fractions in (0, 1]: the integer length of a
 *     row of extent T is ceil(fp32(frac) * T)  (models.py:611-614).
 */
#ifndef CONVASR_B200_H
#define CONVASR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cab_stream_t; /* cudaStream_t */

#define CAB_ABI_VERSION 3

int cab_abi_version(void);
const char* cab_last_error(void);
/* number of kernels launched by this library since load (bench.py reports it) */
int64_t cab_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * A1 + A2: signal normalisation + log-mel filterbank frontend
 *   replaces models.normalize_signal (models.py:684-686) and
 *   LogFilterBankFrontend.forward (models.py:565-597): x/(max|x|+1e-5) -> pre-emphasis
 *   (y0=x0) -> *mask -> reflect pad (nfft/2) left / zero pad right -> STFT(nfft, hop, win
 *   centred in nfft, center=False) -> re^2+im^2 -> mel matmul + eps -> log.
 *   signal: [B, T] fp32 or int16 (int16 is cast without rescaling, models.py:568)
 *   xlen_frac: [B] or NULL (no mask)
 *   window: [win_length] fp32, mel_fb: [n_mels, nfft/2+1] fp32 row-major
 *   mel_band: [n_mels, 2] int32, first / one-past-last non-zero bin of each mel filter
 *   twiddle: [nfft/2] float2 (cos, -sin)(2*pi*k/nfft) computed by the host in fp64
 *   out_logmel: [B, n_mels, F] fp32, F = T / hop + 1
 *   ws_absmax: [B] fp32 workspace (written)
 * ------------------------------------------------------------------------------------- */
int cab_frontend_logmel(const void* signal, int signal_is_int16, const float* xlen_frac, int B,
                        int T, int win_length, int hop, int nfft, int n_mels,
                        const float* window, const float* mel_fb, const int32_t* mel_band,
                        const float* twiddle, float preemphasis, float log_eps, int normalize_signal,
                        float denom_multiplier, float* out_logmel, float* ws_absmax,
                        cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A3 + A4: masked instance norm (models.py:694-719, called at :298-301) fused with the
 *   layout change the conv stack wants: fp32 [B, C, F] -> bf16 channels-last [B, F_pad, C].
 *   With xlen_frac: statistics over the valid frames only, biased variance, output exactly 0
 *   for frames >= ceil(frac*F).  Without: plain biased instance norm over all F frames.
 *   normalize: 0 = layout change only (model built with normalize_features=False)
 *   out_hi: NULL, or bf16 [B, F_pad, C_pad]  (frames F..F_pad-1 and channels C..C_pad-1 are zeroed)
 *   out_lo: NULL, or bf16 residual (x - float(hi)) for the split-bf16 "fp32" tier
 *   out_f32: NULL, or fp32 [B, C, F] normalised features in the reference layout
 *   ws_stats: [B, C, 2] fp32 workspace (mean, rstd)
 * ------------------------------------------------------------------------------------- */
int cab_instnorm_pack(const float* feat, const float* xlen_frac, int B, int C, int F, float eps,
                      int normalize, int F_pad, int C_pad, void* out_hi, void* out_lo, float* out_f32,
                      float* ws_stats, cab_stream_t stream);

/* A1-A4 in one call (what JasperNet.forward does at models.py:286-301 before the backbone): signal -> per-utterance
 * normalisation -> log-mel (ws_logmel: fp32 [B, n_mels, F], also a valid output) -> masked instance norm -> bf16
 * channels-last features.  Three launches: abs-max, the STFT / mel / log kernel (which also emits per-tile instance-norm
 * partial statistics), normalise + pack.  normalize_features: 0 = layout change only; norm_masked: statistics over the valid
 * frames (normalize_features_temporal_mask).  ws_partials: fp32 [B, ceil(F / 64) + 1, n_mels, 2]; ws_absmax: 2 * B floats.  Other arguments as in
 * cab_frontend_logmel / cab_instnorm_pack. */
int cab_frontend_features(const void* signal, int signal_is_int16, const float* xlen_frac, int B, int T,
                          int win_length, int hop, int nfft, int n_mels, const float* window,
                          const float* mel_fb, const int32_t* mel_band, const float* twiddle, float preemphasis,
                          float log_eps, int normalize_signal, float denom_multiplier, int normalize_features,
                          int norm_masked, float norm_eps, float* ws_logmel, int F_pad, int C_pad, void* out_hi,
                          void* out_lo, float* out_f32, float* ws_absmax, float* ws_partials,
                          cab_stream_t stream);

/* cab_frontend_features under FIXED normalisation (nfft = 256 frontend only): every sample is multiplied by
 * signal_scale[b] instead of being divided by the utterance's abs-max, and the instance norm applies the caller's
 * statistics: out = (logmel - mean) * invstd with norm_stats fp32 [B, n_mels, 2] = (mean, invstd).  Two launches, no
 * statistics are computed.  norm_masked: frames >= ceil(xlen_frac * F) are written as 0 (as cab_frontend_features).
 * ws_logmel: fp32 [B, n_mels, T / hop + 1]. */
int cab_frontend_features_fixed(const void* signal, int signal_is_int16, const float* xlen_frac, int B, int T, int win_length,
                                int hop, int nfft, int n_mels, const float* window, const float* mel_fb,
                                const int32_t* mel_band, const float* twiddle, float preemphasis, float log_eps,
                                const float* signal_scale, const float* norm_stats, int norm_masked, float* ws_logmel,
                                int F_pad, int C_pad, void* out_hi, void* out_lo, cab_stream_t stream);

/* Streaming frontend (convasr_b200/streaming.py): the frames of cab_frontend_features_fixed, computed from per-stream
 * staged samples.  staged: fp32 [B, pitch] (16-byte aligned, pitch a multiple of 4); rows: device int32 [B, 5] =
 * (first frame, frames, base, staged, reflect): row b holds samples [base, base + staged) of its stream, emits frames
 * [first, first + frames) to out rows [0, frames) (rows up to F - 1 are written and are don't-care), samples at or past
 * base + staged read as 0 (the right zero pad at the end of the stream) and reflect selects the reflect (1) or constant
 * (0) left pad.  Frames whose window starts before sample 0 need base = 0.  out_hi / out_lo: bf16 [B, F, C_pad];
 * ws_logmel: fp32 [B, n_mels, F]. */
int cab_frontend_stream(const float* staged, int pitch, const int32_t* rows, int B, int F, int win_length, int hop, int nfft,
                        int n_mels, const float* window, const float* mel_fb, const int32_t* mel_band, const float* twiddle,
                        float preemphasis, float log_eps, const float* signal_scale, const float* norm_stats,
                        float* ws_logmel, int C_pad, void* out_hi, void* out_lo, cab_stream_t stream);

/* Batched device copies of the streaming model: jobs is a device int64 [n_jobs, 3] of (dst, src, bytes); src 0 writes
 * zeros.  Pointers and sizes are multiples of 16 bytes, max_bytes bounds every size, and no two ranges of one call
 * overlap.  One launch for all jobs (gather of launch inputs, append of new rows, rebase of stream buffers). */
int cab_stream_copy(const int64_t* jobs, int n_jobs, int64_t max_bytes, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A5-A9: Conv1d (+folded BatchNorm) + residual 1x1 convs + activation + temporal mask as ONE
 *   tcgen05/TMEM implicit GEMM.  Replaces ConvBn1d.forward (models.py:127-139) in its
 *   fuse_conv_bn_eval form (models.py:141-151), ResidualActivation.forward (models.py:357-371)
 *   and the Decoder 1x1 projection + log_softmax + argmax
 *   (models.py:23-44, :316; transcript_generators.py:27).
 *
 *   out[b, t, :] = act( bias + sum_src sum_tap W_src[tap] . x_src[b, t + tap*dil - pad_left, :] )
 *                  * (t < ceil(frac_b * T_out))
 *   Activations are bf16 channels-last; a "source" is one (activation tensor, packed weight)
 *   pair: the main conv, each residual 1x1 conv, and -- in the split-bf16 "fp32" tier -- the
 *   hi*hi, hi*lo, lo*hi partial products.  Stride-2 convs are expressed by the host as
 *   stride-1 convs over the frame-pair view [B, T/2, 2C] with re-packed weights.
 * ------------------------------------------------------------------------------------- */
#define CAB_MAX_CONV_SOURCES 18

typedef struct {
    const void* act;   /* bf16 [B, T_rows, ld_ch]; rows >= T_in are never read (zero fill) */
    const void* wgt;   /* bf16 [taps, w_rows, w_ld_ch] (K-major: channel contiguous) */
    int32_t T_in;      /* valid rows per utterance */
    int32_t T_rows;    /* allocated rows per utterance (batch stride = T_rows * ld_ch) */
    int32_t ld_ch;     /* channels per activation row (allocation) */
    int32_t ch_off;    /* first channel of this source inside the row */
    int32_t C_in;      /* channels contracted, multiple of 64 */
    int32_t w_rows;    /* output-channel rows in the packed weight */
    int32_t w_ld_ch;   /* channels per weight row (allocation) */
    int32_t w_ch_off;  /* first channel inside the weight row */
    int32_t taps, dilation, pad_left;
} cab_conv_source_t;

enum { CAB_ACT_NONE = 0, CAB_ACT_RELU = 1, CAB_ACT_HARDTANH = 2, CAB_ACT_LEAKY_RELU = 3 };
enum {
    CAB_EPI_ACT_BF16 = 0,   /* bf16 channels-last activation (+ optional lo residual) */
    CAB_EPI_LOGSOFTMAX = 1, /* fp32 [B,C,T] logits + log_probs + int32 argmax, C <= 256 */
    CAB_EPI_LOGITS_F32 = 2, /* fp32 [B,C,T] logits only */
    CAB_EPI_LOGITS_ROWS = 3 /* large vocabularies: fp32 logits in CLASS-CONTIGUOUS memory [B, T_out, out_ld_ch] (TMA stores),
                               plus per-row log-sum-exp (written to `log_probs`, here fp32 [B, T_out]) and argmax from an
                               online softmax across the N tiles; cab_log_softmax_rows then writes the log-probs */
};

typedef struct {
    int32_t B, T_out, C_out; /* C_out: real output channels / classes */
    int32_t block_n;         /* N tile: multiple of 16 (32 for ACT_BF16), <= 256; 0 = auto */
    int32_t epilogue;        /* CAB_EPI_* */
    int32_t act;             /* CAB_ACT_* */
    float act_a, act_b;      /* hardtanh (min,max) or leaky slope in act_a */
    const float* bias;       /* [C_out] fp32 or NULL */
    const float* xlen_frac;  /* [B] or NULL: temporal mask (ACT_BF16 only) */
    void* out_hi;            /* ACT_BF16: bf16 [B, out_T_rows, out_ld_ch] */
    void* out_lo;            /* ACT_BF16: NULL or bf16 residual of the fp32 value */
    int32_t out_T_rows, out_ld_ch;
    float* logits;           /* LOGSOFTMAX / LOGITS_F32: fp32 [B, C_out, T_out] or NULL */
    float* log_probs;        /* LOGSOFTMAX: fp32 [B, C_out, T_out] or NULL */
    int32_t* argmax;         /* LOGSOFTMAX: int32 [B, T_out] or NULL (ties -> lowest id) */
    double* stats;           /* ACT_BF16: NULL, or fp64 [2][C_out]: the call zeroes it and the epilogue
                                accumulates per-channel sum / sum of squares of the stored outputs (bf16-rounded;
                                hi + lo in the split tier) over all B*T_out rows -- BatchNorm batch statistics for
                                training.  fp64 so that the order of the atomics cannot reach the fp32 result:
                                the forward pass is reproducible run to run and GPU to GPU */
    const float* skip_frac;  /* ACT_BF16: NULL, or [B]: output rows t >= ceil(skip_frac[b]*skip_T) + skip_margin of
                                utterance b are structural zeros (padding of a ragged batch whose input rows are
                                zero there, or gradient rows nobody reads): 128-row tiles lying entirely in that
                                range are not computed and are stored as zeros.  With xlen_frac set and skip_frac
                                NULL the launch's own temporal mask implies (xlen_frac, T_out, 0). */
    int32_t skip_T, skip_margin;
    /* Training, bf16 tier: BatchNorm-backward reduction folded into the dgrad launch that produces g = dL/d(out) of a
     * ConvBn1d repeat (models.py:127-139 under autograd).  bnr_partials (NULL = off): fp64
     * [CAB_BN_SUM_REPLICAS][2][bnr_C]; the call zeroes it and the epilogue accumulates, per channel, sum(dz) and
     * sum(dz * y) with dz = g * act'(y*scale + shift) * (t < ceil(bnr_xlen_frac[b]*T_out)), g as stored (bf16).
     * bnr_y: that repeat's pre-BatchNorm conv output, bf16 with the geometry of out_hi ([B, out_T_rows, out_ld_ch]);
     * bnr_ss: fp32 [4][bnr_C] as written by cab_bn_finalize / cab_bn_act_mask_fwd_stats (scale, shift, ...).
     * cab_bn_act_mask_bwd_apply then finishes the BatchNorm backward without re-reading (y, g) for the sums.
     * Needs out_lo == NULL and stats == NULL. */
    const void* bnr_y;
    const float* bnr_ss;
    const float* bnr_xlen_frac;
    double* bnr_partials;
    int32_t bnr_C, bnr_act;       /* real channel count; CAB_ACT_* of the repeat */
    float bnr_act_a, bnr_act_b;
} cab_conv_epilogue_t;

int cab_conv1d_fused(const cab_conv_source_t* sources_host, int n_sources,
                     const cab_conv_epilogue_t* epilogue_host, cab_stream_t stream);

/* FP8 inference tier: the same launch with E4M3 operands (tcgen05.mma kind::f8f6f4, fp32 accumulation in TMEM).
 *   Sources: act and wgt are E4M3 (1 byte per element); C_in a multiple of 128; ld_ch, w_ld_ch multiples of 16.
 *   Each source j carries activation scale s_j folded into its weights by the caller:
 *   wgt_j = e4m3(W_j * s_j / alpha[n]), alpha[n] = max_j(s_j * max|W_j[n, :]|) / 448, so that
 *   acc[t, n] * alpha[n] = sum_j s_j * x_q_j . W_j  (x_q_j: the stored E4M3 activation).
 *   alpha: fp32 [C_out], applied to the accumulator before the bias in every epilogue.
 *   CAB_EPI_ACT_BF16 here stores E4M3: out_hi = e4m3(act(acc * alpha + bias) * mask * out_scale_inv), saturating to
 *   +-448 (cvt.rn.satfinite), out_ld_ch a multiple of 16.  LOGSOFTMAX / LOGITS_F32 / LOGITS_ROWS write fp32 as above.
 *   Not available here: out_lo, stats, skip_frac, the folded BatchNorm-backward reduction. */
int cab_conv1d_fused_fp8(const cab_conv_source_t* sources_host, int n_sources,
                         const cab_conv_epilogue_t* epilogue_host, const float* alpha, float out_scale_inv,
                         cab_stream_t stream);
/* calibration of the FP8 tier: out[0] = max |x| over n bf16 elements (n < 2^31) */
int cab_absmax_bf16(const void* x, int64_t n, float* out, cab_stream_t stream);
/* out = e4m3(x * scale_inv) elementwise, saturating to +-448 (cvt.rn.satfinite); x bf16, n a multiple of 16, both 16-byte aligned */
int cab_quantize_e4m3(const void* x, int64_t n, float scale_inv, void* out, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Training: Conv1d weight gradient (autograd's wgrad behind loss.backward(), train.py:770-774)
 *   out[tap][m][n] = sum_{b,t} a[b, t, m] * bx[b, t + tap*dilation - pad_left, n]
 *   a: bf16 [B, a_T_rows, a_ld] (gradient w.r.t. the conv output), bx: bf16 [B, b_T_rows, b_ld]
 *   (conv input) -- or swapped by the caller, whichever side should be the 128-row M side.
 *   out: fp32 [taps, M_total, out_ld].  n_splits = 0 picks a batch split for >= 4 waves;
 *   with n_splits > 1 partial sums are reduced in L2 (the call zeroes `out` first).
 *   skip_frac (or NULL): frames t >= ceil(skip_frac[b]*skip_T) + skip_margin of utterance b contribute
 *   exact zeros (one operand is zero there: ragged batch padding) and are left out of the contraction.
 *   accumulate_into != 0: the products are ADDED to what `out` holds (split-bf16 tier: hi*hi, then hi*lo, lo*hi).
 * ------------------------------------------------------------------------------------- */
int cab_conv1d_wgrad(const void* a, int a_T, int a_T_rows, int a_ld, int M_total, const void* bx,
                     int b_T, int b_T_rows, int b_ld, int N_total, int B, int taps, int dilation,
                     int pad_left, float* out, int out_ld, int n_splits, const float* skip_frac, int skip_T,
                     int skip_margin, int accumulate_into, cab_stream_t stream);

/* Training-mode BatchNorm1d + activation + temporal mask around the conv GEMMs
 * (nn.BatchNorm1d(momentum, eps) inside ConvBn1d.forward, models.py:112-113,127-139):
 *   cab_bn_batch_stats : biased batch statistics over all B*T rows of y (bf16 [B,T,ld]); writes
 *                        out_ss = [scale, shift, mean, invstd] (fp32 [4][C]) and updates the running
 *                        statistics (unbiased running_var) when the pointers are non-NULL.
 *   cab_bn_act_mask_fwd: out = act(y*scale + shift) * (t < ceil(frac*T))
 *   cab_bn_act_mask_bwd: given grad_out w.r.t. `out`: sums = [dbeta, dgamma] (fp32 [2][C]) and
 *                        grad_y = scale * (dz - mean(dz) - xhat * mean(dz*xhat)),
 *                        dz = grad_out * act'(z) * mask  (hardtanh: a < z < b strictly).
 *   dropout_p > 0 applies F.dropout after the activation (ResidualActivation.forward, models.py:357-371):
 *   out *= keep / (1 - p) with a counter-based keep decision from (*seed, salt, element index) that
 *   the backward recomputes; *seed lives in device memory so CUDA-graph replays draw new masks.
 *   Both are HBM-bound streaming kernels: persistent CTAs pull whole rows through shared-memory stages
 *   with bulk async copies.  The backward's channel sums are accumulated in CAB_BN_SUM_REPLICAS copies
 *   (ws_partials) to keep same-address atomics short; with ws_partials == NULL a slower variant runs. */
#define CAB_BN_SUM_REPLICAS 8
int cab_bn_batch_stats(const void* y, int B, int T, int C, int ld, const float* gamma, const float* beta,
                       float eps, float momentum, float* running_mean, float* running_var,
                       double* ws_sums, float* out_ss, cab_stream_t stream);
/* same as cab_bn_batch_stats but from sums the conv epilogue already accumulated (cab_conv_epilogue_t.stats) */
int cab_bn_finalize(const double* sums, int n_rows, int C, const float* gamma, const float* beta, float eps,
                    float momentum, float* running_mean, float* running_var, float* out_ss,
                    cab_stream_t stream);
/* *_lo: NULL, or the bf16 residual halves of the split-bf16 "fp32" tier (value = hi + lo) -- all of a call's
 * tensors together. */
int cab_bn_act_mask_fwd(const void* y, const void* y_lo, const float* ss, int B, int T, int C, int ld, int act,
                        float act_a, float act_b, const float* xlen_frac, void* out, void* out_lo,
                        float dropout_p, const int64_t* seed, int64_t salt, cab_stream_t stream);
/* frozen != 0: the BatchNorm is in eval mode inside a training model (model.freeze, models.py:328-339): it
 * normalised with its running statistics, so grad_y = scale * dz without the batch-statistics terms. */
int cab_bn_act_mask_bwd(const void* y, const void* y_lo, const void* grad_out, const void* grad_out_lo,
                        const float* ss, int B, int T, int C, int ld, int act, float act_a, float act_b,
                        const float* xlen_frac, float* sums, void* grad_y, void* grad_y_lo, float dropout_p,
                        const int64_t* seed, int64_t salt, int frozen,
                        double* ws_partials /* fp64 [CAB_BN_SUM_REPLICAS][2][C] scratch, or NULL */,
                        cab_stream_t stream);
/* Second half of cab_bn_act_mask_bwd alone: `partials` (fp64 [CAB_BN_SUM_REPLICAS][2][C]) already hold the channel sums --
 * accumulated by the dgrad launch that produced grad_out (cab_conv_epilogue_t.bnr_partials) -- so only the apply pass runs:
 * sums = [dbeta, dgamma], grad_y.  bf16 tier or split tier alike; dropout_p must be what the sums were taken with (0 for the
 * folded reduction). */
int cab_bn_act_mask_bwd_apply(const void* y, const void* y_lo, const void* grad_out, const void* grad_out_lo,
                              const float* ss, int B, int T, int C, int ld, int act, float act_a, float act_b,
                              const float* xlen_frac, float* sums, void* grad_y, void* grad_y_lo, float dropout_p,
                              const int64_t* seed, int64_t salt, int frozen, const double* partials,
                              cab_stream_t stream);
/* Host-only query (no device work): 1 when cab_bn_act_mask_bwd_apply covers an activation of R = B*T rows with row pitch ld in
 * the given tier (split != 0: split-bf16), else 0 -- the caller then keeps the separate reduce pass (cab_bn_act_mask_bwd) instead of
 * folding the reduction into the dgrad launch. */
int cab_bn_bwd_apply_covers(int R, int ld, int split);
/* cab_bn_finalize + cab_bn_act_mask_fwd in one launch: every CTA derives the coefficients of its channels from
 * the raw sums of the conv epilogue (raw_sums: fp32 [2][sums_ld]); CTA 0 also writes out_ss and moves the
 * running statistics. */
int cab_bn_act_mask_fwd_stats(const void* y, const void* y_lo, const double* raw_sums, int sums_ld, int n_rows,
                              const float* gamma, const float* beta, float eps, float momentum,
                              float* running_mean, float* running_var, float* out_ss, int B, int T, int C,
                              int ld, int act, float act_a, float act_b, const float* xlen_frac, void* out,
                              void* out_lo, float dropout_p, const int64_t* seed, int64_t salt,
                              cab_stream_t stream);
/* Residual topologies (ConvBn1d.forward models.py:129-133, ResidualActivation.forward :357-371): on the last
 * repeat of a block every residual source passes its own 1x1 conv + BatchNorm and is added before the
 * activation ('flat' residuals are added unchanged: ss == NULL).
 *   cab_bn_multi_act_mask_fwd: out = mask(dropout(act(sum_i (scale_i * y_i + shift_i))))
 *   cab_act_mask_bwd_dz      : dz = grad_out * act'(z) * mask * dropout, the gate read off the stored `out`;
 *                              each BatchNorm branch then runs cab_bn_act_mask_bwd(y_i, dz, act = NONE). */
#define CAB_MAX_BN_BRANCHES 12
typedef struct {
    const void* y;    /* bf16 [B, T, ld] branch input (conv output) */
    const void* y_lo; /* NULL or its split-bf16 residual */
    const float* ss;  /* [4][C] scale, shift, mean, invstd -- or NULL for an identity branch */
} cab_bn_branch_t;
int cab_bn_multi_act_mask_fwd(const cab_bn_branch_t* branches_host, int n_branches, int B, int T, int C, int ld,
                              int act, float act_a, float act_b, const float* xlen_frac, void* out,
                              void* out_lo, float dropout_p, const int64_t* seed, int64_t salt,
                              cab_stream_t stream);
int cab_act_mask_bwd_dz(const void* out, const void* out_lo, const void* grad_out, const void* grad_out_lo,
                        int B, int T, int C, int ld, int act, float act_a, float act_b,
                        const float* xlen_frac, void* dz, void* dz_lo, float dropout_p, const int64_t* seed,
                        int64_t salt, cab_stream_t stream);
/* fp32 [Co,Ci,K] -> bf16 tap-major [K,Co,ci_ld] (forward operand) and/or [K,Ci,co_ld] with flipped
 * taps (dgrad operand); and the inverse for a packed fp32 gradient ([K,Co,ld] or, transposed,
 * [K,Ci,ld]) into the parameter layout. */
int cab_pack_weight(const float* w, int Co, int Ci, int K, void* fwd, int ci_ld, void* dgrad, int co_ld,
                    cab_stream_t stream);
/* the same for up to 32 weights in one launch (all layers of a model at the start of a training step) */
typedef struct {
    const float* w;  /* fp32 [Co, Ci, K] */
    void* fwd;       /* bf16 [K, Co, ci_ld] or NULL */
    void* dgrad;     /* bf16 [K, Ci, co_ld] (taps flipped) or NULL */
    void* fwd_lo;    /* NULL, or the split-bf16 residual of fwd */
    void* dgrad_lo;  /* NULL, or the split-bf16 residual of dgrad */
    int32_t Co, Ci, K, ci_ld, co_ld;
    int32_t mode;    /* 0: plain; 1: stride-2 conv as a stride-1 conv over frame pairs -- fwd is
                        [ (K + 1) / 2 + (pad odd), Co, ci_ld = 2 * ci_alloc ] zero-initialised by the caller,
                        tap kk -> pair tap floor((kk - pad) / 2) - floor(-pad / 2), channel block (kk - pad) mod 2 */
    int32_t pad;     /* mode 1: the strided conv's padding */
} cab_pack_item_t;
int cab_pack_weights_batched(const cab_pack_item_t* items_host, int n_items, cab_stream_t stream);
/* transposed: 0 packed = [K, Co, ld]; 1 packed = [K, Ci, ld]; 2 packed = the stride-2 pair layout of pack mode 1
 * (pair_pad = the conv's padding, pair_ci_alloc = channels per pair half) */
int cab_unpack_wgrad(const float* packed, int K, int Co, int Ci, int ld, int transposed, float* grad,
                     int accumulate, int pair_pad, int pair_ci_alloc, cab_stream_t stream);
/* the same for up to 32 gradients in one launch (every layer of a model at the end of the backward) */
typedef struct {
    const float* packed; /* fp32 packed gradient as cab_conv1d_wgrad wrote it */
    float* grad;         /* fp32 [Co, Ci, K] */
    int32_t K, Co, Ci, ld, transposed, pair_pad, pair_ci_alloc;
} cab_unpack_item_t;
int cab_unpack_wgrad_batched(const cab_unpack_item_t* items_host, int n_items, cab_stream_t stream);
/* fp32 [B,C,T] (gradient w.r.t. the logits) -> bf16 channels-last [B,T,ld]; class_sums (fp32 [C],
 * optional) receives the sums over (b,t) = the decoder bias gradient. */
int cab_bct_to_btc(const float* x, int B, int C, int T, int ld, void* out, void* out_lo, float* class_sums,
                   cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * section 8f "next" #3: multi-tensor optimizer step with gradient-norm clipping folded in.
 *   mode 0: torch.optim.SGD(momentum, dampening, weight_decay, nesterov)   (train.py:657-662)
 *   mode 1: NovoGrad (optimizers.py:66-90); `momentum` = beta1, `dampening` != 0 = the dampening flag
 *   mode 2: gradient norm only -- total_norm_out = ||all gradients of the table||, nothing is updated
 *   max_grad_norm > 0: torch.nn.utils.clip_grad_norm_ (train.py:776-779) applied first; the norm is this
 *   table's own, or *ext_total_norm (device fp32) when given -- clipping is global over all parameter groups,
 *   so a multi-group optimizer first runs mode 2 over every parameter and passes the result to each group.
 *   Tensors are described by DEVICE tables: param/grad/momentum pointers (int64 [n]), element counts
 *   (int64 [n]) and a flat chunk list (tensor index int32 [n_chunks], element offset int64
 *   [n_chunks], chunk_elems elements per chunk, multiple of 4).  ema: fp32 [n] NovoGrad state.
 *   step_cell: int64 device cell counting steps (0 = first step initialises ema / momentum);
 *   lr_dev: fp32 device scalar (so CUDA-graph replays can change it); ws_sumsq: n + n_chunks floats (per-tensor sums, then the
 *   per-chunk partials they are summed from in a fixed order: no atomics, bit-reproducible norms), ws_scale: n floats, ws_first: one int32; total_norm_out: fp32 [1] or NULL (pre-clip global gradient norm).
 * ------------------------------------------------------------------------------------- */
int cab_optimizer_step(int mode, int n_tensors, const int64_t* param_ptrs, const int64_t* grad_ptrs,
                       const int64_t* mom_ptrs, const int64_t* numels, int n_chunks,
                       const int32_t* chunk_tensor, const int64_t* chunk_off, int chunk_elems,
                       float* ws_sumsq, float* ema, float* ws_scale, int64_t* step_cell, int32_t* ws_first,
                       const float* lr_dev, float momentum, float beta2, float eps, float weight_decay,
                       float dampening, int nesterov, float max_grad_norm, float* total_norm_out,
                       const float* ext_total_norm, cab_stream_t stream);

/* grouped Conv1d (+ bias + ReLU when relu != 0) of the separable blocks (models.py:50-64): bf16 channels-last
 * in [B, T_rows, ld_in] / out [B, out_T_rows, ld_out] (channels C_out..ld_out-1 are zeroed),
 * weight fp32 [C_out, C_in/groups, k] (PyTorch layout), stride 1, dilation 1, T frames in and out.
 * act_lo / out_lo: NULL, or the bf16 residual halves of the split-bf16 "fp32" tier.
 * relu == 0 with in-group transposed, tap-flipped weights is the conv's input gradient (training). */
int cab_grouped_conv1d(const void* act, const void* act_lo, int B, int T, int T_rows, int C_in,
                       int ld_in, const float* wgt, const float* bias, int C_out, int groups,
                       int k, int pad_left, void* out, void* out_lo, int out_T_rows, int ld_out, int relu,
                       cab_stream_t stream);
/* FP8 inference tier: the same grouped conv + bias + ReLU with E4M3 input (x = q * in_scale, ld_in a multiple of 16) and
 * E4M3 output e4m3(v * out_scale_inv), saturating; odd k in 3..27 with the input window of 64 outputs at most 208 channels. */
int cab_grouped_conv1d_fp8(const void* act, int B, int T, int T_rows, int C_in, int ld_in, float in_scale,
                           const float* wgt, const float* bias, int C_out, int groups, int k, int pad_left,
                           void* out, int out_T_rows, int ld_out, float out_scale_inv, cab_stream_t stream);
/* training: weight / bias gradient of that grouped conv (autograd's grouped wgrad behind loss.backward(),
 * train.py:770-774):  dw[co, j, k] = sum_{b,t} dy[b,t,co] * x[b, t + k - pad, g(co)*cin_g + j]  (fp32 [C_out, C_in/groups, k],
 * zeroed by the call), db[co] = sum_{b,t} dy[b,t,co] (fp32 [C_out] or NULL).  Odd k with pad = k / 2. */
int cab_grouped_conv1d_wgrad(const void* dy, const void* dy_lo, int dy_T_rows, int ld_dy, const void* x,
                             const void* x_lo, int B, int T, int T_rows, int C_in, int ld_in, int C_out,
                             int groups, int k, int pad_left, float* dw, float* db, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A10 (+A13/A14 argmax): log_softmax over the class dim of [B, C, T] (models.py:316) fused
 *   with the per-frame argmax (transcript_generators.py:27).  in_dtype: 0 fp32, 1 bf16.
 * ------------------------------------------------------------------------------------- */
int cab_log_softmax_argmax(const void* logits, int in_dtype, int B, int C, int T,
                           float* out_log_probs, int32_t* out_argmax, cab_stream_t stream);
/* second half of the fused large-vocabulary head: out[r, c] = logits[r, c] - lse[r] over R rows of C classes (row pitch ld) */
int cab_log_softmax_rows(const float* logits, const float* lse, int64_t R, int C, int ld, float* out_log_probs,
                         cab_stream_t stream);
/* backward of log_softmax over dim 1: gin = gout - exp(lp) * sum_c gout */
int cab_log_softmax_bwd(const float* log_probs, const float* grad_out, int B, int C, int T,
                        float* grad_in, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A11: CTC loss, the arithmetic of torch.nn.functional.ctc_loss(reduction='none',
 *   zero_infinity=False) as called at models.py:323.  log_probs is addressed through
 *   element strides so both [T,B,C] and the permuted [B,C,T] view work without a copy.
 *   targets: int64 [B, L_max] padded; input_lengths / target_lengths: int64 [B].
 *   ws_alpha / ws_beta: fp32 [B, T, 2*L_max+1] workspaces.  nll: fp32 [B].
 *   ws_offsets: fp64 [B, 2, (T+7)/8 + 2] workspace (re-centring offsets of the recursions and the
 *   log-likelihood; alpha/beta are stored relative to them so fp32 stays accurate for long inputs).
 *   cab_ctc_loss_fwd with a non-NULL ws_beta also runs the beta recursion, concurrently with
 *   alpha in the same grid (the caller then passes beta_ready=1 to cab_ctc_loss_bwd).
 *   The backward returns ATen's convention: (exp(lp) - occupancy) * grad_out, zero for
 *   t >= input_length, laid out like log_probs (grad strides given separately).
 * ------------------------------------------------------------------------------------- */
int cab_ctc_loss_fwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                     const int64_t* targets, const int64_t* input_lengths,
                     const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                     float* ws_alpha, float* ws_beta_or_null, double* ws_offsets, float* nll,
                     cab_stream_t stream);
int cab_ctc_loss_bwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                     const int64_t* targets, const int64_t* input_lengths,
                     const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                     const float* ws_alpha, float* ws_beta, int beta_ready, double* ws_offsets,
                     const float* grad_out, float* grad, int64_t gstride_t, int64_t gstride_b,
                     int64_t gstride_c, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A11, long targets: the same loss and gradient for L_max <= 65535 (about an hour of speech).
 *   cab_ctc_loss_fwd/bwd take a batch when cab_ctc_loss_one_cta_covers(L_max) returns 1 (host only:
 *   L_max <= 1345, where one CTA stages 8 frames of emissions in shared memory); beyond, these run
 *   one thread-block cluster of up to 16 CTAs per utterance and direction, the extended states in
 *   contiguous slices, neighbouring slices exchanging boundary values through distributed shared
 *   memory at every frame.  The nll is bit-identical to cab_ctc_loss_fwd wherever both run; the
 *   gradient differs only in the order of its atomic additions.
 *   ws_alpha: fp32 [B, T, 2*L_max+1], cab_ctc_loss_long_workspace gives its size in bytes (host only,
 *   64-bit; fails for L_max > 65535).  cab_ctc_loss_long_fwd with ws_alpha NULL computes the loss
 *   only and needs no [B, T, S] workspace; with ws_alpha it stores alpha for cab_ctc_loss_long_bwd,
 *   which recomputes beta and writes the gradient without a second workspace.  ws_offsets, nll,
 *   grad and the strides as for cab_ctc_loss_fwd/bwd; ws_offsets carries the forward's offsets and
 *   log-likelihood to the backward.  states_per_cta as for cab_ctc_alignment_long.  No host
 *   synchronisation and no allocation: both can be captured into a CUDA graph.
 * ------------------------------------------------------------------------------------- */
int cab_ctc_loss_one_cta_covers(int L_max);
int cab_ctc_loss_long_workspace(int B, int T, int L_max, int64_t* bytes);
int cab_ctc_loss_long_fwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                          const int64_t* targets, const int64_t* input_lengths,
                          const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                          float* ws_alpha_or_null, double* ws_offsets, float* nll, int states_per_cta,
                          cab_stream_t stream);
int cab_ctc_loss_long_bwd(const float* log_probs, int64_t stride_t, int64_t stride_b, int64_t stride_c,
                          const int64_t* targets, const int64_t* input_lengths,
                          const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                          const float* ws_alpha, double* ws_offsets, const float* grad_out, float* grad,
                          int64_t gstride_t, int64_t gstride_b, int64_t gstride_c, int states_per_cta,
                          cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A12: forced alignment, ctc.alignment (ctc.py:6-75) with all of its quirks: finite "zero"
 *   (finfo.min), logsumexp alpha with argmax back-pointers (stay preferred on ties), the
 *   recursion runs over all T frames of the padded batch, terminal state read at global T-1,
 *   back-trace from input_length-1, output = last frame index per target label.
 *   ws_backptr: uint8 [B, T, 2*L_max+1] workspace.  out: int64 [B, L_max].
 *   fp16_arithmetic != 0: log_probs are the fp32 images of an fp16 tensor and the recursion rounds to
 *   fp16 after every operation, "zero" = finfo(float16).min -- what the reference computes when it is
 *   handed fp16 log_probs (ctc.py:29).  fp16_exp_table / fp16_log_table (both or neither; device, uint16
 *   [65536]): exp and log as maps from fp16 bit pattern to fp16 bit pattern, e.g. tabulated with the host's torch --
 *   the recursion then equals that implementation's fp16 arithmetic bit for bit; NULL: expf / logf rounded to fp16.
 * ------------------------------------------------------------------------------------- */
int cab_ctc_alignment(const float* log_probs, int64_t stride_t, int64_t stride_b,
                      int64_t stride_c, const int64_t* targets, const int64_t* input_lengths,
                      const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                      uint8_t* ws_backptr, int64_t* out_alignment, int fp16_arithmetic,
                      const uint16_t* fp16_exp_table, const uint16_t* fp16_log_table, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A12, long targets: the same alignment (same arguments, same result wherever both run) for
 *   L_max <= 65535 (S_max = 2*L_max+1 <= 131071); cab_ctc_alignment stops at S_max <= 4096.
 *   One thread-block cluster of up to 16 CTAs per utterance, the extended states split into
 *   contiguous slices, neighbouring slices exchanging their boundary alpha through distributed
 *   shared memory at every frame; then a back-trace launch (one warp per utterance).
 *   ws_backptr: packed back-pointers, 2 bits per state, 4 states per byte (state s in bits 2*(s%4)),
 *   uint8 [B, T, ceil((2*L_max+1)/4)]; cab_ctc_alignment_long_workspace gives its size in bytes
 *   (host only, no device work) and fails, like cab_ctc_alignment_long, for L_max > 65535.
 *   states_per_cta: 0 = the library picks the slice size; > 0 (a multiple of 4) forces it, and
 *   slices beyond 16 CTAs go round-robin over the cluster (at most 8192 states per CTA).
 * ------------------------------------------------------------------------------------- */
int cab_ctc_alignment_long_workspace(int B, int T, int L_max, int64_t* bytes);
int cab_ctc_alignment_long(const float* log_probs, int64_t stride_t, int64_t stride_b,
                           int64_t stride_c, const int64_t* targets, const int64_t* input_lengths,
                           const int64_t* target_lengths, int B, int T, int C, int L_max, int blank,
                           uint8_t* ws_backptr, int64_t* out_alignment, int fp16_arithmetic,
                           const uint16_t* fp16_exp_table, const uint16_t* fp16_log_table,
                           int states_per_cta, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A13: GreedyDecoder.decode (decoders.py:5-16): per-frame top-K class ids of [B, C, T],
 *   out int32 [B, K, T], ordered by descending value, ties -> lowest id first.
 * ------------------------------------------------------------------------------------- */
int cab_topk_ids(const float* log_probs, int B, int C, int T, int K, int32_t* out_ids,
                 cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * A14: the collapse state machine of GreedyCTCGenerator.generate
 *   (transcript_generators.py:32-83) on device: a segmented warp scan, one utterance per warp.
 *   ids: int32 [B, T] per-frame argmax; lengths: int32 [B] (loop bound, "sample_len").
 *   is_silence / is_word_start: uint8 [C] token class tables.
 *   out_tokens / out_frames: int32 [B, T_cap]; out_frames[i] is the frame the token came
 *   from, or -(frame+1) for a space synthesised by the blank_amount_to_space rule.
 *   out_counts: int32 [B]; -1 marks "only silence in the whole row" (empty transcript).
 * ------------------------------------------------------------------------------------- */
int cab_greedy_collapse(const int32_t* ids, const int32_t* lengths, int B, int T, int C,
                        int eps_id, int space_id, const uint8_t* is_silence,
                        const uint8_t* is_word_start, int blank_amount_to_space,
                        int32_t* out_tokens, int32_t* out_frames, int T_cap, int32_t* out_counts,
                        cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * section 8(f) "next" #1: uncertainty reductions on log_probs (models.py:645-678), fused:
 *   per utterance entropy (masked mean) and weighted_mean_entropy with eps_id weights.
 * ------------------------------------------------------------------------------------- */
/* models.margin (models.py:676-677): the two largest probabilities per frame, out fp32 [B, 2, T] = exp(top-2 of log_probs over
 * the class dim); log_probs [B, C, T] through element strides. */
int cab_top2_probs(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t, int B, int C, int T,
                   float* out, cab_stream_t stream);
int cab_entropy(const float* log_probs, const int64_t* lengths, int B, int C, int T, int eps_id,
                float* out_entropy, float* out_weighted_entropy, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * CTC prefix beam search without a language model (decoders.BeamSearchDecoder; the acoustic
 *   part of ctcdecode's CTCBeamDecoder, alpha = beta = 0).  fp32 log domain, full-precision
 *   expf / logf: the result of an utterance does not depend on the batch it is in.
 *   log_probs [B, C, T] through element strides; output_lengths int64 [B] (frames searched,
 *   clamped to [0, T]).  Per frame the top N = min(cutoff_top_n, C) classes are kept (ties ->
 *   lower class id), then, with cutoff_prob < 1, only those (by descending probability) until
 *   the fp32 running sum of probabilities reaches cutoff_prob, the class that crosses it
 *   included.  W beams per utterance; candidates are ranked by log(p_blank + p_nonblank), ties
 *   to the lower (source beam rank, class id); probability zero is never a candidate.
 *   out_tokens / out_frames: int32 [B, K, L_cap], the K best hypotheses best first, with the
 *   frame at which each token's prefix was created; -1 past the hypothesis' length.
 *   out_lengths: int32 [B, K]; out_scores: fp32 [B, K] = log(p_blank + p_nonblank) at the last
 *   frame, -inf (length 0) where fewer than K hypotheses have nonzero probability.
 *   Refused before any launch: W outside [1, 128], N outside [1, 64] or above C, K outside
 *   [1, W], blank outside [0, C), cutoff_prob outside (0, 1], a workspace smaller than
 *   cab_ctc_beam_search_workspace reports (host only, no device work).  Three launches.
 * ------------------------------------------------------------------------------------- */
int cab_ctc_beam_search_workspace(int B, int T, int C, int N, int W, int K, int blank, float cutoff_prob,
                                  int64_t* bytes);
int cab_ctc_beam_search(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t,
                        const int64_t* output_lengths, int B, int T, int C, int N, float cutoff_prob,
                        int blank, int W, int K, void* workspace, int64_t workspace_bytes,
                        int32_t* out_tokens, int32_t* out_frames, int L_cap, int32_t* out_lengths,
                        float* out_scores, cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * The same search with a word n-gram language model fused in (shallow fusion, ctcdecode's
 *   word-level scorer rules; convasr_b200/lm.py builds the tables from an ARPA file).
 *   Labels are single characters; `space` is the label that ends a word.
 *   N-gram tables: one per order k = 1..order, open addressing with linear probing, `sizes[k-1]`
 *   entries (a power of two) of 16 bytes {uint64 key, float log10 p, float log10 back-off};
 *   key 0 marks an empty slot.  The key of the word-id sequence (w1 .. wk) folds the ids
 *   newest first: h = 0; for id = wk .. w1: h = splitmix64(h + 0x9E3779B97F4A7C15 * (id + 1));
 *   the slot probed first is key & (size - 1).  Each table needs at least one empty slot, or a
 *   key it does not hold is only found absent after a full pass (lm.py builds at load <= 1/2).
 *   Dictionary trie over label ids: child int32 [num_nodes, num_classes] (-1 = no child), node 0
 *   the root; word int32 [num_nodes], the word id a node spells or -1.
 *   A prefix is admissible when every run of labels a space follows is a word, the last run
 *   is a prefix of a word, and no space is first or follows a space; other extensions are not
 *   candidates.  Extending a beam whose current word w is complete by `space` adds
 *   alpha * ln(10) * log10 P(w | last order-1 words, <s>-padded) + beta to the extension (and
 *   to a merge into a beam holding that prefix).  After the last frame each non-empty beam
 *   not ending in a space gets the same term for its last word (-1000 before alpha if that
 *   word is incomplete), and the beams are re-ranked by it (ties to the earlier rank);
 *   out_scores are these fused scores.  Uses cab_ctc_beam_search_workspace's workspace.
 *   Refused before any launch, besides the checks above: a null lm or table, order outside
 *   [1, 6], a table size that is not a power of two, num_classes != C, space outside [0, C)
 *   or equal to blank, num_nodes < 1, a negative bos, non-finite alpha or beta.  Three launches.
 * ------------------------------------------------------------------------------------- */
#define CAB_NGRAM_MAX_ORDER 6
typedef struct {
    int32_t order;         /* n, 1..CAB_NGRAM_MAX_ORDER */
    int32_t num_classes;   /* C of the trie */
    int32_t num_nodes;
    int32_t bos;           /* word id of <s> */
    const void* tables[CAB_NGRAM_MAX_ORDER];  /* order k at [k - 1] */
    int64_t sizes[CAB_NGRAM_MAX_ORDER];
    const int32_t* child;  /* [num_nodes, num_classes] */
    const int32_t* word;   /* [num_nodes] */
} cab_ngram_lm_t;

int cab_ctc_beam_search_lm(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t,
                           const int64_t* output_lengths, int B, int T, int C, int N, float cutoff_prob,
                           int blank, int W, int K, void* workspace, int64_t workspace_bytes,
                           int32_t* out_tokens, int32_t* out_frames, int L_cap, int32_t* out_lengths,
                           float* out_scores, const cab_ngram_lm_t* lm, float alpha, float beta, int space,
                           cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Streaming (resumable) CTC prefix beam search, acoustic only (lm null) or with the word n-gram
 *   LM above.  A stream's log-probs arrive in chunks; each call advances every row's stream by
 *   that row's `frames` (0 allowed) and returns its current K best hypotheses.  After the call
 *   that consumed frames 0..t of a stream, tokens, frames, lengths and scores equal bit for bit
 *   what cab_ctc_beam_search (cab_ctc_beam_search_lm) returns for frames 0..t of that stream
 *   with the same arguments: with an LM they include the last word's term and the re-rank,
 *   computed for the outputs only; the stored state stays the search's beam set.
 *   State block (device, cab_ctc_beam_search_stream_state_bytes(W, lm_order) bytes, zeroed
 *   before the stream's first call): int32 {t0, beam count, finished, 0}, then per beam the
 *   prefix hash and parent hash (uint64), p_blank, p_nonblank (fp32), last class, node id and
 *   parent rank (int32), and with an LM the trie node, the bonus and the order - 1 context
 *   word ids.  Node table (device): `capacity` frames of W entries {int32 parent, int32 class},
 *   indexed by the stream's absolute frame (node id = frame * W + rank); out_frames count from
 *   the stream's start.  The caller keeps t0 and finished in the descriptor in step with the
 *   state (t0 += frames, finished = is_eos after each call) and grows a node table by copying
 *   its first t0 frames into a larger one.
 *   log_probs [B, C, T] through element strides (null allowed when T = 0); workspace of
 *   cab_ctc_beam_search_stream_workspace bytes; outputs as cab_ctc_beam_search.
 *   Refused before any launch: W, N, K, blank, cutoff_prob and the LM as above; a null row
 *   array, state or node table; a state block smaller than the state bytes; frames outside
 *   [0, T]; a finished stream; t0 + frames above capacity; capacity * W above INT32_MAX; two
 *   rows with one state block.  Three launches (prune, search, back-trace).
 * ------------------------------------------------------------------------------------- */
typedef struct {
    void* state;          /* device state block */
    void* nodes;          /* device node table, capacity * W entries of 8 bytes */
    int64_t state_bytes;  /* bytes of the state block */
    int64_t capacity;     /* frames the node table holds */
    int64_t t0;           /* frames the stream consumed before this call */
    int32_t frames;       /* frames of this call, [0, T] */
    int32_t is_eos;       /* nonzero: this call ends the stream */
    int32_t finished;     /* nonzero: an earlier call ended the stream (refused) */
    int32_t reserved;
} cab_beam_stream_t;

int cab_ctc_beam_search_stream_state_bytes(int W, int lm_order, int64_t* bytes);
int cab_ctc_beam_search_stream_workspace(int B, int T, int N, int W, int K, int64_t* bytes);
int cab_ctc_beam_search_stream(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t,
                               const cab_beam_stream_t* rows, int B, int T, int C, int N, float cutoff_prob,
                               int blank, int W, int K, void* workspace, int64_t workspace_bytes,
                               int32_t* out_tokens, int32_t* out_frames, int L_cap, int32_t* out_lengths,
                               float* out_scores, const cab_ngram_lm_t* lm, float alpha, float beta, int space,
                               cab_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Incremental streaming search: the same search and state block as cab_ctc_beam_search_stream,
 *   with a per-call cost that does not grow with the stream.  Every later hypothesis of a stream
 *   descends from one of the beams live after a call, so the deepest common ancestor of those
 *   beams (the commit node) and the labels on its chain are final.  Each call writes the part
 *   of that chain between the previous and the new commit node (out_final_*: int32 tokens and
 *   int64 absolute emission frames [B, L_cap], -1 past out_final_lengths [B]) and each
 *   hypothesis only from the commit node on (out_tokens int32 / out_frames int64
 *   [B, K, L_cap], out_lengths, out_scores as cab_ctc_beam_search_stream).  The final
 *   segments of a stream concatenated, followed by tail k, are bit for bit hypothesis k of
 *   cab_ctc_beam_search (_lm) on the stream's frames so far, where that hypothesis has
 *   nonzero probability; final tokens are never retracted.  out_commit [B] (device): the new
 *   commit node, window-relative after the shift, -1 the root.
 *   Node table: a window of the stream.  Node ids and the block's t0 count from the window's
 *   first frame, at absolute frame `base`.  `shift` > 0 drops the window's first `shift`
 *   frames before the search (one more launch): frames [shift, t0) move to the front, parents
 *   before the window become -2 (below the commit node, never followed), node ids and t0 in
 *   the state block are rebased.  The caller then keeps, for the next call, base += shift,
 *   t0 += frames - shift, commit = out_commit, finished = is_eos; it grows a node table by
 *   copying its first t0 frames into a larger one.  The state block's int32 hdr[3] becomes 1
 *   once the stream has consumed a frame (a live beam set whatever t0 is); a block used here
 *   is not passed to cab_ctc_beam_search_stream, whose node ids are absolute.
 *   Refused before any launch, besides cab_ctc_beam_search_stream's checks (t0 counted in
 *   the window): a negative base; commit outside [-1, t0 * W); shift outside [0, the commit
 *   node's frame] or, when positive, below t0 - shift (the moved frames must not overlap
 *   their destination); t0 - shift + frames above capacity; L_cap below the frames after
 *   the commit node (t0 - shift + frames - (commit >= 0 ? commit / W - shift + 1 : 0)).
 *   Four launches (prune, search, commit, tail back-trace), five with a shift.
 * ------------------------------------------------------------------------------------- */
typedef struct {
    void* state;          /* device state block (cab_ctc_beam_search_stream_state_bytes) */
    void* nodes;          /* device node table of the window, capacity * W entries of 8 bytes */
    int64_t state_bytes;  /* bytes of the state block */
    int64_t capacity;     /* frames the node table holds */
    int64_t base;         /* absolute frame of the window's first frame, before the shift */
    int64_t t0;           /* frames of the window consumed before this call, before the shift */
    int32_t commit;       /* commit node after the previous call, before the shift; -1 = the root */
    int32_t shift;        /* frames dropped from the window's front before this call, 0 = none */
    int32_t frames;       /* frames of this call, [0, T] */
    int32_t is_eos;       /* nonzero: this call ends the stream */
    int32_t finished;     /* nonzero: an earlier call ended the stream (refused) */
    int32_t reserved;
} cab_beam_stream_incremental_t;

int cab_ctc_beam_search_stream_incremental_workspace(int B, int T, int N, int W, int K, int64_t* bytes);
int cab_ctc_beam_search_stream_incremental(const float* log_probs, int64_t stride_b, int64_t stride_c,
                                           int64_t stride_t, const cab_beam_stream_incremental_t* rows,
                                           int B, int T, int C, int N, float cutoff_prob, int blank, int W,
                                           int K, void* workspace, int64_t workspace_bytes,
                                           int32_t* out_final_tokens, int64_t* out_final_frames,
                                           int32_t* out_final_lengths, int32_t* out_commit,
                                           int32_t* out_tokens, int64_t* out_frames, int L_cap,
                                           int32_t* out_lengths, float* out_scores, const cab_ngram_lm_t* lm,
                                           float alpha, float beta, int space, cab_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CONVASR_B200_H */
