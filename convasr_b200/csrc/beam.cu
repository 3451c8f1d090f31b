// CTC prefix beam search (decoders.BeamSearchDecoder, ctcdecode's CTCBeamDecoder), acoustic only or with a word n-gram
// language model fused in (ctcdecode's word-level scorer rules, tables built by convasr_b200/lm.py).
//
// Three launches per call:
//   beam_prune_kernel      one warp per frame: the top N = min(cutoff_top_n, C) classes by log-prob (ties -> lower class
//                          id), cut further by cutoff_prob as ctcdecode does, written in ascending class order.
//   beam_search_kernel     one CTA per utterance, T sequential frames: W <= 128 beams in shared memory, candidates scored,
//                          extensions merged into existing beams, the top W selected by a block-wide radix select, and
//                          one node (parent, class) allocated per surviving new prefix in a [T, W] table.  The LM
//                          instance also holds each beam's trie node and word context, refuses extensions that leave
//                          the dictionary, adds the word score when a space completes a word, and adds the last word's
//                          score and re-ranks after the last frame.
//   beam_backtrace_kernel  one thread per hypothesis walks the parent chain into tokens and emission frames.
//
// Log domain in fp32 with full-precision expf / logf, so the result is deterministic and does not depend on the batch.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>
#include <cmath>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

constexpr int kBeamMaxW = 128;
constexpr int kBeamMaxN = 64;
constexpr int kBeamThreads = 512;
constexpr int kPruneWarps = 8;

__device__ __forceinline__ float beam_lse(float a, float b) {
    const float m = fmaxf(a, b);
    if (m == -INFINITY) return -INFINITY;
    return logf(expf(a - m) + expf(b - m)) + m;
}

// order-preserving fp32 -> uint32 (larger value, larger key); -0 is folded into +0
__device__ __forceinline__ uint32_t beam_fkey(float v) {
    const uint32_t u = __float_as_uint(v + 0.f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// candidate key: 0 = not a candidate (probability zero, or NaN)
__device__ __forceinline__ uint32_t beam_ckey(float v) { return v > -INFINITY ? beam_fkey(v) : 0u; }

// Prefix hash of a labeling: extending by class c.  Two beams are the same prefix iff their hashes are equal (64 bits).
__device__ __forceinline__ uint64_t beam_hash(uint64_t h, int c) {
    uint64_t z = h + 0x9E3779B97F4A7C15ull * (uint64_t)(c + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// shared-memory histogram increment, aggregated over the lanes of a warp that hit the same bin (scores of one frame
// mostly share their top bits)
__device__ __forceinline__ void hist_add(uint32_t* hist, uint32_t bin) {
    const unsigned peers = __match_any_sync(__activemask(), bin);
    if ((peers & ((1u << (threadIdx.x & 31u)) - 1u)) == 0) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
}

// Warp: given 256 bin counts in hist, the digit d with count(bins > d) < need <= count(bins >= d), and count(bins > d).
__device__ __forceinline__ void warp_find_digit(const uint32_t* hist, uint32_t need, int lane, int* digit_out, uint32_t* above_out) {
    uint32_t loc[8], s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { loc[j] = hist[lane * 8 + j]; s += loc[j]; }
    uint32_t suf = s;  // inclusive suffix sum over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += v;
    }
    uint32_t acc = suf - s;
    int digit = -1;
    uint32_t above = 0;
#pragma unroll
    for (int j = 7; j >= 0; --j) {
        if (digit < 0 && acc < need && acc + loc[j] >= need) { digit = lane * 8 + j; above = acc; }
        acc += loc[j];
    }
    const unsigned found = __ballot_sync(0xffffffffu, digit >= 0);
    const int src = found ? __ffs(found) - 1 : 0;
    *digit_out = __shfl_sync(0xffffffffu, digit, src);
    *above_out = __shfl_sync(0xffffffffu, above, src);
}

// ------------------------------------------------------------------------------------------
// prune: one warp per (utterance, frame).  Radix select of the N-th largest key over the C classes (4 passes of 8
// bits, reading log_probs through element strides), then one pass in class order that keeps every key above the
// threshold and the lowest class ids among those equal to it.  With cutoff_prob < 1 the kept classes are ranked by
// value and summed in that order in fp32 (exp of each log-prob); a class is kept while the sum before it is below
// cutoff_prob, so the class that crosses it is kept (ctcdecode's rule).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kPruneWarps * 32)
beam_prune_kernel(const float* __restrict__ x, int64_t sb, int64_t sc, int64_t st, int C, int T, int N, float cutoff_prob,
                  int* __restrict__ out_cls, float* __restrict__ out_lp, int* __restrict__ out_cnt) {
    __shared__ uint32_t s_hist[kPruneWarps][256];
    __shared__ int s_cls[kPruneWarps][kBeamMaxN];
    __shared__ float s_lp[kPruneWarps][kBeamMaxN];
    __shared__ float s_sorted[kPruneWarps][kBeamMaxN];
    __shared__ int s_rank[kPruneWarps][kBeamMaxN];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.y, t = blockIdx.x * kPruneWarps + warp;
    if (t >= T) return;  // warp-uniform; the kernel only synchronises warps
    const float* xf = x + (int64_t)b * sb + (int64_t)t * st;
    uint32_t* hist = s_hist[warp];
    const unsigned lt_mask = (1u << lane) - 1u;

    uint32_t prefix = 0, mask = 0, need = (uint32_t)N;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = lane; i < 256; i += 32) hist[i] = 0;
        __syncwarp();
        for (int c = lane; c < C; c += 32) {
            const uint32_t k = beam_fkey(xf[(int64_t)c * sc]);
            if ((k & mask) == prefix) hist_add(hist, (k >> shift) & 255u);
        }
        __syncwarp();
        int digit;
        uint32_t above;
        warp_find_digit(hist, need, lane, &digit, &above);
        prefix |= (uint32_t)digit << shift;
        mask |= 255u << shift;
        need -= above;
        __syncwarp();
    }
    // keys > prefix: all; keys == prefix: the first `need` in class order
    int n_sel = 0, eq_seen = 0;
    for (int c0 = 0; c0 < C; c0 += 32) {
        const int c = c0 + lane;
        float v = -INFINITY;
        uint32_t k = 0;
        if (c < C) { v = xf[(int64_t)c * sc]; k = beam_fkey(v); }
        const bool eq = c < C && k == prefix;
        const unsigned beq = __ballot_sync(0xffffffffu, eq);
        const bool take = (c < C && k > prefix) || (eq && (uint32_t)(eq_seen + __popc(beq & lt_mask)) < need);
        const unsigned bt = __ballot_sync(0xffffffffu, take);
        if (take) {
            const int pos = n_sel + __popc(bt & lt_mask);
            s_cls[warp][pos] = c;
            s_lp[warp][pos] = v;
        }
        n_sel += __popc(bt);
        eq_seen += __popc(beq);
    }
    __syncwarp();
    int n_keep = N;
    if (cutoff_prob < 1.f) {
        for (int e = lane; e < N; e += 32) {
            const uint32_t ke = beam_fkey(s_lp[warp][e]);
            int r = 0;
            for (int f = 0; f < N; ++f) {
                const uint32_t kf = beam_fkey(s_lp[warp][f]);
                r += (kf > ke) || (kf == ke && f < e);
            }
            s_rank[warp][e] = r;
            s_sorted[warp][r] = expf(s_lp[warp][e]);
        }
        __syncwarp();
        if (lane == 0) {
            float acc = 0.f;
            for (int r = 0; r < N; ++r) {
                acc += s_sorted[warp][r];
                if (acc >= cutoff_prob) { n_keep = r + 1; break; }
            }
        }
        n_keep = __shfl_sync(0xffffffffu, n_keep, 0);
    }
    const size_t row = (size_t)b * T + t;
    int* oc = out_cls + row * N;
    float* ol = out_lp + row * N;
    int n_out = 0;
    for (int e0 = 0; e0 < N; e0 += 32) {
        const int e = e0 + lane;
        const bool keep = e < N && (n_keep == N || s_rank[warp][e] < n_keep);
        const unsigned bk = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const int pos = n_out + __popc(bk & lt_mask);
            oc[pos] = s_cls[warp][e];
            ol[pos] = s_lp[warp][e];
        }
        n_out += __popc(bk);
    }
    for (int e = n_out + lane; e < N; e += 32) { oc[e] = -1; ol[e] = -INFINITY; }
    if (lane == 0) out_cnt[row] = n_out;
}

// ------------------------------------------------------------------------------------------
// search: one CTA of kBeamThreads per utterance.  A beam is (log p_blank, log p_nonblank, last class, node id, prefix
// hash, hash of the prefix without its last class, rank of that shorter prefix among the beams or -1).  Per frame:
//  (1) per beam, the prefix it keeps: p_b' = lse(p_b, p_nb) + lp[blank], p_nb' = p_nb + lp[last]; when the prefix minus
//      its last class c is beam p, the extension of p by c IS this beam: it adds (c == last(p) ? p_b(p) : lse(p_b(p),
//      p_nb(p))) + lp[c] to p_nb' and is marked in the (source beam, class) map so it is not a candidate of its own;
//  (2) candidate q = i * (n + 1) + s of source beam i: s = 0 keeps the prefix (score lse(p_b', p_nb')), s = 1 + k
//      extends it by the k-th pruned class (ascending class order; a repeat of the last class extends only from p_b);
//      probability zero is not a candidate;
//  (3) the top W by score, ties to the lower q: a radix select (4 x 8 bits) finds the threshold key, a block scan
//      in q order takes the lowest q among keys equal to it, and the chosen ones are ranked by (score, -q);
//  (4) the new beams in rank order; a new prefix gets node t * W + rank in the node table.
// ------------------------------------------------------------------------------------------
struct BeamNode {
    int parent;  // node id, -1 = the empty prefix
    int cls;
};

// ------------------------------------------------------------------------------------------
// Word n-gram LM (the LM instance).  A beam also holds the trie node of its current word, the last order - 1 completed
// words (oldest first, <s>-padded) and the bonus that the extension creating its prefix carried (nonzero only when that
// extension was a space; step (1)'s merge into the beam adds it again).  Per frame, before step (2):
//  (a) when `space` is among the frame's classes and the beam's node spells a word w, the space bonus
//      alpha * lm(w | context) + beta; otherwise a space is not a candidate of that beam;
//  (b) a non-space class c is a candidate only if child[node][c] >= 0.
// A new prefix takes node' = child[node][c], or after a space the root and the context shifted by w.
// ------------------------------------------------------------------------------------------
constexpr int kLmMaxOrder = CAB_NGRAM_MAX_ORDER;
constexpr float kLmOovScore = -1000.f;  // ctcdecode's OOV_SCORE (natural log, before alpha)

struct NgramEntry {
    uint64_t key;  // 0 = empty slot
    float log10_p;
    float log10_bo;
};

struct BeamLm {
    const NgramEntry* table[kLmMaxOrder];
    uint64_t mask[kLmMaxOrder];
    const int* child;
    const int* word;
    int order, C, space, bos;
    float alpha, beta;
};

// linear probing from the first probe e (slot key & mask) until the key or an empty slot; at most one pass over the
// table, so a table without an empty slot ends the search as "not listed" instead of spinning
__device__ __forceinline__ NgramEntry ngram_probe(const NgramEntry* table, uint64_t mask, uint64_t key, NgramEntry e) {
    uint64_t slot = key & mask;
    for (uint64_t i = 0; i < mask && e.key != key && e.key != 0; ++i) {
        slot = (slot + 1) & mask;
        e = table[slot];
    }
    return e;
}

// lm(w | ctx) in natural log: ARPA back-off over the order tables.  Every first probe (n for log10 p of the suffixes
// (ctx[n-k..], w), n - 1 for the back-offs of the context suffixes) is issued before any is used; keys are folded
// newest first, so each suffix's key extends the next shorter one's.
__device__ float lm_word_score(const BeamLm& lm, const int* ctx, int w) {
    const int n = lm.order;
    uint64_t pk[kLmMaxOrder], bk[kLmMaxOrder];
    NgramEntry pe[kLmMaxOrder], be[kLmMaxOrder];
    pk[0] = beam_hash(0, w);
    bk[0] = 0;
#pragma unroll
    for (int k = 1; k < kLmMaxOrder; ++k) {
        if (k < n) {
            const int id = ctx[n - 1 - k];
            pk[k] = beam_hash(pk[k - 1], id);
            bk[k] = beam_hash(bk[k - 1], id);
        }
    }
#pragma unroll
    for (int k = 0; k < kLmMaxOrder; ++k) {
        if (k < n) pe[k] = lm.table[k][pk[k] & lm.mask[k]];
        if (k >= 1 && k < n) be[k] = lm.table[k - 1][bk[k] & lm.mask[k - 1]];
    }
    float p = 0.f, bo = 0.f;
    bool found = false;
#pragma unroll
    for (int k = kLmMaxOrder - 1; k >= 0; --k) {
        if (k < n && !found) {
            // (ctx[n-1-k..], w) at order k + 1; back-off of the context suffix of length k (order k)
            const NgramEntry e = ngram_probe(lm.table[k], lm.mask[k], pk[k], pe[k]);
            if (e.key == pk[k]) {
                p = e.log10_p;
                found = true;
            } else if (k >= 1) {
                const NgramEntry c = ngram_probe(lm.table[k - 1], lm.mask[k - 1], bk[k], be[k]);
                if (c.key == bk[k]) bo += c.log10_bo;
            }
        }
    }
    return found ? 2.302585093f * (bo + p) : kLmOovScore;
}

template <bool LM>
__global__ void __launch_bounds__(kBeamThreads, 1)
beam_search_kernel(const int* __restrict__ p_cls, const float* __restrict__ p_lp, const int* __restrict__ p_cnt,
                   const int64_t* __restrict__ lengths, int T, int N, int blank, int W, int K,
                   BeamNode* __restrict__ nodes, int* __restrict__ final_node, float* __restrict__ out_scores, const BeamLm lm) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = kBeamThreads / 32;
    // layout: two beam sets, then per-frame scratch
    uint64_t* s_hash = reinterpret_cast<uint64_t*>(smem);  // [2][W]
    uint64_t* s_phash = s_hash + 2 * W;                     // [2][W]
    float* s_pb = reinterpret_cast<float*>(s_phash + 2 * W);  // [2][W]
    float* s_pnb = s_pb + 2 * W;                             // [2][W]
    int* s_last = reinterpret_cast<int*>(s_pnb + 2 * W);     // [2][W]
    int* s_node = s_last + 2 * W;                            // [2][W]
    int* s_prank = s_node + 2 * W;                           // [2][W]
    float* s_kpb = reinterpret_cast<float*>(s_prank + 2 * W);  // [W] kept p_b'
    float* s_kpnb = s_kpb + W;                                 // [W] kept p_nb'
    int* s_newrank = reinterpret_cast<int*>(s_kpnb + W);       // [W] new rank of old beam i's keep candidate, or -1
    int* s_sel_q = s_newrank + W;                              // [W] selected candidates (unordered)
    uint32_t* s_sel_key = reinterpret_cast<uint32_t*>(s_sel_q + W);  // [W]
    int* s_order = reinterpret_cast<int*>(s_sel_key + W);      // [W] candidate of each new rank
    int* s_fcls = s_order + W;                                 // [N] this frame's pruned classes
    float* s_flp = reinterpret_cast<float*>(s_fcls + N);       // [N]
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_flp + N); // [256]
    int* s_misc = reinterpret_cast<int*>(s_hist + 256);        // [kWarps + 8]
    int16_t* s_merged = reinterpret_cast<int16_t*>(s_misc + kWarps + 8);  // [W * N]
    uint32_t* s_keys = reinterpret_cast<uint32_t*>(s_merged + ((W * N + 1) & ~1));  // [W * (N + 1)]
    int& s_valid = s_misc[kWarps + 0];
    int& s_nsel = s_misc[kWarps + 1];
    int& s_prefix = s_misc[kWarps + 2];
    int& s_need = s_misc[kWarps + 3];
    // LM instance only, after the acoustic layout
    constexpr int kCtx = kLmMaxOrder - 1;
    int* s_tnode = reinterpret_cast<int*>(s_keys + W * (N + 1));  // [2][W] trie node of the current word
    int* s_ctx = s_tnode + 2 * W;                                   // [2][W][kCtx] completed words, oldest first
    float* s_bonus = reinterpret_cast<float*>(s_ctx + 2 * W * kCtx);  // [2][W] bonus of the extension that made the prefix
    float* s_spb = s_bonus + 2 * W;                                  // [W] this frame's space bonus, -inf = no space
    int* s_word = reinterpret_cast<int*>(s_spb + W);                // [W] word id of the beam's node, or -1

    const int64_t len64 = lengths ? lengths[b] : T;
    const int len = len64 < 0 ? 0 : (len64 > T ? T : (int)len64);
    if (tid == 0) {
        s_hash[0] = 0; s_phash[0] = 0; s_pb[0] = 0.f; s_pnb[0] = -INFINITY; s_last[0] = -1; s_node[0] = -1; s_prank[0] = -1;
        if constexpr (LM) {
            s_tnode[0] = 0;
            s_bonus[0] = 0.f;
            for (int k = 0; k < kCtx; ++k) s_ctx[k] = lm.bos;
        }
    }
    int cur = 0, nb = 1;
    const size_t frame0 = (size_t)b * T;
    BeamNode* bnodes = nodes + frame0 * W;
    // next frame's pruned classes, prefetched into registers by threads < N
    int nx_cls = -1, nx_cnt = 0;
    float nx_lp = -INFINITY;
    if (len > 0) {
        if (tid < N) { nx_cls = p_cls[frame0 * N + tid]; nx_lp = p_lp[frame0 * N + tid]; }
        nx_cnt = p_cnt[frame0];
    }
    for (int t = 0; t < len; ++t) {
        const int n = nx_cnt;
        const int M1 = n + 1;
        if (tid < N) { s_fcls[tid] = nx_cls; s_flp[tid] = nx_lp; }
        if (t + 1 < len) {
            if (tid < N) { nx_cls = p_cls[(frame0 + t + 1) * N + tid]; nx_lp = p_lp[(frame0 + t + 1) * N + tid]; }
            nx_cnt = p_cnt[frame0 + t + 1];
        }
        for (int i = tid; i < nb * N; i += kBeamThreads) s_merged[i] = -1;
        for (int i = tid; i < 256; i += kBeamThreads) s_hist[i] = 0;
        if (tid < nb) s_newrank[tid] = -1;
        if (tid == 0) { s_valid = 0; s_nsel = 0; }
        __syncthreads();
        const float* pb = s_pb + cur * W;
        const float* pnb = s_pnb + cur * W;
        const int* last = s_last + cur * W;
        // (1) kept prefixes and merged extensions
        if (tid < nb) {
            const int j = tid, lj = last[j];
            int kb = -1, kl = -1;
            for (int k = 0; k < n; ++k) {
                const int c = s_fcls[k];
                if (c == blank) kb = k;
                if (c == lj) kl = k;
            }
            s_kpb[j] = kb >= 0 ? beam_lse(pb[j], pnb[j]) + s_flp[kb] : -INFINITY;
            float x = kl >= 0 ? pnb[j] + s_flp[kl] : -INFINITY;
            const int p = s_prank[cur * W + j];
            if (p >= 0 && kl >= 0) {
                float e = (last[p] == lj ? pb[p] : beam_lse(pb[p], pnb[p])) + s_flp[kl];
                if constexpr (LM) e += s_bonus[cur * W + j];
                x = beam_lse(x, e);
                s_merged[p * N + kl] = (int16_t)j;
            }
            s_kpnb[j] = x;
        }
        if constexpr (LM) {
            // (a) the space bonus, by the threads step (1) leaves idle
            const int j = tid - kBeamMaxW;
            if (j >= 0 && j < nb) {
                bool has_space = false;
                for (int k = 0; k < n; ++k) has_space |= s_fcls[k] == lm.space;
                const int w = lm.word[s_tnode[cur * W + j]];
                s_word[j] = w;
                s_spb[j] = has_space && w >= 0 ? lm.alpha * lm_word_score(lm, s_ctx + (cur * W + j) * kCtx, w) + lm.beta : -INFINITY;
            }
        }
        __syncthreads();
        // (2) candidate keys; the first radix pass's histogram on the way
        const int M = nb * M1;
        int my_valid = 0;
        for (int q = tid; q < M; q += kBeamThreads) {
            const int i = q / M1, s = q - i * M1;
            float v;
            if (s == 0) {
                v = beam_lse(s_kpb[i], s_kpnb[i]);
            } else {
                const int k = s - 1, c = s_fcls[k];
                if (c == blank || s_merged[i * N + k] >= 0) v = -INFINITY;
                else v = (c == last[i] ? pb[i] : beam_lse(pb[i], pnb[i])) + s_flp[k];
                if constexpr (LM) {
                    // (b) the dictionary constraint; a space carries the word's bonus (-inf: no word to end)
                    if (c == lm.space) v += s_spb[i];
                    else if (c != blank && lm.child[(size_t)s_tnode[cur * W + i] * lm.C + c] < 0) v = -INFINITY;
                }
            }
            const uint32_t key = beam_ckey(v);
            s_keys[q] = key;
            if (key) {
                ++my_valid;
                hist_add(s_hist, key >> 24);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_valid += __shfl_xor_sync(0xffffffffu, my_valid, o);
        if (lane == 0 && my_valid) atomicAdd(&s_valid, my_valid);
        __syncthreads();
        const int n_valid = s_valid;
        const int Kn = n_valid < W ? n_valid : W;
        uint32_t thr = 1u, need_eq = 0xffffffffu;  // every valid key when they all fit
        if (n_valid > W) {
            // (3) radix select of the W-th largest key
            uint32_t prefix = 0, mask = 0;
            for (int shift = 24; shift >= 0; shift -= 8) {
                if (shift != 24) {
                    for (int q = tid; q < M; q += kBeamThreads) {
                        const uint32_t key = s_keys[q];
                        if (key && (key & mask) == prefix) hist_add(s_hist, (key >> shift) & 255u);
                    }
                    __syncthreads();
                }
                if (warp == 0) {
                    const uint32_t need = shift == 24 ? (uint32_t)W : (uint32_t)s_need;
                    int digit;
                    uint32_t above;
                    warp_find_digit(s_hist, need, lane, &digit, &above);
                    for (int i = lane; i < 256; i += 32) s_hist[i] = 0;
                    if (lane == 0) {
                        s_prefix = (int)(prefix | ((uint32_t)digit << shift));
                        s_need = (int)(need - above);
                    }
                }
                __syncthreads();
                prefix = (uint32_t)s_prefix;
                mask |= 255u << shift;
            }
            thr = prefix;
            need_eq = (uint32_t)s_need;
        }
        // take keys > thr, and keys == thr in q order while fewer than need_eq were taken: a contiguous chunk of
        // candidates per thread and an exclusive scan of the per-thread counts of keys equal to thr
        const int per = (M + kBeamThreads - 1) / kBeamThreads;
        const int q0 = tid * per, q1 = min(M, q0 + per);
        int eq = 0;
        for (int q = q0; q < q1; ++q) eq += s_keys[q] == thr;
        int incl = eq;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_misc[warp] = incl;
        __syncthreads();
        int eq_before = incl - eq;
        for (int w = 0; w < warp; ++w) eq_before += s_misc[w];
        for (int q = q0; q < q1; ++q) {
            const uint32_t key = s_keys[q];
            bool take = key > thr;
            if (key == thr) take = (uint32_t)(eq_before++) < need_eq;
            if (take) {
                const int slot = atomicAdd(&s_nsel, 1);
                s_sel_q[slot] = q;
                s_sel_key[slot] = key;
            }
        }
        __syncthreads();
        // rank the chosen: 4 threads per candidate, each comparing a quarter of them
        {
            const int r = tid >> 2, part = tid & 3;
            int rank = 0;
            uint32_t kr = 0;
            int qr = 0;
            if (r < Kn) {
                kr = s_sel_key[r];
                qr = s_sel_q[r];
                for (int f = part; f < Kn; f += 4) {
                    const uint32_t kf = s_sel_key[f];
                    rank += (kf > kr) || (kf == kr && s_sel_q[f] < qr);
                }
            }
            rank += __shfl_xor_sync(0xffffffffu, rank, 1);
            rank += __shfl_xor_sync(0xffffffffu, rank, 2);
            if (r < Kn && part == 0) s_order[rank] = qr;
        }
        __syncthreads();
        // (4) the new beam set
        const int nxt = cur ^ 1;
        int src = -1, keep = 0;
        if (tid < Kn) {
            const int r = tid, q = s_order[r], i = q / M1, s = q - i * M1;
            src = i;
            if (s == 0) {
                keep = 1;
                s_pb[nxt * W + r] = s_kpb[i];
                s_pnb[nxt * W + r] = s_kpnb[i];
                s_last[nxt * W + r] = last[i];
                s_node[nxt * W + r] = s_node[cur * W + i];
                s_hash[nxt * W + r] = s_hash[cur * W + i];
                s_phash[nxt * W + r] = s_phash[cur * W + i];
                s_newrank[i] = r;
                if constexpr (LM) {
                    s_tnode[nxt * W + r] = s_tnode[cur * W + i];
                    s_bonus[nxt * W + r] = s_bonus[cur * W + i];
                    for (int k = 0; k < lm.order - 1; ++k) s_ctx[(nxt * W + r) * kCtx + k] = s_ctx[(cur * W + i) * kCtx + k];
                }
            } else {
                const int k = s - 1, c = s_fcls[k];
                s_pb[nxt * W + r] = -INFINITY;
                float v = (c == last[i] ? pb[i] : beam_lse(pb[i], pnb[i])) + s_flp[k];
                if constexpr (LM) {
                    const int* ctx = s_ctx + (cur * W + i) * kCtx;
                    int* nctx = s_ctx + (nxt * W + r) * kCtx;
                    const int nc = lm.order - 1;
                    if (c == lm.space) {
                        v += s_spb[i];
                        s_tnode[nxt * W + r] = 0;
                        s_bonus[nxt * W + r] = s_spb[i];
                        for (int m = 0; m + 1 < nc; ++m) nctx[m] = ctx[m + 1];
                        if (nc > 0) nctx[nc - 1] = s_word[i];
                    } else {
                        s_tnode[nxt * W + r] = lm.child[(size_t)s_tnode[cur * W + i] * lm.C + c];
                        s_bonus[nxt * W + r] = 0.f;
                        for (int m = 0; m < nc; ++m) nctx[m] = ctx[m];
                    }
                }
                s_pnb[nxt * W + r] = v;
                s_last[nxt * W + r] = c;
                const int id = t * W + r;
                s_node[nxt * W + r] = id;
                bnodes[id] = BeamNode{s_node[cur * W + i], c};
                s_hash[nxt * W + r] = beam_hash(s_hash[cur * W + i], c);
                s_phash[nxt * W + r] = s_hash[cur * W + i];
            }
        }
        __syncthreads();
        if (tid < Kn) {
            const int r = tid;
            int pr;
            if (keep) {
                const int p = s_prank[cur * W + src];
                pr = p >= 0 ? s_newrank[p] : -1;
                if (pr < 0 && s_last[nxt * W + r] >= 0) {
                    // the shorter prefix was not a beam before this frame: it may have come back as a new extension
                    const uint64_t ph = s_phash[nxt * W + r];
                    for (int f = 0; f < Kn; ++f)
                        if (s_hash[nxt * W + f] == ph && s_node[nxt * W + f] == t * W + f) { pr = f; break; }
                }
            } else {
                pr = s_newrank[src];
            }
            s_prank[nxt * W + r] = pr;
        }
        nb = Kn;
        cur = nxt;
        __syncthreads();
        if (nb == 0) break;
    }
    if constexpr (LM) {
        // the last word's term, then re-rank by counting (ties to the earlier rank); hypothesis r is beam s_order[r]
        float* s_fin = s_kpb;
        if (tid < nb) {
            const int l = s_last[cur * W + tid];
            float f = beam_lse(s_pb[cur * W + tid], s_pnb[cur * W + tid]);
            if (l >= 0 && l != lm.space) {
                const int w = lm.word[s_tnode[cur * W + tid]];
                f += lm.alpha * (w >= 0 ? lm_word_score(lm, s_ctx + (cur * W + tid) * kCtx, w) : kLmOovScore) + lm.beta;
            }
            s_fin[tid] = f;
        }
        __syncthreads();
        if (tid < nb) {
            const float f = s_fin[tid];
            int rank = 0;
            for (int g = 0; g < nb; ++g) rank += s_fin[g] > f || (s_fin[g] == f && g < tid);
            s_order[rank] = tid;
        }
        __syncthreads();
        if (tid < K) {
            const size_t o = (size_t)b * K + tid;
            const int r = tid < nb ? s_order[tid] : -1;
            final_node[o] = r >= 0 ? s_node[cur * W + r] : -2;
            out_scores[o] = r >= 0 ? s_fin[r] : -INFINITY;
        }
        return;
    }
    // beams are in rank order: hypothesis r is beam r
    if (tid < K) {
        const size_t o = (size_t)b * K + tid;
        if (tid < nb) {
            final_node[o] = s_node[cur * W + tid];
            out_scores[o] = beam_lse(s_pb[cur * W + tid], s_pnb[cur * W + tid]);
        } else {
            final_node[o] = -2;
            out_scores[o] = -INFINITY;
        }
    }
}

// back-trace: one thread per hypothesis; tokens in order, emission frame = the frame the prefix was created
__global__ void __launch_bounds__(kBeamMaxW)
beam_backtrace_kernel(const BeamNode* __restrict__ nodes, const int* __restrict__ final_node, int T, int W, int K, int L_cap,
                      int* __restrict__ out_tokens, int* __restrict__ out_frames, int* __restrict__ out_lengths) {
    const int b = blockIdx.x, r = threadIdx.x;
    if (r >= K) return;
    const BeamNode* bn = nodes + (size_t)b * T * W;
    const size_t o = (size_t)b * K + r;
    const int start = final_node[o];
    int L = 0;
    for (int id = start; id >= 0; id = bn[id].parent) ++L;
    int* tok = out_tokens + o * L_cap;
    int* frm = out_frames + o * L_cap;
    int pos = L - 1;
    for (int id = start; id >= 0; id = bn[id].parent, --pos) {
        if (pos < L_cap) { tok[pos] = bn[id].cls; frm[pos] = id / W; }
    }
    for (int i = L; i < L_cap; ++i) { tok[i] = -1; frm[i] = -1; }
    out_lengths[o] = L;
}

static size_t beam_align(size_t x) { return (x + 255) & ~(size_t)255; }

// workspace: pruned classes int32 [B, T, N], their log-probs fp32 [B, T, N], counts int32 [B, T], node table
// [B, T, W] of (parent, class), final node of each hypothesis int32 [B, W]
static void beam_workspace_layout(int B, int T, int N, int W, size_t off[5]) {
    const size_t BT = (size_t)B * T;
    off[0] = 0;
    off[1] = beam_align(off[0] + BT * N * 4);
    off[2] = beam_align(off[1] + BT * N * 4);
    off[3] = beam_align(off[2] + BT * 4);
    off[4] = beam_align(off[3] + BT * W * sizeof(BeamNode));
}
static size_t beam_workspace_bytes(int B, int T, int N, int W) {
    size_t off[5];
    beam_workspace_layout(B, T, N, W, off);
    return beam_align(off[4] + (size_t)B * W * 4);
}

static size_t beam_search_smem(int W, int N, bool lm) {
    size_t bytes = 2 * W * 8 * 2 + 2 * W * 4 * 5 + W * 4 * 6 + N * 8 + 256 * 4 + (kBeamThreads / 32 + 8) * 4;
    bytes += (size_t)((W * N + 1) & ~1) * 2 + (size_t)W * (N + 1) * 4;
    if (lm) bytes += (size_t)W * 4 * (2 + 2 * (kLmMaxOrder - 1) + 2 + 2);  // trie node, context, bonus; space bonus, word
    return bytes;
}

// prune -> search -> back-trace; the arguments are checked by the caller
template <bool LM>
static int beam_search_launch(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t, const int64_t* output_lengths,
                              int B, int T, int C, int N, float cutoff_prob, int blank, int W, int K, void* workspace, int32_t* out_tokens,
                              int32_t* out_frames, int L_cap, int32_t* out_lengths, float* out_scores, const BeamLm& lm,
                              cudaStream_t stream) {
    size_t off[5];
    beam_workspace_layout(B, T, N, W, off);
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    int* p_cls = reinterpret_cast<int*>(ws + off[0]);
    float* p_lp = reinterpret_cast<float*>(ws + off[1]);
    int* p_cnt = reinterpret_cast<int*>(ws + off[2]);
    BeamNode* nodes = reinterpret_cast<BeamNode*>(ws + off[3]);
    int* final_node = reinterpret_cast<int*>(ws + off[4]);

    const size_t smem = beam_search_smem(W, N, LM);
    static size_t smem_set = 0;
    if (smem > 48 * 1024 && smem > smem_set) {
        CAB_CHECK_CUDA(cudaFuncSetAttribute(beam_search_kernel<LM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)beam_search_smem(kBeamMaxW, kBeamMaxN, LM)));
        smem_set = beam_search_smem(kBeamMaxW, kBeamMaxN, LM);
    }
    dim3 pgrid((T + kPruneWarps - 1) / kPruneWarps, B);
    beam_prune_kernel<<<pgrid, kPruneWarps * 32, 0, stream>>>(log_probs, stride_b, stride_c, stride_t, C, T, N, cutoff_prob, p_cls,
                                                               p_lp, p_cnt);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    beam_search_kernel<LM><<<B, kBeamThreads, smem, stream>>>(p_cls, p_lp, p_cnt, output_lengths, T, N, blank, W, K, nodes, final_node,
                                                              out_scores, lm);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    beam_backtrace_kernel<<<B, kBeamMaxW, 0, stream>>>(nodes, final_node, T, W, K, L_cap, out_tokens, out_frames, out_lengths);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

}  // namespace cab

using namespace cab;

#define CAB_BEAM_CHECK_ARGS()                                                                                          \
    CAB_CHECK_ARG(B > 0 && T > 0 && C > 0, "bad shape B=%d T=%d C=%d", B, T, C);                                      \
    CAB_CHECK_ARG(W >= 1 && W <= kBeamMaxW, "beam_width=%d out of [1, %d]", W, kBeamMaxW);                            \
    CAB_CHECK_ARG(N >= 1 && N <= kBeamMaxN && N <= C, "N=%d out of [1, %d] (C=%d)", N, kBeamMaxN, C);                 \
    CAB_CHECK_ARG(K >= 1 && K <= W, "K=%d out of [1, beam_width=%d]", K, W);                                           \
    CAB_CHECK_ARG(blank >= 0 && blank < C, "blank=%d out of range (C=%d)", blank, C);                                  \
    CAB_CHECK_ARG(cutoff_prob > 0.f && cutoff_prob <= 1.f, "cutoff_prob=%g out of (0, 1]", (double)cutoff_prob)

#define CAB_BEAM_CHECK_CALL()                                                                                          \
    CAB_CHECK_ARG(log_probs && workspace && out_tokens && out_frames && out_lengths && out_scores, "null pointer argument"); \
    CAB_BEAM_CHECK_ARGS();                                                                                             \
    CAB_CHECK_ARG(L_cap >= 1, "L_cap=%d must be positive", L_cap);                                                     \
    CAB_CHECK_ARG(workspace_bytes >= (int64_t)beam_workspace_bytes(B, T, N, W), "workspace of %lld bytes is too small (%lld needed)", \
                  (long long)workspace_bytes, (long long)beam_workspace_bytes(B, T, N, W))

extern "C" int cab_ctc_beam_search_workspace(int B, int T, int C, int N, int W, int K, int blank, float cutoff_prob, int64_t* bytes) {
    CAB_CHECK_ARG(bytes != nullptr, "null output");
    CAB_BEAM_CHECK_ARGS();
    *bytes = (int64_t)beam_workspace_bytes(B, T, N, W);
    return 0;
}

extern "C" int cab_ctc_beam_search(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t,
                                   const int64_t* output_lengths, int B, int T, int C, int N, float cutoff_prob, int blank,
                                   int W, int K, void* workspace, int64_t workspace_bytes, int32_t* out_tokens,
                                   int32_t* out_frames, int L_cap, int32_t* out_lengths, float* out_scores,
                                   cab_stream_t stream_) {
    CAB_BEAM_CHECK_CALL();
    return beam_search_launch<false>(log_probs, stride_b, stride_c, stride_t, output_lengths, B, T, C, N, cutoff_prob, blank, W, K,
                                     workspace, out_tokens, out_frames, L_cap, out_lengths, out_scores, BeamLm{},
                                     static_cast<cudaStream_t>(stream_));
}

extern "C" int cab_ctc_beam_search_lm(const float* log_probs, int64_t stride_b, int64_t stride_c, int64_t stride_t,
                                      const int64_t* output_lengths, int B, int T, int C, int N, float cutoff_prob, int blank,
                                      int W, int K, void* workspace, int64_t workspace_bytes, int32_t* out_tokens,
                                      int32_t* out_frames, int L_cap, int32_t* out_lengths, float* out_scores,
                                      const cab_ngram_lm_t* lm, float alpha, float beta, int space, cab_stream_t stream_) {
    CAB_BEAM_CHECK_CALL();
    CAB_CHECK_ARG(lm != nullptr, "null lm");
    CAB_CHECK_ARG(lm->order >= 1 && lm->order <= kLmMaxOrder, "lm order=%d out of [1, %d]", lm->order, kLmMaxOrder);
    CAB_CHECK_ARG(lm->num_classes == C, "lm trie has %d classes, log_probs %d", lm->num_classes, C);
    CAB_CHECK_ARG(lm->num_nodes >= 1 && lm->child && lm->word, "lm trie: %d nodes, child %p, word %p", lm->num_nodes,
                  (const void*)lm->child, (const void*)lm->word);
    CAB_CHECK_ARG(lm->bos >= 0, "lm bos=%d negative", lm->bos);
    CAB_CHECK_ARG(space >= 0 && space < C && space != blank, "space=%d out of range (C=%d) or equal to blank=%d", space, C, blank);
    CAB_CHECK_ARG(std::isfinite(alpha) && std::isfinite(beta), "alpha=%g / beta=%g not finite", (double)alpha, (double)beta);
    BeamLm v{};
    for (int k = 0; k < lm->order; ++k) {
        const int64_t n = lm->sizes[k];
        CAB_CHECK_ARG(lm->tables[k] != nullptr, "lm table of order %d is null", k + 1);
        CAB_CHECK_ARG(n > 0 && (n & (n - 1)) == 0, "lm table of order %d: size %lld is not a power of two", k + 1, (long long)n);
        v.table[k] = static_cast<const NgramEntry*>(lm->tables[k]);
        v.mask[k] = (uint64_t)(n - 1);
    }
    v.child = lm->child;
    v.word = lm->word;
    v.order = lm->order;
    v.C = C;
    v.space = space;
    v.bos = lm->bos;
    v.alpha = alpha;
    v.beta = beta;
    return beam_search_launch<true>(log_probs, stride_b, stride_c, stride_t, output_lengths, B, T, C, N, cutoff_prob, blank, W, K,
                                    workspace, out_tokens, out_frames, L_cap, out_lengths, out_scores, v,
                                    static_cast<cudaStream_t>(stream_));
}
