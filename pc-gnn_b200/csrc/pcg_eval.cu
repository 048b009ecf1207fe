// Evaluation pass on the device: the two-class head + sigmoid (PCALayer, GCN) or log-softmax (GraphSage) into a
// whole-set probability buffer, and the binary metrics of src/utils.py:298-333 (AUC, F1, recall, precision, ...) plus
// the ranking metrics of fraud-detection benchmarks (average precision, Recall@K, the best macro-F1 and G-mean cuts)
// and the ROC / PR curve, computed where the probabilities live. Deterministic: integer sums, fp64 sums in a fixed
// order and an order-free arg-max only (no floating-point atomics).
#include <math.h>

#include "pcg_common.cuh"

// ------------------------------------------------------------------------------- head
// l_c = sum_k w[c,k] * emb[k,i] for the rows of plan entry e = *cursor % count that exist (padding rows of the last
// entry are not written), k summed in order 0..E-1, one thread per row. mode 0: prob[c * n_total + e*B + i] =
// sigmoid(l_c); mode 1: log_softmax(l)_c = (l_c - m) - log(exp(l_0 - m) + exp(l_1 - m)) with m = max(l_0, l_1).
__global__ void __launch_bounds__(256) k_eval_head(const float* __restrict__ emb, int E, int B, const float* __restrict__ w,
                                                   int mode, int64_t n_total, const uint32_t* cursor, uint32_t count,
                                                   float* __restrict__ prob) {
    extern __shared__ float sw[];
    for (int k = threadIdx.x; k < 2 * E; k += blockDim.x) sw[k] = w[k];
    __syncthreads();
    const int64_t base = cursor ? (int64_t)(*(volatile const uint32_t*)cursor % count) * B : 0;
    const int64_t rows = n_total - base < (int64_t)B ? n_total - base : (int64_t)B;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    float a0 = 0.f, a1 = 0.f;
    for (int k = 0; k < E; ++k) {
        const float x = __ldg(emb + (int64_t)k * B + i);
        a0 = fmaf(sw[k], x, a0);
        a1 = fmaf(sw[E + k], x, a1);
    }
    if (mode == 0) {
        prob[base + i] = 1.f / (1.f + expf(-a0));
        prob[n_total + base + i] = 1.f / (1.f + expf(-a1));
    } else {
        const float m = fmaxf(a0, a1);
        const float lse = logf(expf(a0 - m) + expf(a1 - m));
        prob[base + i] = (a0 - m) - lse;
        prob[n_total + base + i] = (a1 - m) - lse;
    }
}

extern "C" int pcg_eval_head(const float* emb, int E, int B, const float* w_head, int mode, int64_t n_total,
                             const uint32_t* cursor, uint32_t count, float* prob, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(emb && w_head && prob, "pcg_eval_head: null pointer");
    PCG_REQUIRE(E > 0 && E <= 4096 && B > 0 && n_total > 0, "pcg_eval_head: need 0 < E <= 4096, B > 0, n_total > 0");
    PCG_REQUIRE(mode == 0 || mode == 1, "pcg_eval_head: mode must be 0 (sigmoid) or 1 (log-softmax), got %d", mode);
    PCG_REQUIRE(!cursor || count > 0, "pcg_eval_head: a plan cursor needs count > 0");
    k_eval_head<<<(B + 255) / 256, 256, (size_t)E * 2 * sizeof(float), stream>>>(emb, E, B, w_head, mode, n_total, cursor,
                                                                                  count, prob);
    return pcg_check_launch("pcg_eval_head");
}

// ------------------------------------------------------------------------------- metrics
// prob[1] is sorted ascending with the labels riding along as the "pool" (pcg_sort_pool), then:
//   k_metrics_count  per chunk of CH sorted positions: positives, the AUC rank sum of its positives (tie groups by
//                    lower / upper bound: twice the average rank = lo + hi + 1), and the confusion counts of the
//                    chunk's ORIGINAL positions (pred = prob[1] > prob[0], the argmax of utils.test)
//   k_metrics_best   per chunk: positives in front of every position (chunk prefix from the counts + a block scan),
//                    stored as pre[j]; macro-F1 and G-mean of the cut "positive iff prob[1] >= s[j]" at every tie-group
//                    start j, the chunk's best of each, and the number of group starts in the chunk
//   k_metrics_ap     per chunk, once pre is complete: the chunk's positives' average-precision terms, summed in fp64
//   k_metrics_final  one CTA: sums and arg-max over the chunks, Recall@K, every metric in double
// pcg_binary_curve reads the sorted scores and pre back: k_curve_scan (one CTA) is an exclusive scan of the chunks'
// group-start counts, k_curve_write writes each chunk's groups at that offset (block scan inside the chunk).
//
// Definitions (s = prob[1] sorted ascending, n nodes, P positives, N = n - P):
//   pre[j]      positives among s[0, j); pre[n] = P
//   tie group   a maximal run [lo, hi) of equal s; its cut is "positive iff prob[1] >= s[lo]", so
//               TP = P - pre[lo], FP = (n - lo) - TP
//   ap          sklearn's average_precision_score: sum over groups of (pre[hi] - pre[lo]) / P * TP / (n - lo). Every
//               positive of a group carries the group's precision, so this is summed as (1/P) * sum over positives of
//               TP / (n - lo) with lo = lower_bound(s, s[j]) (no group end needed). NaN when P = 0.
//   recall_at_k K = P alerts: with c = n - P and [lo, hi) the group that contains position c,
//               TP@K = (P - pre[hi]) + (pre[hi] - pre[lo]) * (hi - c) / (hi - lo), the expected count over random
//               orders of the tied scores (independent of the sort's tie order), then / P. NaN when P = 0. Since K = P
//               it is Precision@K as well.
//   best_gmean  sqrt(TP/P * TN/N) maximised over the group cuts (a ratio with a zero denominator is 0), ties to the
//               larger threshold, as best_f1_macro
#define MT_NT 256
#define MT_PER 8
#define MT_CH (MT_NT * MT_PER)

struct MetricsBlk {
    long long auc2;        // sum over the chunk's positives of (lo + hi + 1)
    int pos, tp, fp, tn, fn, pad;
};
struct BestBlk {
    double f1;
    long long at;          // sorted position of the cut (-1: none in this chunk)
    double gm;             // best G-mean and its cut
    long long gat;
    double ap;             // sum over the chunk's positives of TP / (n - lo) (k_metrics_ap)
    long long groups;      // tie-group starts in the chunk
    long long goff;        // group starts in front of the chunk (k_curve_scan)
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct MetricsWs {
    char* sort_ws;
    size_t sort_bytes;
    float* s_score;
    int32_t* s_pos;
    int32_t* s_lab;
    MetricsBlk* blk;
    BestBlk* best;
    int32_t* pre;
    size_t total;
};

static MetricsWs metrics_layout(char* base, int64_t n) {
    MetricsWs w;
    const int64_t nb = (n + MT_CH - 1) / MT_CH;
    size_t o = 0;
    w.sort_bytes = pcg_sort_pool_workspace_bytes((int)n);
    w.sort_ws = base + o;   o += align256(w.sort_bytes);
    w.s_score = (float*)(base + o);   o += align256((size_t)n * 4);
    w.s_pos = (int32_t*)(base + o);   o += align256((size_t)n * 4);
    w.s_lab = (int32_t*)(base + o);   o += align256((size_t)n * 4);
    w.blk = (MetricsBlk*)(base + o);  o += align256((size_t)nb * sizeof(MetricsBlk));
    w.best = (BestBlk*)(base + o);    o += align256((size_t)nb * sizeof(BestBlk));
    w.pre = (int32_t*)(base + o);     o += align256((size_t)n * 4);
    w.total = o;
    return w;
}

// first position with s[pos] >= x (lower) / > x (upper) in the ascending array s[0, n)
__device__ __forceinline__ int64_t bound(const float* __restrict__ s, int64_t n, float x, bool upper) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const float v = s[mid];
        if (upper ? !(x < v) : (v < x)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

template <class T>
__device__ __forceinline__ T block_sum(T v, T* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(PCG_FULL, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    T t = 0;
    if (threadIdx.x == 0)
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    return t;              // valid in thread 0
}

__global__ void __launch_bounds__(MT_NT) k_metrics_count(const float* __restrict__ prob, const int32_t* __restrict__ labels,
                                                         int64_t n, const float* __restrict__ s_score,
                                                         const int32_t* __restrict__ s_lab, MetricsBlk* __restrict__ blk) {
    __shared__ long long red[MT_NT / 32];
    const int64_t j0 = (int64_t)blockIdx.x * MT_CH;
    long long auc2 = 0;
    long long c[5] = {0, 0, 0, 0, 0};     // pos, tp, fp, tn, fn
    for (int u = 0; u < MT_PER; ++u) {
        const int64_t j = j0 + u * MT_NT + threadIdx.x;
        if (j >= n) break;
        if (s_lab[j] != 0) {
            const float x = s_score[j];
            auc2 += bound(s_score, n, x, false) + bound(s_score, n, x, true) + 1;
            c[0] += 1;
        }
        const bool pred = prob[n + j] > prob[j];
        const bool y = labels[j] != 0;
        c[1] += pred && y;
        c[2] += pred && !y;
        c[3] += !pred && !y;
        c[4] += !pred && y;
    }
    const long long a = block_sum(auc2, red);
    long long t[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) t[q] = block_sum(c[q], red);
    if (threadIdx.x == 0) {
        MetricsBlk b;
        b.auc2 = a;
        b.pos = (int)t[0]; b.tp = (int)t[1]; b.fp = (int)t[2]; b.tn = (int)t[3]; b.fn = (int)t[4]; b.pad = 0;
        blk[blockIdx.x] = b;
    }
}

__device__ __forceinline__ double ratio(double a, double b) { return b > 0.0 ? a / b : 0.0; }

// macro-F1 from the confusion counts, with metrics.binary_metrics' arithmetic (sklearn zero_division=0)
__device__ __forceinline__ double f1_pair(double tp, double fp, double tn, double fn, double* f1_pos) {
    const double p1 = ratio(tp, tp + fp), r1 = ratio(tp, tp + fn);
    const double p0 = ratio(tn, tn + fn), r0 = ratio(tn, tn + fp);
    const double f1 = ratio(__dmul_rn(__dmul_rn(2.0, p1), r1), p1 + r1);
    const double f0 = ratio(__dmul_rn(__dmul_rn(2.0, p0), r0), p0 + r0);
    if (f1_pos) *f1_pos = f1;
    return __dmul_rn(0.5, f0 + f1);
}

__device__ __forceinline__ bool better(double f, long long at, double bf, long long bat) {
    return f > bf || (f == bf && at > bat);      // ties: the larger threshold
}

// (bf, bat) <- the better() maximum over the warp, in every lane
__device__ __forceinline__ void argmax_warp(double& bf, long long& bat) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double of = __shfl_xor_sync(PCG_FULL, bf, o);
        const long long oat = __shfl_xor_sync(PCG_FULL, bat, o);
        if (better(of, oat, bf, bat)) { bf = of; bat = oat; }
    }
}

// exclusive prefix sum of v over the CTA's threads in thread order; warp_tot: MT_NT / 32 ints of shared memory, one
// call per kernel
__device__ __forceinline__ int block_excl_scan(int v, int* warp_tot) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(PCG_FULL, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    int run = incl - v;
    for (int q = 0; q < wid; ++q) run += warp_tot[q];
    return run;
}

__global__ void __launch_bounds__(MT_NT) k_metrics_best(int64_t n, const float* __restrict__ s_score,
                                                        const int32_t* __restrict__ s_lab,
                                                        const MetricsBlk* __restrict__ blk, int nb,
                                                        BestBlk* __restrict__ best, int32_t* __restrict__ pre) {
    __shared__ long long red[MT_NT / 32];
    __shared__ int lab_s[MT_CH];
    __shared__ float sc_s[MT_CH + 1];
    __shared__ int warp_tot[MT_NT / 32];
    __shared__ double bf_s[MT_NT / 32], bg_s[MT_NT / 32];
    __shared__ long long bat_s[MT_NT / 32], bgat_s[MT_NT / 32];
    __shared__ long long pos_all, pos_before;
    const int64_t j0 = (int64_t)blockIdx.x * MT_CH;
    // positives over all chunks and in front of this one
    long long all = 0, before = 0;
    for (int c = threadIdx.x; c < nb; c += MT_NT) {
        all += blk[c].pos;
        if (c < (int)blockIdx.x) before += blk[c].pos;
    }
    all = block_sum(all, red);
    if (threadIdx.x == 0) pos_all = all;
    before = block_sum(before, red);
    if (threadIdx.x == 0) pos_before = before;
    for (int u = 0; u < MT_PER; ++u) {
        const int k = u * MT_NT + threadIdx.x;
        const int64_t j = j0 + k;
        lab_s[k] = j < n ? (s_lab[j] != 0) : 0;
        sc_s[k + 1] = j < n ? s_score[j] : 0.f;
    }
    if (threadIdx.x == 0) sc_s[0] = j0 > 0 ? s_score[j0 - 1] : 0.f;
    __syncthreads();
    // exclusive scan of the per-thread counts (thread t owns chunk positions t*MT_PER .. +MT_PER)
    int mine = 0;
#pragma unroll
    for (int u = 0; u < MT_PER; ++u) mine += lab_s[threadIdx.x * MT_PER + u];
    const int run = block_excl_scan(mine, warp_tot);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const double P = (double)pos_all, N = (double)(n - pos_all);
    long long cnt = pos_before + run;          // positives in front of the current position
    double bf = -1.0, bg = -1.0;
    long long bat = -1, bgat = -1, groups = 0;
    for (int u = 0; u < MT_PER; ++u) {
        const int k = threadIdx.x * MT_PER + u;
        const int64_t j = j0 + k;
        if (j >= n) break;
        pre[j] = (int32_t)cnt;
        if (j == 0 || sc_s[k + 1] != sc_s[k]) {
            const double tp = P - (double)cnt, pp = (double)(n - j);
            const double fp = pp - tp, fn = P - tp, tn = N - fp;
            const double f = f1_pair(tp, fp, tn, fn, nullptr);
            if (better(f, j, bf, bat)) { bf = f; bat = j; }
            const double g = sqrt(__dmul_rn(ratio(tp, P), ratio(tn, N)));
            if (better(g, j, bg, bgat)) { bg = g; bgat = j; }
            ++groups;
        }
        cnt += lab_s[k];
    }
    groups = block_sum(groups, red);
    argmax_warp(bf, bat);
    argmax_warp(bg, bgat);
    if (lane == 0) { bf_s[wid] = bf; bat_s[wid] = bat; bg_s[wid] = bg; bgat_s[wid] = bgat; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < MT_NT / 32; ++q) {
            if (better(bf_s[q], bat_s[q], bf, bat)) { bf = bf_s[q]; bat = bat_s[q]; }
            if (better(bg_s[q], bgat_s[q], bg, bgat)) { bg = bg_s[q]; bgat = bgat_s[q]; }
        }
        BestBlk& b = best[blockIdx.x];
        b.f1 = bf;
        b.at = bat;
        b.gm = bg;
        b.gat = bgat;
        b.groups = groups;
    }
}

// Average-precision terms of the chunk's positives (see the definitions above): sum of TP / (n - lo) over the
// positives at sorted positions j of the chunk, lo = the start of j's tie group. Needs pre of every chunk.
__global__ void __launch_bounds__(MT_NT) k_metrics_ap(int64_t n, const float* __restrict__ s_score,
                                                      const int32_t* __restrict__ s_lab, const int32_t* __restrict__ pre,
                                                      BestBlk* __restrict__ best) {
    __shared__ double red[MT_NT / 32];
    const int64_t j0 = (int64_t)blockIdx.x * MT_CH;
    const long long P = (long long)pre[n - 1] + (s_lab[n - 1] != 0);
    double acc = 0.0;
    for (int u = 0; u < MT_PER; ++u) {
        const int64_t j = j0 + u * MT_NT + threadIdx.x;
        if (j >= n) break;
        if (s_lab[j] != 0) {
            const int64_t lo = bound(s_score, n, s_score[j], false);
            acc += (double)(P - pre[lo]) / (double)(n - lo);
        }
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) best[blockIdx.x].ap = acc;
}

// TP@K of the top K = n - c positions: with [lo, hi) the tie group that contains position c, the positives above the
// group plus the group's positives by their expected share (hi - c) / (hi - lo) of its slots above the cut
__device__ __forceinline__ double tp_at_k_of(long long P, long long plo, long long phi, int64_t lo, int64_t hi, int64_t c) {
    return (double)(P - phi) + (double)(phi - plo) * (double)(hi - c) / (double)(hi - lo);
}

__device__ __forceinline__ double tp_at_k(int64_t n, const float* __restrict__ s_score, const int32_t* __restrict__ pre,
                                          long long P, int64_t c) {
    const float x = s_score[c];
    const int64_t lo = bound(s_score, n, x, false), hi = bound(s_score, n, x, true);
    return tp_at_k_of(P, pre[lo], hi < n ? (long long)pre[hi] : P, lo, hi, c);
}

__global__ void __launch_bounds__(MT_NT) k_metrics_final(int64_t n, const float* __restrict__ s_score,
                                                         const int32_t* __restrict__ pre,
                                                         const MetricsBlk* __restrict__ blk, const BestBlk* __restrict__ best,
                                                         int nb, double* __restrict__ out) {
    __shared__ long long red[MT_NT / 32];
    __shared__ double red_d[MT_NT / 32];
    __shared__ double bf_s[MT_NT / 32], bg_s[MT_NT / 32];
    __shared__ long long bat_s[MT_NT / 32], bgat_s[MT_NT / 32];
    long long c[6] = {0, 0, 0, 0, 0, 0};       // auc2, pos, tp, fp, tn, fn
    double bf = -1.0, bg = -1.0, ap = 0.0;
    long long bat = -1, bgat = -1;
    for (int b = threadIdx.x; b < nb; b += MT_NT) {
        const MetricsBlk m = blk[b];
        c[0] += m.auc2; c[1] += m.pos; c[2] += m.tp; c[3] += m.fp; c[4] += m.tn; c[5] += m.fn;
        const BestBlk k = best[b];
        if (better(k.f1, k.at, bf, bat)) { bf = k.f1; bat = k.at; }
        if (better(k.gm, k.gat, bg, bgat)) { bg = k.gm; bgat = k.gat; }
        ap += k.ap;                           // chunks b, b + MT_NT, ... in order, then a fixed tree: same bits on reruns
    }
    long long t[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) t[q] = block_sum(c[q], red);
    ap = block_sum(ap, red_d);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    argmax_warp(bf, bat);
    argmax_warp(bg, bgat);
    if (lane == 0) { bf_s[wid] = bf; bat_s[wid] = bat; bg_s[wid] = bg; bgat_s[wid] = bgat; }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int q = 1; q < MT_NT / 32; ++q) {
        if (better(bf_s[q], bat_s[q], bf, bat)) { bf = bf_s[q]; bat = bat_s[q]; }
        if (better(bg_s[q], bgat_s[q], bg, bgat)) { bg = bg_s[q]; bgat = bgat_s[q]; }
    }
    const long long P = t[1], N = n - t[1];
    const double tp = (double)t[2], fp = (double)t[3], tn = (double)t[4], fn = (double)t[5];
    // Mann-Whitney U with average ranks: 2U = sum_pos (lo + hi + 1) - P(P+1), exact in int64
    out[PCG_MT_AUC] = (P > 0 && N > 0) ? (double)(t[0] - P * (P + 1)) / (2.0 * (double)P * (double)N) : nan("");
    double f1 = 0.0;
    out[PCG_MT_F1_MACRO] = f1_pair(tp, fp, tn, fn, &f1);
    out[PCG_MT_F1] = f1;
    const double r1 = ratio(tp, tp + fn), p1 = ratio(tp, tp + fp), r0 = ratio(tn, tn + fp), p0 = ratio(tn, tn + fn);
    out[PCG_MT_RECALL] = r1;
    out[PCG_MT_PRECISION] = p1;
    out[PCG_MT_RECALL_MACRO] = __dmul_rn(0.5, r0 + r1);
    out[PCG_MT_PRECISION_MACRO] = __dmul_rn(0.5, p0 + p1);
    out[PCG_MT_ACCURACY] = (tp + tn) / (double)n;
    out[PCG_MT_GMEAN] = sqrt(__dmul_rn(r1, r0));
    out[PCG_MT_BEST_F1_MACRO] = bf;
    out[PCG_MT_BEST_THRESHOLD] = (double)s_score[bat];
    out[PCG_MT_N_POS] = (double)P;
    out[PCG_MT_N_NEG] = (double)N;
    out[PCG_MT_TP] = tp;
    out[PCG_MT_FP] = fp;
    out[PCG_MT_TN] = tn;
    out[PCG_MT_FN] = fn;
    out[PCG_MT_AP] = P > 0 ? ap / (double)P : nan("");
    out[PCG_MT_RECALL_AT_K] = P > 0 ? tp_at_k(n, s_score, pre, P, n - P) / (double)P : nan("");   // K = P
    out[PCG_MT_BEST_GMEAN] = bg;
    out[PCG_MT_BEST_GMEAN_THRESHOLD] = (double)s_score[bgat];
}

// Exclusive scan of the chunks' group-start counts into best[b].goff (one CTA, MT_NT chunks per round); *count = G.
__global__ void __launch_bounds__(MT_NT) k_curve_scan(BestBlk* __restrict__ best, int nb, int64_t* __restrict__ count) {
    __shared__ int warp_tot[MT_NT / 32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    for (int b0 = 0; b0 < nb; b0 += MT_NT) {
        const int b = b0 + threadIdx.x;
        const int g = b < nb ? (int)best[b].groups : 0;
        __syncthreads();                       // carry written, warp_tot free for the next round
        const int run = block_excl_scan(g, warp_tot);
        if (b < nb) best[b].goff = carry + run;
        __syncthreads();
        if (threadIdx.x == MT_NT - 1) carry += run + g;
    }
    __syncthreads();
    if (threadIdx.x == 0) *count = carry;
}

// Each chunk's group starts j, in order, at best[chunk].goff: thr = s[j], tp = P - pre[j], fp = (n - j) - tp.
__global__ void __launch_bounds__(MT_NT) k_curve_write(int64_t n, const float* __restrict__ s_score,
                                                       const int32_t* __restrict__ s_lab, const int32_t* __restrict__ pre,
                                                       const BestBlk* __restrict__ best, float* __restrict__ thr,
                                                       int64_t* __restrict__ tp, int64_t* __restrict__ fp) {
    __shared__ float sc_s[MT_CH + 1];
    __shared__ int warp_tot[MT_NT / 32];
    const int64_t j0 = (int64_t)blockIdx.x * MT_CH;
    for (int u = 0; u < MT_PER; ++u) {
        const int k = u * MT_NT + threadIdx.x;
        const int64_t j = j0 + k;
        sc_s[k + 1] = j < n ? s_score[j] : 0.f;
    }
    if (threadIdx.x == 0) sc_s[0] = j0 > 0 ? s_score[j0 - 1] : 0.f;
    __syncthreads();
    const long long P = (long long)pre[n - 1] + (s_lab[n - 1] != 0);
    int mine = 0;
#pragma unroll
    for (int u = 0; u < MT_PER; ++u) {
        const int k = threadIdx.x * MT_PER + u;
        const int64_t j = j0 + k;
        mine += j < n && (j == 0 || sc_s[k + 1] != sc_s[k]);
    }
    long long at = best[blockIdx.x].goff + block_excl_scan(mine, warp_tot);
    for (int u = 0; u < MT_PER; ++u) {
        const int k = threadIdx.x * MT_PER + u;
        const int64_t j = j0 + k;
        if (j >= n) break;
        if (j == 0 || sc_s[k + 1] != sc_s[k]) {
            const long long t = P - pre[j];
            thr[at] = sc_s[k + 1];
            tp[at] = t;
            fp[at] = (n - j) - t;
            ++at;
        }
    }
}

// ------------------------------------------------------------------------------- operating points
// pcg_binary_points answers caller-chosen requests from the workspace of the last metrics call:
//   k_points        CTAs 1 .. nb, one per chunk, kind 2 (partial AUC): every tie group [lo, hi) that starts in the
//                   chunk adds the ROC segment from (FP(hi)/N, TP(hi)/P) to (FP(lo)/N, TP(lo)/P), clipped at FPR = f,
//                   as a trapezoid. Thread t owns chunk positions t*MT_PER .. +MT_PER (two 16-byte loads each of
//                   scores and pre), so a group's hi is the thread's next group start; after the thread's last start it
//                   is the next thread's first position when that starts a group (distinct scores), else a binary
//                   search in the chunk's shared scores, or the end of the group that runs past the chunk (one warp
//                   search per chunk). One fp64
//                   partial per (request, chunk), part[r * nb + chunk], holding twice the area (the 1/2 of the
//                   trapezoids is applied once, at the end).
//                   CTA 0: kinds 0 and 1 and the NaN words of malformed requests, one warp per request (a few
//                   warp_search calls each), beside the chunk CTAs.
//   k_points_final  one CTA, kind 2: adds the request's chunk partials in a fixed order and standardises (same bits on
//                   reruns).
// Definitions and the output words per kind: include/pcgnn_b200.h.

// The first j in [lo, hi) with !before(j), else hi, for a predicate that holds on a prefix of [lo, hi); called by a
// whole warp with the same arguments, result in every lane. 32 probes per round: ceil(log32(hi - lo)) dependent loads.
template <class F>
__device__ __forceinline__ int64_t warp_search(int64_t lo, int64_t hi, F before) {
    const int lane = threadIdx.x & 31;
    while (lo < hi) {
        const int64_t step = (hi - lo + 31) >> 5;
        const int64_t p = lo + step * (lane + 1) - 1;
        const int64_t nlo = lo + step * __popc(__ballot_sync(PCG_FULL, p < hi && before(p)));
        hi = nlo + step - 1 < hi ? nlo + step - 1 : hi;
        lo = nlo;
    }
    return lo;
}

__device__ __forceinline__ bool point_valid(int kd, double a, int64_t n) {
    if (kd == PCG_POINT_TOP_K) return a >= 1.0 && a <= (double)n && a == floor(a);
    if (kd == PCG_POINT_TPR_AT_FPR) return a >= 0.0 && a <= 1.0;
    if (kd == PCG_POINT_PAUC) return a > 0.0 && a <= 1.0;
    return false;
}

// kinds 0 and 1 (and NaN words for malformed requests other than kind 2), warp w taking requests w, w + 8, ...
__device__ void points_search(int64_t n, const float* __restrict__ s, const int32_t* __restrict__ pre, long long P,
                              const int32_t* kd_s, const double* ar_s, int m, double* __restrict__ out) {
    const long long N = n - P;
    const double nan_ = nan("");
    const int lane = threadIdx.x & 31;
    for (int r = threadIdx.x >> 5; r < m; r += MT_NT / 32) {
        const int kd = kd_s[r];
        const double a = ar_s[r];
        double w[PCG_POINT_WORDS];
#pragma unroll
        for (int q = 0; q < PCG_POINT_WORDS; ++q) w[q] = nan_;
        if (kd == PCG_POINT_PAUC) continue;     // k_points_final (the warp's lanes share r)
        if (kd == PCG_POINT_TOP_K && point_valid(kd, a, n)) {
            const int64_t c = n - (int64_t)a;
            const float x = s[c];
            const int64_t lo = warp_search(0, c, [&](int64_t j) { return s[j] < x; });
            const int64_t hi = warp_search(c + 1, n, [&](int64_t j) { return !(x < s[j]); });
            const double tpk = tp_at_k_of(P, pre[lo], hi < n ? (long long)pre[hi] : P, lo, hi, c);
            w[0] = P > 0 ? tpk / (double)P : nan_;
            w[1] = tpk / a;
            w[2] = (double)x;
            w[3] = tpk;
            w[4] = a - tpk;
        } else if (kd == PCG_POINT_TPR_AT_FPR && point_valid(kd, a, n) && P > 0 && N > 0) {
            const double lim = a * (double)N;   // FP(j) = (n - j) - (P - pre[j]) does not increase; FP(n) = 0
            int64_t j = warp_search(0, n, [&](int64_t i) { return (double)((n - i) - (P - pre[i])) > lim; });
            if (j > 0 && j < n && s[j - 1] == s[j]) {       // inside a tie group: its cut is the next group start
                const float x = s[j];
                j = warp_search(j + 1, n, [&](int64_t i) { return !(x < s[i]); });
            }
            const long long tp = j < n ? P - pre[j] : 0, fp = (n - j) - tp;
            w[0] = (double)tp / (double)P;
            w[1] = (double)fp / (double)N;
            w[2] = j < n ? (double)s[j] : (double)INFINITY;
            w[3] = (double)tp;
            w[4] = (double)fp;
        }
        if (lane < PCG_POINT_WORDS) {
            double v = w[0];
#pragma unroll
            for (int q = 1; q < PCG_POINT_WORDS; ++q) v = lane == q ? w[q] : v;
            out[(size_t)r * PCG_POINT_WORDS + lane] = v;
        }
    }
}

// the requests into shared memory (m <= PCG_POINTS_MAX)
__device__ __forceinline__ void load_points(const int32_t* __restrict__ kind, const double* __restrict__ arg, int m,
                                            int* kd_s, double* ar_s) {
    for (int r = threadIdx.x; r < m; r += MT_NT) {
        kd_s[r] = kind[r];
        ar_s[r] = arg[r];
    }
}

__global__ void __launch_bounds__(MT_NT, 2) k_points(int64_t n, const float* __restrict__ s_score,
                                                     const int32_t* __restrict__ s_lab, const int32_t* __restrict__ pre,
                                                     const int32_t* __restrict__ kind, const double* __restrict__ arg,
                                                     int m, int nb, double* __restrict__ part, double* __restrict__ out) {
    __shared__ float sc_s[MT_CH];
    __shared__ int pf_s[MT_NT];                // pre at each thread's first position
    __shared__ int kd_s[PCG_POINTS_MAX];
    __shared__ double ar_s[PCG_POINTS_MAX];
    __shared__ double red[MT_NT / 32];
    __shared__ long long edge_hi, edge_tp;
    const long long P = (long long)pre[n - 1] + (s_lab[n - 1] != 0);
    load_points(kind, arg, m, kd_s, ar_s);
    __syncthreads();
    if (blockIdx.x == 0) {
        points_search(n, s_score, pre, P, kd_s, ar_s, m, out);
        return;
    }
    const int chunk = (int)blockIdx.x - 1;
    int any = 0;
    for (int r = threadIdx.x; r < m; r += MT_NT) any |= kd_s[r] == PCG_POINT_PAUC && point_valid(kd_s[r], ar_s[r], n);
    if (!__syncthreads_or(any) || P == 0 || P == n) return;   // no partial AUC to compute (NaN: k_points_final)
    const double iP = 1.0 / (double)P, iN = 1.0 / (double)(n - P);
    const int64_t j0 = (int64_t)chunk * MT_CH;
    const int kend = (int)(n - j0 < (int64_t)MT_CH ? n - j0 : (int64_t)MT_CH);
    const int k0 = threadIdx.x * MT_PER;
    float sv[MT_PER];                          // the thread's positions k0 .. k0 + MT_PER, straight from global memory
    int pv[MT_PER];
    if (k0 + MT_PER <= kend) {                 // 32-byte aligned: chunks start at multiples of MT_CH
        const float4* s4 = (const float4*)(s_score + j0 + k0);
        const int4* p4 = (const int4*)(pre + j0 + k0);
        const float4 a0 = s4[0], a1 = s4[1];
        const int4 b0 = p4[0], b1 = p4[1];
        sv[0] = a0.x; sv[1] = a0.y; sv[2] = a0.z; sv[3] = a0.w; sv[4] = a1.x; sv[5] = a1.y; sv[6] = a1.z; sv[7] = a1.w;
        pv[0] = b0.x; pv[1] = b0.y; pv[2] = b0.z; pv[3] = b0.w; pv[4] = b1.x; pv[5] = b1.y; pv[6] = b1.z; pv[7] = b1.w;
    } else {
#pragma unroll
        for (int u = 0; u < MT_PER; ++u) {
            sv[u] = k0 + u < kend ? s_score[j0 + k0 + u] : 0.f;
            pv[u] = k0 + u < kend ? pre[j0 + k0 + u] : 0;
        }
    }
#pragma unroll
    for (int u = 0; u < MT_PER; ++u) sc_s[k0 + u] = sv[u];
    pf_s[threadIdx.x] = pv[0];
    if (threadIdx.x < 32) {                    // the end of the chunk's last group, which may run past the chunk
        const int64_t e = j0 + kend;
        const float v = s_score[e - 1];
        const int64_t hi = e < n && !(v < s_score[e]) ? warp_search(e + 1, n, [&](int64_t j) { return !(v < s_score[j]); })
                                                      : e;
        if (threadIdx.x == 0) {
            edge_hi = hi;
            edge_tp = hi < n ? P - pre[hi] : 0;
        }
    }
    const float before = k0 == 0 && j0 > 0 ? s_score[j0 - 1] : 0.f;   // thread 0: the previous chunk's last score
    __syncthreads();
    double x[MT_PER], y[MT_PER];               // ROC point of the group starting at k0 + u; x < 0: no group start there
    bool started = false;
    float v = 0.f;                             // score of the thread's last group start
#pragma unroll
    for (int u = 0; u < MT_PER; ++u) {
        const int k = k0 + u;
        const float prev = u > 0 ? sv[u - 1] : (k0 > 0 ? sc_s[k0 - 1] : before);
        x[u] = -1.0;
        y[u] = 0.0;
        if (k < kend && (j0 + k == 0 || sv[u] != prev)) {
            const long long tp = P - pv[u];
            x[u] = (double)((n - j0 - k) - tp) * iN;
            y[u] = (double)tp * iP;
            started = true;
            v = sv[u];
        }
    }
    double xe = 0.0, ye = 0.0;                 // the point of the group start after the thread's last one
    if (started) {
        int a = k0 + MT_PER < kend ? k0 + MT_PER : kend;
        long long tp;
        if (a < kend && v < sc_s[a]) {         // the next thread's first position starts a group (distinct scores)
            tp = P - pf_s[threadIdx.x + 1];
        } else {                               // first larger score in the chunk, else kend
            int b = kend;
            while (a < b) {
                const int mid = (a + b) >> 1;
                if (!(v < sc_s[mid])) a = mid + 1; else b = mid;
            }
            tp = a < kend ? P - pre[j0 + a] : edge_tp;
        }
        const int64_t hi = a < kend ? j0 + a : edge_hi;
        xe = (double)((n - hi) - tp) * iN;
        ye = (double)tp * iP;
    }
    for (int r = 0; r < m; ++r) {
        const double f = ar_s[r];
        if (kd_s[r] != PCG_POINT_PAUC || !point_valid(PCG_POINT_PAUC, f, n)) continue;   // the same for every thread
        double acc = 0.0, xh = xe, yh = ye;
#pragma unroll
        for (int u = MT_PER - 1; u >= 0; --u) {
            if (x[u] < 0.0) continue;
            if (xh < f) {
                if (x[u] <= f) {
                    acc += (x[u] - xh) * (y[u] + yh);
                } else {                       // TPR at f on the segment, linearly
                    const double yf = yh + (y[u] - yh) * (f - xh) / (x[u] - xh);
                    acc += (f - xh) * (yf + yh);
                }
            }
            xh = x[u];
            yh = y[u];
        }
        acc = block_sum(acc, red);
        if (threadIdx.x == 0) part[(size_t)r * nb + chunk] = acc;
    }
}

__global__ void __launch_bounds__(MT_NT) k_points_final(int64_t n, const int32_t* __restrict__ s_lab,
                                                        const int32_t* __restrict__ pre, const int32_t* __restrict__ kind,
                                                        const double* __restrict__ arg, int m, int nb,
                                                        const double* __restrict__ part, double* __restrict__ out) {
    __shared__ int kd_s[PCG_POINTS_MAX];
    __shared__ double ar_s[PCG_POINTS_MAX];
    __shared__ double red[MT_NT / 32];
    const long long P = (long long)pre[n - 1] + (s_lab[n - 1] != 0), N = n - P;
    load_points(kind, arg, m, kd_s, ar_s);
    __syncthreads();
    for (int r = 0; r < m; ++r) {
        if (kd_s[r] != PCG_POINT_PAUC) continue;
        const double f = ar_s[r];
        const bool ok = point_valid(PCG_POINT_PAUC, f, n) && P > 0 && N > 0;
        double acc = 0.0;
        if (ok) {
#pragma unroll 4
            for (int b = threadIdx.x; b < nb; b += MT_NT) acc += part[(size_t)r * nb + b];
        }
        acc = block_sum(acc, red);
        if (threadIdx.x == 0) {
            double* o = out + (size_t)r * PCG_POINT_WORDS;
            const double A = 0.5 * acc, lo_area = 0.5 * f * f, nan_ = nan("");
            o[0] = ok ? 0.5 * (1.0 + (A - lo_area) / (f - lo_area)) : nan_;     // sklearn's McClish correction
            o[1] = ok ? A : nan_;
            for (int q = 2; q < PCG_POINT_WORDS; ++q) o[q] = nan_;
        }
    }
}

static size_t points_part_bytes(int64_t n, int m) {
    return align256((size_t)m * (size_t)((n + MT_CH - 1) / MT_CH) * sizeof(double));
}

extern "C" size_t pcg_binary_metrics_workspace_bytes(int64_t n) {
    if (n <= 0 || n > 0x7fffffff) return 0;
    return metrics_layout(nullptr, n).total;
}

extern "C" int pcg_binary_metrics(const float* prob, const int32_t* labels, int64_t n, double* out, void* workspace,
                                  size_t workspace_bytes, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(prob && labels && out && workspace, "pcg_binary_metrics: null pointer");
    PCG_REQUIRE(n > 0 && n <= 0x7fffffff, "pcg_binary_metrics: need 0 < n < 2^31 (n=%lld)", (long long)n);
    const MetricsWs w = metrics_layout((char*)workspace, n);
    PCG_REQUIRE(((uintptr_t)workspace & 255) == 0 && workspace_bytes >= w.total,
                "pcg_binary_metrics: workspace must be 256-byte aligned and pcg_binary_metrics_workspace_bytes(n) long");
    const int nb = (int)((n + MT_CH - 1) / MT_CH);
    int rc = pcg_sort_pool(prob + n, labels, (int)n, w.s_score, w.s_pos, w.s_lab, w.sort_ws, w.sort_bytes, stream_);
    if (rc) return rc;
    k_metrics_count<<<nb, MT_NT, 0, stream>>>(prob, labels, n, w.s_score, w.s_lab, w.blk);
    k_metrics_best<<<nb, MT_NT, 0, stream>>>(n, w.s_score, w.s_lab, w.blk, nb, w.best, w.pre);
    k_metrics_ap<<<nb, MT_NT, 0, stream>>>(n, w.s_score, w.s_lab, w.pre, w.best);
    k_metrics_final<<<1, MT_NT, 0, stream>>>(n, w.s_score, w.pre, w.blk, w.best, nb, out);
    return pcg_check_launch("pcg_binary_metrics");
}

extern "C" int pcg_binary_curve(const void* workspace, size_t workspace_bytes, int64_t n, float* thr, int64_t* tp,
                                int64_t* fp, int64_t* count, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(workspace && thr && tp && fp && count, "pcg_binary_curve: null pointer");
    PCG_REQUIRE(n > 0 && n <= 0x7fffffff, "pcg_binary_curve: need 0 < n < 2^31 (n=%lld)", (long long)n);
    const MetricsWs w = metrics_layout((char*)workspace, n);
    PCG_REQUIRE(((uintptr_t)workspace & 255) == 0 && workspace_bytes >= w.total,
                "pcg_binary_curve: workspace must be 256-byte aligned and pcg_binary_metrics_workspace_bytes(n) long");
    const int nb = (int)((n + MT_CH - 1) / MT_CH);
    k_curve_scan<<<1, MT_NT, 0, stream>>>(w.best, nb, count);
    k_curve_write<<<nb, MT_NT, 0, stream>>>(n, w.s_score, w.s_lab, w.pre, w.best, thr, tp, fp);
    return pcg_check_launch("pcg_binary_curve");
}

extern "C" size_t pcg_binary_points_workspace_bytes(int64_t n, int m) {
    if (n <= 0 || n > 0x7fffffff || m <= 0 || m > PCG_POINTS_MAX) return 0;
    return points_part_bytes(n, m);
}

extern "C" int pcg_binary_points(const void* metrics_ws, size_t metrics_ws_bytes, int64_t n, const int32_t* kind,
                                 const double* arg, int m, double* out, void* ws, size_t ws_bytes, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(metrics_ws && kind && arg && out && ws, "pcg_binary_points: null pointer");
    PCG_REQUIRE(n > 0 && n <= 0x7fffffff, "pcg_binary_points: need 0 < n < 2^31 (n=%lld)", (long long)n);
    PCG_REQUIRE(m > 0 && m <= PCG_POINTS_MAX, "pcg_binary_points: need 0 < m <= %d requests (m=%d)", PCG_POINTS_MAX, m);
    const MetricsWs w = metrics_layout((char*)metrics_ws, n);
    PCG_REQUIRE(((uintptr_t)metrics_ws & 255) == 0 && metrics_ws_bytes >= w.total,
                "pcg_binary_points: metrics_ws must be 256-byte aligned and pcg_binary_metrics_workspace_bytes(n) long");
    PCG_REQUIRE(((uintptr_t)ws & 7) == 0 && ws_bytes >= points_part_bytes(n, m),
                "pcg_binary_points: ws must be 8-byte aligned and pcg_binary_points_workspace_bytes(n, m) long");
    PCG_REQUIRE(((uintptr_t)kind & 3) == 0 && ((uintptr_t)arg & 7) == 0 && ((uintptr_t)out & 7) == 0,
                "pcg_binary_points: kind, arg and out must be aligned to their element size");
    const int nb = (int)((n + MT_CH - 1) / MT_CH);
    double* part = (double*)ws;
    k_points<<<nb + 1, MT_NT, 0, stream>>>(n, w.s_score, w.s_lab, w.pre, kind, arg, m, nb, part, out);
    k_points_final<<<1, MT_NT, 0, stream>>>(n, w.s_lab, w.pre, kind, arg, m, nb, part, out);
    return pcg_check_launch("pcg_binary_points");
}
