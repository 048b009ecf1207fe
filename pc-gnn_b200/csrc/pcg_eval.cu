// Evaluation pass on the device: the two-class head + sigmoid (PCALayer, GCN) or log-softmax (GraphSage) into a
// whole-set probability buffer, and the binary metrics of src/utils.py:298-333 (AUC, F1, recall, precision, ...) plus
// a best-threshold macro-F1, computed where the probabilities live. Deterministic: integer sums and an order-free
// arg-max only (no floating-point atomics).
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
//                    macro-F1 of the cut "positive iff prob[1] >= s[j]" at every tie-group start j, the chunk's best
//   k_metrics_final  one CTA: sums and arg-max over the chunks, every metric in double
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

__global__ void __launch_bounds__(MT_NT) k_metrics_best(int64_t n, const float* __restrict__ s_score,
                                                        const int32_t* __restrict__ s_lab,
                                                        const MetricsBlk* __restrict__ blk, int nb,
                                                        BestBlk* __restrict__ best) {
    __shared__ long long red[MT_NT / 32];
    __shared__ int lab_s[MT_CH];
    __shared__ float sc_s[MT_CH + 1];
    __shared__ int warp_tot[MT_NT / 32];
    __shared__ double bf_s[MT_NT / 32];
    __shared__ long long bat_s[MT_NT / 32];
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
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(PCG_FULL, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    int run = incl - mine;
    for (int q = 0; q < wid; ++q) run += warp_tot[q];
    const double P = (double)pos_all, N = (double)(n - pos_all);
    long long cnt = pos_before + run;          // positives in front of the current position
    double bf = -1.0;
    long long bat = -1;
    for (int u = 0; u < MT_PER; ++u) {
        const int k = threadIdx.x * MT_PER + u;
        const int64_t j = j0 + k;
        if (j >= n) break;
        if (j == 0 || sc_s[k + 1] != sc_s[k]) {
            const double tp = P - (double)cnt, pp = (double)(n - j);
            const double fp = pp - tp, fn = P - tp, tn = N - fp;
            const double f = f1_pair(tp, fp, tn, fn, nullptr);
            if (better(f, j, bf, bat)) { bf = f; bat = j; }
        }
        cnt += lab_s[k];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double of = __shfl_xor_sync(PCG_FULL, bf, o);
        const long long oat = __shfl_xor_sync(PCG_FULL, bat, o);
        if (better(of, oat, bf, bat)) { bf = of; bat = oat; }
    }
    if (lane == 0) { bf_s[wid] = bf; bat_s[wid] = bat; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < MT_NT / 32; ++q)
            if (better(bf_s[q], bat_s[q], bf, bat)) { bf = bf_s[q]; bat = bat_s[q]; }
        best[blockIdx.x].f1 = bf;
        best[blockIdx.x].at = bat;
    }
}

__global__ void __launch_bounds__(MT_NT) k_metrics_final(int64_t n, const float* __restrict__ s_score,
                                                         const MetricsBlk* __restrict__ blk, const BestBlk* __restrict__ best,
                                                         int nb, double* __restrict__ out) {
    __shared__ long long red[MT_NT / 32];
    __shared__ double bf_s[MT_NT / 32];
    __shared__ long long bat_s[MT_NT / 32];
    long long c[6] = {0, 0, 0, 0, 0, 0};       // auc2, pos, tp, fp, tn, fn
    double bf = -1.0;
    long long bat = -1;
    for (int b = threadIdx.x; b < nb; b += MT_NT) {
        const MetricsBlk m = blk[b];
        c[0] += m.auc2; c[1] += m.pos; c[2] += m.tp; c[3] += m.fp; c[4] += m.tn; c[5] += m.fn;
        if (better(best[b].f1, best[b].at, bf, bat)) { bf = best[b].f1; bat = best[b].at; }
    }
    long long t[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) t[q] = block_sum(c[q], red);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double of = __shfl_xor_sync(PCG_FULL, bf, o);
        const long long oat = __shfl_xor_sync(PCG_FULL, bat, o);
        if (better(of, oat, bf, bat)) { bf = of; bat = oat; }
    }
    if (lane == 0) { bf_s[wid] = bf; bat_s[wid] = bat; }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int q = 1; q < MT_NT / 32; ++q)
        if (better(bf_s[q], bat_s[q], bf, bat)) { bf = bf_s[q]; bat = bat_s[q]; }
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
    k_metrics_best<<<nb, MT_NT, 0, stream>>>(n, w.s_score, w.s_lab, w.blk, nb, w.best);
    k_metrics_final<<<1, MT_NT, 0, stream>>>(n, w.s_score, w.blk, w.best, nb, out);
    return pcg_check_launch("pcg_binary_metrics");
}
