// Fused dense part of the step, one kernel per tile of TM targets:
//
//   self rows + aggregated rows -> per-relation Linear+ReLU -> concat -> inter-relation combine (+ReLU,
//   transposed store) -> label_clf head -> [train] PCALayer head, both cross-entropies, and the whole
//   activation backward (dZ, dH) plus the head / label_clf weight gradients.
//
// Reference (/root/reference/src): layers.py:616-629 (relu(cat(self, agg_r) @ W_r)), :273-289
// (relu(cat(self, h_1..h_R) @ W).t()), :236-243 (label_clf on the batch), model.py:38 (W_head @ combined),
// :54-61 (loss = CE(gnn) + lambda * CE(label)), and what autograd derives from them. There each step is a
// separate cat / mm / relu library call with its autograd twin; the first round of this repo used one GEMM
// kernel per step (csrc/pcg_dense.cu, csrc/pcg_head.cu: 8 launches with every activation round-tripping global
// memory). Here a tile's activations never leave shared memory:
//
//   * the tile's operand rows (feat[target], agg[r][target]) are loaded once into shared memory,
//   * the weights stream through a ring of [32 x E] chunks filled by cp.async.bulk (TMA bulk copies: a chunk is
//     32 consecutive weight rows = ONE contiguous 32*E*4-byte copy) completing on mbarriers; a dedicated producer
//     warp runs ahead across GEMM boundaries, so the weight stream is one continuous pipeline per tile; the ring
//     is as deep as shared memory allows (C2: all 19 chunks of a tile are in flight at once, 152 KB),
//   * 8 consumer warps own (8 rows x 64 columns) register tiles (16 accumulators per lane, operands read from
//     shared memory as float4 with broadcast) and split K among themselves when the tile has fewer than 8 such
//     blocks; partial sums meet in shared memory in a fixed order (deterministic),
//   * in training mode dLoss == 1 is known at forward time, so the kernel goes on: softmax / cross-entropy per
//     target, dZ = (W_head^T dl) * relu', dH = (dZ @ W[F:]^T) * relu', and the per-tile partial sums of the
//     head and label_clf weight gradients.
// What is left for a second kernel is only the batch-reduction of the weight gradients (k_wgrad below):
// cat^T @ dZ and [self | agg_r]^T @ dH_r, split over the batch across a thread-block CLUSTER whose CTAs add
// their partial tiles through distributed shared memory in rank order (no global partials, no atomics), plus
// one cluster that adds the tiles' small partial sums in tile order.
//
// fp32 FFMA on purpose: parity with the reference is 1e-5 relative (north_star), which tf32 / bf16 tensor-core
// paths do not meet, and the whole dense part is 80 MFLOP (C2) to 1.5 GFLOP (C3) per step.
#include "pcg_common.cuh"

#include <cooperative_groups.h>
namespace cg = cooperative_groups;

#define TILE_KC 32                         // weight rows per chunk
#define TILE_NWC 8                         // consumer warps
#define TILE_NT (32 * (TILE_NWC + 1))      // + one producer warp
#define TILE_MAX_STAGE 32                  // deepest ring of weight chunks
#define TILE_MAX_E 256
#define TILE_SMEM_MAX (227 * 1024)

struct TileP {
    const float* feat; int64_t ldf; int F;
    const int32_t* targets; int B, R, E;
    const float* agg; int64_t lda;         // [R*B, lda], row of item w is agg[rep ? rep[w] : w]
    const int32_t* rep;
    const float* w_intra[PCG_MAX_REL];     // [2F, E] each
    const float* w_inter;                  // [F + R*E, E]
    const float* w_head;                   // [2, E]            (mode 2)
    const float* w_clf; const float* b_clf;  // [2, F], [2]     (NULL: no center scores)
    const int64_t* labels; float lambda;   // (mode 2)
    int mode;                              // 0 inference | 1 forward that keeps cat for pcg_dense_bwd | 2 train
    int nstage;                            // ring depth (<= TILE_MAX_STAGE)
    float* out;                            // [E, B]
    float* center;                         // [B, 2] or NULL
    float* cat; int64_t ldcat;             // mode 1: [B, F + R*E] (unpadded) ; mode 2: [B, Fp + R*E] (padded)
    float* dz;                             // [B, E]      (mode 2)
    float* dh;                             // [B, R*E]    (mode 2)
    float* partial;                        // [n_tiles, PS] per-tile sums of the small gradients and losses (mode 2)
    float* logits;                         // [B, 2] or NULL (mode 2)
};

// per-tile partial record: [loss_gnn, loss_label, d b_clf[2], d W_head[2][E], d W_clf[2][F]], padded to 4 floats
__host__ __device__ __forceinline__ int tile_ps(int F, int E) { return (4 + 2 * E + 2 * F + 3) & ~3; }

// ---- mbarrier / bulk copy / named barrier primitives (PTX; sm_90+) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// one contiguous global -> shared copy by the TMA unit, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(float* dst_smem, const float* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(TILE_NWC * 32) : "memory"); }
__device__ __forceinline__ void grid_dependency_wait() { pcg_grid_dependency_wait(); }

__host__ __device__ __forceinline__ int ld_pad(int x) { return x + ((4 - (x & 15)) & 15); }   // multiple of 4 -> = 4 (mod 16)

// Shared-memory plan (floats), the same arithmetic on host and device.
struct TileSmem {
    int Fp, K2p, LDC, LDA, LDO, LDB;
    size_t cat, agg, o, dzs, stage, scratch, wh, wc, rows, bars, total_bytes;
};
__host__ __device__ inline TileSmem tile_smem(int TM, int F, int R, int E, int mode, int nstage) {
    TileSmem s;
    s.Fp = (F + 3) & ~3;
    s.K2p = s.Fp + R * E;
    s.LDC = ld_pad(s.K2p); s.LDA = ld_pad(s.Fp); s.LDO = E + 4;
    s.LDB = E;                                   // chunk rows unpadded: one bulk copy per chunk
    size_t o = 0;
    s.cat = o; o += (size_t)TM * s.LDC;
    s.agg = o; o += (size_t)R * TM * s.LDA;
    s.o = o; o += (size_t)TM * s.LDO;
    s.dzs = o; o += mode == 2 ? (size_t)TM * s.LDO : 0;
    s.stage = o; o += (size_t)nstage * TILE_KC * s.LDB;
    // K-split partial sums, double buffered; not needed when every GEMM phase has at least as many tasks as warps
    const int tpg = (TM / 8) * (E / 64);
    s.scratch = o; o += tpg >= TILE_NWC ? 0 : 2 * (size_t)TILE_NWC * 16 * 32;
    s.wh = o; o += 2 * (size_t)E;
    s.wc = o; o += 2 * (size_t)s.Fp + 4;
    s.rows = o; o += (size_t)TM * 8;
    s.bars = o; o += 4 * TILE_MAX_STAGE;         // 2 * MAX_STAGE uint64
    s.total_bytes = o * 4;
    return s;
}
__host__ __device__ inline int tile_chunks(int F, int R, int E, int mode) {
    const int Fp = (F + 3) & ~3, K2p = Fp + R * E;
    return R * ((2 * Fp + TILE_KC - 1) / TILE_KC) + (K2p + TILE_KC - 1) / TILE_KC + (mode == 2 ? R * (E / TILE_KC) : 0);
}

// Source row of weight-chunk row k' (padded K index); -1: no source (the operand column it multiplies is
// exactly zero: the chunk row only has to be finite).
//   A (relation transform, W_r [2F,E]):   k' in [0,Fp) -> self row k' ; [Fp, 2Fp) -> row F + (k'-Fp)
//   B (combine, W [F+RE, E]):             k' in [0,Fp) -> row k'      ; >= Fp     -> row F + (k'-Fp)
__device__ __forceinline__ int wrow_A(int kp, int F, int Fp) {
    if (kp < Fp) return kp < F ? kp : -1;
    const int q = kp - Fp;
    return q < F ? F + q : -1;
}
__device__ __forceinline__ int wrow_B(int kp, int F, int Fp) {
    if (kp < Fp) return kp < F ? kp : -1;
    return F + (kp - Fp);
}

#ifdef PCG_TRACE
// Debug build only (make trace): phase timestamps of tile 0, 16 int64.
__device__ long long* g_tile_trace = nullptr;
__device__ __forceinline__ long long tile_now() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TTRACE(slot) do { if (g_tile_trace && threadIdx.x == 0 && blockIdx.x == 0) g_tile_trace[(slot)] = tile_now(); } while (0)
extern "C" __attribute__((visibility("default"))) int pcg_debug_set_tile_trace(long long* buf) {
    return (int)cudaMemcpyToSymbol(g_tile_trace, &buf, sizeof(buf));
}
#else
#define TTRACE(slot) do {} while (0)
#endif

template <int TM>
__global__ void __launch_bounds__(TILE_NT, 1) k_tile(TileP p) {
    extern __shared__ __align__(128) float sm[];
    const int NS = p.nstage;
    const TileSmem L = tile_smem(TM, p.F, p.R, p.E, p.mode, NS);
    const int F = p.F, Fp = L.Fp, E = p.E, R = p.R, K2p = L.K2p;
    const int LDC = L.LDC, LDA = L.LDA, LDO = L.LDO, LDB = L.LDB;
    float* catS = sm + L.cat;
    float* aggS = sm + L.agg;
    float* oS = sm + L.o;
    float* dzS = sm + L.dzs;
    float* stage = sm + L.stage;
    float* scratch = sm + L.scratch;
    float* whS = sm + L.wh;
    float* wcS = sm + L.wc;
    float* rowS = sm + L.rows;
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + L.bars);
    uint64_t* empty = full + TILE_MAX_STAGE;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.x * TM;
    const int mode = p.mode;
    const int nchA = (2 * Fp + TILE_KC - 1) / TILE_KC, nchB = (K2p + TILE_KC - 1) / TILE_KC, nchD = E / TILE_KC;

    TTRACE(0);
    pcg_launch_dependents();                 // the weight-gradient kernel's CTAs may queue up behind this tile
    if (tid == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], TILE_NWC); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (F != Fp) {
        // the chunk rows that face the zero padding of the operand rows are never copied: make them finite once
        for (int x = tid; x < NS * TILE_KC * LDB; x += TILE_NT) stage[x] = 0.f;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (wid == TILE_NWC) {
        // ------------------------------------------------------------------ producer warp: the weight stream
        // (weights are not written by the kernel in front of this one, so the stream starts before the
        // grid-dependency wait of the consumers).
        // A chunk is TILE_KC consecutive rows of the padded operand; its source rows are consecutive rows of the
        // weight matrix except across the F -> Fp padding, so a chunk is ONE bulk copy (two or three when F is not
        // a multiple of 4): lane j looks at chunk row j, the first lane of every run of consecutive source rows
        // issues the copy of the whole run. (One copy per row was measured first: 600 small TMA requests per tile
        // made the kernel 29 us; the TMA unit wants few, large requests.)
        int it = 0;
        auto fill = [&](int nrows, const float* W, auto row_of) {      // row_of(j) -> source row of chunk row j, or -1
            const int s = it % NS, round = it / NS;
            if (round > 0) mbar_wait(&empty[s], (uint32_t)((round - 1) & 1));
            const int row = lane < nrows ? row_of(lane) : -1;
            const int prev = __shfl_up_sync(PCG_FULL, row, 1);
            const bool head = row >= 0 && (lane == 0 || prev < 0 || prev + 1 != row);
            const unsigned valid = __ballot_sync(PCG_FULL, row >= 0);
            const unsigned heads = __ballot_sync(PCG_FULL, head);
            if (lane == 0) mbar_expect_tx(&full[s], (uint32_t)(__popc(valid) * E * 4));
            __syncwarp();
            if (head) {
                // run = from this lane up to (not including) the next head or the first row without a source
                const unsigned after = lane == 31 ? 0u : ~((2u << lane) - 1u);   // lanes above this one
                const unsigned stop = (heads | ~valid) & after;
                const int end = stop ? __ffs(stop) - 1 : 32;
                bulk_g2s(stage + ((size_t)s * TILE_KC + lane) * LDB, W + (size_t)row * E, (uint32_t)((end - lane) * E * 4),
                         &full[s]);
            }
            ++it;
        };
        for (int r = 0; r < R; ++r)
            for (int c = 0; c < nchA; ++c)
                fill(min(TILE_KC, 2 * Fp - c * TILE_KC), p.w_intra[r], [&](int j) { return wrow_A(c * TILE_KC + j, F, Fp); });
        for (int c = 0; c < nchB; ++c)
            fill(min(TILE_KC, K2p - c * TILE_KC), p.w_inter, [&](int j) { return wrow_B(c * TILE_KC + j, F, Fp); });
        if (mode == 2)
            for (int r = 0; r < R; ++r)
                for (int c = 0; c < nchD; ++c)          // rows of W[F + r*E + n], n = 32c .. 32c+31: the transposed operand of dH
                    fill(TILE_KC, p.w_inter, [&](int j) { return F + r * E + c * TILE_KC + j; });
#ifdef PCG_TRACE
        if (g_tile_trace && blockIdx.x == 0 && lane == 0) {     // when has the weight stream landed? (peek; ring all-resident)
            const int total = tile_chunks(F, R, E, mode);
            if (total <= NS) {
                mbar_wait(&full[(R * nchA - 1) % NS], 0); g_tile_trace[9] = tile_now();
                mbar_wait(&full[(R * nchA + nchB - 1) % NS], 0); g_tile_trace[10] = tile_now();
                mbar_wait(&full[(total - 1) % NS], 0); g_tile_trace[11] = tile_now();
            }
        }
#endif
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    // small weights (heads) into shared memory
    if (p.w_clf)
        for (int x = tid; x < 2 * Fp + 2; x += TILE_NWC * 32) {
            float v;
            if (x < 2 * Fp) { const int c = x / Fp, f = x - c * Fp; v = f < F ? __ldg(p.w_clf + c * F + f) : 0.f; }
            else v = __ldg(p.b_clf + (x - 2 * Fp));
            wcS[x] = v;
        }
    if (mode == 2)
        for (int x = tid; x < 2 * E; x += TILE_NWC * 32) whS[x] = __ldg(p.w_head + x);
    grid_dependency_wait();                 // the aggregate kernel's rows (and everything before it) are visible
    TTRACE(1);
    {
        const int V = Fp >> 2;
        for (int idx = tid; idx < (1 + R) * TM * V; idx += TILE_NWC * 32) {
            const int q = idx % V, rowi = idx / V, which = rowi / TM, m = rowi - which * TM;
            const int i = m0 + m;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < p.B) {
                if (which == 0) {
                    v = ld_f4(p.feat + (int64_t)__ldg(p.targets + i) * p.ldf + 4 * q);
                } else {
                    const int64_t w = (int64_t)(which - 1) * p.B + i;
                    v = ld_f4(p.agg + (p.rep ? (int64_t)__ldg(p.rep + w) : w) * p.lda + 4 * q);
                }
            }
            float* dst = which == 0 ? catS + m * LDC + 4 * q : aggS + ((size_t)(which - 1) * TM + m) * LDA + 4 * q;
            *reinterpret_cast<float4*>(dst) = v;
        }
    }
    consumer_sync();
    TTRACE(2);

    // ---- label_clf on the tile's own rows (layers.py:236-243): center[m][c] -> rowS[m][0..1]
    if (p.w_clf) {
        for (int m = wid; m < TM; m += TILE_NWC) {
            float a0 = 0.f, a1 = 0.f;
            for (int f = lane; f < Fp; f += 32) {
                const float x = catS[m * LDC + f];
                a0 = fmaf(x, wcS[f], a0);
                a1 = fmaf(x, wcS[Fp + f], a1);
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                a0 += __shfl_xor_sync(PCG_FULL, a0, off);
                a1 += __shfl_xor_sync(PCG_FULL, a1, off);
            }
            if (lane == 0) {
                a0 += wcS[2 * Fp]; a1 += wcS[2 * Fp + 1];
                rowS[m * 8 + 0] = a0; rowS[m * 8 + 1] = a1;
                if (p.center && m0 + m < p.B) *reinterpret_cast<float2*>(p.center + 2 * (int64_t)(m0 + m)) = make_float2(a0, a1);
            }
        }
    }

    // ---- K-chunked GEMMs. A task = (operand group, row block of 8, column block of 64): one warp, 16 accumulators
    // per lane. Phase A has R groups (the relations, each with its own weight chunks), phase B one. With fewer
    // tasks than warps the spare warps split K by WHOLE chunks (chunk c of a group belongs to split c % ksplit), so a
    // warp waits for few barriers and runs long independent FMA streams; the splits meet in shared memory in split
    // order. With more tasks than warps (<= 32) a warp runs up to four tasks of different groups one after the other.
    // Ring protocol: every consumer warp visits every chunk in stream order (wait full / arrive empty) unless the
    // ring holds the whole stream, in which case chunks a warp does not use are not touched at all.
    constexpr int RB = TM / 8;
    const int CB = E >> 6, tpg = RB * CB;              // tasks per group
    const bool resident = tile_chunks(F, R, E, mode) <= NS;
    const int lr = lane >> 3, lc = lane & 7;
    int it = 0, st = 0, phase = 0;
    uint32_t par = 0;
    auto advance = [&]() { ++it; if (++st == NS) { st = 0; par ^= 1u; } };
    auto release = [&]() { if (!resident) { __syncwarp(); if (lane == 0) mbar_arrive(&empty[st]); } };
    auto skip_to = [&](int target) {                    // pass over chunks this warp does not use
        if (resident) { st += target - it; it = target; return; }
        while (it < target) { mbar_wait(&full[st], par); release(); advance(); }
    };
    float acc[16];

    // one chunk: acc += A[rows row0, row0+1][k' in chunk] * chunk[k'][this lane's 8 columns]
    auto chunk_fma = [&](int kg0, int kv, const float* A0, int ld0, int split, const float* A1, int ld1, int row0, int col_lo) {
        const float* Bs = stage + (size_t)st * TILE_KC * LDB + col_lo;
#pragma unroll 2
        for (int kk = 0; kk < kv; kk += 4) {
            const int kg = kg0 + kk;
            const float* Ar = kg < split ? A0 + (size_t)row0 * ld0 + kg : A1 + (size_t)row0 * ld1 + (kg - split);
            const int lda_ = kg < split ? ld0 : ld1;
            const float4 a0 = *reinterpret_cast<const float4*>(Ar);
            const float4 a1 = *reinterpret_cast<const float4*>(Ar + lda_);
            const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 bl = *reinterpret_cast<const float4*>(Bs + (size_t)(kk + j) * LDB);
                const float4 bh = *reinterpret_cast<const float4*>(Bs + (size_t)(kk + j) * LDB + 32);
                acc[0] = fmaf(av0[j], bl.x, acc[0]); acc[1] = fmaf(av0[j], bl.y, acc[1]);
                acc[2] = fmaf(av0[j], bl.z, acc[2]); acc[3] = fmaf(av0[j], bl.w, acc[3]);
                acc[4] = fmaf(av0[j], bh.x, acc[4]); acc[5] = fmaf(av0[j], bh.y, acc[5]);
                acc[6] = fmaf(av0[j], bh.z, acc[6]); acc[7] = fmaf(av0[j], bh.w, acc[7]);
                acc[8] = fmaf(av1[j], bl.x, acc[8]); acc[9] = fmaf(av1[j], bl.y, acc[9]);
                acc[10] = fmaf(av1[j], bl.z, acc[10]); acc[11] = fmaf(av1[j], bl.w, acc[11]);
                acc[12] = fmaf(av1[j], bh.x, acc[12]); acc[13] = fmaf(av1[j], bh.y, acc[13]);
                acc[14] = fmaf(av1[j], bh.z, acc[14]); acc[15] = fmaf(av1[j], bh.w, acc[15]);
            }
        }
    };

    // One phase: groups x tpg tasks; group g multiplies A_g = [A0 (k' < split) | A1 + g*a1_stride] (TM x Kp) with its nch
    // chunks and writes relu(.) to dst + g*dst_stride (row stride ld).
    auto phase_k = [&](int groups, int Kp, int nch, const float* A0, int ld0, int split, const float* A1, int ld1,
                       size_t a1_stride, float* dst, int ld, int dst_stride) {
        const int ntask = groups * tpg;
        int ksplit = 1;
        while (ksplit * 2 * ntask <= TILE_NWC) ksplit *= 2;
        const int first = it;
        float* sc = scratch + (size_t)(phase & 1) * TILE_NWC * 16 * 32;
        int my_task = -1, my_ks = 0;
        for (int slot = 0; slot < 4; ++slot) {
            int t, ks;
            if (ntask <= TILE_NWC) { t = wid % ntask; ks = wid / ntask; if (slot >= 1 || ks >= ksplit) break; }
            else { t = wid + TILE_NWC * slot; ks = 0; if (t >= ntask) break; }
            const int g = t / tpg, rem = t - g * tpg, rb = rem / CB, cb = rem - rb * CB;
            const int row0 = rb * 8 + 2 * lr, col_lo = cb * 64 + lc * 4;
            skip_to(first + g * nch);
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[j] = 0.f;
            for (int c = 0; c < nch; ++c) {
                if (c % ksplit == ks) {
                    if (phase == 0) TTRACE(20);
                    mbar_wait(&full[st], par);
                    if (phase == 0) TTRACE(21);
                    chunk_fma(c * TILE_KC, min(TILE_KC, Kp - c * TILE_KC), A0, ld0, split, A1 + g * a1_stride, ld1, row0, col_lo);
                    if (phase == 0) TTRACE(22);
                    release();
                    advance();
                } else {
                    skip_to(it + 1);
                }
            }
            float* d0 = dst + (size_t)g * dst_stride + (size_t)row0 * ld + col_lo;
            if (ksplit == 1) {
                *reinterpret_cast<float4*>(d0) = make_float4(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f), fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f));
                *reinterpret_cast<float4*>(d0 + 32) = make_float4(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f), fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f));
                *reinterpret_cast<float4*>(d0 + ld) = make_float4(fmaxf(acc[8], 0.f), fmaxf(acc[9], 0.f), fmaxf(acc[10], 0.f), fmaxf(acc[11], 0.f));
                *reinterpret_cast<float4*>(d0 + ld + 32) = make_float4(fmaxf(acc[12], 0.f), fmaxf(acc[13], 0.f), fmaxf(acc[14], 0.f), fmaxf(acc[15], 0.f));
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) sc[((size_t)wid * 16 + j) * 32 + lane] = acc[j];
                my_task = t; my_ks = ks;
            }
        }
        skip_to(first + groups * nch);
        if (phase == 0) TTRACE(23);
        if (ksplit > 1) {
            // every warp of a task adds 16/ksplit of the lanes' slots over the splits, in split order (deterministic).
            // The scratch buffer alternates between phases, so one barrier here and one behind the phase are enough.
            consumer_sync();
            if (phase == 0) TTRACE(24);
            if (my_task >= 0) {
                const int g = my_task / tpg, rem = my_task - g * tpg, rb = rem / CB, cb = rem - rb * CB;
                float* d0 = dst + (size_t)g * dst_stride + (size_t)(rb * 8 + 2 * lr) * ld + cb * 64 + lc * 4;
                const int per = 16 / ksplit;
                // slot j of a lane: row (j >> 3), columns 32 * ((j >> 2) & 1) + (j & 3) of its 2 x 8 block: slots come
                // in groups of 4 consecutive columns (one float4 store) unless the task has 8 splits (2 slots each)
                auto slot_sum = [&](int j) {
                    float v[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) v[q] = q < ksplit ? sc[((size_t)(my_task + q * ntask) * 16 + j) * 32 + lane] : 0.f;
                    float a = v[0];
#pragma unroll
                    for (int q = 1; q < 8; ++q) if (q < ksplit) a += v[q];
                    return fmaxf(a, 0.f);
                };
                if (per >= 4) {
                    for (int j = my_ks * per; j < (my_ks + 1) * per; j += 4)
                        *reinterpret_cast<float4*>(d0 + (size_t)(j >> 3) * ld + 32 * ((j >> 2) & 1)) =
                            make_float4(slot_sum(j), slot_sum(j + 1), slot_sum(j + 2), slot_sum(j + 3));
                } else {
                    for (int j = my_ks * per; j < (my_ks + 1) * per; ++j)
                        d0[(size_t)(j >> 3) * ld + 32 * ((j >> 2) & 1) + (j & 3)] = slot_sum(j);
                }
            }
        }
        if (phase == 0) TTRACE(25);
        ++phase;
        consumer_sync();
    };

    // h_r = relu([self | agg_r] @ W_r) -> catS[:, Fp + r*E ...]   (layers.py:625-629), all relations side by side
    phase_k(R, 2 * Fp, nchA, catS, LDC, Fp, aggS, LDA, (size_t)TM * LDA, catS + Fp, LDC, E);
    TTRACE(3);
    // combined = relu(cat @ W) -> oS ; out[e][i] (layers.py:284-289, transposed)
    phase_k(1, K2p, nchB, catS, LDC, K2p, catS, LDC, 0, oS, LDO, 0);
    TTRACE(4);
    if ((p.B & 3) == 0 && TM % 4 == 0) {
        for (int idx = tid; idx < (TM / 4) * E; idx += TILE_NWC * 32) {       // 4 consecutive targets per store
            const int h = idx % (TM / 4), e = idx / (TM / 4), m = 4 * h;
            if (m0 + m < p.B)                                                   // B % 4 == 0: all four or none
                *reinterpret_cast<float4*>(p.out + (int64_t)e * p.B + m0 + m) =
                    make_float4(oS[m * LDO + e], oS[(m + 1) * LDO + e], oS[(m + 2) * LDO + e], oS[(m + 3) * LDO + e]);
        }
    } else {
        for (int idx = tid; idx < TM * E; idx += TILE_NWC * 32) {
            const int m = idx % TM, e = idx / TM;
            if (m0 + m < p.B) p.out[(int64_t)e * p.B + m0 + m] = oS[m * LDO + e];
        }
    }
    if (mode == 1) {          // cat rows for pcg_dense_bwd: unpadded columns [self F | h ...]
        const int ncol = F + R * E;
        for (int idx = tid; idx < TM * ncol; idx += TILE_NWC * 32) {
            const int m = idx / ncol, c = idx - m * ncol;
            if (m0 + m < p.B) p.cat[(int64_t)(m0 + m) * p.ldcat + c] = catS[m * LDC + (c < F ? c : c - F + Fp)];
        }
    }
    if (mode != 2) return;
    {                         // padded cat rows for k_wgrad, 16 bytes per store
        const int V = K2p >> 2;
        for (int idx = tid; idx < TM * V; idx += TILE_NWC * 32) {
            const int m = idx / V, q = idx - m * V;
            if (m0 + m < p.B)
                *reinterpret_cast<float4*>(p.cat + (int64_t)(m0 + m) * p.ldcat + 4 * q) = *reinterpret_cast<const float4*>(catS + m * LDC + 4 * q);
        }
    }
    TTRACE(5);

    // ---- heads + losses per target (model.py:38, :54-61), dLoss == 1: dl = (softmax - onehot) / B
    const float inv_b = 1.0f / (float)p.B;
    for (int m = wid; m < TM; m += TILE_NWC) {
        float g0 = 0.f, g1 = 0.f;
        for (int e = lane; e < E; e += 32) {
            const float x = oS[m * LDO + e];
            g0 = fmaf(whS[e], x, g0);
            g1 = fmaf(whS[E + e], x, g1);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            g0 += __shfl_xor_sync(PCG_FULL, g0, off);
            g1 += __shfl_xor_sync(PCG_FULL, g1, off);
        }
        const bool valid = m0 + m < p.B;
        float dl1 = 0.f, dc1 = 0.f, lg = 0.f, ll = 0.f;
        if (valid) {
            const int y = __ldg(p.labels + m0 + m) == 1 ? 1 : 0;
            {
                const float mx = fmaxf(g0, g1);
                const float e0 = expf(g0 - mx), e1 = expf(g1 - mx);
                lg = mx + logf(e0 + e1) - (y ? g1 : g0);
                dl1 = (e1 / (e0 + e1) - (float)y) * inv_b;
            }
            {
                const float c0 = rowS[m * 8 + 0], c1 = rowS[m * 8 + 1];
                const float mx = fmaxf(c0, c1);
                const float e0 = expf(c0 - mx), e1 = expf(c1 - mx);
                ll = mx + logf(e0 + e1) - (y ? c1 : c0);
                dc1 = p.lambda * (e1 / (e0 + e1) - (float)y) * inv_b;
            }
            if (lane == 0 && p.logits) *reinterpret_cast<float2*>(p.logits + 2 * (int64_t)(m0 + m)) = make_float2(g0, g1);
        }
        __syncwarp();
        if (lane == 0) {
            rowS[m * 8 + 2] = -dl1; rowS[m * 8 + 3] = dl1;      // d logits
            rowS[m * 8 + 4] = -dc1; rowS[m * 8 + 5] = dc1;      // d center
            rowS[m * 8 + 6] = lg; rowS[m * 8 + 7] = ll;
        }
        // dZ = (W_head^T dl) * (combined > 0)
        for (int e = lane; e < E; e += 32)
            dzS[m * LDO + e] = oS[m * LDO + e] > 0.f ? fmaf(whS[e], -dl1, whS[E + e] * dl1) : 0.f;
    }
    consumer_sync();
    TTRACE(6);
    {
        const int V = E >> 2;
        for (int idx = tid; idx < TM * V; idx += TILE_NWC * 32) {
            const int m = idx / V, q = idx - m * V;
            if (m0 + m < p.B)
                *reinterpret_cast<float4*>(p.dz + (int64_t)(m0 + m) * E + 4 * q) = *reinterpret_cast<const float4*>(dzS + m * LDO + 4 * q);
        }
    }
    // per-tile partial sums of the small gradients (k_wgrad's last cluster adds the tiles in tile order)
    {
        const int PS = tile_ps(F, E);
        float* mine = p.partial + (size_t)blockIdx.x * PS;
        for (int x = tid; x < 4 + 2 * E + 2 * F; x += TILE_NWC * 32) {
            float a = 0.f;
            if (x < 2) {                                             // loss sums (gnn, label)
#pragma unroll
                for (int m = 0; m < TM; ++m) a += rowS[m * 8 + 6 + x];
            } else if (x < 4) {                                      // d b_clf
#pragma unroll
                for (int m = 0; m < TM; ++m) a += rowS[m * 8 + 4 + (x - 2)];
            } else if (x < 4 + 2 * E) {                              // d W_head[c][e] = sum_m dl[m][c] * combined[m][e]
                const int c = (x - 4) / E, e = (x - 4) - c * E;
#pragma unroll
                for (int m = 0; m < TM; ++m) a = fmaf(rowS[m * 8 + 2 + c], oS[m * LDO + e], a);
            } else {                                                 // d W_clf[c][f] = sum_m dc[m][c] * self[m][f]
                const int c = (x - 4 - 2 * E) / F, f = (x - 4 - 2 * E) - c * F;
#pragma unroll
                for (int m = 0; m < TM; ++m) a = fmaf(rowS[m * 8 + 4 + c], catS[m * LDC + f], a);
            }
            mine[x] = a;
        }
    }

    // ---- dH_r = (dZ @ W[F + r*E ..]^T) * (h_r > 0): a weight chunk holds 32 output columns n with all K = E; the
    // chunks are dealt to the warps (chunk d belongs to warp d % 8): 8 columns x RB rows per lane, K walked from a
    // per-row-group offset so that the four chunk rows a warp reads per instruction fall into different banks
    {
        const int jj = lane >> 3, mrow = lane & 7;
        const int nD = R * nchD, firstD = it;
        for (int d = 0; d < nD; ++d) {
            if ((d & (TILE_NWC - 1)) != wid) { skip_to(it + 1); continue; }
            mbar_wait(&full[st], par);
            const float* Bt = stage + (size_t)st * TILE_KC * LDB;
            float a2[RB][8];
#pragma unroll
            for (int i = 0; i < RB; ++i)
#pragma unroll
                for (int u = 0; u < 8; ++u) a2[i][u] = 0.f;
            for (int k0 = 0; k0 < E; k0 += 4) {
                const int kr = k0 + 4 * jj;
                const int kx = kr >= E ? kr - E : kr;
                float4 a[RB];
#pragma unroll
                for (int i = 0; i < RB; ++i) a[i] = *reinterpret_cast<const float4*>(dzS + (size_t)(mrow + 8 * i) * LDO + kx);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float4 b = *reinterpret_cast<const float4*>(Bt + (size_t)(jj + 4 * u) * LDB + kx);
#pragma unroll
                    for (int i = 0; i < RB; ++i) {
                        a2[i][u] = fmaf(a[i].x, b.x, a2[i][u]); a2[i][u] = fmaf(a[i].y, b.y, a2[i][u]);
                        a2[i][u] = fmaf(a[i].z, b.z, a2[i][u]); a2[i][u] = fmaf(a[i].w, b.w, a2[i][u]);
                    }
                }
            }
            release();
            advance();
            const int r = d / nchD, c = d - r * nchD;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int n = r * E + c * TILE_KC + jj + 4 * u;
#pragma unroll
                for (int i = 0; i < RB; ++i) {
                    const int m = mrow + 8 * i;
                    float* hc = catS + m * LDC + Fp + n;       // h[m][n] is read (relu mask) and replaced by dH[m][n] by this lane only
                    *hc = *hc > 0.f ? a2[i][u] : 0.f;
                }
            }
        }
        skip_to(firstD + nD);
    }
    consumer_sync();
    TTRACE(7);
    {
        const int V = (R * E) >> 2;
        for (int idx = tid; idx < TM * V; idx += TILE_NWC * 32) {
            const int m = idx / V, q = idx - m * V;
            if (m0 + m < p.B)
                *reinterpret_cast<float4*>(p.dh + (int64_t)(m0 + m) * (R * E) + 4 * q) = *reinterpret_cast<const float4*>(catS + m * LDC + Fp + 4 * q);
        }
    }
    TTRACE(8);
}

// ------------------------------------------------------------------------------------------------
// Weight gradients of the two GEMM levels, split over the batch across a thread-block cluster:
//   job 0      dW'  [K2p, E] = cat^T  @ dZ          (cat padded: [B, K2p])
//   job 1 + r  dW_r'[2Fp, E] = [self | agg_r]^T @ dH_r
//   job R + 1  the tiles' small partial sums (d W_head, d W_clf, d b_clf, losses) added in tile order
// The grid is a flat list of clusters of S CTAs: first one cluster for job R + 1, then one per W x W output block of
// jobs 0..R (built from each job's real row count, so no CTA is launched only to return). CTA `rank` of a cluster
// multiplies batch slice `rank` (one fmaf chain per output element over the slice's rows in ascending order, from 0),
// leaves its partial block in its own shared memory, and after one cluster barrier every CTA adds W/S rows of the
// block over the S CTAs through distributed shared memory in rank order (deterministic) and stores the rows of the
// unpadded gradient. No global partials, no atomics, no tickets. The block width W only decides which CTA computes an
// element, never how: every W gives the same bits. The operand slice comes in 16-byte cp.async chunks of WG_KC rows:
// all at once behind one wait when the slice fits the CTA's buffers, else through a two-stage ring.
// (Round 1: k_gemm_v to global split partials + a separate k_dense_reduce launch.)
struct WgP {
    const float* cat; int64_t ldcat;        // [B, K2p]
    const float* agg; int64_t lda; const int32_t* rep;
    const float* dz; const float* dh;       // [B, E], [B, R*E]
    int B, F, Fp, R, E, S;                  // S = cluster size = batch slices
    float* grad[PCG_MAX_REL + 1];           // job 0: [F + R*E, E]; job 1+r: [2F, E]
    const float* partial; int n_tiles, PS;  // k_tile's per-tile records
    float lambda;
    float* loss; float* d_w_head; float* d_w_clf; float* d_b_clf;
};

__device__ __forceinline__ void cp_async16_(float* smem_dst, const float* gsrc, int bytes) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}

#define WG_KC 32                            // batch rows per operand chunk
#define WG_BUF_BYTES (48 * 1024)            // operand buffers of one CTA

template <int W> struct WgShape {
    static constexpr int T = W / 16;                          // a thread's T x T accumulators (16 x 16 threads)
    static constexpr int LD = W + 4;
    static constexpr int CHUNK = 2 * WG_KC * LD;              // floats: A rows | B rows
    static constexpr int NBUF = WG_BUF_BYTES / (CHUNK * 4);   // chunks held at once
    static_assert(NBUF >= 2 && W * LD <= NBUF * CHUNK, "wgrad buffers");
};

template <int T> __device__ __forceinline__ void ld_vec(float (&v)[T], const float* s) {
    if constexpr (T == 4) { const float4 x = *reinterpret_cast<const float4*>(s); v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; }
    else { static_assert(T == 2, "T"); const float2 x = *reinterpret_cast<const float2*>(s); v[0] = x.x; v[1] = x.y; }
}

template <int W>   // 3 CTAs per SM: room for 80 registers, which k_wgrad<64> needs to run without spills
__global__ void __launch_bounds__(256, 3) k_wgrad(WgP p) {
    using SH = WgShape<W>;
    constexpr int T = SH::T, LD = SH::LD, NBUF = SH::NBUF;
    __shared__ __align__(16) float smw[NBUF * SH::CHUNK];   // chunk c: A [KC][LD] | B [KC][LD]; later the C block [W][LD]
    float* Cs = smw;
    cg::cluster_group cl = cg::this_cluster();
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int S = p.S;
    const int cluster = blockIdx.x / S, split = blockIdx.x - cluster * S;   // split == rank in the cluster (dims S,1,1)
    const int E = p.E, RE = p.R * p.E;
    if (cluster == 0) {
        // ---- job R + 1, small gradients: sum over the tiles in tile order. CTA `split` owns a slice of the record's
        // columns; thread (g, c): column c, tiles [g*n/8, (g+1)*n/8) of n in order; the 8 group sums are added in group order.
        grid_dependency_wait();
        float* red = smw;                                              // [8][32] group sums, then the column totals
        const int n_real = 4 + 2 * E + 2 * p.F;
        const int g = tid >> 5, c = tid & 31;
        const int per_t = (p.n_tiles + 7) / 8, t0 = min(p.n_tiles, g * per_t), t1 = min(p.n_tiles, t0 + per_t);
        for (int base = split * 32; base < n_real; base += S * 32) {
            const int x = base + c;
            float a = 0.f;
            if (x < n_real)
                for (int q0 = t0; q0 < t1; q0 += 16) {
                    float v[16];
#pragma unroll
                    for (int u = 0; u < 16; ++u) v[u] = q0 + u < t1 ? __ldcg(p.partial + (size_t)(q0 + u) * p.PS + x) : 0.f;
#pragma unroll
                    for (int u = 0; u < 16; ++u) a += v[u];
                }
            red[g * 32 + c] = a;
            __syncthreads();
            if (g == 0 && x < n_real) {
                float s = 0.f;
#pragma unroll
                for (int q = 0; q < 8; ++q) s += red[q * 32 + c];
                red[256 + c] = s;
                if (x >= 4 + 2 * E) p.d_w_clf[x - 4 - 2 * E] = s;
                else if (x >= 4) p.d_w_head[x - 4] = s;
                else if (x >= 2) p.d_b_clf[x - 2] = s;
            }
            __syncthreads();
            if (base == 0 && tid == 0)      // model.py:54-61: both cross-entropies are batch means
                p.loss[0] = red[256] / (float)p.B + p.lambda * (red[257] / (float)p.B);
            __syncthreads();
        }
        return;
    }
    // ---- which output block: job 0 has ceil(K2p / W) row blocks, jobs 1..R ceil(2Fp / W) each, all ceil(E / W) columns
    const int K2p = p.Fp + p.R * p.E;
    const int ncb = (E + W - 1) / W, nb0 = (K2p + W - 1) / W * ncb, nb1 = (2 * p.Fp + W - 1) / W * ncb;
    int blk = cluster - 1, job = 0;
    if (blk >= nb0) { blk -= nb0; job = 1 + blk / nb1; blk -= (job - 1) * nb1; }
    const int rows = job == 0 ? K2p : 2 * p.Fp;
    const int m0 = blk / ncb * W, n0 = (blk % ncb) * W;
    pcg_launch_dependents();                // the exchange + Adam kernel may queue up
    grid_dependency_wait();
    const int per = (p.B + S - 1) / S;
    const int kb = min(p.B, split * per), ke = min(p.B, kb + per);
    const int nt = (ke - kb + WG_KC - 1) / WG_KC;
    // chunk t (rows kb + t*KC ..) -> buffer `buf`; rows past the slice are zero-filled (they add fmaf(0, 0, acc) == acc)
    auto issue = [&](int t, int buf) {
        float* As = smw + buf * SH::CHUNK;
        float* Bs = As + WG_KC * LD;
        const int k0 = kb + t * WG_KC;
#pragma unroll
        for (int j = 0; j < WG_KC * W / 4 / 256; ++j) {
            const int c = tid + 256 * j;
            const int kk = c / (W / 4), q4 = (c % (W / 4)) * 4;
            const int i = k0 + kk;
            const bool krow = i < ke;
            const int m = m0 + q4, n = n0 + q4;
            const int ba = krow ? min(16, max(0, (rows - m) * 4)) : 0;
            const int bb = krow ? min(16, max(0, (E - n) * 4)) : 0;
            const float* a = p.cat;
            if (ba > 0) {
                if (job == 0 || m < p.Fp) a = p.cat + (int64_t)i * p.ldcat + m;
                else {
                    const int64_t w = (int64_t)(job - 1) * p.B + i;
                    a = p.agg + (p.rep ? (int64_t)__ldg(p.rep + w) : w) * p.lda + (m - p.Fp);
                }
            }
            const float* b = p.dz;
            if (bb > 0) b = job == 0 ? p.dz + (int64_t)i * E + n : p.dh + (int64_t)i * RE + (job - 1) * E + n;
            cp_async16_(As + kk * LD + q4, a, ba);
            cp_async16_(Bs + kk * LD + q4, b, bb);
        }
    };
    float acc[T][T];
#pragma unroll
    for (int a = 0; a < T; ++a)
#pragma unroll
        for (int b = 0; b < T; ++b) acc[a][b] = 0.f;
    auto chunk_fma = [&](int buf) {
        const float* As = smw + buf * SH::CHUNK;
        const float* Bs = As + WG_KC * LD;
#pragma unroll
        for (int kk = 0; kk < WG_KC; ++kk) {
            float av[T], bv[T];
            ld_vec<T>(av, As + kk * LD + ty * T);
            ld_vec<T>(bv, Bs + kk * LD + tx * T);
#pragma unroll
            for (int a = 0; a < T; ++a)
#pragma unroll
                for (int b = 0; b < T; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
        }
    };
    if (NBUF > 2 && nt <= NBUF) {
        // the whole slice fits: every copy in flight at once, one wait (with two buffers the ring below does the same)
        for (int t = 0; t < nt; ++t) issue(t, t);
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        for (int t = 0; t < nt; ++t) chunk_fma(t);
        __syncthreads();
    } else {
        issue(0, 0);
        asm volatile("cp.async.commit_group;" ::: "memory");
        for (int t = 0; t < nt; ++t) {
            if (t + 1 < nt) issue(t + 1, (t + 1) & 1);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncthreads();
            chunk_fma(t & 1);
            __syncthreads();
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    // this CTA's partial block -> its shared memory (the operand buffers are free behind the last barrier)
#pragma unroll
    for (int a = 0; a < T; ++a) {
        float* c = Cs + (ty * T + a) * LD + tx * T;
        if constexpr (T == 4) *reinterpret_cast<float4*>(c) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
        else *reinterpret_cast<float2*>(c) = make_float2(acc[a][0], acc[a][1]);
    }
    cl.sync();
    // map a padded row to the row of the real gradient (or -1 for a pad row)
    auto real_row = [&](int m) -> int {
        if (m < p.Fp) return m < p.F ? m : -1;
        if (job == 0) return p.F + (m - p.Fp);
        const int q = m - p.Fp;
        return q < p.F ? p.F + q : -1;
    };
    float* grad = p.grad[job];
    const int rpc = W / S;                   // rows of the block this CTA adds up (S in {1, 2, 4, 8})
    for (int idx = tid; idx < rpc * (W / 4); idx += 256) {
        const int lr = idx / (W / 4), q4 = (idx % (W / 4)) * 4;
        const int ml = split * rpc + lr, m = m0 + ml, n = n0 + q4;
        const int rr = m < rows ? real_row(m) : -1;
        if (rr < 0 || n >= E) continue;
        float4 v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
            v[q] = q < S ? *reinterpret_cast<const float4*>(cl.map_shared_rank(Cs, q) + ml * LD + q4) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 sacc = v[0];
#pragma unroll
        for (int q = 1; q < 8; ++q) if (q < S) f4_add(sacc, v[q]);
        float* g = grad + (int64_t)rr * E + n;
        if (((uintptr_t)g & 15) == 0) *reinterpret_cast<float4*>(g) = sacc;
        else { g[0] = sacc.x; g[1] = sacc.y; g[2] = sacc.z; g[3] = sacc.w; }
    }
    cl.sync();                               // nobody leaves while a peer may still read its block
}

// ------------------------------------------------------------------------------------------- C ABI
// rows per tile and ring depth: small batches get 8-row tiles so that the tiles cover the GPU, larger ones 16 / 32
// rows (weights amortised over more targets) as long as (row blocks x column blocks) fits the 8 consumer warps;
// the ring takes what is left of shared memory (all chunks of the tile when they fit).
static int tile_plan(int B, int F, int R, int E, int mode, int* nstage_out, size_t* smem_out) {
    const int sms = pcg_device_sms();
    const int chunks = tile_chunks(F, R, E, mode);
    const int cands[3] = {32, 16, 8};
    for (int c = 0; c < 3; ++c) {
        const int tm = cands[c];
        if (tm > 8 && (B + tm - 1) / tm < sms - sms / 5) continue;          // would leave too many SMs idle
        if ((tm / 8) * (E / 64) > TILE_NWC || R * (tm / 8) * (E / 64) > 4 * TILE_NWC) continue;
        int ns = chunks < TILE_MAX_STAGE ? chunks : TILE_MAX_STAGE;
        while (ns >= 3 && tile_smem(tm, F, R, E, mode, ns).total_bytes > TILE_SMEM_MAX) --ns;
        const TileSmem s = tile_smem(tm, F, R, E, mode, ns);
        if (s.total_bytes > TILE_SMEM_MAX) continue;
        *nstage_out = ns;
        *smem_out = s.total_bytes;
        return tm;
    }
    return 0;
}

// k_wgrad's launch: S batch slices (= cluster size) of >= 64 targets, and the output block width W. 64 x 64 blocks
// when their clusters already cover the SMs (C3: 40 blocks x 8 slices); otherwise 32 x 32 blocks (C2: 7 -> 26 blocks
// x 8 slices), which cut each CTA's fmaf chains to a quarter and let a C2-sized slice load behind a single wait.
// Smaller blocks read more shared memory per FMA, so they are used only where they buy parallelism.
struct WgradPlan { int S, W, clusters; };
static WgradPlan wgrad_plan(int B, int F, int R, int E) {
    WgradPlan w;
    w.S = 8;
    while (w.S > 1 && (B + w.S - 1) / w.S < 64) w.S >>= 1;
    const int Fp = (F + 3) & ~3, K2p = Fp + R * E;
    auto blocks = [&](int W) { return ((K2p + W - 1) / W + R * ((2 * Fp + W - 1) / W)) * ((E + W - 1) / W); };
    w.W = blocks(64) * w.S >= pcg_device_sms() ? 64 : 32;
    w.clusters = 1 + blocks(w.W);            // + the small-gradient cluster
    return w;
}

extern "C" int pcg_tile_supported(int B, int R, int F, int E) {
    if (B <= 0 || R < 1 || R > PCG_MAX_REL || F < 1 || E < 64 || E > TILE_MAX_E || E % 64 != 0) return 0;
    size_t smem;
    int ns;
    return tile_plan(B, F, R, E, 2, &ns, &smem) > 0 ? 1 : 0;
}

// floats of scratch for one train step: cat [B,K2p] | dz [B,E] | dh [B,RE] | tile partial records
struct TileScratch { size_t cat, dz, dh, partial, total; };
static TileScratch tile_scratch(int B, int R, int F, int E) {
    TileScratch t;
    const int Fp = (F + 3) & ~3, K2p = Fp + R * E;
    size_t o = 0;
    auto al = [](size_t x) { return (x + 3) & ~(size_t)3; };
    t.cat = o; o = al(o + (size_t)B * K2p);
    t.dz = o; o = al(o + (size_t)B * E);
    t.dh = o; o = al(o + (size_t)B * R * E);
    t.partial = o; o = al(o + (size_t)((B + 7) / 8) * tile_ps(F, E));
    t.total = o + 64;
    return t;
}

extern "C" size_t pcg_tile_scratch_floats(int B, int R, int F, int E) { return tile_scratch(B, R, F, E).total; }

template <int TM>
static cudaError_t launch_tile(const TileP& p, size_t smem, cudaStream_t stream, int pdl) {
    static size_t configured_dev[PCG_MAX_DEVICES];
    size_t& configured = configured_dev[pcg_current_device()];
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(k_tile<TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((p.B + TM - 1) / TM));
    cfg.blockDim = dim3(TILE_NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k_tile<TM>, p);
}

static cudaError_t launch_tile_any(int tm, const TileP& p, size_t smem, cudaStream_t stream, int pdl) {
    return tm == 32 ? launch_tile<32>(p, smem, stream, pdl) : tm == 16 ? launch_tile<16>(p, smem, stream, pdl)
                                                                      : launch_tile<8>(p, smem, stream, pdl);
}

extern "C" int pcg_tile_fwd(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, int R, int E,
                            const float* agg, int64_t lda, const int32_t* agg_rep, const float* const* w_intra_host,
                            const float* w_inter, const float* w_clf, const float* b_clf, int keep_cat, float* out,
                            float* center, float* cat, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B == 0) return 0;
    PCG_REQUIRE(feat && targets && agg && w_intra_host && w_inter && out, "pcg_tile_fwd: null pointer");
    PCG_REQUIRE(pcg_tile_supported(B, R, F, E), "pcg_tile_fwd: unsupported sizes R=%d F=%d E=%d", R, F, E);
    PCG_REQUIRE(!keep_cat || cat, "pcg_tile_fwd: keep_cat without a cat buffer");
    PCG_REQUIRE(ldf % 4 == 0 && lda % 4 == 0 && ldf >= ((F + 3) & ~3) && lda >= ((F + 3) & ~3) &&
                    ((uintptr_t)feat & 15) == 0 && ((uintptr_t)agg & 15) == 0 && ((uintptr_t)w_inter & 15) == 0 &&
                    ((uintptr_t)out & 15) == 0,
                "pcg_tile_fwd: feat / agg / weights / out must be 16-byte aligned with padded rows");
    TileP p = {};
    p.feat = feat; p.ldf = ldf; p.F = F; p.targets = targets; p.B = B; p.R = R; p.E = E;
    p.agg = agg; p.lda = lda; p.rep = agg_rep;
    for (int r = 0; r < R; ++r) {
        PCG_REQUIRE(((uintptr_t)w_intra_host[r] & 15) == 0, "pcg_tile_fwd: W_r must be 16-byte aligned");
        p.w_intra[r] = w_intra_host[r];
    }
    p.w_inter = w_inter; p.w_clf = w_clf; p.b_clf = b_clf;
    p.mode = keep_cat ? 1 : 0;
    p.out = out; p.center = center; p.cat = cat; p.ldcat = F + R * E;
    size_t smem;
    const int tm = tile_plan(B, F, R, E, p.mode, &p.nstage, &smem);
    cudaError_t e = launch_tile_any(tm, p, smem, stream, 0);
    if (e != cudaSuccess) { pcg_set_error("pcg_tile_fwd: launch: %s", cudaGetErrorString(e)); return (int)e; }
    return pcg_check_launch("pcg_tile_fwd");
}

extern "C" int pcg_tile_train(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, int R, int E,
                              const float* agg, int64_t lda, const int32_t* agg_rep, const float* const* w_intra_host,
                              const float* w_inter, const float* w_clf, const float* b_clf, const float* w_head,
                              const int64_t* labels, float lambda, float* out, float* center, float* logits,
                              float* loss, float* const* d_w_intra_host, float* d_w_inter, float* d_w_clf,
                              float* d_b_clf, float* d_w_head, float* scratch, int pdl, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(B > 0, "pcg_tile_train: empty batch");
    PCG_REQUIRE(feat && targets && agg && w_intra_host && w_inter && w_clf && b_clf && w_head && labels && out && loss &&
                    d_w_intra_host && d_w_inter && d_w_clf && d_b_clf && d_w_head && scratch,
                "pcg_tile_train: null pointer");
    PCG_REQUIRE(pcg_tile_supported(B, R, F, E), "pcg_tile_train: unsupported sizes R=%d F=%d E=%d", R, F, E);
    PCG_REQUIRE(ldf % 4 == 0 && lda % 4 == 0 && ldf >= ((F + 3) & ~3) && lda >= ((F + 3) & ~3) &&
                    ((uintptr_t)feat & 15) == 0 && ((uintptr_t)agg & 15) == 0 && ((uintptr_t)w_inter & 15) == 0 &&
                    ((uintptr_t)scratch & 15) == 0 && ((uintptr_t)out & 15) == 0,
                "pcg_tile_train: feat / agg / weights / out / scratch must be 16-byte aligned with padded rows");
    const TileScratch ts = tile_scratch(B, R, F, E);
    const int Fp = (F + 3) & ~3, K2p = Fp + R * E;
    TileP p = {};
    p.feat = feat; p.ldf = ldf; p.F = F; p.targets = targets; p.B = B; p.R = R; p.E = E;
    p.agg = agg; p.lda = lda; p.rep = agg_rep;
    for (int r = 0; r < R; ++r) {
        PCG_REQUIRE(((uintptr_t)w_intra_host[r] & 15) == 0, "pcg_tile_train: W_r must be 16-byte aligned");
        p.w_intra[r] = w_intra_host[r];
    }
    p.w_inter = w_inter; p.w_head = w_head; p.w_clf = w_clf; p.b_clf = b_clf; p.labels = labels; p.lambda = lambda;
    p.mode = 2;
    p.out = out; p.center = center; p.logits = logits;
    p.cat = scratch + ts.cat; p.ldcat = K2p; p.dz = scratch + ts.dz; p.dh = scratch + ts.dh;
    p.partial = scratch + ts.partial;
    size_t smem;
    const int tm = tile_plan(B, F, R, E, 2, &p.nstage, &smem);
    const int mask = pcg_pdl_enabled() | (pdl ? 6 : 0);
    cudaError_t e = launch_tile_any(tm, p, smem, stream, (mask & 2) != 0);
    if (e != cudaSuccess) { pcg_set_error("pcg_tile_train: launch: %s", cudaGetErrorString(e)); return (int)e; }

    WgP w = {};
    w.cat = p.cat; w.ldcat = K2p; w.agg = agg; w.lda = lda; w.rep = agg_rep; w.dz = p.dz; w.dh = p.dh;
    w.B = B; w.F = F; w.Fp = Fp; w.R = R; w.E = E;
    const WgradPlan wp = wgrad_plan(B, F, R, E);
    w.S = wp.S;
    w.grad[0] = d_w_inter;
    for (int j = 1; j <= R; ++j) w.grad[j] = d_w_intra_host[j - 1];
    w.partial = p.partial; w.n_tiles = (B + tm - 1) / tm; w.PS = tile_ps(F, E);
    w.lambda = lambda; w.loss = loss; w.d_w_head = d_w_head; w.d_w_clf = d_w_clf; w.d_b_clf = d_b_clf;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(wp.clusters * wp.S));
    cfg.blockDim = dim3(256);
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)wp.S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (mask & 4) ? 2 : 1;
    e = wp.W == 64 ? cudaLaunchKernelEx(&cfg, k_wgrad<64>, w) : cudaLaunchKernelEx(&cfg, k_wgrad<32>, w);
    if (e != cudaSuccess) { pcg_set_error("pcg_tile_train: wgrad launch: %s", cudaGetErrorString(e)); return (int)e; }
    return pcg_check_launch("pcg_tile_train");
}
