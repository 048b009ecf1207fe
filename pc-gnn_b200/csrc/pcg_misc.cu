// Error plumbing, the label-score table and the label-balanced pick step.
#include <stdarg.h>

#include <cub/device/device_radix_sort.cuh>

#include "pcg_common.cuh"

static thread_local char g_err[512] = "";

void pcg_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int pcg_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        pcg_set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}

extern "C" const char* pcg_last_error(void) { return g_err; }

static int g_pdl = 0;
int pcg_pdl_enabled() { return g_pdl; }
extern "C" int pcg_set_pdl(int enabled) {
    const int old = g_pdl;
    g_pdl = enabled;
    return old;
}
extern "C" int pcg_version(void) { return 102; }

// ------------------------------------------------------------------------------- score table
// score[v] = <feat[v, :], w> + b. Eight lanes per row, float4 loads, fixed reduction tree (so the
// table is bit-reproducible run to run). The weight vector is zero-padded to ldf in shared memory.
// Reference: label_clf = nn.Linear(F, 2) (src/layers.py:200) applied at :236-237; only output
// column 0 feeds the choose step.
__global__ void __launch_bounds__(256) k_score_table(const float* __restrict__ feat, int64_t n, int F, int64_t ldf,
                                                     const float* __restrict__ w, const float* __restrict__ b, float* __restrict__ score) {
    extern __shared__ float sw[];
    pcg_launch_dependents();                 // the pool sort behind this kernel may start its prologue
    for (int c = threadIdx.x; c < ldf; c += blockDim.x) sw[c] = c < F ? w[c] : 0.f;
    const float bias = b ? b[0] : 0.f;
    __syncthreads();
    const int l = threadIdx.x & 7;
    const int V = (int)(ldf >> 2);
    const int64_t rows_per_block = blockDim.x >> 3;
    // vb is warp-uniform (4 rows per warp), so every lane runs the same trip count for the shuffles
    for (int64_t vb = (int64_t)blockIdx.x * rows_per_block + ((threadIdx.x >> 5) << 2); vb < n;
         vb += (int64_t)gridDim.x * rows_per_block) {
        const int64_t v = vb + ((threadIdx.x & 31) >> 3);
        float acc = 0.f;
        if (v < n) {
            const float* rowp = feat + v * ldf;
            for (int c = l; c < V; c += 8) {
                float4 x = ld_f4(rowp + 4 * c);
                const float4 ww = *reinterpret_cast<const float4*>(sw + 4 * c);
                acc = fmaf(x.x, ww.x, acc); acc = fmaf(x.y, ww.y, acc);
                acc = fmaf(x.z, ww.z, acc); acc = fmaf(x.w, ww.w, acc);
            }
        }
        acc += __shfl_xor_sync(PCG_FULL, acc, 4);
        acc += __shfl_xor_sync(PCG_FULL, acc, 2);
        acc += __shfl_xor_sync(PCG_FULL, acc, 1);
        if (l == 0 && v < n) score[v] = acc + bias;
    }
}

// Scores of the pool members only, with EXACTLY the arithmetic of k_score_table (same lanes, same order, same
// reduction tree: the values are bit-identical to score[pool[i]]). It lets the pool sort run NEXT TO the score-table
// kernel instead of behind it (and, on a row-partitioned graph, next to the score exchange: features are replicated),
// and it is the common predecessor from which the step's three front branches fork.
// Staging rider: the CTAs behind the first `score_blocks` copy `stage_words` 32-bit words from stage_src to stage_dst
// (the batch's ids / labels out of mapped pinned host memory, see pcg_stage): the step's first kernel fetches the
// batch while it computes, so a host batch needs no copy node in front of the recorded step.
__device__ __forceinline__ uint32_t ld_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void stage_copy(const uint32_t* src, uint32_t* dst, int64_t n, int64_t first, int64_t stride) {
    // four independent loads in flight per thread (a PCIe round trip each when src is host memory)
    for (int64_t i = first; i < n; i += 4 * stride) {
        uint32_t v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = i + u * stride < n ? ld_sys(src + i + u * stride) : 0u;
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (i + u * stride < n) st_sys(dst + i + u * stride, v[u]);
    }
}

// cursor != NULL: entry (*cursor % count) of a plan: src / dst advance by that many strides (32-bit words); bump: the
// cursor is incremented behind the copy (one CTA only: the indexed form copies a few words).
__global__ void __launch_bounds__(256) k_stage(const uint32_t* src, uint32_t* dst, int64_t n, uint32_t* cursor,
                                               uint32_t count, int64_t src_stride, int64_t dst_stride, int bump) {
    // no fence behind the stores: the consumer (a later kernel, or the host after an event / stream wait) is ordered
    // behind the END of this kernel, which makes them visible (a system-scope fence here cost 5 us: ncu, membar 100 %)
    uint32_t at = 0;
    if (cursor) {
        at = *(volatile uint32_t*)cursor;
        src += (int64_t)(at % count) * src_stride;
        dst += (int64_t)(at % count) * dst_stride;
    }
    stage_copy(src, dst, n, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);
    if (cursor && bump) {
        __syncthreads();                     // single CTA (enforced by the launcher): every thread has read the cursor
        if (threadIdx.x == 0) *(volatile uint32_t*)cursor = at + 1u;
    }
}

__global__ void __launch_bounds__(256) k_pool_scores(const float* __restrict__ feat, int F, int64_t ldf,
                                                     const float* __restrict__ w, const float* __restrict__ b,
                                                     const int32_t* __restrict__ pool, int P, float* __restrict__ pool_score,
                                                     int score_blocks, const uint32_t* stage_src, uint32_t* stage_dst,
                                                     int64_t stage_words, const uint32_t* cursor, uint32_t count,
                                                     int64_t src_stride) {
    if ((int)blockIdx.x >= score_blocks) {
        const int64_t nb = gridDim.x - score_blocks;
        if (cursor) stage_src += (int64_t)(*(volatile const uint32_t*)cursor % count) * src_stride;   // plan entry
        stage_copy(stage_src, stage_dst, stage_words, (int64_t)(blockIdx.x - score_blocks) * blockDim.x + threadIdx.x,
                   nb * blockDim.x);
        return;
    }
    extern __shared__ float sw[];
    for (int c = threadIdx.x; c < ldf; c += blockDim.x) sw[c] = c < F ? w[c] : 0.f;
    const float bias = b ? b[0] : 0.f;
    __syncthreads();
    const int l = threadIdx.x & 7;
    const int V = (int)(ldf >> 2);
    const int rows_per_block = blockDim.x >> 3;
    for (int ib = blockIdx.x * rows_per_block + ((threadIdx.x >> 5) << 2); ib < P; ib += score_blocks * rows_per_block) {
        const int i = ib + ((threadIdx.x & 31) >> 3);
        float acc = 0.f;
        if (i < P) {
            const float* rowp = feat + (int64_t)__ldg(pool + i) * ldf;
            for (int c = l; c < V; c += 8) {
                float4 x = ld_f4(rowp + 4 * c);
                const float4 ww = *reinterpret_cast<const float4*>(sw + 4 * c);
                acc = fmaf(x.x, ww.x, acc); acc = fmaf(x.y, ww.y, acc);
                acc = fmaf(x.z, ww.z, acc); acc = fmaf(x.w, ww.w, acc);
            }
        }
        acc += __shfl_xor_sync(PCG_FULL, acc, 4);
        acc += __shfl_xor_sync(PCG_FULL, acc, 2);
        acc += __shfl_xor_sync(PCG_FULL, acc, 1);
        if (l == 0 && i < P) pool_score[i] = acc + bias;
    }
}

__global__ void k_gather_pool(const float* __restrict__ score, const int32_t* __restrict__ pool, int P,
                              float* __restrict__ pool_score) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < P) pool_score[p] = score[pool[p]];
}

// ------------------------------------------------------------------------------- pool sort
// The train-positive pool sorted by score (ties by pool position), once per step; the choose kernels
// then find every target's o nearest positives by binary search instead of scanning the pool
// (reference: one torch.sort over all P pool distances per positive target, src/layers.py:685-690).
__device__ __forceinline__ uint32_t orderable(float f) {   // float order -> unsigned order
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ uint32_t unorderable(uint32_t k) {   // inverse of orderable (bit pattern of the float)
    return (k & 0x80000000u) ? (k ^ 0x80000000u) : ~k;
}
// P <= 8192: rank sort. Every CTA stages all P keys (orderable(score) << 32 | position, unique) in
// shared memory and ranks 32 of them by counting smaller keys, 16 lanes per element; the rank is the
// element's place in the sorted order. O(P^2) compares spread over P/32 CTAs: a few microseconds and
// no serial merge chain (a single-CTA bitonic sort of the same pool took ~48 us on B200).
// `gather` != 0: pool_score is the whole score table and entry i's score is pool_score[pool[i]].
#define RANK_NT 512
#define RANK_PER 32      // elements ranked per CTA: 16 threads each
__global__ void __launch_bounds__(RANK_NT) k_sort_pool_rank(const float* __restrict__ pool_score, int gather,
                                                            const int32_t* __restrict__ pool, int P,
                                                            float* __restrict__ ps_score, int32_t* __restrict__ ps_pos,
                                                            int32_t* __restrict__ ps_id) {
    extern __shared__ unsigned long long keys[];
    pcg_grid_dependency_wait();              // the score table in front of this kernel is complete
    // stage all keys: ids first, then the dependent score gathers, 8 of each in flight per thread
    for (int base = 0; base < P; base += RANK_NT * 8) {
        int32_t id[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = base + u * RANK_NT + threadIdx.x;
            id[u] = (i < P && gather) ? __ldg(pool + i) : i;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = base + u * RANK_NT + threadIdx.x;
            if (i < P) keys[i] = ((unsigned long long)orderable(__ldg(pool_score + id[u])) << 32) | (unsigned)i;
        }
    }
    __syncthreads();
    const int e = threadIdx.x >> 4, part = threadIdx.x & 15;
    const int i = blockIdx.x * RANK_PER + e;
    const unsigned long long mine = i < P ? keys[i] : ~0ull;
    int cnt = 0;
#pragma unroll 4
    for (int j = part; j < P; j += 16) cnt += keys[j] < mine;
    cnt += __shfl_xor_sync(PCG_FULL, cnt, 1);
    cnt += __shfl_xor_sync(PCG_FULL, cnt, 2);
    cnt += __shfl_xor_sync(PCG_FULL, cnt, 4);
    cnt += __shfl_xor_sync(PCG_FULL, cnt, 8);
    if (part == 0 && i < P) {
        ps_score[cnt] = __uint_as_float(unorderable((uint32_t)(mine >> 32)));
        ps_pos[cnt] = i;
        ps_id[cnt] = pool[i];
    }
}

__global__ void k_sort_prepare(const float* __restrict__ pool_score, int P, uint32_t* __restrict__ keys,
                               int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P) { keys[i] = orderable(pool_score[i]); vals[i] = i; }
}

__global__ void k_sort_finish(const float* __restrict__ pool_score, const int32_t* __restrict__ pool,
                              const int32_t* __restrict__ order, int P, float* __restrict__ ps_score,
                              int32_t* __restrict__ ps_pos, int32_t* __restrict__ ps_id) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P) { const int pos = order[i]; ps_score[i] = pool_score[pos]; ps_pos[i] = pos; ps_id[i] = pool[pos]; }
}

#define PCG_SORT_SMALL_MAX 8192

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static size_t cub_sort_temp_bytes(int P) {
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, P);
    return temp;
}

extern "C" size_t pcg_sort_pool_workspace_bytes(int P) {
    // [gathered pool scores][keys in/out][vals in/out][cub temp]; the last three only for big pools
    size_t o = align256((size_t)(P > 0 ? P : 1) * 4);
    if (P > PCG_SORT_SMALL_MAX) o += 4 * align256((size_t)P * 4) + align256(cub_sort_temp_bytes(P));
    return o;
}

static int sort_pool_impl(const float* pool_score, int gather, const int32_t* pool, int P, float* ps_score, int32_t* ps_pos,
                          int32_t* ps_id, char* ws, size_t ws_bytes, cudaStream_t stream) {
    if (P <= 0) return 0;
    if (P <= PCG_SORT_SMALL_MAX) {
        const size_t smem = (size_t)P * 8;
        static bool configured_dev[PCG_MAX_DEVICES];
        bool& configured = configured_dev[pcg_current_device()];
        if (!configured) {
            cudaError_t e = cudaFuncSetAttribute(k_sort_pool_rank, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 PCG_SORT_SMALL_MAX * 8);
            if (e != cudaSuccess) { pcg_set_error("pcg_sort_pool: smem attr: %s", cudaGetErrorString(e)); return (int)e; }
            configured = true;
        }
        cudaError_t le = pcg_launch(k_sort_pool_rank, dim3((P + RANK_PER - 1) / RANK_PER), dim3(RANK_NT), smem, stream,
                                    gather && (pcg_pdl_enabled() & 1), pool_score, gather, pool, P, ps_score, ps_pos, ps_id);
        if (le != cudaSuccess) { pcg_set_error("pcg_sort_pool: launch: %s", cudaGetErrorString(le)); return (int)le; }
        return 0;
    }
    const size_t a = align256((size_t)P * 4);
    size_t temp = cub_sort_temp_bytes(P);
    PCG_REQUIRE(ws && ws_bytes >= 4 * a + align256(temp), "pcg_sort_pool: workspace too small");
    uint32_t* k_in = (uint32_t*)ws;
    uint32_t* k_out = (uint32_t*)(ws + a);
    int32_t* v_in = (int32_t*)(ws + 2 * a);
    int32_t* v_out = (int32_t*)(ws + 3 * a);
    void* d_temp = ws + 4 * a;
    k_sort_prepare<<<(P + 255) / 256, 256, 0, stream>>>(pool_score, P, k_in, v_in);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(d_temp, temp, k_in, k_out, v_in, v_out, P, 0, 32, stream);
    if (e != cudaSuccess) { pcg_set_error("pcg_sort_pool: cub: %s", cudaGetErrorString(e)); return (int)e; }
    k_sort_finish<<<(P + 255) / 256, 256, 0, stream>>>(pool_score, pool, v_out, P, ps_score, ps_pos, ps_id);
    return 0;
}

extern "C" int pcg_sort_pool(const float* pool_score, const int32_t* pool, int P, float* ps_score, int32_t* ps_pos,
                             int32_t* ps_id, void* workspace, size_t workspace_bytes, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (P <= 0) return 0;
    PCG_REQUIRE(pool_score && pool && ps_score && ps_pos && ps_id, "pcg_sort_pool: null pointer");
    size_t skip = align256((size_t)P * 4);   // the gathered-score slot of the shared layout is unused here
    char* ws = workspace ? (char*)workspace + skip : nullptr;
    int rc = sort_pool_impl(pool_score, 0, pool, P, ps_score, ps_pos, ps_id, ws,
                            workspace_bytes > skip ? workspace_bytes - skip : 0, stream);
    if (rc) return rc;
    return pcg_check_launch("pcg_sort_pool");
}

static int pool_scores_impl(const char* who, const float* feat, int F, int64_t ldf, const float* w, const float* b,
                            const int32_t* pool, int P, float* pool_score, const void* stage_src, void* stage_dst,
                            size_t stage_bytes, const uint32_t* cursor, uint32_t count, int64_t src_stride_bytes,
                            cudaStream_t stream) {
    PCG_REQUIRE(stage_bytes == 0 || (stage_src && stage_dst), "%s: staging pointers missing", who);
    PCG_REQUIRE(stage_bytes % 4 == 0 && ((uintptr_t)stage_src & 3) == 0 && ((uintptr_t)stage_dst & 3) == 0,
                "%s: the staged copy works on aligned 32-bit words", who);
    PCG_REQUIRE(!cursor || (count > 0 && src_stride_bytes % 4 == 0), "%s: a plan cursor needs count > 0 and a stride of whole words", who);
    if (P <= 0) {
        if (stage_bytes) {
            const int64_t n = (int64_t)(stage_bytes / 4);
            k_stage<<<(int)((n + 1023) / 1024 < 64 ? (n + 1023) / 1024 : 64), 256, 0, stream>>>(
                (const uint32_t*)stage_src, (uint32_t*)stage_dst, n, const_cast<uint32_t*>(cursor), count, src_stride_bytes / 4, 0, 0);
            return pcg_check_launch(who);
        }
        return 0;
    }
    PCG_REQUIRE(feat && w && pool && pool_score, "%s: null pointer", who);
    PCG_REQUIRE(ldf % 4 == 0 && F <= ldf && F > 0 && ldf * 4 <= 48 * 1024 && ((uintptr_t)feat & 15) == 0,
                "%s: need F <= ldf, ldf %% 4 == 0, 16-byte aligned rows (F=%d ldf=%lld)", who, F, (long long)ldf);
    int blocks = (P + 31) / 32;
    const int sms = pcg_device_sms();
    if (blocks > sms * 16) blocks = sms * 16;
    const int64_t words = (int64_t)(stage_bytes / 4);
    int64_t rider = (words + 1023) / 1024;            // four words per thread
    if (rider > 64) rider = 64;
    k_pool_scores<<<blocks + (int)rider, 256, (size_t)ldf * 4, stream>>>(feat, F, ldf, w, b, pool, P, pool_score, blocks,
                                                                         (const uint32_t*)stage_src, (uint32_t*)stage_dst,
                                                                         words, cursor, count, src_stride_bytes / 4);
    return pcg_check_launch(who);
}

extern "C" int pcg_pool_scores(const float* feat, int F, int64_t ldf, const float* w, const float* b, const int32_t* pool,
                               int P, float* pool_score, pcg_stream_t stream_) {
    return pool_scores_impl("pcg_pool_scores", feat, F, ldf, w, b, pool, P, pool_score, nullptr, nullptr, 0, nullptr, 0, 0,
                            (cudaStream_t)stream_);
}

extern "C" int pcg_pool_scores_stage(const float* feat, int F, int64_t ldf, const float* w, const float* b,
                                     const int32_t* pool, int P, float* pool_score, const void* stage_src, void* stage_dst,
                                     size_t stage_bytes, const uint32_t* cursor, uint32_t count, int64_t src_stride_bytes,
                                     pcg_stream_t stream_) {
    return pool_scores_impl("pcg_pool_scores_stage", feat, F, ldf, w, b, pool, P, pool_score, stage_src, stage_dst,
                            stage_bytes, cursor, count, src_stride_bytes, (cudaStream_t)stream_);
}

extern "C" void* pcg_host_device_ptr(void* host_ptr) {
    void* dev = nullptr;
    cudaError_t e = cudaHostGetDevicePointer(&dev, host_ptr, 0);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        pcg_set_error("pcg_host_device_ptr: %s (not page-locked / not mapped)", cudaGetErrorString(e));
        return nullptr;
    }
    return dev;
}

extern "C" int pcg_stage(const void* src, void* dst, size_t bytes, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (bytes == 0) return 0;
    PCG_REQUIRE(src && dst, "pcg_stage: null pointer");
    PCG_REQUIRE(bytes % 4 == 0 && ((uintptr_t)src & 3) == 0 && ((uintptr_t)dst & 3) == 0,
                "pcg_stage: the copy works on aligned 32-bit words");
    const int64_t n = (int64_t)(bytes / 4);
    int64_t blocks = (n + 1023) / 1024;
    if (blocks > 64) blocks = 64;
    k_stage<<<(int)blocks, 256, 0, stream>>>((const uint32_t*)src, (uint32_t*)dst, n, nullptr, 0, 0, 0, 0);
    return pcg_check_launch("pcg_stage");
}

extern "C" int pcg_stage_indexed(const void* src, void* dst, size_t bytes, uint32_t* cursor, uint32_t count,
                                 int64_t src_stride_bytes, int64_t dst_stride_bytes, int bump, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (bytes == 0) return 0;
    PCG_REQUIRE(src && dst && cursor && count > 0, "pcg_stage_indexed: null pointer or empty plan");
    PCG_REQUIRE(bytes % 4 == 0 && ((uintptr_t)src & 3) == 0 && ((uintptr_t)dst & 3) == 0 && src_stride_bytes % 4 == 0 &&
                    dst_stride_bytes % 4 == 0,
                "pcg_stage_indexed: the copy works on aligned 32-bit words");
    const int64_t n = (int64_t)(bytes / 4);
    int64_t blocks = (n + 1023) / 1024;
    if (blocks > 64) blocks = 64;
    PCG_REQUIRE(!bump || blocks == 1, "pcg_stage_indexed: a copy that advances the cursor is at most 4 KB (one CTA)");
    k_stage<<<(int)blocks, 256, 0, stream>>>((const uint32_t*)src, (uint32_t*)dst, n, cursor, count, src_stride_bytes / 4,
                                             dst_stride_bytes / 4, bump);
    return pcg_check_launch("pcg_stage_indexed");
}

extern "C" int pcg_score_table(const float* feat, int64_t n_nodes, int F, int64_t ldf, const float* w, const float* b,
                               float* score, const int32_t* pool, int P, float* ps_score, int32_t* ps_pos,
                               int32_t* ps_id, void* workspace, size_t workspace_bytes, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(feat && w && score, "pcg_score_table: null pointer");
    PCG_REQUIRE(ldf % 4 == 0 && F <= ldf && F > 0, "pcg_score_table: need F <= ldf, ldf %% 4 == 0 (F=%d ldf=%lld)", F,
                (long long)ldf);
    PCG_REQUIRE(ldf * 4 <= 48 * 1024, "pcg_score_table: rows wider than 12288 floats unsupported");
    PCG_REQUIRE(((uintptr_t)feat & 15) == 0, "pcg_score_table: feat must be 16-byte aligned");
    if (n_nodes > 0) {
        int64_t blocks = (n_nodes + 31) / 32;
        const int sms = pcg_device_sms();
        if (blocks > (int64_t)sms * 16) blocks = (int64_t)sms * 16;
        k_score_table<<<(int)blocks, 256, (size_t)ldf * 4, stream>>>(feat, n_nodes, F, ldf, w, b, score);
    }
    if (P > 0 && pool) {
        PCG_REQUIRE(ps_score && ps_pos && ps_id, "pcg_score_table: sorted pool outputs missing");
        const size_t skip = align256((size_t)P * 4);
        PCG_REQUIRE(workspace && workspace_bytes >= skip, "pcg_score_table: workspace too small");
        int rc;
        if (P <= PCG_SORT_SMALL_MAX) {      // the rank sort reads score[pool[i]] itself
            rc = sort_pool_impl(score, 1, pool, P, ps_score, ps_pos, ps_id, nullptr, 0, stream);
        } else {
            float* gathered = (float*)workspace;
            k_gather_pool<<<(P + 255) / 256, 256, 0, stream>>>(score, pool, P, gathered);
            rc = sort_pool_impl(gathered, 0, pool, P, ps_score, ps_pos, ps_id, (char*)workspace + skip,
                                workspace_bytes - skip, stream);
        }
        if (rc) return rc;
    }
    return pcg_check_launch("pcg_score_table");
}

// ------------------------------------------------------------------------------- pick step
// index = bisect_right(cum, x, 0, n-1): first position in [0, n-1) with x < cum[pos], else n-1
// (CPython random.choices: bisect(cum_weights, random() * total, 0, hi) with hi = n - 1).
__device__ __forceinline__ int64_t bisect_right_hi(const double* __restrict__ cum, int64_t n, double x) {
    int64_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (x < cum[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__global__ void k_pick_replay(const double* __restrict__ cum, int64_t n, const double* __restrict__ u, int64_t k,
                              const int32_t* __restrict__ idx_train, int32_t* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= k) return;
    const double total = cum[n - 1] + 0.0;
    const int64_t pos = bisect_right_hi(cum, n, __dmul_rn(u[t], total));
    out[t] = idx_train ? idx_train[pos] : (int32_t)pos;
}

// Philox4x32-10 (Salmon et al., SC'11): counter = (offset + t, 0), key = seed.
__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0,
                                             uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__global__ void k_pick_philox(const double* __restrict__ cum, int64_t n, uint64_t seed, uint64_t offset, int64_t k,
                              const int32_t* __restrict__ idx_train, int32_t* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= k) return;
    const uint64_t ctr = offset + (uint64_t)t;
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0, c3 = 0;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    // 53-bit double in [0,1), built the way CPython's random() builds it from two 32-bit words
    const double u = ((double)(c0 >> 5) * 67108864.0 + (double)(c1 >> 6)) * (1.0 / 9007199254740992.0);
    const double total = cum[n - 1] + 0.0;
    const int64_t pos = bisect_right_hi(cum, n, __dmul_rn(u, total));
    out[t] = idx_train ? idx_train[pos] : (int32_t)pos;
}

extern "C" int pcg_pick_step(const double* cum, int64_t n, const double* u, int64_t k, const int32_t* idx_train,
                             int32_t* out, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(cum && u && out && n > 0, "pcg_pick_step: null pointer or empty population");
    if (k > 0) k_pick_replay<<<(int)((k + 255) / 256), 256, 0, stream>>>(cum, n, u, k, idx_train, out);
    return pcg_check_launch("pcg_pick_step");
}

extern "C" int pcg_pick_step_philox(const double* cum, int64_t n, uint64_t seed, uint64_t offset, int64_t k,
                                    const int32_t* idx_train, int32_t* out, pcg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PCG_REQUIRE(cum && out && n > 0, "pcg_pick_step_philox: null pointer or empty population");
    if (k > 0) k_pick_philox<<<(int)((k + 255) / 256), 256, 0, stream>>>(cum, n, seed, offset, k, idx_train, out);
    return pcg_check_launch("pcg_pick_step_philox");
}
