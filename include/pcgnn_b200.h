/*
 * pcgnn_b200 — C ABI of the B200-native pick-and-choose message-passing path.
 *
 * One shared library (libpcgnn_b200.so, built from pc-gnn_b200/csrc/ for sm_100a). Every entry
 * point takes plain device pointers and sizes, is asynchronous on the given stream, never
 * allocates or frees, and returns 0 on success or a non-zero cudaError_t-compatible code
 * (pcg_last_error() then holds the message; thread-local). The caller owns every buffer.
 *
 * Host-side state (all of it): per DEVICE ordinal, the forked side streams / events of pcg_choose (created on first
 * use) and the probe results cached per kernel (shared-memory opt-in, 16-CTA clusters, SM count); process-wide, the
 * pcg_set_pdl switch. Calls launch on the CURRENT device (cudaSetDevice is the caller's) and are not thread-safe per
 * device: one host thread at a time drives a device, which is how the reference runs (single-threaded,
 * src/model_handler.py:142-156) and how every multi-GPU run of this package is laid out (one process per GPU;
 * pc-gnn_b200/engine.py refuses an engine for a device other than the current one).
 *
 * The reference (h22hyeon/PC-GNN) is pure Python; each function below names the reference
 * lines whose work it replaces (paths relative to /root/reference/).
 *
 * Conventions
 *   work item   w = r * B + i        (relation r of target i; relation-major)
 *   graph       stacked CSR: row r*N+v of `indptr` (int64 [R*N+1]) / `indices` (int32, ids
 *               ascending inside a row) is the neighbour list of node v under relation r
 *   feat        fp32 [N, ldf], ldf % 4 == 0, 16-byte aligned, columns >= F are zero
 *   slot        PCG_SLOT consecutive selected ids of ONE item; items own whole slots
 */
#ifndef PCGNN_B200_H
#define PCGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCG_SLOT 64          /* selected ids per aggregation slot */
#define PCG_MAX_REL 8        /* relations per graph (reference ships 1, 3 and 5) */
#define PCG_NORM_MEAN 0      /* sum / n        (src/layers.py:612-614, src/graphsage.py:86-88) */
#define PCG_NORM_RSQRT 1     /* sum / sqrt(n)  (src/graphsage.py:224-226) */

/* status words written by the kernels (int32 device array of PCG_STATUS_WORDS) */
#define PCG_STATUS_WORDS 12
#define PCG_ST_SLOTS 0       /* slots handed out (aggregation consumes [0, this)) */
#define PCG_ST_OVERFLOW 3    /* != 0: `cap_slots` was too small, results are incomplete */

typedef void* pcg_stream_t;  /* a cudaStream_t */

#define PCG_API __attribute__((visibility("default")))

PCG_API const char* pcg_last_error(void);
PCG_API int pcg_version(void);
/* SM count of the current device (grid sizing), or a negative error. */
PCG_API int pcg_device_sms(void);
/* Programmatic dependent launch for the step's linear kernel chain (score table -> pool sort, aggregate -> fused
 * dense kernel -> weight gradients -> exchange + Adam): each kernel's prologue overlaps the tail of the kernel in
 * front; results are only touched behind griddepcontrol.wait. `mask` selects the dependent launches: 1 pool sort,
 * 2 fused dense kernel, 4 weight gradients, 8 exchange + Adam. Process-wide; returns the previous setting. */
PCG_API int pcg_set_pdl(int mask);

/*
 * Label-aware score table, column 0 only: score[v] = dot(feat[v, :F], w) + b[0] for all N nodes (w, b
 * device pointers), then the train-positive pool sorted by that score (see pcg_sort_pool).
 * Replaces src/layers.py:231-237 (label_clf over the batch's unique nodes and over train_pos);
 * only column 0 is ever compared (src/layers.py:649-650, 685, 714-715).
 *   workspace  pcg_sort_pool_workspace_bytes(P) bytes
 */
PCG_API int pcg_score_table(const float* feat, int64_t n_nodes, int F, int64_t ldf, const float* w, const float* b,
                    float* score, const int32_t* pool, int P, float* ps_score, int32_t* ps_pos, int32_t* ps_id,
                    void* workspace, size_t workspace_bytes, pcg_stream_t stream);

/*
 * Scores of the pool members only: pool_score[i] = dot(feat[pool[i], :F], w) + b[0], bit-identical to what
 * pcg_score_table writes for those nodes (same arithmetic). With it the pool sort (pcg_sort_pool) does not have to
 * wait for the score table: the two run side by side (src/layers.py:232, :237: pos_scores = label_clf(features(train_pos))).
 */
PCG_API int pcg_pool_scores(const float* feat, int F, int64_t ldf, const float* w, const float* b, const int32_t* pool,
                    int P, float* pool_score, pcg_stream_t stream);

/*
 * Host batches without copy nodes. The reference hands every batch over as host data (model_handler.py:142-150:
 * Python lists of ids, a LongTensor of labels made on the spot). pcg_stage copies `bytes` (a multiple of 4, 4-byte
 * aligned pointers) with a KERNEL, so that src or dst may be page-locked host memory (cudaHostAlloc / torch pinned
 * memory: device-addressable under unified addressing) and a captured step graph stays a graph of kernel nodes only
 * (graphs with memcpy nodes were measured to launch their branches several microseconds apart). Used for the loss
 * word on its way out. pcg_pool_scores_stage is pcg_pool_scores with the same copy riding on extra CTAs of the kernel:
 * the first kernel of the training step fetches the batch's ids and labels while it computes, which takes the host
 * to device copy off the step's critical path altogether. The source must stay unchanged until the kernel has
 * finished (the caller's event / synchronisation), like the source of any asynchronous copy.
 *
 * Epoch plans (the batch loop of src/model_handler.py:128-150 with the whole epoch's batches uploaded once): with a
 * device-resident `cursor` word the copy takes entry (*cursor % count) of a plan: pcg_pool_scores_stage reads its
 * source at stage_src + entry * src_stride_bytes (cursor NULL: plain); pcg_stage_indexed offsets source and destination
 * by entry * stride each and, with bump != 0 (copies of at most 4 KB), increments the cursor behind the copy. A recorded
 * step that fetches its batch through the cursor and ends with a bumping copy of its loss word into a per-step array
 * replays a whole epoch without the host touching a batch.
 */
PCG_API int pcg_stage(const void* src, void* dst, size_t bytes, pcg_stream_t stream);
/* Device address of a page-locked host buffer (cudaHostGetDevicePointer), or NULL + pcg_last_error(). */
PCG_API void* pcg_host_device_ptr(void* host_ptr);
PCG_API int pcg_pool_scores_stage(const float* feat, int F, int64_t ldf, const float* w, const float* b, const int32_t* pool,
                          int P, float* pool_score, const void* stage_src, void* stage_dst, size_t stage_bytes,
                          const uint32_t* cursor, uint32_t count, int64_t src_stride_bytes, pcg_stream_t stream);
PCG_API int pcg_stage_indexed(const void* src, void* dst, size_t bytes, uint32_t* cursor, uint32_t count,
                      int64_t src_stride_bytes, int64_t dst_stride_bytes, int bump, pcg_stream_t stream);

/*
 * Pool sorted by score: ps_score ascending with ties in pool-position order, ps_pos[i] = position in
 * `pool` of sorted entry i, ps_id[i] = pool[ps_pos[i]]. One sort per step replaces the reference's
 * torch.sort over all P pool distances for EVERY positive target (src/layers.py:683-690): with the pool
 * sorted, a target's nearest positives are a window around lower_bound(score[target]).
 */
PCG_API size_t pcg_sort_pool_workspace_bytes(int P);
PCG_API int pcg_sort_pool(const float* pool_score, const int32_t* pool, int P, float* ps_score, int32_t* ps_pos,
                  int32_t* ps_id, void* workspace, size_t workspace_bytes, pcg_stream_t stream);

/* pool_pos_of[v] = position of node v in `pool`, -1 for every other node (once per pool; pool ids distinct). */
PCG_API int pcg_pool_positions(const int32_t* pool, int P, int64_t n_nodes, int32_t* pool_pos_of, pcg_stream_t stream);
/* entry_pool_pos[e] = pool_pos_of[indices[e]] for every CSR entry (once per pool; same size as `indices`). */
PCG_API int pcg_entry_pool_positions(const int32_t* indices, int64_t nnz, const int32_t* pool_pos_of,
                             int32_t* entry_pool_pos, pcg_stream_t stream);

/* Bytes of scratch pcg_choose needs for B targets x R relations on a graph of n_nodes nodes whose largest
 * row has max_degree entries. The first n_nodes*4 bytes hold a per-node table that carries state between
 * calls (all bytes 0x7f between calls; pcg_choose restores it): call pcg_choose_workspace_init once after
 * allocating the buffer, and again if the same buffer is later used with another n_nodes. */
/* pcg_choose_sticky_offset(n_nodes): byte offset in the workspace of an int32 that every pcg_choose call ORs its
 * status[PCG_ST_OVERFLOW] into (the status block itself is rewritten by every call); the host reads and clears it. */
PCG_API size_t pcg_choose_workspace_bytes(int B, int R, int64_t max_degree, int64_t n_nodes);
PCG_API size_t pcg_choose_sticky_offset(int64_t n_nodes);
PCG_API int pcg_choose_workspace_init(void* workspace, size_t workspace_bytes, int64_t n_nodes, pcg_stream_t stream);

/*
 * Choose step for a batch: per item keep the ceil(d*thresh[r]) neighbours nearest in label score
 * (ties by position == id) when d > that + 1, else all; for positive targets in train mode add the
 * int(ceil(d*thresh)*rho) nearest train positives (ties by pool position) that are not already kept.
 * Replaces src/layers.py:216-227 (neighbour lookup), :246-262 (per-relation prep),
 * :633-697 choose_step_neighs, :700-738 choose_step_test and the set-union of :594/:694.
 *
 *   indptr/indices  stacked CSR of R relations over n_nodes ROWS each (row r*n_nodes + (v - row_lo)); a row
 *                partition of a larger graph passes its first global node id as row_lo (else 0); neighbour
 *                ids, targets, the score table and the pool always use GLOBAL node ids. A target outside
 *                [row_lo, row_lo + n_nodes) yields an empty item and status[PCG_ST_OVERFLOW] = 2.
 *   score        [N] table, or NULL with entry_score/center_score given (explicit scores, the
 *                IntraAgg.forward calling convention of src/layers.py:562)
 *   entry_score  per CSR entry (same indexing as `indices`) or NULL
 *   center_score [B] or NULL (then score[targets[i]])
 *   labels       int64 [B] (== 1 means positive) or NULL; ignored unless train != 0
 *   thresh_host  HOST array of R doubles (src/layers.py:193 hard-codes 0.5)
 *   k_override   int32 [R*B] explicit num_sample per item (src/layers.py:260-262) or NULL
 *   ps_score/ps_pos/ps_id  the score-sorted pool from pcg_score_table / pcg_sort_pool (P entries)
 *   entry_pool_pos  int32 [nnz] from pcg_entry_pool_positions (pool position of every CSR entry's node, -1 if
 *                it is not in the pool), or NULL: "already kept" is then tested by binary search in the row
 *                instead of a per-item bitmap over pool positions
 * Outputs
 *   sel_idx      int32 [cap_slots * PCG_SLOT]; item w's ids are sel_idx[it_base[w] .. + it_m[w])
 *   sel_dist     optional fp32 [cap_slots * PCG_SLOT] (NULL to skip): the distances the reference returns as
 *                samp_scores (src/layers.py:666-672, 691): at it_base[w] + [0,k) the kept neighbours' |Δ|
 *                (aligned with sel_idx), at it_base[w] + k + [0,o) the o nearest pool members' |Δ| (duplicates of kept ids
 *                included, as in the reference's list; unordered)
 *   slot_item    int32 [cap_slots]  owning item of each handed-out slot, or -1
 *   it_slot0/it_m int32 [R*B], it_base int64 [R*B], it_done int32 [R*B] (zeroed; aggregation tickets)
 *   it_rep       int32 [R*B]: targets that repeat an earlier id of the batch (pick_step samples with
 *                replacement) are not processed again; it_rep[w] is the item whose list w shares (w itself
 *                for first occurrences). Only representatives (it_rep[w] == w) carry it_slot0/it_m/it_base;
 *                pcg_aggregate copies the aggregated row of a repeated target from its representative.
 *   status       int32 [PCG_STATUS_WORDS] (every word written here)
 * The slots of the items are handed out by a prefix sum in item order, so the layout of sel_idx is the same
 * on every run.
 *   phases       3: the whole step. 1: only the preparation (folding of repeated targets, item sizes, slot prefix
 *                sum, tier queues), which reads targets / labels / indptr but NO scores, so a caller can run it on a
 *                second stream next to pcg_score_table; 2: only the selection, after a phases == 1 call with the
 *                same arguments has completed (stream order / event).
 * Threading / devices: the call launches on the current device; its forked side streams are kept per device, the
 * workspace (barrier words, queues) belongs to the caller, so two devices can be driven from one process with one
 * workspace each, but concurrent pcg_choose calls for the SAME device from several threads are not supported (the
 * reference is single-threaded, src/model_handler.py:142-156; multi-GPU runs of this package are one process per GPU).
 */
PCG_API int pcg_choose(const int64_t* indptr, const int32_t* indices, int64_t n_nodes, int64_t row_lo, int R,
               const float* score,
               const float* entry_score, const float* center_score, const int32_t* targets,
               const int64_t* labels, int B, const double* thresh_host, const int32_t* k_override, double rho,
               const float* ps_score, const int32_t* ps_pos, const int32_t* ps_id, const int32_t* entry_pool_pos, int P,
               int train, int64_t max_degree,
               int32_t* sel_idx, float* sel_dist, int64_t cap_slots, int32_t* slot_item, int32_t* it_slot0,
               int32_t* it_m, int64_t* it_base, int32_t* it_done, int32_t* it_rep, void* workspace,
               size_t workspace_bytes, int32_t* status, int phases, pcg_stream_t stream);

/*
 * Select-all variant for the GraphSAGE / GCN baselines: the item list IS the CSR row (no copy);
 * with add_self the target itself is added when its row lacks it.
 * Replaces src/graphsage.py:69-80 (MeanAggregator neighbour handling) and :206-212 (GCNAggregator).
 * it_extra[w] = node id to add on top of the row, or -1. Items index `indices` directly.
 */
PCG_API int pcg_select_all(const int64_t* indptr, const int32_t* indices, int64_t n_nodes, int R, const int32_t* targets,
                   int B, int add_self, int64_t cap_slots, int32_t* slot_item, int32_t* it_slot0, int32_t* it_m,
                   int64_t* it_base, int32_t* it_extra, int32_t* it_done, int32_t* status, pcg_stream_t stream);

/*
 * Segmented aggregation: agg[w, :] = norm(sum of feat rows of item w's id list).
 * Replaces the dense-mask matmul of src/layers.py:593-624 and src/graphsage.py:80-95, 212-231.
 *   idx       the id array the items index (sel_idx from pcg_choose, or CSR indices from select_all)
 *   it_extra / it_rep  from pcg_select_all / pcg_choose, or NULL
 *   copy_dups  != 0: rows of repeated targets (it_rep[w] != w) are filled with their representative's row by a
 *              second kernel; 0: they are left unwritten and the consumer reads row it_rep[w] instead
 *              (pcg_dense_fwd / pcg_dense_bwd take it_rep as `agg_rep`)
 *   partial   fp32 [cap_slots, ldf] scratch, it_done int32 [n_items] tickets zeroed by choose/select
 *   agg       fp32 [n_items, ldf]
 */
PCG_API int pcg_aggregate(const float* feat, int64_t ldf, const int32_t* idx, const int32_t* slot_item,
                  const int32_t* it_slot0, const int32_t* it_m, const int64_t* it_base, const int32_t* it_extra,
                  const int32_t* it_rep, int copy_dups, int n_items, int64_t cap_slots, const int32_t* status,
                  int norm, float* partial, int32_t* it_done, float* agg, pcg_stream_t stream);

/*
 * Backward of pcg_aggregate w.r.t. the feature table (only needed when `features` is trainable; the
 * reference freezes it, src/model_handler.py:85-86): feat_grad[j, :] += d_agg[w, :] * norm(n_w) for
 * every j in item w's list (vector red.global.add, one row per lane group).
 */
PCG_API int pcg_aggregate_bwd(const float* d_agg, int64_t ldf, const int32_t* idx, const int32_t* slot_item,
                      const int32_t* it_slot0, const int32_t* it_m, const int64_t* it_base, const int32_t* it_extra,
                      int n_items, int64_t cap_slots, const int32_t* status, int norm, float* feat_grad,
                      pcg_stream_t stream);

/*
 * Fused relation transforms + inter-relation combine, forward:
 *   cat[i, 0:F]            = feat[targets[i], :F]
 *   cat[i, F+rE:F+(r+1)E]  = relu([feat[targets[i]], agg[r*B+i]] @ W_r)      (src/layers.py:616-629)
 *   out[e, i]              = relu(cat[i, :] @ W)[e]                          (src/layers.py:273-289, [E,B])
 *   w_intra_host  HOST array of R device pointers, each the reference's IntraAgg.weight [2F, E] row-major
 *   w_inter       device [F+R*E, E]
 *   cat           fp32 [B, F+R*E] (kept for backward), out fp32 [E, B]
 *   agg_rep       int32 [R*B] or NULL: row of `agg` that holds item w's aggregate (pcg_choose's it_rep)
 */
PCG_API int pcg_dense_fwd(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, int R, int E,
                  const float* agg, const int32_t* agg_rep, const float* const* w_intra_host, const float* w_inter,
                  float* cat, float* out, pcg_stream_t stream);

/*
 * Backward of pcg_dense_fwd w.r.t. the weights (the reference's features are frozen, src/model_handler.py:85-86,
 * so these are the only gradients the path produces): d_w_intra_host[r] [2F,E] and d_w_inter [F+R*E,E] are
 * OVERWRITTEN; the reduction over the batch is split-K with a fixed summation order (deterministic).
 *   d_out    fp32 [E,B] gradient of `out`;  scratch  pcg_dense_bwd_scratch_floats(B,R,F,E) floats
 */
PCG_API size_t pcg_dense_bwd_scratch_floats(int B, int R, int F, int E);
PCG_API int pcg_dense_bwd(int64_t ldf, int F, int B, int R, int E, const float* agg, const int32_t* agg_rep,
                  const float* w_inter,
                  const float* cat, const float* out, const float* d_out, float* const* d_w_intra_host,
                  float* d_w_inter, float* scratch, pcg_stream_t stream);

/*
 * Fused dense part of the step (csrc/pcg_tile.cu), one kernel per tile of targets: relation transforms
 * (src/layers.py:616-629), inter-relation combine (src/layers.py:273-289, out is [E,B]) and the label_clf head on
 * the batch (src/layers.py:236-243); activations stay in shared memory, weights stream in by TMA bulk copies.
 * Supported when E is a multiple of 64 (<= 256) and the tile fits shared memory: pcg_tile_supported() != 0;
 * other shapes use pcg_dense_fwd / pcg_center_fwd.
 *   agg [R*B, lda] from pcg_aggregate (row of item w: agg_rep ? agg_rep[w] : w); feat / agg rows zero padded to
 *   a multiple of 4 floats; w_clf [2,F], b_clf [2] or NULL (then no center scores)
 *   keep_cat != 0: cat [B, F+R*E] is written for pcg_dense_bwd (autograd path), else cat may be NULL
 */
PCG_API int pcg_tile_supported(int B, int R, int F, int E);
PCG_API int pcg_tile_fwd(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, int R, int E,
                 const float* agg, int64_t lda, const int32_t* agg_rep, const float* const* w_intra_host,
                 const float* w_inter, const float* w_clf, const float* b_clf, int keep_cat, float* out,
                 float* center, float* cat, pcg_stream_t stream);
/*
 * Training form: the same forward, then (dLoss == 1 is known at forward time) PCALayer's head and both
 * cross-entropies (src/model.py:38, :54-61: loss = CE(W_head @ combined, y) + lambda * CE(center, y)), the
 * activation backward and EVERY weight gradient of the step (what autograd derives from the calls above):
 * d_w_head [2,E], d_w_clf [2,F], d_b_clf [2] by the tile kernel, d_w_inter [F+R*E,E] and d_w_intra_host[r] [2F,E]
 * by a weight-gradient kernel that follows it (batch split over a thread-block cluster, partial tiles added
 * through distributed shared memory). All gradients are OVERWRITTEN; reductions run in a
 * fixed order (deterministic). logits [B,2] / center [B,2] may be NULL.
 *   scratch  pcg_tile_scratch_floats(B,R,F,E) floats, 16-byte aligned
 *   pdl != 0: launch with programmatic stream serialization (the kernels' prologues overlap the previous
 *   kernel's tail; they wait for it with griddepcontrol.wait before touching its results)
 */
PCG_API size_t pcg_tile_scratch_floats(int B, int R, int F, int E);
PCG_API int pcg_tile_train(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, int R, int E,
                   const float* agg, int64_t lda, const int32_t* agg_rep, const float* const* w_intra_host,
                   const float* w_inter, const float* w_clf, const float* b_clf, const float* w_head,
                   const int64_t* labels, float lambda, float* out, float* center, float* logits, float* loss,
                   float* const* d_w_intra_host, float* d_w_inter, float* d_w_clf, float* d_b_clf, float* d_w_head,
                   float* scratch, int pdl, pcg_stream_t stream);

/*
 * label_clf similarity head on the batch's targets (src/layers.py:200, :236, :243):
 *   center[i][c] = dot(feat[targets[i], :F], w[c, :]) + b[c],  w [2,F], b [2] (nn.Linear layout)
 * and its backward: d_w [2,F], d_b [2] from d_center [B,2] (features are frozen). Deterministic.
 *   scratch  pcg_head_scratch_floats(B,F,E) floats; ticket: one int32, zero before the first call
 */
PCG_API size_t pcg_head_scratch_floats(int B, int F, int E);
PCG_API int pcg_center_fwd(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, const float* w,
                   const float* b, float* center, pcg_stream_t stream);
PCG_API int pcg_center_bwd(const float* feat, int64_t ldf, int F, const int32_t* targets, int B, const float* d_center,
                   float* d_w, float* d_b, float* scratch, int32_t* ticket, pcg_stream_t stream);

/*
 * PCALayer head + loss (src/model.py:38, :54-61): logits[i][c] = dot(w[c, :], emb[:, i]) with emb [E,B];
 * loss = mean_i CE(logits[i], labels[i]) + lambda * mean_i CE(center[i], labels[i]).
 * p1 / q1 [B] receive the class-1 softmax probabilities of the two heads (inputs of the backward).
 * Backward: d_emb [E,B], d_center [B,2], d_w [2,E] from the scalar d_loss (device pointer).
 */
PCG_API int pcg_head_loss_fwd(const float* emb, int E, int B, const float* w, const float* center,
                      const int64_t* labels, float lambda, float* logits, float* p1, float* q1, float* loss,
                      float* scratch, int32_t* ticket, pcg_stream_t stream);
PCG_API int pcg_head_loss_bwd(const float* emb, int E, int B, const float* w, const int64_t* labels, const float* p1,
                      const float* q1, float lambda, const float* d_loss, float* d_emb, float* d_center, float* d_w,
                      float* scratch, int32_t* ticket, pcg_stream_t stream);

/*
 * Encoder of the GraphSAGE / GCN baselines (src/graphsage.py:149 Encoder, :274 GCNEncoder):
 *   out[e][i] = relu(sum_f w[e][f] * X[i][f]),  X = agg rows (GCN; GraphSAGE with gcn=True) or [feat[targets[i]] | agg]
 *   (GraphSAGE with gcn=False, the cat of src/graphsage.py:145; pass feat/targets, else NULL), w [E, F or 2F].
 * Backward: d_w [E, F or 2F] from d_out [E,B] (relu mask from out); deterministic two-stage reduction.
 *   scratch  pcg_encoder_scratch_floats(B, F_in, E) floats; ticket: one int32, zero before the first call.
 * The head and cross-entropy behind the encoder (src/graphsage.py:169, :176-178) are pcg_head_loss_fwd/_bwd with
 * lambda = 0.
 */
PCG_API size_t pcg_encoder_scratch_floats(int B, int F_in, int E);
PCG_API int pcg_encoder_fwd(const float* agg, int64_t lda, const float* feat, int64_t ldf, const int32_t* targets, int F,
                    const float* w, int B, int E, float* out, pcg_stream_t stream);
PCG_API int pcg_encoder_bwd(const float* agg, int64_t lda, const float* feat, int64_t ldf, const int32_t* targets, int F,
                    int B, int E, const float* out, const float* d_out, float* d_w, float* scratch, int32_t* ticket,
                    pcg_stream_t stream);

/*
 * Label-balanced pick step, replay form: out[t] = idx_train[bisect_right(cum, u[t]*total, 0, n-1)],
 * total = cum[n-1]. Bit-compatible with random.choices(idx_train, weights, k) of
 * src/utils.py:274-278 when `u` are the doubles random.random() would have produced and `cum` is
 * the sequential fp64 prefix sum of the weights. idx_train may be NULL (positions are returned).
 */
PCG_API int pcg_pick_step(const double* cum, int64_t n, const double* u, int64_t k, const int32_t* idx_train,
                  int32_t* out, pcg_stream_t stream);
/* Same draw with device-generated uniforms (Philox4x32-10 counter RNG, 53-bit doubles): matches the
 * reference in distribution only. */
PCG_API int pcg_pick_step_philox(const double* cum, int64_t n, uint64_t seed, uint64_t offset, int64_t k,
                         const int32_t* idx_train, int32_t* out, pcg_stream_t stream);

/*
 * Data-parallel gradient exchange + Adam step as one kernel over NVLink peer memory (new design: the
 * reference is single-GPU, model_handler.py:87, and steps with torch.optim.Adam, model_handler.py:124,153).
 * Every rank owns a REGION of pcg_comm_region_bytes(n) bytes allocated with pcg_comm_alloc (cudaMalloc, zeroed),
 * exported with pcg_comm_export (64-byte CUDA IPC handle) and mapped by the peers with pcg_comm_import.
 * pcg_allreduce_adam(grad, param, m, v, n, regions[world] (HOST array of this process's mappings, own region
 * at [rank]), rank, world, epoch, ticket, lr, beta1, beta2, eps, weight_decay, do_adam, stream):
 *   grad <- mean over ranks of grad (summed in rank order: bit-identical on every rank); with do_adam the
 *   torch.optim.Adam update (L2 weight decay, bias correction with step = *epoch + 1) is applied to param / m / v
 *   and grad is cleared. epoch (uint32, zero before the first step) and ticket (int32, zero) live in device
 *   memory so that CUDA-graph replays advance them. n must be a multiple of 4; world <= 8. All ranks must call
 *   it the same number of times (the kernels wait for one another through flags in the regions).
 */
PCG_API size_t pcg_comm_region_bytes(int64_t n_params);
PCG_API int pcg_comm_alloc(void** ptr, size_t bytes);
PCG_API int pcg_comm_free(void* ptr);
PCG_API int pcg_comm_export(void* ptr, unsigned char* handle64);
PCG_API int pcg_comm_import(const unsigned char* handle64, void** ptr);
PCG_API int pcg_comm_unmap(void* ptr);
PCG_API int pcg_allreduce_adam(float* grad, float* param, float* m, float* v, int64_t n_params,
                       void* const* peer_regions_host, int rank, int world, uint32_t* epoch, int32_t* ticket,
                       float lr, float beta1, float beta2, float eps, float weight_decay, int do_adam,
                       pcg_stream_t stream);

/*
 * Label scores of a row partition + halo exchange in one kernel (config C5). Every rank owns a region of
 * pcg_score_region_bytes(n_global) bytes ([n_global] fp32 score table + arrival counters; pcg_comm_alloc /
 * _export / _import as above). pcg_score_bcast scores the n_rows feature rows at feat_rows (global ids row_lo ..)
 * with w[0..F), b[0] (src/layers.py:236-237, column 0) and stores them into the table of EVERY rank, then waits
 * (on the stream) until every peer's slice has arrived in the own table. Equal n_rows on all ranks. Safe to call
 * once per training step: the gradient exchange of the step orders it against the peers' readers.
 */
PCG_API size_t pcg_score_region_bytes(int64_t n_global);
PCG_API int pcg_score_bcast(const float* feat_rows, int64_t n_rows, int F, int64_t ldf, const float* w, const float* b,
                    int64_t row_lo, int64_t n_global, void* const* regions_host, int rank, int world,
                    uint32_t* epoch, pcg_stream_t stream);

/*
 * Evaluation pass (the batch loop of src/utils.py:298-312 and its metrics, :313-333) with every batch of the node set
 * resident in HBM. pcg_eval_head is the two-class head and to_prob's output on one recorded batch: with entry
 * e = *cursor % count (cursor NULL: e = 0) and l_c = sum_k w_head[c,k] * emb[k,i] (k summed in order 0..E-1), row
 * i < min(B, n_total - e*B) writes
 *   mode 0: prob[c * n_total + e*B + i] = sigmoid(l_c)     PCALayer (src/model.py:38, :41-45), GCN (src/graphsage.py:154-178)
 *   mode 1: prob[c * n_total + e*B + i] = (l_c - m) - log(exp(l_0 - m) + exp(l_1 - m)),  m = max(l_0, l_1)
 *           the log_softmax of GraphSage.to_prob (src/graphsage.py:16-39, over dim 1)
 * emb [E,B] from pcg_tile_fwd or pcg_encoder_fwd, w_head [2,E]; prob is planar [2, n_total] and padding rows are not
 * written. The cursor is not advanced (a trailing pcg_stage_indexed with bump != 0 does that).
 *
 * pcg_binary_metrics computes every metric of prob [2,n] (planar, as above) against int32 labels [n] (0 / 1) into
 * out[PCG_METRICS_WORDS] doubles: prob[1] is sorted with pcg_sort_pool (labels as the pool), AUC is the Mann-Whitney
 * statistic with average ranks for ties (NaN when one class is absent), the confusion counts take pred = 1 iff
 * prob[1] > prob[0], F1 / recall / precision follow sklearn's zero_division=0, and the best threshold is the distinct
 * value t of prob[1] whose cut "positive iff prob[1] >= t" has the largest macro-F1 (ties: the larger t).
 * Ranking words, with s = prob[1] sorted ascending, P positives, N = n - P, pre[j] = positives among s[0, j)
 * (pre[n] = P), a tie group = a maximal run [lo, hi) of equal s and its cut "positive iff prob[1] >= s[lo]"
 * (TP = P - pre[lo], FP = (n - lo) - TP):
 *   PCG_MT_AP           sklearn's average_precision_score: sum over groups of (pre[hi]-pre[lo])/P * TP/(n-lo); NaN if P = 0
 *   PCG_MT_RECALL_AT_K  K = P: with c = n - P and [lo, hi) the group containing c,
 *                       TP@K = (P - pre[hi]) + (pre[hi]-pre[lo]) * (hi-c)/(hi-lo) (the expected count over random
 *                       orders of the tied scores), then / P; NaN if P = 0. With K = P it is also Precision@K.
 *   PCG_MT_BEST_GMEAN   sqrt(TP/P * TN/N) maximised over the group cuts (0 where a denominator is 0), ties to the larger
 *                       threshold; PCG_MT_BEST_GMEAN_THRESHOLD is that s[lo]
 * Deterministic (integer sums, fp64 sums in a fixed order, an order-free arg-max); 0 < n < 2^31.
 *   workspace  pcg_binary_metrics_workspace_bytes(n) bytes, 256-byte aligned
 * Words 17-20 were appended in version 101 (PCG_METRICS_WORDS was 17); words 0-16 are unchanged, so a caller that
 * sizes `out` with PCG_METRICS_WORDS only needs to recompile.
 *
 * pcg_binary_curve: the ROC / PR curve of the last pcg_binary_metrics call on `workspace` (same n, ordered after it on
 * the stream), read from the sorted scores and pre that call left there (no further sort). For the G tie groups in
 * ascending order of threshold it writes thr[g] = s[lo], tp[g] = TP, fp[g] = FP of the group's cut, and G into the
 * device word *count. thr, tp and fp must hold n entries (G <= n).
 *
 * pcg_binary_points: operating points the caller chooses, read like pcg_binary_curve from the workspace of the last
 * pcg_binary_metrics call (same n, ordered after it on the stream; no further sort). Request r is kind[r] with the
 * argument arg[r]; both arrays live in device memory, so a recorded graph keeps reading them and the caller may change
 * them in place between replays. Request r writes out[r * PCG_POINT_WORDS + 0 .. 4]:
 *   kind 0  top K (arg = K, an integer, 1 <= K <= n): with c = n - K and [lo, hi) the group containing c,
 *           TP@K = (P - pre[hi]) + (pre[hi]-pre[lo]) * (hi-c)/(hi-lo) (PCG_MT_RECALL_AT_K's rule for any K).
 *           Words {recall = TP@K / P (NaN if P = 0), precision = TP@K / K, threshold = s[c] (the K-th highest score),
 *           TP@K, K - TP@K}. With K = P, recall has the bits of PCG_MT_RECALL_AT_K.
 *   kind 1  TPR at FPR <= f (arg = f, 0 <= f <= 1): of the group cuts with FP(lo) <= f * N (compared in fp64) the one
 *           with the largest TPR, i.e. the smallest such lo; when none has, nothing is flagged (TP = FP = 0, threshold
 *           +inf). Words {TPR = TP / P, FPR = FP / N, threshold = s[lo], TP, FP}; all NaN if P = 0 or N = 0.
 *   kind 2  standardised partial AUC (arg = max_fpr f, 0 < f <= 1), sklearn's roc_auc_score(max_fpr=f): A = the
 *           trapezoid area under the ROC points (FP(lo)/N, TP(lo)/P) of the group starts and (0, 0), up to FPR = f
 *           with TPR interpolated linearly at f. Words {0.5 * (1 + (A - f^2/2) / (f - f^2/2)), A, NaN, NaN, NaN};
 *           with f = 1 the first is the AUC. NaN if P = 0 or N = 0.
 * A request whose argument is out of its range, or whose kind is not 0, 1 or 2, writes PCG_POINT_WORDS NaN; words a
 * kind does not define are NaN. Two launches whatever m is (0 < m <= PCG_POINTS_MAX); kind 2 sums fp64 partials per
 * chunk in a fixed order, so reruns give the same bits.
 *   metrics_ws  the workspace of pcg_binary_metrics (pcg_binary_metrics_workspace_bytes(n) bytes), not modified
 *   ws          pcg_binary_points_workspace_bytes(n, m) bytes, 8-byte aligned (kind 2's partials)
 */
#define PCG_METRICS_WORDS 21
#define PCG_MT_AUC 0
#define PCG_MT_F1 1
#define PCG_MT_F1_MACRO 2
#define PCG_MT_RECALL 3
#define PCG_MT_PRECISION 4
#define PCG_MT_RECALL_MACRO 5
#define PCG_MT_PRECISION_MACRO 6
#define PCG_MT_ACCURACY 7
#define PCG_MT_GMEAN 8
#define PCG_MT_BEST_F1_MACRO 9
#define PCG_MT_BEST_THRESHOLD 10
#define PCG_MT_N_POS 11
#define PCG_MT_N_NEG 12
#define PCG_MT_TP 13
#define PCG_MT_FP 14
#define PCG_MT_TN 15
#define PCG_MT_FN 16
#define PCG_MT_AP 17
#define PCG_MT_RECALL_AT_K 18
#define PCG_MT_BEST_GMEAN 19
#define PCG_MT_BEST_GMEAN_THRESHOLD 20
/* pcg_binary_points: doubles per request, most requests per call, request kinds */
#define PCG_POINT_WORDS 5
#define PCG_POINTS_MAX 1024
#define PCG_POINT_TOP_K 0
#define PCG_POINT_TPR_AT_FPR 1
#define PCG_POINT_PAUC 2
PCG_API int pcg_eval_head(const float* emb, int E, int B, const float* w_head, int mode, int64_t n_total,
                  const uint32_t* cursor, uint32_t count, float* prob, pcg_stream_t stream);
PCG_API size_t pcg_binary_metrics_workspace_bytes(int64_t n);
PCG_API int pcg_binary_metrics(const float* prob, const int32_t* labels, int64_t n, double* out, void* workspace,
                       size_t workspace_bytes, pcg_stream_t stream);
PCG_API int pcg_binary_curve(const void* workspace, size_t workspace_bytes, int64_t n, float* thr, int64_t* tp,
                     int64_t* fp, int64_t* count, pcg_stream_t stream);
PCG_API size_t pcg_binary_points_workspace_bytes(int64_t n, int m);
PCG_API int pcg_binary_points(const void* metrics_ws, size_t metrics_ws_bytes, int64_t n, const int32_t* kind,
                      const double* arg, int m, double* out, void* ws, size_t ws_bytes, pcg_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PCGNN_B200_H */
