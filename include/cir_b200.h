/* cir_b200.h -- C-ABI of the B200-native stage-II candidate re-ranker hot path.
 *
 * The reference (Cuberick-Orion/Candidate-Reranking-CIR) has no FFI/plugin registry: its
 * boundary for this path is the Python method surface of BLIP_NLVR / BLIP_Retrieval
 * (src/blip_stage2.py:57-136, src/blip_stage1.py:48-92) plus the metric functions of
 * src/validate_stage2.py:33-66,153-206 and the similarity/top-K lines of
 * src/validate.py:54-59,198-210.  Each entry point below names the reference code it
 * replaces; the Python host modules in candidate-reranking-cir_b200/ mirror the reference's
 * method signatures and call ONLY these functions (ctypes), with raw device pointers taken
 * from torch tensors.  See INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative CIR_E* code on failure; the message is
 *     retrievable with cir_last_error() (thread-local).  Nothing throws across the ABI.
 *   - all pointers are DEVICE pointers unless the name ends in _host.
 *   - functions are asynchronous on the context's stream and never synchronise it, never
 *     allocate device memory: the caller supplies a workspace (size from *_workspace_bytes).
 *   - "act" tensors (activations / image tokens) have the context's dtype: bf16 in
 *     CIR_DTYPE_BF16 mode, fp32 in CIR_DTYPE_F32 (the fp32 check mode).  Weight matrices have
 *     the same dtype; biases / LayerNorm parameters / embedding tables are always fp32.
 *   - matrices are row-major; Linear weights keep PyTorch's [out, in] layout (K-major).
 *   - one context per (device, stream); a context is not thread-safe.
 */
#ifndef CIR_B200_H
#define CIR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CIR_OK            0
#define CIR_EINVAL       -1   /* bad argument / unsupported shape */
#define CIR_ECUDA        -2   /* CUDA runtime / driver error */
#define CIR_EWORKSPACE   -3   /* workspace too small */
#define CIR_EUNSUPPORTED -4   /* device is not sm_100 or feature unavailable */

#define CIR_DTYPE_F32   0     /* fp32 check mode: CUDA-core FMA GEMMs, fp32 activations */
#define CIR_DTYPE_BF16  1     /* production: tcgen05 bf16 GEMMs with fp32 accumulation */

#define CIR_GEMM_AUTO    0    /* bf16 -> tcgen05, fp32 -> simt */
#define CIR_GEMM_SIMT    1    /* force the CUDA-core GEMM (debug / cross-check) */
#define CIR_GEMM_TCGEN05 2
#define CIR_GEMM_TCGEN05_1CTA 3   /* tcgen05 but never the cta_group::2 pair tile (cross-check) */

#define CIR_ACT_NONE 0
/* GELU of the reference (transformers ACT2FN["gelu"] = erf form; src/nlvr_encoder.py:376, src/vit.py:38).  fp32 contexts evaluate
 * 0.5 x (1 + erf(x / sqrt 2)) with erff.  bf16 contexts evaluate the tanh form 0.5 x (1 + tanh(0.79788456 (x + 0.044715 x^3)))
 * with the hardware tanh.approx in the GEMM epilogue: |gelu_tanh - gelu_erf| <= 5e-4 absolute (at |x| ~ 2), tanh.approx adds
 * <= 2^-11 relative -- both below the bf16 rounding of the stored activation (2^-9 relative) for |x| >= 0.3; measured effect on
 * stage-II scores: inside the 2e-2 tolerance with the same margin as an erf epilogue (DESIGN.md section 5). */
#define CIR_ACT_GELU 1
#define CIR_ACT_RELU 2

#define CIR_HIDDEN   768
#define CIR_HEADS    12
#define CIR_HEAD_DIM 64
#define CIR_FFN      3072
#define CIR_LAYERS   12
#define CIR_EMBED    256

typedef struct cir_ctx cir_ctx;

/* ---- context ------------------------------------------------------------------------ */
const char* cir_last_error(void);
int  cir_version(void);
int  cir_create(cir_ctx** out, int device, int dtype);
int  cir_destroy(cir_ctx* ctx);
int  cir_set_stream(cir_ctx* ctx, void* cuda_stream);       /* cudaStream_t */
int  cir_set_gemm_impl(cir_ctx* ctx, int impl);              /* CIR_GEMM_* */
int  cir_set_attention_impl(cir_ctx* ctx, int impl);      /* 0 auto (tcgen05 where eligible, else mma.sync), 1 CUDA-core kernel, 2 mma.sync only */
/* stage II: compute layer 11 only for the two CLS query rows that the encoder returns (default on; 0 = all rows) */
int  cir_set_prune_last_layer(cir_ctx* ctx, int enable);
/* stage II: layer 0's self-attention block and cross query projection depend on the query only (both streams are expanded
 * copies, src/blip_stage2.py:118-124): run them once per unique query of a chunk and expand (default on; exact) */
int  cir_set_dedup_first_layer(cir_ctx* ctx, int enable);
/* bf16 mode, captions of 8, 16, 24 or 32 tokens: the query/key/value Linears and the masked text self-attention run as ONE kernel
 * (cir_qkv_attention) -- the [rows, 2304] projection never reaches HBM.  Default on; 0 = GEMM + attention kernel (bit-equal). */
int  cir_set_fuse_qkv_attention(cir_ctx* ctx, int enable);
/* bf16 contexts, galleries of >= 16,384 rows: cir_stage1_topk and cir_stage1_index_topk compute the similarities on the tensor
 * cores (bf16 operands) only to FILTER candidates with a rigorous error margin, then re-compute the survivors in fp32 -- results
 * are bit-identical to the fp32 path.  Default on; 0 = fp32 CUDA-core similarities for every gallery row. */
int  cir_set_stage1_tensor_cores(cir_ctx* ctx, int enable);
/* 1 (default): bf16 GEMM outputs leave the tcgen05 epilogue through TMA bulk tensor stores; 0: per-lane 16 B stores. */
int  cir_set_gemm_tma_store(cir_ctx* ctx, int enable);
int  cir_get_dtype(const cir_ctx* ctx);
/* number of kernel launches issued through this context since the last reset (bench.py's gpu_launches) */
int64_t cir_launch_count(cir_ctx* ctx, int reset);

/* per-launch timing of the tcgen05 GEMM (CUDA events on the context's stream around every GEMM launch);
 * cir_profile_gemm(ctx,1) resets and starts, (ctx,0) stops; _read synchronises on the recorded events and
 * returns summed duration, summed algorithmic FLOPs (2*M*N*K*batch) and the launch count. */
int  cir_profile_gemm(cir_ctx* ctx, int enable);
int  cir_profile_gemm_read(cir_ctx* ctx, double* total_ms, double* total_flops, int64_t* launches);
/* the same event pairs are recorded around the other kernels that matter for the step time; `kind` selects them:
 * total_work = algorithmic FLOPs for CIR_PROF_GEMM / CIR_PROF_ATTN_TC (4*Lq*Lk*64 per (batch, head)) / CIR_PROF_ATTN_SELF /
 * CIR_PROF_QKV_ATTN (projection + attention), algorithmic bytes (rows * 768 * (bytes read + bytes written)) for CIR_PROF_LAYERNORM. */
#define CIR_PROF_GEMM      0
#define CIR_PROF_ATTN_TC   1   /* tcgen05 cross-attention / ViT attention */
#define CIR_PROF_ATTN_SELF 2   /* masked text self-attention (mma.sync kernels) */
#define CIR_PROF_LAYERNORM 3
#define CIR_PROF_QKV_ATTN  4   /* fused QKV projection + masked self-attention */
#define CIR_PROF_KINDS     5
int  cir_profile_read(cir_ctx* ctx, int kind, double* total_ms, double* total_work, int64_t* launches);

/* ---- primitive ops (each replaces one ATen call of the reference; used by the pipelines
 *      below and individually by the parity tests) ------------------------------------- */

/* C[b] = act(A[b] * W[b]^T + bias[b]) (+ residual[b]);  replaces nn.Linear / torch.matmul
 * (e.g. src/nlvr_encoder.py:150,158-159,250-254,381,394; src/vit.py:37-40,72,83).
 * A: [batch][M, K] act dtype, row stride lda, batch stride a_bstride (elements; 0 = shared)
 * W: [batch][N, K] act dtype, row stride ldw, batch stride w_bstride
 * C: [batch][M, N] bf16/fp32 (c_f32), row stride ldc, batch stride c_bstride
 * bias: fp32 [batch][N] or NULL; residual: [batch][M,N] (fp32 if res_f32 else act dtype) or NULL */
typedef struct cir_gemm_args {
  const void* A; const void* W; void* C;
  const float* bias; const void* residual;
  int64_t M, N, K;
  int64_t lda, ldw, ldc, ldres;
  int64_t a_bstride, w_bstride, c_bstride, bias_bstride, res_bstride;
  int32_t batch;
  int32_t act;       /* CIR_ACT_* */
  int32_t c_f32;     /* 1: C is fp32 regardless of ctx dtype */
  int32_t res_f32;   /* 1: residual is fp32 */
} cir_gemm_args;
int cir_gemm(cir_ctx* ctx, const cir_gemm_args* args);

/* y[r] = LayerNorm(x[r % x_rows] + res[r]) * gamma[g] + beta[g], g = r / rows_per_group;
 * replaces nn.LayerNorm incl. the twin LayerNormA/B of src/nlvr_encoder.py:256,260-264.
 * x: fp32 if x_f32 else act dtype; res: act dtype or NULL; y: act dtype (fp32 if y_f32). */
int cir_add_layernorm(cir_ctx* ctx, const void* x, int x_f32, int64_t x_rows, const void* res,
                      const float* gamma, const float* beta, int64_t rows_per_group,
                      void* y, int y_f32, int64_t rows, float eps);

/* softmax(Q K^T * scale + mask) V per (batch, head); dh = 64.  Replaces
 * BertSelfAttention.forward (src/nlvr_encoder.py:175-217) and vit Attention (src/vit.py:74-82).
 * q/k/v/o: act dtype; element strides: *_bs batch, *_rs row; head h lives at column h*64.
 * kv_index: optional int32[B] -> batch index used for K/V (candidate gather); key_mask: optional
 * int32 [B, Lk] (1 = attend, 0 -> additive -10000, src/nlvr_encoder.py:774). */
typedef struct cir_attn_args {
  const void* q; const void* k; const void* v; void* o;
  int64_t q_bs, q_rs, k_bs, k_rs, v_bs, v_rs, o_bs, o_rs;
  const int32_t* kv_index; const int32_t* key_mask;
  const int32_t* mask_index;   /* optional int32[B] -> row of key_mask used for batch b (default b) */
  /* optional K/V-sharing work list, int32 [num_work][4] = {first batch, first 16-row unit, units in
   * the run, 0}: one CTA per entry; all batches of a run MUST name the same K/V batch (candidate-
   * major triplets).  A unit is (batch, 16-row query tile): unit u -> batch first+u/mt, tile u%mt,
   * mt = ceil(Lq/16).  NULL: every batch is its own run. */
  const int32_t* work; int32_t num_work;
  /* tcgen05 path (bf16, no key_mask): optional tile list int32 [num_tiles][4] = {first batch, batches in
   * the tile, first query row, rows per batch RB = min(256, smallest power of two >= Lq)}: a tile is 256 query
   * rows = (256/RB) batches sharing one K/V batch x RB rows starting at `first query row` (two 128-row UMMA tiles
   * that share every K/V chunk).  NULL: one batch per tile, 256-row slices.
   * kv_batches = number of K/V batches behind k/v (rows = kv_batches*Lk, k_bs must equal Lk*k_rs). */
  const int32_t* tiles; int32_t num_tiles; int32_t kv_batches;
  int32_t B, H, Lq, Lk;
  float scale;
} cir_attn_args;
int cir_attention(cir_ctx* ctx, const cir_attn_args* args);

/* Fused self-attention block input side: out[b][c*L + l, h*64 + d] = softmax(Q_h K_h^T * scale + mask) V_h with
 * [Q|K|V] = x[b] w[b]^T + bias[b] (query / key / value Linears stacked as [2304, 768], PyTorch [out, in] layout);
 * replaces BertSelfAttention.forward for text self-attention (src/nlvr_encoder.py:140-222, src/med.py:112-216).
 * bf16 context only; L in {8, 16, 24, 32}; rows of x / out are caption-major (row = caption*L + token), row stride 768 / out_rs.
 * key_mask int32 [*, L] (1 = attend, 0 -> additive -10000), row mask_index[c] (NULL: c) belongs to caption c. */
typedef struct cir_qkv_attn_args {
  const void* x; int64_t x_bs;          /* [batch][captions*L, 768] bf16; batch stride in elements */
  const void* w;                        /* [batch][2304, 768] bf16 */
  const float* bias;                    /* [batch][2304] fp32 or NULL */
  void* out; int64_t out_rs, out_bs;    /* [batch][captions*L, 768] bf16 context */
  const int32_t* key_mask; const int32_t* mask_index;
  int64_t captions; int32_t L; int32_t batch;
  float scale;
} cir_qkv_attn_args;
int cir_qkv_attention(cir_ctx* ctx, const cir_qkv_attn_args* args);

/* out[q,l,:] = LayerNorm(word[ids[q,l]] + pos[l]); src/nlvr_encoder.py:68-91, src/med.py:86-110 */
int cir_bert_embeddings(cir_ctx* ctx, const int32_t* ids, int64_t Q, int64_t L, const float* word_emb,
                        const float* pos_emb, const float* gamma, const float* beta, void* out);

/* dst[i, :] = src[index[i], :] for rows of `row_elems` act elements (expand / candidate gather:
 * src/blip_stage2.py:118-124, src/validate_stage2.py:251). index NULL = identity copy. */
int cir_gather_rows(cir_ctx* ctx, const void* src, const int32_t* index, void* dst, int64_t rows,
                    int64_t row_elems);
int cir_cast_f32_to_act(cir_ctx* ctx, const float* src, void* dst, int64_t n);
int cir_cast_act_to_f32(cir_ctx* ctx, const void* src, float* dst, int64_t n);

/* y = x / max(||x||_2, 1e-12) per row (F.normalize, src/blip_stage1.py:57,83; src/validate.py:311) */
int cir_l2_normalize(cir_ctx* ctx, const float* x, float* y, int64_t rows, int64_t dim);

/* ---- re-sort, top-K, merge, recall (src/validate_stage2.py:53-62,174-203; src/validate.py:57-59,202-210) */

/* order[q,:] = argsort(scores[q,:], descending), ties -> lowest index first. K <= 2048. */
int cir_rerank_sort(cir_ctx* ctx, const float* scores, int64_t Q, int64_t K, int32_t* order);

/* From a distance matrix dist[Q, G] (row stride ldd): the K smallest per row in ascending order,
 * ties -> lowest index, skipping column exclude[q] (-1 = none).  `col_offset` is added to the
 * output indices (gallery shard offset).  K <= 1024.  Bit-exact integer selection. */
int cir_topk_from_dist(cir_ctx* ctx, const float* dist, int64_t Q, int64_t G, int64_t ldd,
                       const int32_t* exclude, int64_t col_offset, int64_t K,
                       float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes);
size_t cir_topk_workspace_bytes(int64_t Q, int64_t G, int64_t K);

/* Fused stage-I retrieval: dist = 1 - q_emb @ g_emb^T computed tile-wise (never materialising
 * [Q, G]), running top-K per query.  q_emb [Q,256] fp32, g_emb [G,256] fp32. */
int cir_stage1_topk(cir_ctx* ctx, const float* q_emb, const float* g_emb, int64_t Q, int64_t G,
                    const int32_t* exclude, int64_t col_offset, int64_t K,
                    float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes);
size_t cir_stage1_topk_workspace_bytes(int64_t Q, int64_t G, int64_t K);

/* Resident stage-I gallery index: the gallery embeddings (the `index_features` of src/utils.py:56-70, pooled and normalised)
 * converted once and searched by many query batches (src/validate.py:198-203).  A search returns exactly what cir_stage1_topk
 * returns over the same rows, bit for bit.  The blob (cir_stage1_index_bytes, 256-byte aligned) is owned by the caller; the struct
 * points into it.  _init and _add enqueue work on the context's stream.
 *   _add appends n rows (device fp32 [n,256]): copies them and, in bf16 contexts, converts only the new rows to bf16 and raises
 *        the gallery maxima the filter bound uses.  Past `capacity`: CIR_EINVAL.  `rows` counts on the host.
 *   _topk searches the first `rows` rows with the tensor-core filter (bf16 context, cir_set_stage1_tensor_cores on, rows >= 16,384)
 *        or the fp32 tile loop, chosen per call.  It never synchronises and never copies to the host, so it can be captured in a
 *        CUDA graph; a graph captured before an _add still searches the row count of its capture.  exact_rows (optional, [Q]):
 *        1 where a query's candidate list overflowed and its list came from the exact scan of the whole index, else 0.
 *        The workspace size depends on the capacity, not on `rows`: one workspace serves the index as it grows. */
typedef struct cir_stage1_index {
  int64_t capacity, rows;   /* rows added so far (host-side count) */
  float*  g_f32;            /* [capacity,256] fp32 rows, owned copy (the exact re-check reads them) */
  void*   g_bf16;           /* [capacity,256] bf16 copy; NULL in fp32 contexts */
  uint32_t* gmax;           /* device: {max ||g||, max ||g - bf16(g)||} as float bits, updated by _add only */
} cir_stage1_index;
size_t cir_stage1_index_bytes(const cir_ctx* ctx, int64_t capacity);
int    cir_stage1_index_init(cir_ctx* ctx, void* blob, size_t bytes, int64_t capacity, cir_stage1_index* out);
int    cir_stage1_index_add(cir_ctx* ctx, cir_stage1_index* index, const float* g_emb, int64_t n);
size_t cir_stage1_index_topk_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* index, int64_t Q, int64_t K);
int    cir_stage1_index_topk(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q, const int32_t* exclude,
                             int64_t col_offset, int64_t K, float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                             void* workspace, size_t workspace_bytes);
/* Filtered search: row r of the index is eligible for query q iff (row_tags[r] & query_masks[q]) != 0; otherwise as
 * cir_stage1_index_topk.  The result is exactly what cir_stage1_topk returns over the eligible rows compacted in their original
 * order, with indices mapped back (col_offset + local row), ties to the lowest eligible row; a query with fewer than K eligible
 * rows gets (+inf, -1) in the remaining slots (a mask of 0: all of them).  `exclude` applies on top of eligibility; exact_rows
 * flags queries whose eligible-row candidate list overflowed.  Eligibility is applied before a row enters a query's candidate
 * list (tensor-core filter, exact scan and fp32 path alike).  The workspace is cir_stage1_index_topk_workspace_bytes, so one
 * workspace (and one captured graph) serves both calls.  Tags and masks belong to the caller and are read when the search runs:
 * a captured graph follows in-place edits of both, which is how rows are removed (tag 0) or re-categorised.  Never synchronises.
 * NULL row_tags or query_masks: CIR_EINVAL. */
int    cir_stage1_index_topk_filtered(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q,
                                      const uint32_t* row_tags,     /* device [index->rows], local row order */
                                      const uint32_t* query_masks,  /* device [Q] */
                                      const int32_t* exclude, int64_t col_offset, int64_t K,
                                      float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                                      void* workspace, size_t workspace_bytes);
/* Compaction and subsets: copy the rows r of `src` with (src_tags[r] & keep_mask) != 0, in their order, into `dst` -- an initialised,
 * EMPTY index in a different blob (overlap: CIR_EINVAL) of the context's dtype -- with their tags in dst_tags and their ids in dst_ids
 * (device [dst->capacity]).  The id of row r is src_ids[r], or r when src_ids is NULL.  keep_mask 0xFFFFFFFF drops the removed rows
 * (tag 0); a narrower mask extracts a subset.  dst's blob is byte for byte what cir_stage1_index_add of the kept rows builds: fp32 rows,
 * bf16 copy and the maxima of the kept rows only.  The call synchronises the stream ONCE to read the kept count (dst->rows is a host
 * count): a maintenance call, not capturable in a CUDA graph (CIR_EINVAL while the stream captures).  More kept rows than
 * dst->capacity: CIR_EINVAL and nothing written.  Zero kept rows is valid.  workspace: _compact_workspace_bytes(src). */
size_t cir_stage1_index_compact_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* src);
int    cir_stage1_index_compact(cir_ctx* ctx, const cir_stage1_index* src, const uint32_t* src_tags, const int32_t* src_ids,
                                uint32_t keep_mask, cir_stage1_index* dst, uint32_t* dst_tags, int32_t* dst_ids,
                                void* workspace, size_t workspace_bytes);
/* Search an index whose physical row p carries the permanent id row_ids[p] (device [index->rows], strictly increasing, all < id_end --
 * e.g. the number of rows ever added; compaction keeps the order, so its ids stay increasing).  exclude[q] and the returned indices
 * are col_offset + id; an excluded id that no row holds excludes nothing.  row_tags and query_masks: both NULL (unfiltered, as
 * cir_stage1_index_topk) or both set (as cir_stage1_index_topk_filtered).  Because ids increase with the physical rows, ties resolve
 * as they would over the ids: the result equals the same search over an index that was never compacted, bit for bit.  Never
 * synchronises (graph-capturable).  col_offset + id_end > 2^31: CIR_EINVAL.  workspace: _topk_ids_workspace_bytes, which is
 * cir_stage1_index_topk_workspace_bytes plus 4 bytes per query (256-byte aligned). */
size_t cir_stage1_index_topk_ids_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* index, int64_t Q, int64_t K);
int    cir_stage1_index_topk_ids(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q,
                                 const int32_t* row_ids, int64_t id_end,
                                 const uint32_t* row_tags, const uint32_t* query_masks,   /* both NULL or both set */
                                 const int32_t* exclude, int64_t col_offset, int64_t K,
                                 float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                                 void* workspace, size_t workspace_bytes);

/* In-batch contrastive logits of the stage-I forward: logits[Q, G] = q_emb[Q,256] @ t_emb[G,256]^T / temp, all fp32.
 * Replaces `predicted_features @ target_features.T / self.temp` (src/blip_stage1.py:90-91), forward only. */
int cir_stage1_logits(cir_ctx* ctx, const float* q_emb, const float* t_emb, int64_t Q, int64_t G, float temp, float* logits);

/* Stage-I ranking of P named gallery rows per query (the CIRR "img_set" group members without the reference image):
 * member_dist[q,j] = 1 - q_emb[q] . g_emb[members[q,j]] with the arithmetic of cir_stage1_topk, member_order[q,r] = slot j of
 * the r-th closest member (ties -> lowest gallery row).  Yields `group_labels` of the stage-I top-K file without the full
 * [Q,G] sort: src/validate.py:213-218 (labels[group_mask]), written at :256-263 and read at src/data_utils.py:301.  P <= 32. */
int cir_stage1_rank_members(cir_ctx* ctx, const float* q_emb, const float* g_emb, const int32_t* members, int64_t Q,
                            int64_t P, float* member_dist, int32_t* member_order);

/* Merge P per-shard sorted lists pairs[p][Q][K] -> best K per query (ascending dist, ties ->
 * lowest global index).  The NCCL all-gather that assembles `dist_in/idx_in` is done by the host. */
int cir_topk_merge(cir_ctx* ctx, const float* dist_in, const int32_t* idx_in, int64_t P, int64_t Q,
                   int64_t K, float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes);
                   /* workspace: cir_topk_workspace_bytes(Q, 0, K) */

/* hits[j] = sum_q any(labels[q, order[q, :ks[j]]]); labels uint8 [Q,K].  Recall@k = 100*hits/Q. */
int cir_recall_counts(cir_ctx* ctx, const uint8_t* labels, const int32_t* order, int64_t Q, int64_t K,
                      const int32_t* ks_host, int32_t num_ks, int64_t* hits);

/* ---- model pipelines ------------------------------------------------------------------ */

/* ViT-B/16 weights (src/vit.py:113-161), packed by the host: per block i in [0,12). */
typedef struct cir_vit_weights {
  const void*  patch_w;  const float* patch_b;      /* [768, 3*16*16] act, [768] */
  const float* cls_token; const float* pos_embed;   /* [768], [N,768] fp32 */
  const float* norm1_g[CIR_LAYERS]; const float* norm1_b[CIR_LAYERS];
  const void*  qkv_w[CIR_LAYERS];   const float* qkv_b[CIR_LAYERS];     /* [2304,768] */
  const void*  proj_w[CIR_LAYERS];  const float* proj_b[CIR_LAYERS];    /* [768,768] */
  const float* norm2_g[CIR_LAYERS]; const float* norm2_b[CIR_LAYERS];
  const void*  fc1_w[CIR_LAYERS];   const float* fc1_b[CIR_LAYERS];     /* [3072,768] */
  const void*  fc2_w[CIR_LAYERS];   const float* fc2_b[CIR_LAYERS];     /* [768,3072] */
  const float* norm_g; const float* norm_b;
} cir_vit_weights;

/* VisionTransformer.forward (src/vit.py:180-194) == BLIP_NLVR.img_embed / BLIP_Retrieval.img_embed.
 * images fp32 [B,3,S,S] -> tokens act [B, N=(S/16)^2+1, 768]. */
size_t cir_vit_workspace_bytes(const cir_ctx* ctx, int64_t B, int64_t image_size);
int cir_vit_forward(cir_ctx* ctx, const cir_vit_weights* w, const float* images, int64_t B,
                    int64_t image_size, void* tokens, void* workspace, size_t workspace_bytes);

/* Stage-I single-stream MED encoder weights (src/med.py:335-398) + projections (src/blip_stage1.py:40-43). */
typedef struct cir_stage1_weights {
  const float* word_emb; const float* pos_emb; const float* emb_ln_g; const float* emb_ln_b;
  const void*  self_qkv_w[CIR_LAYERS];  const float* self_qkv_b[CIR_LAYERS];    /* [2304,768] q;k;v */
  const void*  self_out_w[CIR_LAYERS];  const float* self_out_b[CIR_LAYERS];
  const float* self_ln_g[CIR_LAYERS];   const float* self_ln_b[CIR_LAYERS];
  const void*  cross_q_w[CIR_LAYERS];   const float* cross_q_b[CIR_LAYERS];
  const void*  cross_kv_w[CIR_LAYERS];  const float* cross_kv_b[CIR_LAYERS];    /* [1536,768] k;v */
  const void*  cross_out_w[CIR_LAYERS]; const float* cross_out_b[CIR_LAYERS];
  const float* cross_ln_g[CIR_LAYERS];  const float* cross_ln_b[CIR_LAYERS];
  const void*  ffn1_w[CIR_LAYERS];      const float* ffn1_b[CIR_LAYERS];
  const void*  ffn2_w[CIR_LAYERS];      const float* ffn2_b[CIR_LAYERS];
  const float* ffn_ln_g[CIR_LAYERS];    const float* ffn_ln_b[CIR_LAYERS];
  const void*  text_proj_w;  const float* text_proj_b;     /* [256,768] */
  const void*  vision_proj_w; const float* vision_proj_b;  /* [256,768] */
} cir_stage1_weights;

/* BLIP_Retrieval.img_txt_fusion(train=False) (src/blip_stage1.py:67-88 -> src/med.py:685-821):
 * per query q the text cross-attends the tokens of gallery image ref_index[q].
 * gallery_tokens act [G,N,768]; ids/mask int32 [Q,L].  Outputs (either may be NULL):
 * z_t act [Q,L,768] (= last_hidden_state, return_raw=True) and q_emb fp32 [Q,256]
 * (= normalize(text_proj(CLS)); normalize_twice=1 reproduces src/validate.py:311). */
size_t cir_stage1_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t L, int64_t N);
int cir_stage1_encode(cir_ctx* ctx, const cir_stage1_weights* w, const void* gallery_tokens,
                      const int32_t* ref_index, const int32_t* ids, const int32_t* mask,
                      int64_t Q, int64_t L, int64_t N, void* z_t, float* q_emb, int normalize_twice,
                      void* workspace, size_t workspace_bytes);

/* normalize(vision_proj(tokens[:,0,:])): src/blip_stage1.py:57.  tokens act [G,N,768] -> g_emb fp32 [G,256].
 * workspace: cir_stage1_workspace_bytes(ctx, G, 1, 1). */
int cir_stage1_gallery_embed(cir_ctx* ctx, const cir_stage1_weights* w, const void* tokens, int64_t G,
                             int64_t N, float* g_emb, void* workspace, size_t workspace_bytes);

/* Stage-II dual-stream encoder weights (src/nlvr_encoder.py:225-476) + cls_head (src/blip_stage2.py:50-54).
 * Host-side packing (see candidate-reranking-cir_b200/engine.py):
 *   self_qkv_w[i]   : [2][2304,768]  stream-major (self0 q;k;v then self1 q;k;v)
 *   cross_kv_w[i]   : [3072,768]     rows K0;V0;K1;V1 (both streams read the SAME candidate tokens)
 *   cross_out_w[i]  : [768,1536]     dense0|dense1 with the merge folded in:
 *                      i <  6: 0.5*[W0 | W1], bias 0.5*(b0+b1)                      (mergeAvg  :257-258)
 *                      i >= 6: [Wm[:, :768] W0 | Wm[:, 768:] W1], bias Wm[b0;b1]+bm  (mergeMLP :252-254)
 *   *_ln_g/_b       : [2][768]       LayerNormA then LayerNormB */
typedef struct cir_stage2_weights {
  const float* word_emb; const float* pos_emb; const float* emb_ln_g; const float* emb_ln_b;
  const void*  self_qkv_w[CIR_LAYERS];  const float* self_qkv_b[CIR_LAYERS];
  const void*  self_out_w[CIR_LAYERS];  const float* self_out_b[CIR_LAYERS];    /* [2][768,768] */
  const float* self_ln_g[CIR_LAYERS];   const float* self_ln_b[CIR_LAYERS];
  const void*  cross_q_w[CIR_LAYERS];   const float* cross_q_b[CIR_LAYERS];     /* [2][768,768] */
  const void*  cross_kv_w[CIR_LAYERS];  const float* cross_kv_b[CIR_LAYERS];
  const void*  cross_out_w[CIR_LAYERS]; const float* cross_out_b[CIR_LAYERS];
  const float* cross_ln_g[CIR_LAYERS];  const float* cross_ln_b[CIR_LAYERS];
  const void*  ffn1_w[CIR_LAYERS];      const float* ffn1_b[CIR_LAYERS];
  const void*  ffn2_w[CIR_LAYERS];      const float* ffn2_b[CIR_LAYERS];
  const float* ffn_ln_g[CIR_LAYERS];    const float* ffn_ln_b[CIR_LAYERS];
  const void*  cls0_w; const float* cls0_b;      /* [768,1536], [768] */
  const float* cls2_w; const float* cls2_b;      /* row 0 of cls_head.2: [768] fp32, [1] */
} cir_stage2_weights;

/* BLIP_NLVR.img_txt_fusion_val (src/blip_stage2.py:101-136 -> src/nlvr_encoder.py:777-909) for a
 * batch of T triplets that share C unique candidate images (candidate-major scheduling: the
 * cross-attention K/V projections -- 69% of the reference's FLOPs, src/nlvr_encoder.py:158-159 --
 * are computed once per candidate and reused by every triplet that names it).
 *   gallery_tokens act [G,N,768]; cand_list int32 [C] gallery rows of the chunk's candidates
 *   z_t act [Q,L,768]; ids/mask int32 [Q,L]
 *   trip_query int32 [T] -> row of z_t/ids/mask; trip_slot int32 [T] -> position in cand_list
 *   attn_work int32 [W,4] / attn_tiles int32 [W',4] optional cross-attention work lists (see
 *   cir_attn_args.work / .tiles; both require trip_slot sorted so that triplets naming the same candidate
 *   are adjacent); attn_tiles_cls: the tile list for one query row per triplet (last layer, CLS only)
 *   scores fp32 [T] (class-0 logit); feats fp32 [T,1536] optional (cat(CLS0,CLS1), nlvr_encoder.py:909) */
size_t cir_stage2_workspace_bytes(const cir_ctx* ctx, int64_t T, int64_t C, int64_t Q, int64_t L, int64_t N);
int cir_stage2_score(cir_ctx* ctx, const cir_stage2_weights* w, const void* gallery_tokens,
                     const int32_t* cand_list, int64_t C, const void* z_t, const int32_t* ids,
                     const int32_t* mask, int64_t Q, int64_t L, int64_t N,
                     const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                     const int32_t* attn_work, int64_t num_attn_work,
                     const int32_t* attn_tiles, int64_t num_attn_tiles,
                     const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                     float* scores, float* feats, void* workspace, size_t workspace_bytes);
/* Layer 0's query-only part for a whole query set (same arithmetic as inside cir_stage2_score, which otherwise repeats it
 * for the unique queries of every chunk): self-attention block of both streams -> a0, cross query projection -> qc0,
 * both act [2][Q*L][768].  Feed them to cir_stage2_score_prefixed, whose trip_query then indexes these Q rows. */
size_t cir_stage2_prefix_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t L);
int cir_stage2_prefix(cir_ctx* ctx, const cir_stage2_weights* w, const void* z_t, const int32_t* ids,
                      const int32_t* mask, int64_t Q, int64_t L, void* a0, void* qc0,
                      void* workspace, size_t workspace_bytes);
int cir_stage2_score_prefixed(cir_ctx* ctx, const cir_stage2_weights* w, const void* gallery_tokens,
                              const int32_t* cand_list, int64_t C, const void* a0, const void* qc0,
                              const int32_t* mask, int64_t Q, int64_t L, int64_t N,
                              const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                              const int32_t* attn_work, int64_t num_attn_work,
                              const int32_t* attn_tiles, int64_t num_attn_tiles,
                              const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                              float* scores, float* feats, void* workspace, size_t workspace_bytes);

/* Resident cross-attention K/V gallery: the K0|V0|K1|V1 projections of every layer depend on the gallery image only
 * (src/nlvr_encoder.py:158-159), so they can be computed once per image and read by every later scoring call.  The blob
 * (cir_stage2_kv_cache_bytes, 256-byte aligned) is owned by the caller; the struct points into it.  Per layer i the cache holds
 * act [rows * N][3072] at kv + i * rows * N * 3072 elements: row (r - row0) * N + t is token t of gallery row r, in exactly the
 * layout cir_stage2_score projects per chunk.  12 * rows * N * 3072 elements: 42.5 MB per image in bf16 at N = 577.
 *   _init records the row range, N and the context's dtype; it enqueues nothing.  Blob too small or misaligned: CIR_EINVAL.
 *   _fill projects gallery rows [first, first + n) (tokens act [n, N, 768]) with the cross_kv_w GEMM of each layer, straight
 *        into the cache; no workspace.  In bf16 contexts it always takes the cta_group::2 pair tile (unless cir_set_gemm_impl
 *        chose CIR_GEMM_TCGEN05_1CTA), so the bytes do not depend on how the rows are sliced into calls.  Rows outside
 *        [row0, row0 + rows) or a cache of the other dtype: CIR_EINVAL. */
typedef struct cir_stage2_kv_cache {
  int64_t row0, rows;     /* gallery rows [row0, row0 + rows) */
  int64_t num_tokens;     /* N (577 at 384 px) */
  int32_t dtype;          /* CIR_DTYPE_* of the context that initialised it */
  void*   kv;             /* act dtype, per layer i: [rows * N][3072] = K0|V0|K1|V1, at kv + i * rows * N * 3072 */
} cir_stage2_kv_cache;
size_t cir_stage2_kv_cache_bytes(const cir_ctx* ctx, int64_t rows, int64_t N);
int    cir_stage2_kv_cache_init(cir_ctx* ctx, void* blob, size_t bytes, int64_t row0, int64_t rows, int64_t N, cir_stage2_kv_cache* out);
int    cir_stage2_kv_cache_fill(cir_ctx* ctx, const cir_stage2_weights* w, cir_stage2_kv_cache* cache,
                                const void* tokens /* act [n, N, 768]: gallery rows first..first+n-1 */, int64_t first, int64_t n);
/* cir_stage2_score / cir_stage2_score_prefixed with the candidates' K/V read from a filled cache: no token gather and no K/V
 * GEMMs, one small kernel maps each triplet to its cache row.  Same chunk description and results; N comes from the cache.
 * PRECONDITION (not checked on the device): every cand_list entry lies in [cache->row0, cache->row0 + cache->rows) and the cache
 * was filled with the K/V weights of `w`.  a0 / qc0: optional cir_stage2_prefix pair (then z_t / ids may be NULL); otherwise z_t
 * and ids are required.  A missing half of the pair, missing z_t / ids or a cache of the other dtype: CIR_EINVAL.  The workspace
 * has no candidate term.  Never synchronises. */
size_t cir_stage2_score_cached_workspace_bytes(const cir_ctx* ctx, int64_t T, int64_t Q, int64_t L, int64_t N);
int cir_stage2_score_cached(cir_ctx* ctx, const cir_stage2_weights* w, const cir_stage2_kv_cache* cache,
                            const int32_t* cand_list, int64_t C, const void* z_t, const int32_t* ids,
                            const void* a0, const void* qc0,
                            const int32_t* mask, int64_t Q, int64_t L,
                            const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                            const int32_t* attn_work, int64_t num_attn_work, const int32_t* attn_tiles, int64_t num_attn_tiles,
                            const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                            float* scores, float* feats, void* workspace, size_t workspace_bytes);

/* Re-ranking a top-K list that lives on the device (e.g. the top_idx of cir_stage1_index_topk) through a filled K/V cache, with no
 * host round trip: every call below only enqueues kernels, never synchronises and never touches host memory, so the whole
 * "stage-I search -> stage-II scores -> re-ranked list" sequence can be captured in one CUDA graph.
 *   _plan_topk plans one call on the device: the candidate-major schedule that the host planner (schedule.plan_chunks as one chunk +
 *        build_attn_tiles) computes for cand int32 [Q,K], T = Q*K <= 16,384, 1 <= L <= 256, a cache of rows [row0, row0 + rows),
 *        rows <= 2^18 - 2.  Outputs (device, T entries each unless noted):
 *          flat_pos    the triplets q*K+k sorted by candidate, ties in q*K+k order (a stable sort)
 *          kv_row      cand[flat_pos] - row0 (the cross-attention's kv_index)
 *          trip_query  flat_pos / K
 *          tiles       int32 [<= T][4] tcgen05 tile list for RB = the smallest power of two >= L (cir_attn_args.tiles)
 *          tiles_cls   int32 [<= T][4] tile list for one query row per triplet (RB = 1)
 *          counts      int32 [3]: number of tiles, number of cls tiles, number of invalid entries
 *        An entry is invalid if it is negative (-1: the padding of a filtered search) or outside the cache's rows.  Invalid entries
 *        sort after every valid one and read kv_row 0; nothing traps.  Bad shapes or a NULL pointer: CIR_EINVAL.
 *   _rerank_cached runs _plan_topk, the stage-II scoring of all T triplets as one chunk through the cache (layer-0 dedup as in
 *        cir_stage2_score; the cross-attentions read the device tile counts), scatters the scores to scores fp32 [Q,K] (-99999.99
 *        at invalid entries, src/validate_stage2.py:123,258), sorts them with cir_rerank_sort into order int32 [Q,K] and, when
 *        ranked is not NULL, writes ranked[q,r] = cand[q, order[q,r]].  z_t act [Q,L,768], ids / mask int32 [Q,L].  counts
 *        (optional, int32 [3]) receives the plan's counts, so a caller can check the invalid entries after the fact.  Scores and
 *        order equal those of the host-planned cir_stage2_score_cached call of the same single chunk, bit for bit.
 *        PRECONDITION (not checked on the device): the cache was filled with the K/V weights of `w`.  Q*K > 16,384, K > 2048,
 *        L > 256, a cache of the other dtype or of more than 2^18 - 2 rows, or a NULL z_t / ids / mask: CIR_EINVAL before anything
 *        is enqueued.  workspace: _rerank_cached_workspace_bytes(Q, K, L, cache->num_tokens). */
int    cir_stage2_plan_topk(cir_ctx* ctx, const int32_t* cand, int64_t Q, int64_t K, int64_t L, int64_t row0, int64_t rows,
                            int32_t* flat_pos, int32_t* kv_row, int32_t* trip_query, int32_t* tiles, int32_t* tiles_cls, int32_t* counts);
size_t cir_stage2_rerank_cached_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t K, int64_t L, int64_t N);
int    cir_stage2_rerank_cached(cir_ctx* ctx, const cir_stage2_weights* w, const cir_stage2_kv_cache* cache, const int32_t* cand,
                                int64_t Q, int64_t K, const void* z_t, const int32_t* ids, const int32_t* mask, int64_t L,
                                float* scores, int32_t* order, int32_t* ranked, int32_t* counts, void* workspace, size_t workspace_bytes);


/* ---- weight packing: reference state_dict tensors -> the packed structs above ------------------------------------------
 * A consumer that does not go through the Python host layer binds the reference's checkpoints here: every field of a
 * cir_*_state is a DEVICE pointer to one fp32 tensor of the reference `state_dict()` (key in the comment; PyTorch [out, in]
 * layout, contiguous).  cir_pack_* casts GEMM weights to the context's activation dtype, stacks twin-stream / q;k;v tensors
 * as the kernels expect, folds the cross-attention output projections and the stream merge into one [768,1536] matrix per
 * layer in fp64 (src/nlvr_encoder.py:250-258), and lays everything out in ONE caller-provided device blob
 * (cir_pack_*_bytes); the returned struct points into the blob.  Work is enqueued on the context's stream; the state
 * tensors may be freed once the stream has passed the call. */
typedef struct cir_vit_state {              /* prefix visual_encoder. (src/vit.py:113-161) */
  const float* patch_w; const float* patch_b;          /* patch_embed.proj.weight [768,3,16,16], .bias [768] */
  const float* cls_token; const float* pos_embed;      /* cls_token [1,1,768], pos_embed [1,N,768] */
  int64_t num_tokens;                                   /* N = (image_size/16)^2 + 1 */
  const float* norm1_g[CIR_LAYERS]; const float* norm1_b[CIR_LAYERS];   /* blocks.i.norm1.{weight,bias} */
  const float* qkv_w[CIR_LAYERS];   const float* qkv_b[CIR_LAYERS];     /* blocks.i.attn.qkv */
  const float* proj_w[CIR_LAYERS];  const float* proj_b[CIR_LAYERS];    /* blocks.i.attn.proj */
  const float* norm2_g[CIR_LAYERS]; const float* norm2_b[CIR_LAYERS];
  const float* fc1_w[CIR_LAYERS];   const float* fc1_b[CIR_LAYERS];     /* blocks.i.mlp.fc1 */
  const float* fc2_w[CIR_LAYERS];   const float* fc2_b[CIR_LAYERS];
  const float* norm_g; const float* norm_b;            /* norm.{weight,bias} */
} cir_vit_state;
size_t cir_pack_vit_bytes(const cir_ctx* ctx, int64_t num_tokens);
int cir_pack_vit_weights(cir_ctx* ctx, const cir_vit_state* sd, void* blob, size_t blob_bytes, cir_vit_weights* out);

typedef struct cir_text_embed_state {       /* text_encoder.embeddings.* */
  const float* word_emb; int64_t vocab_rows;           /* word_embeddings.weight [vocab,768] */
  const float* pos_emb; int64_t pos_rows;              /* position_embeddings.weight [512,768] */
  const float* ln_g; const float* ln_b;                /* LayerNorm.{weight,bias} */
} cir_text_embed_state;

typedef struct cir_stage1_state {           /* BLIP_Retrieval (src/blip_stage1.py:16-46; src/med.py:335-398), layer prefix text_encoder.encoder.layer.i. */
  cir_text_embed_state emb;
  const float* self_q_w[CIR_LAYERS]; const float* self_q_b[CIR_LAYERS];     /* attention.self.query */
  const float* self_k_w[CIR_LAYERS]; const float* self_k_b[CIR_LAYERS];
  const float* self_v_w[CIR_LAYERS]; const float* self_v_b[CIR_LAYERS];
  const float* self_out_w[CIR_LAYERS]; const float* self_out_b[CIR_LAYERS]; /* attention.output.dense */
  const float* self_ln_g[CIR_LAYERS]; const float* self_ln_b[CIR_LAYERS];   /* attention.output.LayerNorm */
  const float* cross_q_w[CIR_LAYERS]; const float* cross_q_b[CIR_LAYERS];   /* crossattention.self.query */
  const float* cross_k_w[CIR_LAYERS]; const float* cross_k_b[CIR_LAYERS];
  const float* cross_v_w[CIR_LAYERS]; const float* cross_v_b[CIR_LAYERS];
  const float* cross_out_w[CIR_LAYERS]; const float* cross_out_b[CIR_LAYERS];
  const float* cross_ln_g[CIR_LAYERS]; const float* cross_ln_b[CIR_LAYERS];
  const float* ffn1_w[CIR_LAYERS]; const float* ffn1_b[CIR_LAYERS];         /* intermediate.dense */
  const float* ffn2_w[CIR_LAYERS]; const float* ffn2_b[CIR_LAYERS];         /* output.dense */
  const float* ffn_ln_g[CIR_LAYERS]; const float* ffn_ln_b[CIR_LAYERS];     /* output.LayerNorm */
  const float* text_proj_w; const float* text_proj_b;                       /* text_proj [256,768] */
  const float* vision_proj_w; const float* vision_proj_b;
} cir_stage1_state;
size_t cir_pack_stage1_bytes(const cir_ctx* ctx, int64_t vocab_rows, int64_t pos_rows);
int cir_pack_stage1_weights(cir_ctx* ctx, const cir_stage1_state* sd, void* blob, size_t blob_bytes, cir_stage1_weights* out);

typedef struct cir_stage2_state {           /* BLIP_NLVR (src/blip_stage2.py:19-54; src/nlvr_encoder.py:225-476); index [s] = stream (self0/self1, dense0/dense1, LayerNormA/B) */
  cir_text_embed_state emb;
  const float* self_q_w[2][CIR_LAYERS]; const float* self_q_b[2][CIR_LAYERS];       /* attention.self{s}.query */
  const float* self_k_w[2][CIR_LAYERS]; const float* self_k_b[2][CIR_LAYERS];
  const float* self_v_w[2][CIR_LAYERS]; const float* self_v_b[2][CIR_LAYERS];
  const float* self_out_w[2][CIR_LAYERS]; const float* self_out_b[2][CIR_LAYERS];   /* attention.output.dense{s} */
  const float* self_ln_g[2][CIR_LAYERS]; const float* self_ln_b[2][CIR_LAYERS];     /* attention.output.LayerNorm{A,B} */
  const float* cross_q_w[2][CIR_LAYERS]; const float* cross_q_b[2][CIR_LAYERS];     /* crossattention.self{s}.query */
  const float* cross_k_w[2][CIR_LAYERS]; const float* cross_k_b[2][CIR_LAYERS];
  const float* cross_v_w[2][CIR_LAYERS]; const float* cross_v_b[2][CIR_LAYERS];
  const float* cross_out_w[2][CIR_LAYERS]; const float* cross_out_b[2][CIR_LAYERS]; /* crossattention.output.dense{s} */
  const float* merge_w[CIR_LAYERS]; const float* merge_b[CIR_LAYERS];               /* crossattention.output.merge_layer [768,1536]; layers 6..11 (NULL below) */
  const float* cross_ln_g[2][CIR_LAYERS]; const float* cross_ln_b[2][CIR_LAYERS];   /* crossattention.output.LayerNorm{A,B} */
  const float* ffn1_w[CIR_LAYERS]; const float* ffn1_b[CIR_LAYERS];
  const float* ffn2_w[CIR_LAYERS]; const float* ffn2_b[CIR_LAYERS];
  const float* ffn_ln_g[CIR_LAYERS]; const float* ffn_ln_b[CIR_LAYERS];
  const float* cls0_w; const float* cls0_b;                                         /* cls_head.0 [768,1536] */
  const float* cls2_w; const float* cls2_b;                                         /* cls_head.2 [2,768], [2] (row 0 is used, src/blip_stage2.py:136) */
} cir_stage2_state;
size_t cir_pack_stage2_bytes(const cir_ctx* ctx, int64_t vocab_rows, int64_t pos_rows);
/* CIR_EINVAL with a message naming merge_layer when a layer >= 6 carries no merge tensors (a BLIP base checkpoint). */
int cir_pack_stage2_weights(cir_ctx* ctx, const cir_stage2_state* sd, void* blob, size_t blob_bytes, cir_stage2_weights* out);

#ifdef __cplusplus
}
#endif
#endif /* CIR_B200_H */
