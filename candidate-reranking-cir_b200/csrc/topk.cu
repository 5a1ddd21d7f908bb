// Re-sort, top-K selection, shard merge and recall counting -- all integer work on composite
// 64-bit keys (order-preserving float bits << 32 | index), so results are bit-exact and ties
// break towards the lowest index (torch.sort(stable=True) order).
//   cir_rerank_sort      argsort(scores, descending)                 src/validate_stage2.py:53,174,190
//   cir_topk_from_dist   K smallest of a distance row, minus `exclude` src/validate.py:58,203-210,257
//   cir_stage1_topk      fused 1 - q @ G^T tiles + running top-K       src/validate.py:57-58,202-203
//   cir_stage1_index_*   the same search over a resident gallery index (built once, grown by appends); _filtered restricts each
//                        query to the rows whose tag shares a bit with its mask
//   cir_topk_merge       merge of per-shard (dist, idx) lists after the NCCL all-gather
//   cir_recall_counts    sum(labels[:, :k]) over sorted labels         src/validate_stage2.py:56-62,178-203
#include <algorithm>
#include "common.cuh"

int cir_gemm_simt_f32(cir_ctx* ctx, const cir_gemm_args* a);   // gemm_simt.cu

namespace {

constexpr int CH = 2048;          // columns per sorted chunk
constexpr int MAXK = 1024;
constexpr int THREADS = 256;
constexpr uint64_t KEY_MAX = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ uint32_t ordered_bits(float f) {
  f = f + 0.0f;                                 // -0.0 -> +0.0 (torch compares them equal)
  uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float from_ordered_bits(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o ^ 0x80000000u) : ~o;
  return __uint_as_float(u);
}

// in-place ascending bitonic sort of n (power of two) keys in shared memory
__device__ void bitonic_sort(uint64_t* s, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int partner = i ^ j;
        if (partner > i) {
          const uint64_t a = s[i], b = s[partner];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { s[i] = b; s[partner] = a; }
        }
      }
    }
  }
  __syncthreads();
}
// s holds a bitonic sequence of n keys -> ascending
__device__ void bitonic_merge(uint64_t* s, int n) {
  for (int j = n >> 1; j > 0; j >>= 1) {
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int partner = i ^ j;
      if (partner > i) {
        const uint64_t a = s[i], b = s[partner];
        if (a > b) { s[i] = b; s[partner] = a; }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(THREADS)
rerank_sort_kernel(const float* __restrict__ scores, int64_t K, int n_pad, int32_t* __restrict__ order) {
  extern __shared__ uint64_t skeys[];
  const int64_t q = blockIdx.x;
  for (int i = threadIdx.x; i < n_pad; i += blockDim.x)
    skeys[i] = (i < K) ? (((uint64_t)(~ordered_bits(scores[q * K + i])) << 32) | (uint32_t)i) : KEY_MAX;
  bitonic_sort(skeys, n_pad);
  for (int i = threadIdx.x; i < K; i += blockDim.x) order[q * K + i] = (int32_t)(skeys[i] & 0xFFFFFFFFu);
}

struct TopkParams {
  const float* vals; int64_t ld; int64_t ncols;     // this call's [Q, ncols] slab
  const int32_t* col_idx;                            // optional explicit global index per (row, col), same ld
  int64_t col_base;                                  // global index of column 0 (when col_idx == NULL)
  const int32_t* exclude;                            // optional per-row excluded global index
  int one_minus;                                     // key value = 1 - v (distance from similarity)
  int K, Kp;                                         // K and K padded to a power of two
  uint64_t* best;                                    // [Q][Kp] running sorted lists
  int init;                                          // 1: start from empty lists
  float* out_dist; int32_t* out_idx;                 // optional final outputs [Q][K]
  // topk_rows_filtered_kernel only: column c of row q is a candidate iff (row_tags[c] & query_masks[q]) != 0 (row_tags starts at
  // this slab's column 0).  Last in the struct, so the other fields keep their offsets in topk_rows_kernel.
  const uint32_t* row_tags; const uint32_t* query_masks;
};

template <bool TAGS>
__device__ __forceinline__ void topk_rows(const TopkParams& p) {
  __shared__ uint64_t sbest[MAXK];
  __shared__ uint64_t schunk[CH];
  __shared__ int s_any;
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  for (int i = tid; i < p.Kp; i += THREADS) sbest[i] = p.init ? KEY_MAX : p.best[q * p.Kp + i];
  const int64_t excl = p.exclude ? (int64_t)p.exclude[q] : -1;
  const float* row = p.vals + q * p.ld;
  const int32_t* irow = p.col_idx ? p.col_idx + q * p.ld : nullptr;
  const uint32_t qmask = TAGS ? p.query_masks[q] : 0u;
  __syncthreads();
  for (int64_t c0 = 0; c0 < p.ncols; c0 += CH) {
    if (tid == 0) s_any = 0;
    __syncthreads();
    const uint64_t thresh = sbest[p.K - 1];            // current K-th best (KEY_MAX while not full)
    // compact the keys that can still enter the top-K (usually a handful once the lists have warmed up)
    for (int i = tid; i < CH; i += THREADS) {
      const int64_t c = c0 + i;
      if (c < p.ncols && (!TAGS || (p.row_tags[c] & qmask) != 0)) {
        float v = row[c];
        if (p.one_minus) v = 1.0f - v;
        const int64_t gi = irow ? (int64_t)irow[c] : p.col_base + c;
        const uint64_t key = ((uint64_t)ordered_bits(v) << 32) | (uint32_t)gi;
        if (gi != excl && key < thresh) schunk[atomicAdd(&s_any, 1)] = key;
      }
    }
    __syncthreads();
    const int n = s_any;
    __syncthreads();                                    // s_any is rewritten at the top of the next chunk
    if (n == 0) continue;                               // nothing in this chunk beats the K-th best
    int m = 32;
    while (m < n) m <<= 1;                              // sort only the survivors (order of arrival is irrelevant: keys are unique)
    for (int i = n + tid; i < m; i += THREADS) schunk[i] = KEY_MAX;
    bitonic_sort(schunk, m);
    // K smallest of (best U survivors): min(best[i], cand[Kp-1-i]) is bitonic
    for (int i = tid; i < p.Kp; i += THREADS) {
      const int j = p.Kp - 1 - i;
      const uint64_t a = sbest[i], b = j < m ? schunk[j] : KEY_MAX;
      sbest[i] = a < b ? a : b;
    }
    bitonic_merge(sbest, p.Kp);
  }
  for (int i = tid; i < p.Kp; i += THREADS) p.best[q * p.Kp + i] = sbest[i];
  if (p.out_idx) {
    for (int i = tid; i < p.K; i += THREADS) {
      const uint64_t key = sbest[i];
      p.out_idx[q * p.K + i] = (key == KEY_MAX) ? -1 : (int32_t)(key & 0xFFFFFFFFu);
      p.out_dist[q * p.K + i] = (key == KEY_MAX) ? INFINITY : from_ordered_bits((uint32_t)(key >> 32));
    }
  }
}
__global__ void __launch_bounds__(THREADS) topk_rows_kernel(TopkParams p) { topk_rows<false>(p); }
__global__ void __launch_bounds__(THREADS) topk_rows_filtered_kernel(TopkParams p) { topk_rows<true>(p); }

// Merge of P per-shard lists in ONE pass: the P*K composite keys of a query (<= 8192) are sorted once in shared memory and the first K
// leave.  Keys are unique across shards (disjoint global indices), so the result equals the sequential merge bit for bit.
__global__ void __launch_bounds__(THREADS)
merge_lists_kernel(const float* __restrict__ dist_in, const int32_t* __restrict__ idx_in, int P, int64_t Q, int K, int n_pad,
                   float* __restrict__ out_dist, int32_t* __restrict__ out_idx) {
  extern __shared__ uint64_t skeys[];
  const int64_t q = blockIdx.x;
  for (int i = threadIdx.x; i < n_pad; i += THREADS) {
    uint64_t key = KEY_MAX;
    if (i < P * K) {
      const int s = i / K, j = i - s * K;
      const int32_t gi = idx_in[((int64_t)s * Q + q) * K + j];
      if (gi >= 0) key = ((uint64_t)ordered_bits(dist_in[((int64_t)s * Q + q) * K + j]) << 32) | (uint32_t)gi;   // -1: empty slot of a short shard
    }
    skeys[i] = key;
  }
  bitonic_sort(skeys, n_pad);
  for (int i = threadIdx.x; i < K; i += THREADS) {
    const uint64_t key = skeys[i];
    out_idx[q * K + i] = (key == KEY_MAX) ? -1 : (int32_t)(key & 0xFFFFFFFFu);
    out_dist[q * K + i] = (key == KEY_MAX) ? INFINITY : from_ordered_bits((uint32_t)(key >> 32));
  }
}

struct RecallParams { int32_t ks[16]; int32_t num; };
__global__ void recall_counts_kernel(const uint8_t* __restrict__ labels, const int32_t* __restrict__ order, int64_t Q, int64_t K,
                                     RecallParams rp, unsigned long long* __restrict__ hits) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  for (int64_t i = 0; i < K; i++) {
    if (labels[q * K + order[q * K + i]]) {
      for (int j = 0; j < rp.num; j++)
        if (i < rp.ks[j]) atomicAdd(&hits[j], 1ull);
    }
  }
}

// One thread per query: fp32 distances 1 - q . g[member] of P <= 32 named gallery rows (the dot product accumulates k = 0..255 in
// order with fmaf, exactly like the similarity tiles of cir_stage1_topk), then the members' slots ranked by (distance, gallery index).
__global__ void rank_members_kernel(const float* __restrict__ q_emb, const float* __restrict__ g_emb, const int32_t* __restrict__ members,
                                    int64_t Q, int P, float* __restrict__ out_dist, int32_t* __restrict__ out_order) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  uint64_t keys[32];
  const float4* qv = reinterpret_cast<const float4*>(q_emb + q * CIR_EMBED);
  for (int j = 0; j < P; j++) {
    const int32_t gi = members[q * P + j];
    const float4* gv = reinterpret_cast<const float4*>(g_emb + (int64_t)gi * CIR_EMBED);
    float acc = 0.f;
    for (int k = 0; k < CIR_EMBED / 4; k++) {
      const float4 a = qv[k], b = __ldg(gv + k);
      acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
    }
    const float d = 1.0f - acc;
    out_dist[q * P + j] = d;
    keys[j] = ((uint64_t)ordered_bits(d) << 32) | (uint32_t)gi;
  }
  // rank r of slot j = number of members with a smaller key (equal gallery rows keep slot order)
  for (int j = 0; j < P; j++) {
    int r = 0;
    for (int i = 0; i < P; i++) r += (keys[i] < keys[j]) || (keys[i] == keys[j] && i < j);
    out_order[q * P + r] = j;
  }
}

inline int pow2_at_least(int64_t k) { int p = 1; while (p < k) p <<= 1; return p; }

}  // namespace

extern "C" int cir_rerank_sort(cir_ctx* ctx, const float* scores, int64_t Q, int64_t K, int32_t* order) {
  CIR_ENTER(ctx);
  if (Q == 0 || K == 0) return CIR_OK;
  CIR_CHECK_ARG(K <= 2048, "rerank_sort: K=%lld > 2048", (long long)K);
  const int n_pad = pow2_at_least(K);
  rerank_sort_kernel<<<(unsigned)Q, THREADS, n_pad * sizeof(uint64_t), ctx->stream>>>(scores, K, n_pad, order);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

extern "C" size_t cir_topk_workspace_bytes(int64_t Q, int64_t G, int64_t K) {
  (void)G;
  return align_up((size_t)Q * pow2_at_least(K) * sizeof(uint64_t), 256);
}

extern "C" int cir_topk_from_dist(cir_ctx* ctx, const float* dist, int64_t Q, int64_t G, int64_t ldd,
                                  const int32_t* exclude, int64_t col_offset, int64_t K,
                                  float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(K >= 1 && K <= MAXK, "topk: K=%lld out of range [1,%d]", (long long)K, MAXK);
  if (workspace_bytes < cir_topk_workspace_bytes(Q, G, K)) { cir_set_error("topk: workspace too small"); return CIR_EWORKSPACE; }
  TopkParams p{};
  p.vals = dist; p.ld = ldd; p.ncols = G; p.col_idx = nullptr; p.col_base = col_offset; p.exclude = exclude;
  p.one_minus = 0; p.K = (int)K; p.Kp = pow2_at_least(K); p.best = (uint64_t*)workspace; p.init = 1;
  p.out_dist = top_dist; p.out_idx = top_idx;
  topk_rows_kernel<<<(unsigned)Q, THREADS, 0, ctx->stream>>>(p);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

static const int64_t kSimChunk = 8192;    // gallery columns per similarity tile

static size_t stage1_fp32_workspace_bytes(int64_t Q, int64_t G, int64_t K) {
  const int64_t gc = G < kSimChunk ? G : kSimChunk;
  return cir_topk_workspace_bytes(Q, G, K) + align_up((size_t)Q * (size_t)gc * sizeof(float), 256);
}
extern "C" size_t cir_stage1_topk_workspace_bytes(int64_t Q, int64_t G, int64_t K) {
  // the tensor-core path (large galleries, bf16 contexts) and the fp32 path use the same buffer one after the other
  const size_t a = stage1_fp32_workspace_bytes(Q, G, K);
  const size_t b = (G >= 16384 && K >= 1 && K <= MAXK) ? cir_stage1_topk_tc_workspace_bytes(Q, G, K) : 0;
  return a > b ? a : b;
}

// fp32 CUDA-core path: similarity tiles of kSimChunk columns + running top-K (workspace: stage1_fp32_workspace_bytes).
// row_tags [G] / query_masks [Q] (both or neither): query q ranks only the rows with (row_tags[r] & query_masks[q]) != 0.
static int stage1_fp32(cir_ctx* ctx, const float* q_emb, const float* g_emb, int64_t Q, int64_t G, const int32_t* exclude, int64_t col_offset,
                       int64_t K, float* top_dist, int32_t* top_idx, void* workspace, const uint32_t* row_tags = nullptr,
                       const uint32_t* query_masks = nullptr) {
  uint64_t* best = (uint64_t*)workspace;
  float* sim = (float*)((char*)workspace + cir_topk_workspace_bytes(Q, G, K));
  const int64_t gc = G < kSimChunk ? G : kSimChunk;
  if (G == 0) {   // empty shard: emit empty lists
    TopkParams p{};
    p.vals = sim; p.ld = 0; p.ncols = 0; p.K = (int)K; p.Kp = pow2_at_least(K); p.best = best; p.init = 1;
    p.out_dist = top_dist; p.out_idx = top_idx;
    topk_rows_kernel<<<(unsigned)Q, THREADS, 0, ctx->stream>>>(p);
    CIR_LAUNCH_CHECK(ctx);
    return CIR_OK;
  }
  for (int64_t g0 = 0; g0 < G; g0 += gc) {
    const int64_t n = (G - g0) < gc ? (G - g0) : gc;
    cir_gemm_args ga{};
    ga.A = q_emb; ga.W = g_emb + g0 * CIR_EMBED; ga.C = sim;
    ga.M = Q; ga.N = n; ga.K = CIR_EMBED; ga.lda = CIR_EMBED; ga.ldw = CIR_EMBED; ga.ldc = gc;
    ga.batch = 1; ga.act = CIR_ACT_NONE; ga.c_f32 = 1;
    CIR_TRY(cir_gemm_simt_f32(ctx, &ga));      // true fp32 similarities, like the reference's fp32 matmul
    TopkParams p{};
    p.vals = sim; p.ld = gc; p.ncols = n; p.col_idx = nullptr; p.col_base = col_offset + g0; p.exclude = exclude;
    p.one_minus = 1; p.K = (int)K; p.Kp = pow2_at_least(K); p.best = best; p.init = (g0 == 0);
    const bool last = g0 + gc >= G;
    p.out_dist = last ? top_dist : nullptr; p.out_idx = last ? top_idx : nullptr;
    if (row_tags) {
      p.row_tags = row_tags + g0; p.query_masks = query_masks;
      topk_rows_filtered_kernel<<<(unsigned)Q, THREADS, 0, ctx->stream>>>(p);
    } else {
      topk_rows_kernel<<<(unsigned)Q, THREADS, 0, ctx->stream>>>(p);
    }
    CIR_LAUNCH_CHECK(ctx);
  }
  return CIR_OK;
}

extern "C" int cir_stage1_topk(cir_ctx* ctx, const float* q_emb, const float* g_emb, int64_t Q, int64_t G,
                               const int32_t* exclude, int64_t col_offset, int64_t K,
                               float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(K >= 1 && K <= MAXK, "stage1_topk: K=%lld out of range [1,%d]", (long long)K, MAXK);
  if (workspace_bytes < cir_stage1_topk_workspace_bytes(Q, G, K)) { cir_set_error("stage1_topk: workspace too small"); return CIR_EWORKSPACE; }
  // large gallery: candidate filter on the tensor cores + exact fp32 re-check (bit-identical results); queries whose candidate
  // list overflows (adversarial gallery order / thousands of near-duplicates) get an exact scan on the device
  if (cir_stage1_topk_tc_supported(ctx, Q, G, K))
    return cir_stage1_topk_tc(ctx, q_emb, g_emb, Q, G, exclude, col_offset, K, top_dist, top_idx, workspace, workspace_bytes);
  return stage1_fp32(ctx, q_emb, g_emb, Q, G, exclude, col_offset, K, top_dist, top_idx, workspace);
}

// ---- resident stage-I index: blob = [capacity,256] fp32 rows | [capacity,256] bf16 copy (bf16 contexts) | gmax (256 B)
static const int64_t kTcMinRows = 16384;    // cir_stage1_topk_tc_supported's gallery threshold

extern "C" size_t cir_stage1_index_bytes(const cir_ctx* ctx, int64_t capacity) {
  if (!ctx || capacity < 0) return 0;
  const size_t b = ctx->dtype == CIR_DTYPE_BF16 ? align_up((size_t)capacity * CIR_EMBED * 2, 256) : 0;
  return align_up((size_t)capacity * CIR_EMBED * 4, 256) + b + 256;
}

extern "C" int cir_stage1_index_init(cir_ctx* ctx, void* blob, size_t bytes, int64_t capacity, cir_stage1_index* out) {
  CIR_CHECK_ARG(ctx && out && blob, "stage1_index_init: null argument");
  CIR_CHECK_ARG(capacity >= 0 && capacity < (1ll << 31), "stage1_index_init: capacity=%lld out of range [0,2^31)", (long long)capacity);
  CIR_CHECK_ARG(((uintptr_t)blob & 255) == 0, "stage1_index_init: blob must be 256-byte aligned");
  const size_t need = cir_stage1_index_bytes(ctx, capacity);
  if (bytes < need) { cir_set_error("stage1_index_init: blob %zu < %zu bytes", bytes, need); return CIR_EWORKSPACE; }
  CIR_ENTER(ctx);
  char* base = (char*)blob;
  const size_t f32 = align_up((size_t)capacity * CIR_EMBED * 4, 256);
  out->capacity = capacity;
  out->rows = 0;
  out->g_f32 = (float*)base;
  out->g_bf16 = ctx->dtype == CIR_DTYPE_BF16 ? (void*)(base + f32) : nullptr;
  out->gmax = (uint32_t*)(base + need - 256);
  CIR_CUDA(cudaMemsetAsync(out->gmax, 0, 2 * sizeof(uint32_t), ctx->stream));
  return CIR_OK;
}

extern "C" int cir_stage1_index_add(cir_ctx* ctx, cir_stage1_index* index, const float* g_emb, int64_t n) {
  CIR_CHECK_ARG(ctx && index && (g_emb || n == 0), "stage1_index_add: null argument");
  CIR_CHECK_ARG(n >= 0 && index->rows + n <= index->capacity, "stage1_index_add: %lld rows + %lld exceed the capacity %lld",
                (long long)index->rows, (long long)n, (long long)index->capacity);
  if (n == 0) return CIR_OK;
  CIR_ENTER(ctx);
  float* dst = index->g_f32 + index->rows * CIR_EMBED;
  CIR_CUDA(cudaMemcpyAsync(dst, g_emb, (size_t)n * CIR_EMBED * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  if (index->g_bf16) CIR_TRY(cir_stage1_tc_convert(ctx, dst, n, (bf16*)index->g_bf16 + index->rows * CIR_EMBED, index->gmax));
  index->rows += n;
  return CIR_OK;
}

extern "C" size_t cir_stage1_index_topk_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* index, int64_t Q, int64_t K) {
  (void)ctx;
  if (!index || Q < 0 || K < 1 || K > MAXK) return 0;
  // sized for every row count up to the capacity, so that a workspace stays valid while the index grows
  const size_t a = stage1_fp32_workspace_bytes(Q, index->capacity, K);
  const size_t b = (index->g_bf16 && index->capacity >= kTcMinRows) ? cir_stage1_tc_search_bytes(Q, K) : 0;
  return a > b ? a : b;
}

// cir_stage1_index_topk (row_tags == query_masks == NULL) and cir_stage1_index_topk_filtered; `fn` names the entry point in errors
static int index_topk(const char* fn, cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q, const uint32_t* row_tags,
                      const uint32_t* query_masks, const int32_t* exclude, int64_t col_offset, int64_t K, float* top_dist, int32_t* top_idx,
                      int32_t* exact_rows, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(K >= 1 && K <= MAXK, "%s: K=%lld out of range [1,%d]", fn, (long long)K, MAXK);
  const size_t need = cir_stage1_index_topk_workspace_bytes(ctx, index, Q, K);
  if (workspace_bytes < need) { cir_set_error("%s: workspace %zu < %zu bytes", fn, workspace_bytes, need); return CIR_EWORKSPACE; }
  const int64_t G = index->rows;
  if (index->g_bf16 && cir_stage1_topk_tc_supported(ctx, Q, G, K))
    return cir_stage1_tc_search(ctx, q_emb, Q, index->g_f32, (const bf16*)index->g_bf16, G, index->gmax, row_tags, query_masks, exclude,
                                col_offset, K, top_dist, top_idx, exact_rows, workspace, workspace_bytes);
  if (exact_rows) CIR_CUDA(cudaMemsetAsync(exact_rows, 0, (size_t)Q * sizeof(int32_t), ctx->stream));
  return stage1_fp32(ctx, q_emb, index->g_f32, Q, G, exclude, col_offset, K, top_dist, top_idx, workspace, row_tags, query_masks);
}

extern "C" int cir_stage1_index_topk(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q, const int32_t* exclude,
                                     int64_t col_offset, int64_t K, float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                                     void* workspace, size_t workspace_bytes) {
  CIR_CHECK_ARG(ctx && index, "stage1_index_topk: null argument");
  return index_topk("stage1_index_topk", ctx, index, q_emb, Q, nullptr, nullptr, exclude, col_offset, K, top_dist, top_idx, exact_rows,
                    workspace, workspace_bytes);
}

extern "C" int cir_stage1_index_topk_filtered(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q,
                                              const uint32_t* row_tags, const uint32_t* query_masks, const int32_t* exclude,
                                              int64_t col_offset, int64_t K, float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                                              void* workspace, size_t workspace_bytes) {
  CIR_CHECK_ARG(ctx && index, "stage1_index_topk_filtered: null argument");
  CIR_CHECK_ARG(row_tags && query_masks, "stage1_index_topk_filtered: row_tags and query_masks are required (all bits set = no filter)");
  return index_topk("stage1_index_topk_filtered", ctx, index, q_emb, Q, row_tags, query_masks, exclude, col_offset, K, top_dist, top_idx,
                    exact_rows, workspace, workspace_bytes);
}

// ---- compaction and permanent row ids.  Compaction is stable (kept rows keep their order), so the ids stay strictly increasing along
// the physical rows and a search over physical rows ranks ties exactly as a search over ids would.
namespace {

constexpr int CPT_ROWS = 1024;            // rows per block of the count / gather kernels (4 consecutive rows per thread)

__device__ __forceinline__ int kept_row(const uint32_t* __restrict__ tags, int64_t r, int64_t n, uint32_t mask) {
  return r < n && (tags[r] & mask) != 0;
}

// block b: how many rows of [b * CPT_ROWS, (b + 1) * CPT_ROWS) are kept
__global__ void __launch_bounds__(THREADS)
compact_count_kernel(const uint32_t* __restrict__ tags, int64_t n, uint32_t mask, int32_t* __restrict__ block_count) {
  __shared__ int s_count;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const int64_t r0 = (int64_t)blockIdx.x * CPT_ROWS;
  int c = 0;
  for (int i = threadIdx.x; i < CPT_ROWS; i += THREADS) c += kept_row(tags, r0 + i, n, mask);
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_count, c);
  __syncthreads();
  if (threadIdx.x == 0) block_count[blockIdx.x] = s_count;
}

// one block: block_off[b] = sum of block_count[0..b), block_off[nb] = the kept total
__global__ void __launch_bounds__(1024)
compact_scan_kernel(const int32_t* __restrict__ block_count, int64_t nb, int32_t* __restrict__ block_off) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) s_carry = 0;
  for (int64_t b0 = 0; b0 < nb; b0 += 1024) {
    const int64_t b = b0 + tid;
    const int v = b < nb ? block_count[b] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    if (w == 0) {
      const int t = s_warp[lane];
      int x = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += u; }
      s_warp[lane] = x - t;                                  // warps before this one
    }
    __syncthreads();
    const int excl = s_carry + s_warp[w] + incl - v;
    if (b < nb) block_off[b] = excl;
    __syncthreads();                                         // everyone has read s_carry / s_warp
    if (tid == 1023) s_carry = excl + v;
    __syncthreads();
  }
  if (tid == 0) block_off[nb] = s_carry;
}

// Kept row r (in order) -> dst row block_off[b] + (kept rows before it in its block): the 1 KB fp32 row, its tag and its id
// (src_ids[r], or r when src_ids is NULL).  One warp copies a row with two 16-byte loads per lane.
__global__ void __launch_bounds__(THREADS)
compact_gather_kernel(const float* __restrict__ src, const uint32_t* __restrict__ src_tags, const int32_t* __restrict__ src_ids, int64_t n,
                      uint32_t mask, const int32_t* __restrict__ block_off, float* __restrict__ dst, uint32_t* __restrict__ dst_tags,
                      int32_t* __restrict__ dst_ids) {
  __shared__ int s_dst[CPT_ROWS];
  __shared__ int s_warp[THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t b0 = (int64_t)blockIdx.x * CPT_ROWS;
  int k[4], c = 0;
#pragma unroll
  for (int j = 0; j < 4; j++) { k[j] = kept_row(src_tags, b0 + 4 * tid + j, n, mask); c += k[j]; }
  int incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  int d = block_off[blockIdx.x] + incl - c;
  for (int i = 0; i < w; i++) d += s_warp[i];
#pragma unroll
  for (int j = 0; j < 4; j++) s_dst[4 * tid + j] = k[j] ? d++ : -1;
  __syncthreads();
  for (int i = w; i < CPT_ROWS; i += THREADS / 32) {
    const int to = s_dst[i];
    if (to < 0) continue;
    const int64_t r = b0 + i;
    const float4* s4 = reinterpret_cast<const float4*>(src + r * CIR_EMBED);
    float4* d4 = reinterpret_cast<float4*>(dst + (int64_t)to * CIR_EMBED);
    const float4 a = __ldg(s4 + lane), b = __ldg(s4 + lane + 32);
    d4[lane] = a;
    d4[lane + 32] = b;
    if (lane == 0) { dst_tags[to] = src_tags[r]; dst_ids[to] = src_ids ? src_ids[r] : (int32_t)r; }
  }
}

// exclude[q] (col_offset + id, -1 = none) -> the physical row holding that id (binary search of the strictly increasing row_ids), -1 when
// no row holds it
__global__ void map_exclude_kernel(const int32_t* __restrict__ exclude, int64_t Q, const int32_t* __restrict__ row_ids, int64_t rows,
                                   int64_t col_offset, int32_t* __restrict__ out) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const int64_t id = exclude[q] < 0 ? -1 : (int64_t)exclude[q] - col_offset;
  int32_t p = -1;
  if (id >= 0) {
    int64_t lo = 0, hi = rows;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if ((int64_t)row_ids[mid] < id) lo = mid + 1; else hi = mid;
    }
    if (lo < rows && (int64_t)row_ids[lo] == id) p = (int32_t)lo;
  }
  out[q] = p;
}

// physical rows of a finished search -> col_offset + id; -1 (empty slot) passes through
__global__ void map_ids_kernel(int32_t* __restrict__ idx, int64_t n, const int32_t* __restrict__ row_ids, int64_t col_offset) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t v = idx[i];
    if (v >= 0) idx[i] = (int32_t)(col_offset + row_ids[v]);
  }
}

}  // namespace

extern "C" size_t cir_stage1_index_compact_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* src) {
  (void)ctx;
  if (!src) return 0;
  const int64_t nb = (src->rows + CPT_ROWS - 1) / CPT_ROWS;
  return align_up((size_t)nb * 4, 256) + align_up((size_t)(nb + 1) * 4, 256);
}

extern "C" int cir_stage1_index_compact(cir_ctx* ctx, const cir_stage1_index* src, const uint32_t* src_tags, const int32_t* src_ids,
                                        uint32_t keep_mask, cir_stage1_index* dst, uint32_t* dst_tags, int32_t* dst_ids, void* workspace,
                                        size_t workspace_bytes) {
  CIR_CHECK_ARG(ctx && src && dst && dst_tags && dst_ids, "stage1_index_compact: null argument");
  CIR_CHECK_ARG(src_tags || src->rows == 0, "stage1_index_compact: src_tags is required");
  CIR_CHECK_ARG(dst->rows == 0, "stage1_index_compact: dst holds %lld rows; it must be an empty index", (long long)dst->rows);
  const bool bf = ctx->dtype == CIR_DTYPE_BF16;
  CIR_CHECK_ARG((src->g_bf16 != nullptr) == bf && (dst->g_bf16 != nullptr) == bf,
                "stage1_index_compact: src and dst must both be indexes of the context's dtype (%s)", bf ? "bf16" : "fp32");
  // a blob spans [g_f32, gmax + 256): a parallel stable compaction in place would read rows other blocks already overwrote
  const char *s_lo = (const char*)src->g_f32, *s_hi = (const char*)src->gmax + 256;
  const char *d_lo = (const char*)dst->g_f32, *d_hi = (const char*)dst->gmax + 256;
  CIR_CHECK_ARG(s_hi <= d_lo || d_hi <= s_lo, "stage1_index_compact: src and dst blobs overlap; compact into a different blob");
  const size_t need = cir_stage1_index_compact_workspace_bytes(ctx, src);
  if (workspace_bytes < need) { cir_set_error("stage1_index_compact: workspace %zu < %zu bytes", workspace_bytes, need); return CIR_EWORKSPACE; }
  CIR_ENTER(ctx);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  CIR_CUDA(cudaStreamIsCapturing(ctx->stream, &cs));
  CIR_CHECK_ARG(cs == cudaStreamCaptureStatusNone, "stage1_index_compact: synchronises the stream and cannot be captured in a CUDA graph");
  const int64_t n = src->rows, nb = (n + CPT_ROWS - 1) / CPT_ROWS;
  int32_t* count = (int32_t*)workspace;
  int32_t* off = (int32_t*)((char*)workspace + align_up((size_t)nb * 4, 256));
  int32_t kept = 0;
  if (n > 0) {
    compact_count_kernel<<<(unsigned)nb, THREADS, 0, ctx->stream>>>(src_tags, n, keep_mask, count);
    CIR_LAUNCH_CHECK(ctx);
    compact_scan_kernel<<<1, 1024, 0, ctx->stream>>>(count, nb, off);
    CIR_LAUNCH_CHECK(ctx);
    CIR_CUDA(cudaMemcpyAsync(&kept, off + nb, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CIR_CUDA(cudaStreamSynchronize(ctx->stream));             // the one synchronisation: dst->rows is a host-side count
  }
  CIR_CHECK_ARG(kept <= dst->capacity, "stage1_index_compact: %lld kept rows exceed the capacity %lld of dst (nothing written)",
                (long long)kept, (long long)dst->capacity);
  CIR_CUDA(cudaMemsetAsync(dst->gmax, 0, 2 * sizeof(uint32_t), ctx->stream));
  if (kept > 0) {
    compact_gather_kernel<<<(unsigned)nb, THREADS, 0, ctx->stream>>>(src->g_f32, src_tags, src_ids, n, keep_mask, off, dst->g_f32, dst_tags,
                                                                      dst_ids);
    CIR_LAUNCH_CHECK(ctx);
    // the bf16 copy and the maxima of the kept rows only, as cir_stage1_index_add of those rows builds them
    if (dst->g_bf16) CIR_TRY(cir_stage1_tc_convert(ctx, dst->g_f32, kept, (bf16*)dst->g_bf16, dst->gmax));
  }
  dst->rows = kept;
  return CIR_OK;
}

extern "C" size_t cir_stage1_index_topk_ids_workspace_bytes(const cir_ctx* ctx, const cir_stage1_index* index, int64_t Q, int64_t K) {
  const size_t s = cir_stage1_index_topk_workspace_bytes(ctx, index, Q, K);
  return s ? align_up(s, 256) + align_up((size_t)Q * sizeof(int32_t), 256) : 0;
}

extern "C" int cir_stage1_index_topk_ids(cir_ctx* ctx, const cir_stage1_index* index, const float* q_emb, int64_t Q, const int32_t* row_ids,
                                         int64_t id_end, const uint32_t* row_tags, const uint32_t* query_masks, const int32_t* exclude,
                                         int64_t col_offset, int64_t K, float* top_dist, int32_t* top_idx, int32_t* exact_rows,
                                         void* workspace, size_t workspace_bytes) {
  CIR_CHECK_ARG(ctx && index, "stage1_index_topk_ids: null argument");
  CIR_CHECK_ARG(row_ids || index->rows == 0, "stage1_index_topk_ids: row_ids is required");
  CIR_CHECK_ARG((row_tags == nullptr) == (query_masks == nullptr),
                "stage1_index_topk_ids: row_tags and query_masks are both NULL (unfiltered) or both set (filtered)");
  CIR_CHECK_ARG(col_offset >= 0 && id_end >= index->rows && col_offset + id_end <= (1ll << 31),
                "stage1_index_topk_ids: col_offset %lld + ids up to %lld do not fit int32 indices", (long long)col_offset,
                (long long)id_end - 1);
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(K >= 1 && K <= MAXK, "stage1_index_topk_ids: K=%lld out of range [1,%d]", (long long)K, MAXK);
  const size_t need = cir_stage1_index_topk_ids_workspace_bytes(ctx, index, Q, K);
  if (workspace_bytes < need) { cir_set_error("stage1_index_topk_ids: workspace %zu < %zu bytes", workspace_bytes, need); return CIR_EWORKSPACE; }
  const size_t search = align_up(cir_stage1_index_topk_workspace_bytes(ctx, index, Q, K), 256);
  int32_t* ex = nullptr;
  if (exclude) {
    ex = (int32_t*)((char*)workspace + search);
    map_exclude_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, ctx->stream>>>(exclude, Q, row_ids, index->rows, col_offset, ex);
    CIR_LAUNCH_CHECK(ctx);
  }
  CIR_TRY(index_topk("stage1_index_topk_ids", ctx, index, q_emb, Q, row_tags, query_masks, ex, 0, K, top_dist, top_idx, exact_rows,
                     workspace, search));
  const int64_t n = Q * K;
  const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->num_sms * 8);
  map_ids_kernel<<<blocks, 256, 0, ctx->stream>>>(top_idx, n, row_ids, col_offset);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

__global__ void divide_rows_kernel(float* __restrict__ x, int64_t n, float d) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = x[i] / d;
}

extern "C" int cir_stage1_logits(cir_ctx* ctx, const float* q_emb, const float* t_emb, int64_t Q, int64_t G, float temp, float* logits) {
  CIR_ENTER(ctx);
  if (Q == 0 || G == 0) return CIR_OK;
  CIR_CHECK_ARG(temp != 0.f, "stage1_logits: temp must be non-zero");
  cir_gemm_args ga{};
  ga.A = q_emb; ga.W = t_emb; ga.C = logits;
  ga.M = Q; ga.N = G; ga.K = CIR_EMBED; ga.lda = CIR_EMBED; ga.ldw = CIR_EMBED; ga.ldc = G;
  ga.batch = 1; ga.act = CIR_ACT_NONE; ga.c_f32 = 1;
  CIR_TRY(cir_gemm_simt_f32(ctx, &ga));
  const int64_t n = Q * G;
  const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->num_sms * 8);
  divide_rows_kernel<<<blocks, 256, 0, ctx->stream>>>(logits, n, temp);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

extern "C" int cir_stage1_rank_members(cir_ctx* ctx, const float* q_emb, const float* g_emb, const int32_t* members, int64_t Q,
                                       int64_t P, float* member_dist, int32_t* member_order) {
  CIR_ENTER(ctx);
  if (Q == 0 || P == 0) return CIR_OK;
  CIR_CHECK_ARG(P >= 1 && P <= 32, "rank_members: P=%lld out of range [1,32]", (long long)P);
  CIR_CHECK_ARG(q_emb && g_emb && members && member_dist && member_order, "rank_members: null argument");
  rank_members_kernel<<<(unsigned)((Q + 127) / 128), 128, 0, ctx->stream>>>(q_emb, g_emb, members, Q, (int)P, member_dist, member_order);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

extern "C" int cir_topk_merge(cir_ctx* ctx, const float* dist_in, const int32_t* idx_in, int64_t P, int64_t Q,
                              int64_t K, float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0 || P == 0) return CIR_OK;
  CIR_CHECK_ARG(K >= 1 && K <= MAXK, "topk_merge: K=%lld out of range", (long long)K);
  if (workspace_bytes < cir_topk_workspace_bytes(Q, 0, K)) { cir_set_error("topk_merge: workspace too small"); return CIR_EWORKSPACE; }
  if (P * K <= 8192) {                                   // all lists of a query fit one shared-memory sort: a single launch
    const int n_pad = pow2_at_least(P * K);
    if (!(ctx->func_attr_mask & (1u << 7))) {
      CIR_CUDA(cudaFuncSetAttribute(merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * 8));
      ctx->func_attr_mask |= 1u << 7;
    }
    merge_lists_kernel<<<(unsigned)Q, THREADS, (size_t)n_pad * 8, ctx->stream>>>(dist_in, idx_in, (int)P, Q, (int)K, n_pad, top_dist, top_idx);
    CIR_LAUNCH_CHECK(ctx);
    return CIR_OK;
  }
  uint64_t* scratch = (uint64_t*)workspace;
  for (int64_t s = 0; s < P; s++) {
    TopkParams p{};
    p.vals = dist_in + s * Q * K; p.ld = K; p.ncols = K; p.col_idx = idx_in + s * Q * K; p.col_base = 0;
    p.exclude = nullptr; p.one_minus = 0; p.K = (int)K; p.Kp = pow2_at_least(K); p.best = scratch; p.init = (s == 0);
    p.out_dist = (s == P - 1) ? top_dist : nullptr; p.out_idx = (s == P - 1) ? top_idx : nullptr;
    topk_rows_kernel<<<(unsigned)Q, THREADS, 0, ctx->stream>>>(p);
    CIR_LAUNCH_CHECK(ctx);
  }
  return CIR_OK;
}

extern "C" int cir_recall_counts(cir_ctx* ctx, const uint8_t* labels, const int32_t* order, int64_t Q, int64_t K,
                                 const int32_t* ks_host, int32_t num_ks, int64_t* hits) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(num_ks >= 1 && num_ks <= 16, "recall_counts: num_ks=%d out of range [1,16]", num_ks);
  RecallParams rp{};
  rp.num = num_ks;
  for (int i = 0; i < num_ks; i++) rp.ks[i] = ks_host[i];
  CIR_CUDA(cudaMemsetAsync(hits, 0, sizeof(int64_t) * num_ks, ctx->stream));
  if (Q == 0) return CIR_OK;
  recall_counts_kernel<<<(unsigned)((Q + 127) / 128), 128, 0, ctx->stream>>>(labels, order, Q, K, rp, (unsigned long long*)hits);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}
