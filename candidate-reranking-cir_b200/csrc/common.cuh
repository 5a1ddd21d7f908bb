// Shared host/device helpers for libcir_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>

#include "../../include/cir_b200.h"

typedef __nv_bfloat16 bf16;

struct cir_ctx {
  int device;
  int dtype;            // CIR_DTYPE_*
  int gemm_impl;        // CIR_GEMM_*
  int attn_impl;        // 0 = auto (tensor cores in bf16 mode), 1 = force the CUDA-core kernel
  int gemm_pair;        // 1 = allow cta_group::2 pair tiles for large GEMMs (default)
  int gemm_force_pair;  // 1 = take the pair tile whenever gemm_pair allows it, whatever M is (stage-II K/V cache fill)
  int prune_last;       // 1 = stage II computes the last layer for the CLS rows only (default)
  int gemm_tma_store;   // 1 = bf16 GEMM outputs leave through TMA bulk tensor stores (default)
  int fuse_qkv;         // 1 = QKV projection + masked text self-attention as one kernel where eligible (default)
  int stage1_tc;        // 1 = stage-I top-K over large galleries filters on the tensor cores, exact fp32 re-check of the survivors (default)
  int dedup_first;      // 1 = stage II runs layer 0's query-only part once per unique query of a chunk (default)
  unsigned func_attr_mask;   // kernels whose dynamic shared-memory limit was raised on this context's device (bit per kernel)
  cudaStream_t stream;
  int num_sms;
  int64_t launches;
  void* encode_tiled;   // cuTensorMapEncodeTiled entry point (PFN), resolved lazily
  // optional per-launch GEMM timing (bench.py roofline): event pairs around every tcgen05 GEMM launch
  int profiling;
  void* prof;           // ProfState*
};
void cir_prof_gemm_begin(cir_ctx* ctx, double flops);
void cir_prof_gemm_end(cir_ctx* ctx);
void cir_prof_begin(cir_ctx* ctx, int kind, double work);     // kind: CIR_PROF_*; work: algorithmic FLOPs or bytes of the launch
void cir_prof_end(cir_ctx* ctx);

void cir_set_error(const char* fmt, ...);

#define CIR_CHECK_ARG(cond, ...)                      \
  do {                                                \
    if (!(cond)) {                                    \
      cir_set_error(__VA_ARGS__);                     \
      return CIR_EINVAL;                              \
    }                                                 \
  } while (0)

#define CIR_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      cir_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return CIR_ECUDA;                                                                  \
    }                                                                                    \
  } while (0)

#define CIR_LAUNCH_CHECK(ctx)                                                            \
  do {                                                                                   \
    (ctx)->launches++;                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) {                                                            \
      cir_set_error("%s:%d: kernel launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return CIR_ECUDA;                                                                  \
    }                                                                                    \
  } while (0)

// Every C-ABI entry point that touches the device runs on ctx->device and puts the caller's current device back on exit
// (two contexts on different GPUs may be driven from one thread).
struct CirDeviceGuard {
  int prev = -1; bool switched = false;
  explicit CirDeviceGuard(int want) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != want) switched = cudaSetDevice(want) == cudaSuccess;
  }
  ~CirDeviceGuard() { if (switched) cudaSetDevice(prev); }
};
#define CIR_ENTER(ctx) CirDeviceGuard cir_device_guard__((ctx)->device)

#define CIR_TRY(call)            \
  do {                           \
    int r__ = (call);            \
    if (r__ != CIR_OK) return r__; \
  } while (0)

static inline size_t act_size(const cir_ctx* ctx) { return ctx->dtype == CIR_DTYPE_F32 ? 4 : 2; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- device-side scalar conversion helpers, usable with T = float or bf16 ---------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Threshold filter of the tcgen05 similarity tiles (stage-I top-K): every accumulator S[row, col] >= thr[row] is appended to the
// row's candidate list, cand[row * cap + atomicAdd(count[row])] = {col_base + col, float bits of S}; a full list raises *overflow.
// col_tags [N] / row_masks [M] (both or neither): only columns with (col_tags[col] & row_masks[row]) != 0 are appended (a separate
// kernel instantiation, so the untagged filter keeps its code).
struct cir_gemm_filter {
  const float* thr; int32_t* count; uint2* cand; int32_t* overflow;
  int64_t cap; int64_t col_base;
};
int cir_gemm_tcgen05_filter(cir_ctx* ctx, const void* A, const void* W, int64_t M, int64_t N, int64_t K, const cir_gemm_filter* f,
                            const uint32_t* col_tags = nullptr, const uint32_t* row_masks = nullptr);

// internal cross-file entry points
int cir_gemm_simt(cir_ctx* ctx, const cir_gemm_args* a);
int cir_gemm_tcgen05(cir_ctx* ctx, const cir_gemm_args* a);
// 2-D bf16 tensor map over a [rows, K] row-major matrix (row stride ld elements), box [box_rows, 64], SWIZZLE_128B
int cir_make_map_2d(cir_ctx* ctx, CUtensorMap* map, const void* base, int64_t rows, int64_t K, int64_t ld, int box_rows);
// 3-D bf16 map, SWIZZLE_128B: dims (d0 contiguous, d1 stride s1, d2 stride s2; strides in elements), box (b0 <= 64, b1, b2)
int cir_make_map_3d(cir_ctx* ctx, CUtensorMap* map, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t s1, int64_t s2,
                    int b0, int b1, int b2);
int cir_attention_tc(cir_ctx* ctx, const cir_attn_args* a);
int cir_attention_tc_counted(cir_ctx* ctx, const cir_attn_args* a, const int32_t* ntiles_dev);   // tile count read on the device
int cir_attention_counted(cir_ctx* ctx, const cir_attn_args* a, const int32_t* ntiles_dev);      // attention.cu
// stage2_plan.cu: the two kernels after the scoring of an on-device plan (cir_stage2_rerank_cached)
int cir_stage2_scatter_scores(cir_ctx* ctx, const float* sorted, const int32_t* flat_pos, int64_t T, const int32_t* counts, float* scores);
int cir_stage2_gather_ranked(cir_ctx* ctx, const int32_t* cand, const int32_t* order, int64_t Q, int64_t K, int32_t* ranked);
bool cir_qkv_attention_supported(const cir_ctx* ctx, int64_t L);   // qkv_attention.cu
// stage1_topk_tc.cu: tensor-core candidate filter + exact fp32 re-check, per-query exact fallback on the device (never synchronises).
// A gallery "view" is the fp32 rows, their bf16 copy and gmax = {max ||g||, max ||g - bf16(g)||} as float bits.
bool cir_stage1_topk_tc_supported(const cir_ctx* ctx, int64_t Q, int64_t G, int64_t K);
size_t cir_stage1_topk_tc_workspace_bytes(int64_t Q, int64_t G, int64_t K);    // transient view + search
size_t cir_stage1_tc_search_bytes(int64_t Q, int64_t K);
// n more rows of a view: g_bf16[0..n) = bf16(g_emb[0..n)), gmax raised to cover them
int cir_stage1_tc_convert(cir_ctx* ctx, const float* g_emb, int64_t n, bf16* g_bf16, uint32_t* gmax);
// row_tags [G] / query_masks [Q] (both or neither): only rows with (row_tags[r] & query_masks[q]) != 0 are searched for query q
int cir_stage1_tc_search(cir_ctx* ctx, const float* q_emb, int64_t Q, const float* g_emb, const bf16* g_bf16, int64_t G, const uint32_t* gmax,
                         const uint32_t* row_tags, const uint32_t* query_masks, const int32_t* exclude, int64_t col_offset, int64_t K,
                         float* top_dist, int32_t* top_idx, int32_t* exact_rows, void* workspace, size_t workspace_bytes);
int cir_stage1_topk_tc(cir_ctx* ctx, const float* q_emb, const float* g_emb, int64_t Q, int64_t G, const int32_t* exclude, int64_t col_offset,
                       int64_t K, float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes);
