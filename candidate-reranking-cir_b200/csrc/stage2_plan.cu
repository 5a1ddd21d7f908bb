// On-device candidate-major planning of one stage-II call, for a [Q, K] top-K list that already lives on the device
// (cir_stage1_index_topk output): the triplet order, cache rows and cross-attention tile lists that schedule.plan_chunks +
// build_attn_tiles compute on the host for one chunk, without a device -> host read.
//   cir_stage2_plan_topk       one CTA: bitonic sort of (candidate, flat position) keys in shared memory, run starts by a
//                              block max-scan, tile starts every G triplets of a run by a block sum-scan
//   scatter / gather kernels   the sorted scores back to [Q, K] (NEG_FILL at invalid entries), ranked ids from the order
#include "common.cuh"

namespace {

constexpr int PLAN_THREADS = 1024;
constexpr int FLAT_BITS = 14;                     // flat position q*K+k in the low bits of a key: T <= 2^14
constexpr int PLAN_MAX_T = 1 << FLAT_BITS;
constexpr int TILE_ROWS = 256;                    // query rows of one tcgen05 attention tile (schedule.TILE_ROWS)
constexpr float NEG_FILL = -99999.99f;            // src/validate_stage2.py:123,258

// block-wide exclusive scan of one int per thread under `op` (identity `id`); *total receives the reduction of all threads
template <typename Op>
__device__ int block_scan_excl(int v, int id, Op op, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl = op(incl, n);
  }
  int excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = id;
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int w = lane < nw ? s_warp[lane] : id;
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi = op(wi, n);
    }
    s_warp[lane] = wi;                           // inclusive over warps 0..lane
  }
  __syncthreads();
  const int res = op(warp > 0 ? s_warp[warp - 1] : id, excl);
  *total = s_warp[31];
  __syncthreads();                               // s_warp is reused by the next scan
  return res;
}

struct MaxOp { __device__ int operator()(int a, int b) const { return a > b ? a : b; } };
struct SumOp { __device__ int operator()(int a, int b) const { return a + b; } };

// One CTA plans all T = Q*K triplets.  key = (cand_rel << 14) | flat, cand_rel = cand - row0 for a candidate inside the cache,
// `rows` for an invalid one (-1 padding or outside the cache): sorting the keys orders the triplets by candidate, ties by flat
// position (the stable sort of schedule._sorted_triplets), with every invalid entry after every valid one.  Each thread then
// walks a contiguous segment of the sorted keys.
__global__ void __launch_bounds__(PLAN_THREADS)
stage2_plan_kernel(const int32_t* __restrict__ cand, int K, int T, int n_pad, int RB, int64_t row0, int64_t rows,
                   int32_t* __restrict__ flat_pos, int32_t* __restrict__ kv_row, int32_t* __restrict__ trip_query,
                   int4* __restrict__ tiles, int4* __restrict__ tiles_cls, int32_t* __restrict__ counts) {
  extern __shared__ uint32_t skey[];
  __shared__ int s_warp[32];
  __shared__ int s_invalid;
  const int tid = threadIdx.x;
  const uint32_t inv_rel = (uint32_t)rows;
  if (tid == 0) s_invalid = 0;
  for (int i = tid; i < n_pad; i += PLAN_THREADS) {
    uint32_t key = 0xFFFFFFFFu;                  // padding sorts last (rows < 2^18 - 1 keeps every real key below it)
    if (i < T) {
      const int64_t c = cand[i];
      const uint32_t rel = (c >= row0 && c < row0 + rows) ? (uint32_t)(c - row0) : inv_rel;
      key = (rel << FLAT_BITS) | (uint32_t)i;
    }
    skey[i] = key;
  }
  for (int k = 2; k <= n_pad; k <<= 1) {         // ascending bitonic sort
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = tid; i < n_pad; i += PLAN_THREADS) {
        const int partner = i ^ j;
        if (partner > i) {
          const uint32_t a = skey[i], b = skey[partner];
          if ((a > b) == ((i & k) == 0)) { skey[i] = b; skey[partner] = a; }
        }
      }
    }
  }
  __syncthreads();
  const int per = n_pad > PLAN_THREADS ? n_pad / PLAN_THREADS : 1;
  const int lo = min(tid * per, T), hi = min(lo + per, T);
  const int G = TILE_ROWS / RB;
  auto rel_at = [&](int i) { return skey[i] >> FLAT_BITS; };
  auto is_start = [&](int i) { return i == 0 || rel_at(i) != rel_at(i - 1); };
  // run start of every triplet: max-scan of the start positions
  int last_start = -1;
  for (int i = lo; i < hi; i++)
    if (is_start(i)) last_start = i;
  int dummy;
  const int rs_in = block_scan_excl(last_start, -1, MaxOp{}, s_warp, &dummy);
  // tile starts (every G-th triplet of a run, every 256th for the CLS list), packed as main << 16 | cls (each <= 2^14)
  int marks = 0, invalid = 0, rs = rs_in;
  for (int i = lo; i < hi; i++) {
    if (is_start(i)) rs = i;
    const int off = i - rs;
    marks += (off % G == 0 ? 1 << 16 : 0) + (off % TILE_ROWS == 0 ? 1 : 0);
    invalid += rel_at(i) == inv_rel;
  }
  if (invalid) atomicAdd(&s_invalid, invalid);
  int total;
  const int base = block_scan_excl(marks, 0, SumOp{}, s_warp, &total);
  int nm = base >> 16, nc = base & 0xFFFF;
  rs = rs_in;
  for (int i = lo; i < hi; i++) {
    const uint32_t key = skey[i];
    const uint32_t rel = key >> FLAT_BITS;
    const int flat = (int)(key & (PLAN_MAX_T - 1));
    flat_pos[i] = flat;
    kv_row[i] = rel == inv_rel ? 0 : (int)rel;
    trip_query[i] = flat / K;
    if (is_start(i)) rs = i;
    const int off = i - rs;
    const bool run_end = i + 1 == T || rel_at(i + 1) != rel;
    nm += off % G == 0;
    nc += off % TILE_ROWS == 0;
    // the last triplet of a tile writes it: {first triplet, triplets, first query row, RB} (schedule.build_attn_tiles)
    if (run_end || (off + 1) % G == 0) tiles[nm - 1] = make_int4(i - off % G, off % G + 1, 0, RB);
    if (run_end || (off + 1) % TILE_ROWS == 0) tiles_cls[nc - 1] = make_int4(i - off % TILE_ROWS, off % TILE_ROWS + 1, 0, 1);
  }
  if (tid == 0) {
    counts[0] = total >> 16;
    counts[1] = total & 0xFFFF;
    counts[2] = s_invalid;                       // every thread's atomicAdd precedes the scan's barriers
  }
}

__global__ void stage2_scatter_kernel(const float* __restrict__ sorted, const int32_t* __restrict__ flat_pos, int64_t T,
                                      const int32_t* __restrict__ counts, float* __restrict__ scores) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < T) scores[flat_pos[i]] = i < T - counts[2] ? sorted[i] : NEG_FILL;      // invalid entries trail the sorted list
}

// The unique-candidate list of a plan, for caches whose K/V are dequantised per chunk (CIR_KV_MXFP8).  kv_row holds the plan's
// sorted cache rows, its first T - counts[2] entries valid: slot[t] = run number of t among them (invalid entries: 0),
// run_row[r] = row0 + the cache row of run r, *n_runs = number of runs.  Without a valid entry run 0 is cache row 0, so every
// slot names a dequantised row.
__global__ void __launch_bounds__(PLAN_THREADS)
stage2_kv_runs_kernel(const int32_t* __restrict__ kv_row, const int32_t* __restrict__ counts, int T, int64_t row0,
                      int32_t* __restrict__ slot, int32_t* __restrict__ run_row, int32_t* __restrict__ n_runs) {
  __shared__ int s_warp[32];
  const int V = T - counts[2];
  const int per = (T + PLAN_THREADS - 1) / PLAN_THREADS;
  const int lo = min((int)threadIdx.x * per, T), hi = min(lo + per, T);
  auto is_start = [&](int i) { return i < V && (i == 0 || kv_row[i] != kv_row[i - 1]); };
  int starts = 0;
  for (int i = lo; i < hi; i++) starts += is_start(i);
  int total;
  int r = block_scan_excl(starts, 0, SumOp{}, s_warp, &total) - 1;
  for (int i = lo; i < hi; i++) {
    if (is_start(i)) run_row[++r] = (int32_t)(row0 + kv_row[i]);
    slot[i] = i < V ? r : 0;
  }
  if (threadIdx.x == 0) {
    if (total == 0) run_row[0] = (int32_t)row0;
    *n_runs = max(total, 1);
  }
}

__global__ void stage2_gather_ranked_kernel(const int32_t* __restrict__ cand, const int32_t* __restrict__ order, int64_t n, int64_t K,
                                            int32_t* __restrict__ ranked) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ranked[i] = cand[(i / K) * K + order[i]];
}

}  // namespace

extern "C" int cir_stage2_plan_topk(cir_ctx* ctx, const int32_t* cand, int64_t Q, int64_t K, int64_t L, int64_t row0, int64_t rows,
                                    int32_t* flat_pos, int32_t* kv_row, int32_t* trip_query, int32_t* tiles, int32_t* tiles_cls,
                                    int32_t* counts) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(Q >= 1 && K >= 1 && Q * K <= PLAN_MAX_T, "stage2_plan_topk: Q*K = %lld triplets outside [1, %d]", (long long)(Q * K),
                PLAN_MAX_T);
  CIR_CHECK_ARG(L >= 1 && L <= TILE_ROWS, "stage2_plan_topk: L=%lld outside [1, %d]", (long long)L, TILE_ROWS);
  CIR_CHECK_ARG(row0 >= 0 && rows >= 0 && rows < (1ll << (32 - FLAT_BITS)) - 1,
                "stage2_plan_topk: cache rows [%lld, +%lld) out of range (at most 2^18 - 2 rows)", (long long)row0, (long long)rows);
  CIR_CHECK_ARG(cand && flat_pos && kv_row && trip_query && tiles && tiles_cls && counts, "stage2_plan_topk: NULL pointer");
  const int T = (int)(Q * K);
  int n_pad = 32;
  while (n_pad < T) n_pad <<= 1;
  int RB = 1;
  while (RB < L) RB <<= 1;
  const size_t smem = (size_t)n_pad * sizeof(uint32_t);
  if (!(ctx->func_attr_mask & (1u << 5))) {                   // per context: the attribute is per device
    CIR_CUDA(cudaFuncSetAttribute(stage2_plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PLAN_MAX_T * (int)sizeof(uint32_t)));
    ctx->func_attr_mask |= 1u << 5;
  }
  stage2_plan_kernel<<<1, PLAN_THREADS, smem, ctx->stream>>>(cand, (int)K, T, n_pad, RB, row0, rows, flat_pos, kv_row, trip_query,
                                                              reinterpret_cast<int4*>(tiles), reinterpret_cast<int4*>(tiles_cls), counts);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_stage2_scatter_scores(cir_ctx* ctx, const float* sorted, const int32_t* flat_pos, int64_t T, const int32_t* counts, float* scores) {
  stage2_scatter_kernel<<<(unsigned)((T + 255) / 256), 256, 0, ctx->stream>>>(sorted, flat_pos, T, counts, scores);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_stage2_kv_runs(cir_ctx* ctx, const int32_t* kv_row, const int32_t* counts, int64_t T, int64_t row0, int32_t* slot,
                       int32_t* run_row, int32_t* n_runs) {
  stage2_kv_runs_kernel<<<1, PLAN_THREADS, 0, ctx->stream>>>(kv_row, counts, (int)T, row0, slot, run_row, n_runs);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_stage2_gather_ranked(cir_ctx* ctx, const int32_t* cand, const int32_t* order, int64_t Q, int64_t K, int32_t* ranked) {
  const int64_t n = Q * K;
  stage2_gather_ranked_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(cand, order, n, K, ranked);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}
