// Stage-I retrieval on the tensor cores: the K nearest gallery rows of every query under dist = 1 - q . g, bit-identical to the
// fp32 path of topk.cu (src/validate.py:57-58,202-210: `1 - q @ G^T`, ascending argsort, reference image removed, first K),
// without ever forming the [Q, G] matrix and without fp32 CUDA-core GEMM work (2 * 256 * Q * G flop).
//
//   1. q, g -> bf16 copies (one pass), with the exact rounding residuals ||x - bf16(x)|| and norms: a RIGOROUS per-query bound
//      eps_q >= |q . g - bf16(q) . bf16(g)| for every gallery row g (Cauchy-Schwarz) plus accumulation slack.
//   2. The gallery is walked in super-blocks of geometrically growing size.  For each one the tcgen05 GEMM (gemm_tcgen05.cu, FILT
//      epilogue) computes the approximate similarities tile by tile in TMEM and appends to the query's candidate list only the
//      entries >= thr_q.  After each super-block `select_kernel` sorts the (few hundred) candidates of every query, sets
//      thr_q = (K-th best approximate similarity so far) - 2 eps_q, and drops what fell below.  Any gallery row whose EXACT
//      similarity is among the K best has an approximate similarity >= thr_q at every point of the walk, so it survives.
//   3. `finalize_kernel` recomputes the survivors' distances in fp32 -- fmaf over k = 0..255 in order, the arithmetic of
//      sgemm_nt_kernel -- and sorts (distance bits, index) keys: the result equals the fp32 path bit for bit, ties included.
//   4. A query whose candidate list would overflow its capacity (adversarial gallery order, thousands of near-duplicates) stops
//      filtering (threshold +inf) and is listed by `finalize_kernel`; `exact_scan_kernel` / `exact_merge_kernel` then compute
//      the exact top-K of the listed queries only, with the same fp32 arithmetic over the whole gallery.  Nothing is read back to
//      the host, so a search can be captured in a CUDA graph.
// The gallery side (bf16 copy + the maxima {max ||g||, max ||g - bf16(g)||}) is a "view": cir_stage1_index keeps one resident and
// grows it row block by row block (the maxima only grow), cir_stage1_topk builds a transient one in its workspace per call.
// Filtered search (row tags, per-query masks): the tagged FILT GEMM drops ineligible columns before a hit reserves a slot and the exact
// scan skips them, so the lists, thresholds and counts of select_kernel / finalize_kernel only ever hold eligible rows (those two
// kernels are shared unchanged).  gmax stays a valid bound: it covers a superset of the eligible rows.
#include "common.cuh"

namespace s1tc {

constexpr int E = CIR_EMBED;              // 256
constexpr int THREADS = 256;
constexpr int MAX_SORT = 8192;            // candidate list capacity (power of two; 64 KB of keys in shared memory)
constexpr uint64_t KEY_MAX = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ uint32_t ordered_bits(float f) {
  f = f + 0.0f;
  uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float from_ordered_bits(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o ^ 0x80000000u) : ~o;
  return __uint_as_float(u);
}

// one warp per TB_ROWS consecutive rows (all loads issued before the first reduction): bf16 copy, ||x - bf16(x)||_2 and ||bf16(x)||_2
// (fp32, rounded up by the caller's slack); gmax (optional): running maxima {max ||x||, max ||x - bf16(x)||} over all rows as float
// bits (non-negative floats order like uints)
constexpr int TB_ROWS = 4;
__global__ void __launch_bounds__(THREADS)
to_bf16_kernel(const float* __restrict__ x, int64_t rows, bf16* __restrict__ xb, float* __restrict__ row_err, float* __restrict__ row_nrm,
               uint32_t* __restrict__ gmax) {
  const int lane = threadIdx.x & 31;
  const int64_t r0 = ((int64_t)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5)) * TB_ROWS;
  if (r0 >= rows) return;
  float4 v[TB_ROWS][2];
#pragma unroll
  for (int t = 0; t < TB_ROWS; t++)
#pragma unroll
    for (int i = 0; i < 2; i++)
      v[t][i] = r0 + t < rows ? reinterpret_cast<const float4*>(x + (r0 + t) * E)[lane + 32 * i] : make_float4(0.f, 0.f, 0.f, 0.f);
  float mx_full = 0.f, mx_err = 0.f;
#pragma unroll
  for (int t = 0; t < TB_ROWS; t++) {
    const int64_t r = r0 + t;
    if (r >= rows) break;
    float e2 = 0.f, n2 = 0.f, f2 = 0.f;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const float4 w = v[t][i];
      const __nv_bfloat162 lo = __floats2bfloat162_rn(w.x, w.y), hi = __floats2bfloat162_rn(w.z, w.w);
      const float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
      e2 += (w.x - a.x) * (w.x - a.x) + (w.y - a.y) * (w.y - a.y) + (w.z - b.x) * (w.z - b.x) + (w.w - b.y) * (w.w - b.y);
      n2 += a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y;
      f2 += w.x * w.x + w.y * w.y + w.z * w.z + w.w * w.w;
      uint2 o;
      o.x = *reinterpret_cast<const uint32_t*>(&lo); o.y = *reinterpret_cast<const uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(xb + r * E + (lane + 32 * i) * 4) = o;
    }
    e2 = warp_sum(e2); n2 = warp_sum(n2); f2 = warp_sum(f2);
    const float err = sqrtf(e2) * 1.0001f, nrm = sqrtf(n2) * 1.0001f, full = sqrtf(f2) * 1.0001f;
    if (lane == 0 && row_err) { row_err[r] = err; row_nrm[r] = nrm; }
    mx_full = fmaxf(mx_full, full); mx_err = fmaxf(mx_err, err);
  }
  if (lane == 0 && gmax) {                                     // the maxima settle after a few rows: look before paying for an atomic
    if (__float_as_uint(mx_full) > *(volatile uint32_t*)gmax) atomicMax(gmax, __float_as_uint(mx_full));
    if (__float_as_uint(mx_err) > *(volatile uint32_t*)(gmax + 1)) atomicMax(gmax + 1, __float_as_uint(mx_err));
  }
}

__global__ void init_kernel(float* thr, int32_t* count, int64_t Q, int32_t* flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Q) { thr[i] = -INFINITY; count[i] = 0; }
  if (i == 0) { flags[0] = 0; flags[1] = 0; }
}

// descending bitonic sort of n (power of two) keys in shared memory
__device__ void sort_desc(uint64_t* s, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int partner = i ^ j;
        if (partner > i) {
          const uint64_t a = s[i], b = s[partner];
          const bool up = (i & k) == 0;
          if ((a < b) == up) { s[i] = b; s[partner] = a; }
        }
      }
    }
  }
  __syncthreads();
}
__device__ void sort_asc(uint64_t* s, int n) {
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
__device__ void merge_asc(uint64_t* s, int n) {
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

// 1 - q . g in fp32, fmaf over k = 0..255 in order (sgemm_nt_kernel's sum, hence the fp32 path's distance bit for bit); sq in
// shared memory, 16 independent 16-byte loads of the gallery row in flight before each part of the chain
__device__ __forceinline__ float exact_dist(const float* sq, const float* __restrict__ g_row) {
  const float4* gv = reinterpret_cast<const float4*>(g_row);
  const float4* qv = reinterpret_cast<const float4*>(sq);
  float acc = 0.f;
#pragma unroll 1
  for (int k0 = 0; k0 < E / 4; k0 += 16) {
    float4 b[16];
#pragma unroll
    for (int k = 0; k < 16; k++) b[k] = __ldg(gv + k0 + k);
#pragma unroll
    for (int k = 0; k < 16; k++) {
      const float4 a = qv[k0 + k];
      acc = fmaf(a.x, b[k].x, acc); acc = fmaf(a.y, b[k].y, acc); acc = fmaf(a.z, b[k].z, acc); acc = fmaf(a.w, b[k].w, acc);
    }
  }
  return 1.0f - acc;
}

// One CTA per query, after a super-block: find the Ksel-th best approximate similarity among the candidates (radix select on the
// order-preserving bits, 4 passes of 8 bits -- no sort: the list order is irrelevant), move the threshold to it minus 2 eps_q and
// keep what is still above.  Ksel = K (+1 when a reference index is excluded: it may sit in the list).
// An overflowed list (count > cap) is incomplete: the query stops filtering (thr = +inf appends nothing more, so count stays
// above cap) and finalize_kernel hands it to the exact scan.
__global__ void __launch_bounds__(THREADS)
select_kernel(uint2* __restrict__ cand, int32_t* __restrict__ count, float* __restrict__ thr, int64_t cap, int K, const int32_t* __restrict__ exclude,
              const float* __restrict__ q_err, const float* __restrict__ q_nrm, const uint32_t* __restrict__ gmax) {
  extern __shared__ uint64_t skeys[];                                       // n entries: (ordered similarity bits) << 32 | column
  __shared__ int hist[256];
  __shared__ uint32_t s_prefix;
  __shared__ int s_need, s_keep;
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x;
  const int n = count[q];
  if (n > cap) { if (tid == 0) thr[q] = INFINITY; return; }
  const int Ksel = K + ((exclude && exclude[q] >= 0) ? 1 : 0);
  if (n < Ksel) return;                                                     // fewer than K candidates so far: keep all, threshold stays
  uint2* row = cand + q * cap;
  for (int i = tid; i < n; i += THREADS) { const uint2 c = row[i]; skeys[i] = ((uint64_t)ordered_bits(__uint_as_float(c.y)) << 32) | c.x; }
  if (tid == 0) { s_prefix = 0u; s_need = Ksel; }
  // after pass p the top 8 (p + 1) bits of the Ksel-th largest key are known
  for (int pass = 0; pass < 4; pass++) {
    const int shift = 24 - 8 * pass;
    hist[tid] = 0;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    const int need = s_need;
    for (int i = tid; i < n; i += THREADS) {
      const uint32_t k = (uint32_t)(skeys[i] >> 32);
      if (pass == 0 || (k >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(&hist[(k >> shift) & 255], 1);
    }
    __syncthreads();
    if (tid < 32) {                                                         // bins from the top: first bin where the running count reaches `need`
      int c[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) { c[j] = hist[255 - (tid * 8 + j)]; tot += c[j]; }
      int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (tid >= o) incl += t; }
      int run = incl - tot;                                                 // elements in bins above this lane's eight
      if (run < need && incl >= need) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          if (run < need && run + c[j] >= need) { s_prefix = prefix | ((uint32_t)(255 - (tid * 8 + j)) << shift); s_need = need - run; }
          run += c[j];
        }
      }
    }
    __syncthreads();
  }
  const float kth = from_ordered_bits(s_prefix);
  const float g_nrm = __uint_as_float(gmax[0]), g_err = __uint_as_float(gmax[1]);
  // |q.g - bf16(q).bf16(g)| <= ||q - q^|| ||g|| + ||q^|| ||g - g^||; + fp32 accumulation slack of both the tensor-core sum and the exact chain
  const float eps = (q_err[q] * g_nrm + q_nrm[q] * g_err) * 1.001f + 1e-4f * (q_nrm[q] + q_err[q]) * g_nrm;
  const float t_new = fmaxf(thr[q], kth - 2.0f * eps);
  if (tid == 0) s_keep = 0;
  __syncthreads();
  for (int i = tid; i < n; i += THREADS) {
    const uint64_t key = skeys[i];
    const float sv = from_ordered_bits((uint32_t)(key >> 32));
    if (sv >= t_new) row[atomicAdd(&s_keep, 1)] = make_uint2((uint32_t)(key & 0xFFFFFFFFu), __float_as_uint(sv));
  }
  __syncthreads();
  if (tid == 0) { count[q] = s_keep; thr[q] = t_new; }
}

// One CTA per query: exact fp32 distances of the surviving candidates (exact_dist), composite (distance bits, global index) keys,
// ascending sort, first K.  Missing entries: index -1, distance +inf (as topk.cu).  A query whose list overflowed is appended to
// `flagged` (flags[1] counts them) and left to the exact scan; exact_rows (optional) records which queries took that path.
__global__ void __launch_bounds__(THREADS, 2)
finalize_kernel(const uint2* __restrict__ cand, const int32_t* __restrict__ count, int64_t cap, const float* __restrict__ q_emb,
                const float* __restrict__ g_emb, const int32_t* __restrict__ exclude, int64_t col_offset, int K,
                float* __restrict__ out_dist, int32_t* __restrict__ out_idx, int32_t* __restrict__ flags, int32_t* __restrict__ flagged,
                int32_t* __restrict__ exact_rows) {
  extern __shared__ uint64_t skeys[];
  __shared__ __align__(16) float sq[E];
  const int64_t q = blockIdx.x;
  const int n = count[q];
  const bool over = n > cap;
  if (threadIdx.x == 0) {
    if (exact_rows) exact_rows[q] = over ? 1 : 0;
    if (over) flagged[atomicAdd(flags + 1, 1)] = (int32_t)q;
  }
  if (over) return;
  for (int i = threadIdx.x; i < E; i += THREADS) sq[i] = q_emb[q * E + i];
  int m = 32;
  while (m < n || m < K) m <<= 1;
  const int64_t excl = exclude ? (int64_t)exclude[q] : -1;
  __syncthreads();
  const uint2* row = cand + q * cap;
  for (int i = threadIdx.x; i < m; i += THREADS) {
    uint64_t key = KEY_MAX;
    if (i < n) {
      const uint32_t gi = row[i].x;                          // local gallery row
      const int64_t global = col_offset + (int64_t)gi;
      const float d = exact_dist(sq, g_emb + (int64_t)gi * E);
      if (global != excl) key = ((uint64_t)ordered_bits(d) << 32) | (uint32_t)global;
    }
    skeys[i] = key;
  }
  sort_asc(skeys, m);
  for (int i = threadIdx.x; i < K; i += THREADS) {
    const uint64_t key = skeys[i];
    out_idx[q * K + i] = (key == KEY_MAX) ? -1 : (int32_t)(key & 0xFFFFFFFFu);
    out_dist[q * K + i] = (key == KEY_MAX) ? INFINITY : from_ordered_bits((uint32_t)(key >> 32));
  }
}

// Exact top-K of the flagged queries (flags[1] of them, ids in `flagged`), the running-list algorithm of topk.cu's topk_rows_kernel
// on exact_dist keys.  Fixed grid, independent of the data: blockIdx.x = one of `parts` gallery slices of `slice` rows, blockIdx.y
// strides over the flagged queries; every CTA exits at once when nothing is flagged.  Slice p's Kp best keys go to the query's own
// candidate row at [p * Kp, (p + 1) * Kp) (parts * Kp <= cap), which the filter no longer needs.
// TAGS: rows with (row_tags[r] & query_masks[q]) == 0 are skipped next to the excluded one.
constexpr int SCAN_CH = 2048;                  // gallery rows per compaction round
constexpr int MAX_PARTS = 64;
template <bool TAGS>
__device__ __forceinline__ void exact_scan(const int32_t* __restrict__ flags, const int32_t* __restrict__ flagged, const float* __restrict__ q_emb,
                                           const float* __restrict__ g_emb, int64_t G, int64_t slice, const int32_t* __restrict__ exclude,
                                           int64_t col_offset, int K, int Kp, uint2* __restrict__ cand, int64_t cap,
                                           const uint32_t* __restrict__ row_tags, const uint32_t* __restrict__ query_masks) {
  __shared__ __align__(16) float sq[E];
  __shared__ uint64_t sbest[1024];
  __shared__ uint64_t schunk[SCAN_CH];
  __shared__ int s_n;
  const int nflag = flags[1];
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * slice, r1 = r0 + slice < G ? r0 + slice : G;
  for (int f = blockIdx.y; f < nflag; f += gridDim.y) {
    const int64_t q = flagged[f];
    __syncthreads();                                         // the previous query's lists have left shared memory
    for (int i = tid; i < E; i += THREADS) sq[i] = q_emb[q * E + i];
    for (int i = tid; i < Kp; i += THREADS) sbest[i] = KEY_MAX;
    const int64_t excl = exclude ? (int64_t)exclude[q] : -1;
    const uint32_t qmask = TAGS ? query_masks[q] : 0u;
    __syncthreads();
    for (int64_t c0 = r0; c0 < r1; c0 += SCAN_CH) {
      if (tid == 0) s_n = 0;
      __syncthreads();
      const uint64_t thresh = sbest[K - 1];                  // current K-th best (KEY_MAX while not full)
      for (int i = tid; i < SCAN_CH; i += THREADS) {
        const int64_t r = c0 + i;
        if (r < r1 && (!TAGS || (row_tags[r] & qmask) != 0)) {
          const int64_t global = col_offset + r;
          const uint64_t key = ((uint64_t)ordered_bits(exact_dist(sq, g_emb + r * E)) << 32) | (uint32_t)global;
          if (global != excl && key < thresh) schunk[atomicAdd(&s_n, 1)] = key;
        }
      }
      __syncthreads();
      const int n = s_n;
      __syncthreads();                                       // s_n is rewritten at the top of the next round
      if (n == 0) continue;
      int m = 32;
      while (m < n) m <<= 1;
      for (int i = n + tid; i < m; i += THREADS) schunk[i] = KEY_MAX;
      sort_asc(schunk, m);
      for (int i = tid; i < Kp; i += THREADS) {              // K smallest of (best U survivors): min(best[i], cand[Kp-1-i]) is bitonic
        const int j = Kp - 1 - i;
        const uint64_t a = sbest[i], b = j < m ? schunk[j] : KEY_MAX;
        sbest[i] = a < b ? a : b;
      }
      merge_asc(sbest, Kp);
    }
    uint64_t* out = reinterpret_cast<uint64_t*>(cand + q * cap) + (int64_t)blockIdx.x * Kp;
    for (int i = tid; i < Kp; i += THREADS) out[i] = sbest[i];
  }
}
__global__ void __launch_bounds__(THREADS, 2)
exact_scan_kernel(const int32_t* __restrict__ flags, const int32_t* __restrict__ flagged, const float* __restrict__ q_emb,
                  const float* __restrict__ g_emb, int64_t G, int64_t slice, const int32_t* __restrict__ exclude, int64_t col_offset,
                  int K, int Kp, uint2* __restrict__ cand, int64_t cap) {
  exact_scan<false>(flags, flagged, q_emb, g_emb, G, slice, exclude, col_offset, K, Kp, cand, cap, nullptr, nullptr);
}
__global__ void __launch_bounds__(THREADS, 2)
exact_scan_filtered_kernel(const int32_t* __restrict__ flags, const int32_t* __restrict__ flagged, const float* __restrict__ q_emb,
                           const float* __restrict__ g_emb, int64_t G, int64_t slice, const int32_t* __restrict__ exclude, int64_t col_offset,
                           int K, int Kp, uint2* __restrict__ cand, int64_t cap, const uint32_t* __restrict__ row_tags,
                           const uint32_t* __restrict__ query_masks) {
  exact_scan<true>(flags, flagged, q_emb, g_emb, G, slice, exclude, col_offset, K, Kp, cand, cap, row_tags, query_masks);
}

// The flagged queries' `n` = parts * Kp slice keys (a power of two) -> sorted, first K out.
__global__ void __launch_bounds__(THREADS)
exact_merge_kernel(const int32_t* __restrict__ flags, const int32_t* __restrict__ flagged, const uint2* __restrict__ cand, int64_t cap,
                   int n, int K, float* __restrict__ out_dist, int32_t* __restrict__ out_idx) {
  extern __shared__ uint64_t skeys[];
  const int nflag = flags[1];
  for (int f = blockIdx.x; f < nflag; f += gridDim.x) {
    const int64_t q = flagged[f];
    const uint64_t* row = reinterpret_cast<const uint64_t*>(cand + q * cap);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += THREADS) skeys[i] = row[i];
    sort_asc(skeys, n);
    for (int i = threadIdx.x; i < K; i += THREADS) {
      const uint64_t key = skeys[i];
      out_idx[q * K + i] = (key == KEY_MAX) ? -1 : (int32_t)(key & 0xFFFFFFFFu);
      out_dist[q * K + i] = (key == KEY_MAX) ? INFINITY : from_ordered_bits((uint32_t)(key >> 32));
    }
  }
}

static int64_t capacity(int64_t K) { return K <= 512 ? 4096 : MAX_SORT; }
static int pow2_at_least(int64_t k) { int p = 1; while (p < k) p <<= 1; return p; }

// search workspace; `flagged` reuses `thr`: the thresholds are dead once finalize_kernel runs
struct Ws { bf16* qb; float *q_err, *q_nrm, *thr; int32_t *count, *flags, *flagged; uint2* cand; size_t total; };
static Ws plan(void* ws, int64_t Q, int64_t cap) {
  char* base = (char*)ws; size_t off = 0;
  auto take = [&](size_t bytes) { off = align_up(off, 256); void* r = base ? base + off : nullptr; off += bytes; return r; };
  Ws w;
  w.qb = (bf16*)take((size_t)Q * E * 2);
  w.q_err = (float*)take((size_t)Q * 4);
  w.q_nrm = (float*)take((size_t)Q * 4);
  w.thr = (float*)take((size_t)Q * 4);
  w.flagged = (int32_t*)w.thr;
  w.count = (int32_t*)take((size_t)Q * 4);
  w.flags = (int32_t*)take(256);                             // [0] filter overflow word (unused), [1] number of flagged queries
  w.cand = (uint2*)take((size_t)Q * cap * 8);
  w.total = align_up(off, 256);
  return w;
}
// transient gallery view of cir_stage1_topk, in front of the search workspace
static size_t view_bytes(int64_t G) { return align_up((size_t)G * E * 2, 256) + 256; }

}  // namespace s1tc

bool cir_stage1_topk_tc_supported(const cir_ctx* ctx, int64_t Q, int64_t G, int64_t K) {
  return ctx->dtype == CIR_DTYPE_BF16 && ctx->gemm_impl != CIR_GEMM_SIMT && ctx->stage1_tc && Q >= 1 && G >= 16384 && K >= 1 && K <= 1024 &&
         G < (1ll << 31);
}
size_t cir_stage1_tc_search_bytes(int64_t Q, int64_t K) { return s1tc::plan(nullptr, Q, s1tc::capacity(K)).total; }
size_t cir_stage1_topk_tc_workspace_bytes(int64_t Q, int64_t G, int64_t K) { return s1tc::view_bytes(G) + cir_stage1_tc_search_bytes(Q, K); }

int cir_stage1_tc_convert(cir_ctx* ctx, const float* g_emb, int64_t n, bf16* g_bf16, uint32_t* gmax) {
  using namespace s1tc;
  if (n == 0) return CIR_OK;
  to_bf16_kernel<<<(unsigned)((n + 8 * TB_ROWS - 1) / (8 * TB_ROWS)), THREADS, 0, ctx->stream>>>(g_emb, n, g_bf16, nullptr, nullptr, gmax);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_stage1_tc_search(cir_ctx* ctx, const float* q_emb, int64_t Q, const float* g_emb, const bf16* g_bf16, int64_t G, const uint32_t* gmax,
                         const uint32_t* row_tags, const uint32_t* query_masks, const int32_t* exclude, int64_t col_offset, int64_t K,
                         float* top_dist, int32_t* top_idx, int32_t* exact_rows, void* workspace, size_t workspace_bytes) {
  using namespace s1tc;
  const int64_t cap = capacity(K);
  Ws w = plan(workspace, Q, cap);
  if (workspace_bytes < w.total) { cir_set_error("stage1_topk_tc: workspace %zu < %zu", workspace_bytes, w.total); return CIR_EWORKSPACE; }
  cudaStream_t st = ctx->stream;
  init_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, st>>>(w.thr, w.count, Q, w.flags);
  CIR_LAUNCH_CHECK(ctx);
  to_bf16_kernel<<<(unsigned)((Q + 8 * TB_ROWS - 1) / (8 * TB_ROWS)), THREADS, 0, st>>>(q_emb, Q, w.qb, w.q_err, w.q_nrm, nullptr);
  CIR_LAUNCH_CHECK(ctx);
  if (!(ctx->func_attr_mask & (1u << 29))) {                  // per context: the attribute is per device
    CIR_CUDA(cudaFuncSetAttribute(select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SORT * 8));
    CIR_CUDA(cudaFuncSetAttribute(finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SORT * 8));
    CIR_CUDA(cudaFuncSetAttribute(exact_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SORT * 8));
    ctx->func_attr_mask |= 1u << 29;
  }
  // super-blocks: the first one is small (everything passes while thr = -inf), then each is as large as all rows seen so far
  // (expected new candidates per block ~ K), capped so that a block's GEMM stays a few hundred microseconds
  const int64_t first = (cap / 2 / 256) * 256;
  const int64_t kMaxBlock = 262144;
  int64_t g0 = 0;
  while (g0 < G) {
    int64_t n = g0 == 0 ? first : (g0 < kMaxBlock ? g0 : kMaxBlock);
    if (n > G - g0) n = G - g0;
    cir_gemm_filter f{};
    f.thr = w.thr; f.count = w.count; f.cand = w.cand; f.overflow = w.flags; f.cap = cap; f.col_base = g0;
    CIR_TRY(cir_gemm_tcgen05_filter(ctx, w.qb, g_bf16 + g0 * E, Q, n, E, &f, row_tags ? row_tags + g0 : nullptr, query_masks));
    g0 += n;
    if (g0 < G) {
      select_kernel<<<(unsigned)Q, THREADS, (size_t)cap * 8, st>>>(w.cand, w.count, w.thr, cap, (int)K, exclude, w.q_err, w.q_nrm, gmax);
      CIR_LAUNCH_CHECK(ctx);
    }
  }
  finalize_kernel<<<(unsigned)Q, THREADS, (size_t)cap * 8, st>>>(w.cand, w.count, cap, q_emb, g_emb, exclude, col_offset, (int)K, top_dist, top_idx,
                                                                w.flags, w.flagged, exact_rows);
  CIR_LAUNCH_CHECK(ctx);
  // exact fallback of the flagged queries (usually none: both launches exit at once)
  const int Kp = pow2_at_least(K);
  const int parts = (int)(cap / Kp < MAX_PARTS ? cap / Kp : MAX_PARTS);
  const int64_t slice = (G + parts - 1) / parts;
  const int64_t ys = (2 * (int64_t)ctx->num_sms + parts - 1) / parts;
  const unsigned gy = (unsigned)(Q < ys ? Q : ys);
  if (row_tags)
    exact_scan_filtered_kernel<<<dim3((unsigned)parts, gy), THREADS, 0, st>>>(w.flags, w.flagged, q_emb, g_emb, G, slice, exclude, col_offset,
                                                                               (int)K, Kp, w.cand, cap, row_tags, query_masks);
  else
    exact_scan_kernel<<<dim3((unsigned)parts, gy), THREADS, 0, st>>>(w.flags, w.flagged, q_emb, g_emb, G, slice, exclude, col_offset, (int)K, Kp,
                                                                      w.cand, cap);
  CIR_LAUNCH_CHECK(ctx);
  const unsigned gm = (unsigned)(Q < 2 * ctx->num_sms ? Q : 2 * ctx->num_sms);
  exact_merge_kernel<<<gm, THREADS, (size_t)parts * Kp * 8, st>>>(w.flags, w.flagged, w.cand, cap, parts * Kp, (int)K, top_dist, top_idx);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

// cir_stage1_topk's tensor-core branch: a transient view of g_emb (bf16 copy + maxima) in front of the search workspace
int cir_stage1_topk_tc(cir_ctx* ctx, const float* q_emb, const float* g_emb, int64_t Q, int64_t G, const int32_t* exclude, int64_t col_offset,
                       int64_t K, float* top_dist, int32_t* top_idx, void* workspace, size_t workspace_bytes) {
  const size_t vb = s1tc::view_bytes(G);
  if (workspace_bytes < vb) { cir_set_error("stage1_topk_tc: workspace %zu < %zu", workspace_bytes, vb); return CIR_EWORKSPACE; }
  bf16* gb = (bf16*)workspace;
  uint32_t* gmax = (uint32_t*)((char*)workspace + vb - 256);
  CIR_CUDA(cudaMemsetAsync(gmax, 0, 2 * sizeof(uint32_t), ctx->stream));
  CIR_TRY(cir_stage1_tc_convert(ctx, g_emb, G, gb, gmax));
  return cir_stage1_tc_search(ctx, q_emb, Q, g_emb, gb, G, gmax, nullptr, nullptr, exclude, col_offset, K, top_dist, top_idx, nullptr,
                              (char*)workspace + vb, workspace_bytes - vb);
}
