// softmax(Q K^T * scale + mask) V per (batch, head), head dim 64.
//
// attention_simt_kernel: generic CUDA-core kernel (fp32 math, T = float | bf16 storage) used by the
// fp32 check mode for every attention, and by the bf16 mode where no tensor-core specialisation
// exists yet.  One CTA = one (batch, head, 32-query tile); scores for the whole key range live in
// shared memory (Lk <= 1024), so softmax is exact two-pass like the reference
// (src/nlvr_encoder.py:193-199, src/vit.py:74-75).
#include "common.cuh"

namespace {

constexpr int QT = 32;      // queries per CTA
constexpr int KC = 64;      // keys per shared-memory chunk
constexpr int DH = CIR_HEAD_DIM;
constexpr int THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(THREADS)
attention_simt_kernel(cir_attn_args p) {
  extern __shared__ float smem[];
  const int lk_pad = (p.Lk + 3) & ~3;
  float* sQ = smem;                         // [QT][DH]
  float* sKV = sQ + QT * DH;                // [KC][DH+1]
  float* sS = sKV + KC * (DH + 1);          // [QT][lk_pad+1]
  const int ss = lk_pad + 1;

  const int b = blockIdx.x, h = blockIdx.y, q0 = blockIdx.z * QT;
  const int tid = threadIdx.x;
  const int kvb = p.kv_index ? p.kv_index[b] : b;
  const T* Q = (const T*)p.q + (int64_t)b * p.q_bs + h * DH;
  const T* K = (const T*)p.k + (int64_t)kvb * p.k_bs + h * DH;
  const T* V = (const T*)p.v + (int64_t)kvb * p.v_bs + h * DH;
  T* O = (T*)p.o + (int64_t)b * p.o_bs + h * DH;
  const int32_t* mask = p.key_mask ? p.key_mask + (int64_t)(p.mask_index ? p.mask_index[b] : b) * p.Lk : nullptr;

  for (int i = tid; i < QT * DH; i += THREADS) {
    const int q = i / DH, d = i % DH;
    sQ[i] = (q0 + q < p.Lq) ? to_f32<T>(Q[(int64_t)(q0 + q) * p.q_rs + d]) : 0.f;
  }
  const int q = tid / 8, sub = tid % 8;
  // ---- phase 1: S = Q K^T * scale + mask
  for (int k0 = 0; k0 < p.Lk; k0 += KC) {
    __syncthreads();
    for (int i = tid; i < KC * DH; i += THREADS) {
      const int kk = i / DH, d = i % DH;
      sKV[kk * (DH + 1) + d] = (k0 + kk < p.Lk) ? to_f32<T>(K[(int64_t)(k0 + kk) * p.k_rs + d]) : 0.f;
    }
    __syncthreads();
    float acc[8] = {};
#pragma unroll 8
    for (int d = 0; d < DH; d++) {
      const float qv = sQ[q * DH + d];
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] = fmaf(qv, sKV[(sub + 8 * j) * (DH + 1) + d], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int kk = k0 + sub + 8 * j;
      if (kk < p.Lk) {
        float s = acc[j] * p.scale;
        if (mask) s += (1.0f - (float)mask[kk]) * -10000.0f;
        sS[q * ss + kk] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 2: exact softmax per row (one warp handles 4 rows)
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp * 4; r < warp * 4 + 4; r++) {
      float m = -INFINITY;
      for (int k = lane; k < p.Lk; k += 32) m = fmaxf(m, sS[r * ss + k]);
      m = warp_max(m);
      float sum = 0.f;
      for (int k = lane; k < p.Lk; k += 32) { float e = expf(sS[r * ss + k] - m); sS[r * ss + k] = e; sum += e; }
      sum = warp_sum(sum);
      const float inv = 1.0f / sum;
      for (int k = lane; k < p.Lk; k += 32) sS[r * ss + k] *= inv;
    }
  }
  // ---- phase 3: O = P V
  float o[8] = {};
  const int d0 = sub * 8;
  for (int k0 = 0; k0 < p.Lk; k0 += KC) {
    __syncthreads();
    for (int i = tid; i < KC * DH; i += THREADS) {
      const int kk = i / DH, d = i % DH;
      sKV[kk * (DH + 1) + d] = (k0 + kk < p.Lk) ? to_f32<T>(V[(int64_t)(k0 + kk) * p.v_rs + d]) : 0.f;
    }
    __syncthreads();
    const int kn = min(KC, p.Lk - k0);
    for (int kk = 0; kk < kn; kk++) {
      const float pv = sS[q * ss + k0 + kk];
#pragma unroll
      for (int j = 0; j < 8; j++) o[j] = fmaf(pv, sKV[kk * (DH + 1) + d0 + j], o[j]);
    }
  }
  if (q0 + q < p.Lq) {
    T* op = O + (int64_t)(q0 + q) * p.o_rs + d0;
#pragma unroll
    for (int j = 0; j < 8; j++) op[j] = from_f32<T>(o[j]);
  }
}


// ------------------------------------------------------------------------------------------
// attention_mma_kernel: bf16 tensor-core (mma.sync m16n8k16, fp32 accumulate) flash attention with
// online softmax.  One warp = one 16-row query tile ("unit"); the NWARPS warps of a CTA belong to
// one run of batches that share the same K/V (candidate-major triplets of one candidate image, or
// the query tiles of one ViT image), so each 64-key K/V chunk is fetched once per CTA into
// XOR-swizzled shared memory by a 3-stage cp.async pipeline and read by every warp via ldmatrix.
// Scores never leave registers (no [L,577] round trip, no K^T / V transpose copies).
constexpr int FA_KC = 64;                       // keys per chunk
constexpr int FA_STAGES = 3;
constexpr int FA_STAGE_BYTES = 2 * FA_KC * 128; // K chunk + V chunk, 128 B per key row (64 bf16)

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <int NWARPS>
__global__ void __launch_bounds__(NWARPS * 32)
attention_mma_kernel(cir_attn_args p, int mt) {
  extern __shared__ __align__(128) uint8_t fa_smem[];
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(fa_smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  int batch0, unit0, run_units;
  if (p.work) {
    const int4 w = reinterpret_cast<const int4*>(p.work)[blockIdx.x];
    batch0 = w.x; unit0 = w.y; run_units = w.z;
  } else {
    const int cpb = (mt + NWARPS - 1) / NWARPS;
    batch0 = blockIdx.x / cpb; unit0 = (blockIdx.x % cpb) * NWARPS; run_units = mt;
  }
  const int h = blockIdx.y;
  const int u = unit0 + warp;
  const bool active = u < run_units;
  const int b = batch0 + (active ? u / mt : 0);
  const int mi = active ? u % mt : 0;
  const int kvb = p.kv_index ? p.kv_index[batch0] : batch0;
  const bf16* Kg = (const bf16*)p.k + (int64_t)kvb * p.k_bs + h * DH;
  const bf16* Vg = (const bf16*)p.v + (int64_t)kvb * p.v_bs + h * DH;
  const int nchunks = (p.Lk + FA_KC - 1) / FA_KC;

  auto load_chunk = [&](int c) {
    if (c < nchunks) {
      const uint32_t sbase = smem0 + (uint32_t)(c % FA_STAGES) * FA_STAGE_BYTES;
      for (int idx = tid; idx < 2 * FA_KC * 8; idx += NWARPS * 32) {
        const int which = idx >> 9, rem = idx & 511, row = rem >> 3, ch = rem & 7;
        int key = c * FA_KC + row;
        key = key < p.Lk ? key : p.Lk - 1;                       // clamp: rows past Lk are masked below
        const bf16* src = (which ? Vg + (int64_t)key * p.v_rs : Kg + (int64_t)key * p.k_rs) + ch * 8;
        cp_async16(sbase + (uint32_t)which * (FA_KC * 128) + (uint32_t)row * 128 + (uint32_t)((ch ^ (row & 7)) << 4), src);
      }
    }
    cp_async_commit();
  };
#pragma unroll
  for (int c = 0; c < FA_STAGES - 1; c++) load_chunk(c);

  // Q fragments (A operand, 16 rows x 64) straight from global memory
  const int r0 = mi * 16 + g, r1 = r0 + 8;
  const bool v0 = active && r0 < p.Lq, v1 = active && r1 < p.Lq;
  uint32_t qa[4][4];
  {
    const bf16* Qb = (const bf16*)p.q + (int64_t)b * p.q_bs + h * DH;
    const uint32_t* q0 = reinterpret_cast<const uint32_t*>(Qb + (int64_t)r0 * p.q_rs);
    const uint32_t* q1 = reinterpret_cast<const uint32_t*>(Qb + (int64_t)r1 * p.q_rs);
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
      qa[kk][0] = v0 ? q0[kk * 8 + t] : 0u;
      qa[kk][1] = v1 ? q1[kk * 8 + t] : 0u;
      qa[kk][2] = v0 ? q0[kk * 8 + 4 + t] : 0u;
      qa[kk][3] = v1 ? q1[kk * 8 + 4 + t] : 0u;
    }
  }
  const int32_t* mask = (p.key_mask && active) ? p.key_mask + (int64_t)(p.mask_index ? p.mask_index[b] : b) * p.Lk : nullptr;
  const float sl2 = p.scale * 1.4426950408889634f;          // scores in the log2 domain
  const float mask_l2 = -10000.0f * 1.4426950408889634f;    // additive -10000 (src/nlvr_encoder.py:774)
  float o[8][4];
#pragma unroll
  for (int j = 0; j < 8; j++) { o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

  for (int c = 0; c < nchunks; c++) {
    cp_async_wait<FA_STAGES - 2>();
    __syncthreads();                      // chunk c landed for everyone; chunk c-1's stage is free
    load_chunk(c + FA_STAGES - 1);
    if (!active) continue;
    const uint32_t sK = smem0 + (uint32_t)(c % FA_STAGES) * FA_STAGE_BYTES;
    const uint32_t sV = sK + FA_KC * 128;
    // ---- S = Q K^T for 64 keys: 8 n-tiles x 4 k-steps
    float s[8][4];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
      const int krow = j * 8 + (lane & 7);
      const uint32_t rowaddr = sK + (uint32_t)krow * 128;
      uint32_t kb[4];
      ldmatrix_x4(rowaddr + (uint32_t)((((lane >> 3)) ^ (krow & 7)) << 4), kb);          // dh chunks 0..3
      mma_bf16_16816(s[j], qa[0], kb[0], kb[1]);
      mma_bf16_16816(s[j], qa[1], kb[2], kb[3]);
      ldmatrix_x4(rowaddr + (uint32_t)(((4 + (lane >> 3)) ^ (krow & 7)) << 4), kb);      // dh chunks 4..7
      mma_bf16_16816(s[j], qa[2], kb[0], kb[1]);
      mma_bf16_16816(s[j], qa[3], kb[2], kb[3]);
    }
    // ---- scale, mask, online softmax (rows r0 and r1; a row lives in the 4 lanes of a quad)
    float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; j++) {
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int key = c * FA_KC + j * 8 + 2 * t + e;
        float add = 0.f;
        if (key >= p.Lk) add = -INFINITY;
        else if (mask && mask[key] == 0) add = mask_l2;
        s[j][e] = fmaf(s[j][e], sl2, add);
        s[j][2 + e] = fmaf(s[j][2 + e], sl2, add);
        cm0 = fmaxf(cm0, s[j][e]);
        cm1 = fmaxf(cm1, s[j][2 + e]);
      }
    }
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1)); cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1)); cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
    const float nm0 = fmaxf(m0, cm0), nm1 = fmaxf(m1, cm1);
    const float a0 = exp2f(m0 - nm0), a1 = exp2f(m1 - nm1);      // first chunk: exp2(-inf) = 0
    m0 = nm0; m1 = nm1;
    l0 *= a0; l1 *= a1;
#pragma unroll
    for (int j = 0; j < 8; j++) { o[j][0] *= a0; o[j][1] *= a0; o[j][2] *= a1; o[j][3] *= a1; }
    uint32_t pa[4][4];                    // P as bf16 A fragments: k-step kk covers keys 16kk..16kk+15
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float p00 = exp2f(s[j][0] - m0), p01 = exp2f(s[j][1] - m0);
      const float p10 = exp2f(s[j][2] - m1), p11 = exp2f(s[j][3] - m1);
      l0 += p00 + p01; l1 += p10 + p11;
      pa[j >> 1][(j & 1) * 2 + 0] = pack_bf16(p00, p01);
      pa[j >> 1][(j & 1) * 2 + 1] = pack_bf16(p10, p11);
    }
    // ---- O += P V : 4 k-steps (16 keys) x 8 n-tiles (8 dh), V fragments via ldmatrix.trans
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
      const int vrow = kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
      const uint32_t rowaddr = sV + (uint32_t)vrow * 128;
#pragma unroll
      for (int jp = 0; jp < 4; jp++) {
        uint32_t vb[4];
        ldmatrix_x4_trans(rowaddr + (uint32_t)(((2 * jp + (lane >> 4)) ^ (vrow & 7)) << 4), vb);
        mma_bf16_16816(o[2 * jp], pa[kk], vb[0], vb[1]);
        mma_bf16_16816(o[2 * jp + 1], pa[kk], vb[2], vb[3]);
      }
    }
  }
  cp_async_wait<0>();
  if (!active) return;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  bf16* Ob = (bf16*)p.o + (int64_t)b * p.o_bs + h * DH;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    if (v0) *reinterpret_cast<uint32_t*>(Ob + (int64_t)r0 * p.o_rs + j * 8 + 2 * t) = pack_bf16(o[j][0] * i0, o[j][1] * i0);
    if (v1) *reinterpret_cast<uint32_t*>(Ob + (int64_t)r1 * p.o_rs + j * 8 + 2 * t) = pack_bf16(o[j][2] * i1, o[j][3] * i1);
  }
}

// ------------------------------------------------------------------------------------------
// attention_small_kernel: masked text self-attention with Lq, Lk <= 32 (the twin self-attention of the dual-stream
// encoder at the BASELINE caption length).  It is bound by re-reading the QKV projection from HBM, so the kernel is
// built for memory-level parallelism: ONE WARP per (batch, head), no block barriers, Q and K fragments loaded straight
// from global memory into mma.sync operand registers, V staged through a warp-private swizzled 4 KB tile for
// ldmatrix.trans, exact single-pass softmax (all 32 keys are in registers).
constexpr int SM_WARPS = 4;
__global__ void __launch_bounds__(SM_WARPS * 32)
attention_small_kernel(cir_attn_args p) {
  __shared__ __align__(128) uint8_t sv_all[SM_WARPS][32 * 128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int64_t wid = (int64_t)blockIdx.x * SM_WARPS + warp;
  if (wid >= (int64_t)p.B * p.H) return;
  const int b = (int)(wid / p.H), h = (int)(wid % p.H);
  const int kvb = p.kv_index ? p.kv_index[b] : b;
  const bf16* Qb = (const bf16*)p.q + (int64_t)b * p.q_bs + h * DH;
  const bf16* Kg = (const bf16*)p.k + (int64_t)kvb * p.k_bs + h * DH;
  const bf16* Vg = (const bf16*)p.v + (int64_t)kvb * p.v_bs + h * DH;
  bf16* Ob = (bf16*)p.o + (int64_t)b * p.o_bs + h * DH;
  const int32_t* mask = p.key_mask ? p.key_mask + (int64_t)(p.mask_index ? p.mask_index[b] : b) * p.Lk : nullptr;
  // ---- V rows -> warp-private swizzled tile (issued first: longest latency)
  uint8_t* sv = sv_all[warp];
  {
    uint4 vv[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int row = i * 4 + (lane >> 3), ch = lane & 7;
      vv[i] = row < p.Lk ? *reinterpret_cast<const uint4*>(Vg + (int64_t)row * p.v_rs + ch * 8) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int row = i * 4 + (lane >> 3), ch = lane & 7;
      *reinterpret_cast<uint4*>(sv + row * 128 + ((ch ^ (row & 7)) << 4)) = vv[i];
    }
  }
  // ---- K fragments (B operand of Q K^T): n-tile j = keys 8j..8j+7, k-step kk = dh 16kk..16kk+15
  uint32_t kb[4][4][2];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int key = j * 8 + g;
    const uint32_t* kp = reinterpret_cast<const uint32_t*>(Kg + (int64_t)key * p.k_rs);
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
      kb[j][kk][0] = key < p.Lk ? kp[kk * 8 + t] : 0u;
      kb[j][kk][1] = key < p.Lk ? kp[kk * 8 + 4 + t] : 0u;
    }
  }
  // per-thread additive mask (log2 domain) of its 8 key columns: keys 8j + 2t + e
  const float sl2 = p.scale * 1.4426950408889634f;
  float madd[4][2];
#pragma unroll
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int key = j * 8 + 2 * t + e;
      madd[j][e] = key >= p.Lk ? -INFINITY : ((mask && mask[key] == 0) ? -10000.0f * 1.4426950408889634f : 0.f);
    }
  __syncwarp();
  const uint32_t sv_addr = (uint32_t)__cvta_generic_to_shared(sv);
#pragma unroll 1
  for (int mt = 0; mt < 2; mt++) {
    const int r0 = mt * 16 + g, r1 = r0 + 8;
    if (mt * 16 >= p.Lq) break;
    const bool v0 = r0 < p.Lq, v1 = r1 < p.Lq;
    uint32_t qa[4][4];
    {
      const uint32_t* q0 = reinterpret_cast<const uint32_t*>(Qb + (int64_t)r0 * p.q_rs);
      const uint32_t* q1 = reinterpret_cast<const uint32_t*>(Qb + (int64_t)r1 * p.q_rs);
#pragma unroll
      for (int kk = 0; kk < 4; kk++) {
        qa[kk][0] = v0 ? q0[kk * 8 + t] : 0u;
        qa[kk][1] = v1 ? q1[kk * 8 + t] : 0u;
        qa[kk][2] = v0 ? q0[kk * 8 + 4 + t] : 0u;
        qa[kk][3] = v1 ? q1[kk * 8 + 4 + t] : 0u;
      }
    }
    float sc[4][4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 4; kk++) mma_bf16_16816(sc[j], qa[kk], kb[j][kk][0], kb[j][kk][1]);
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        sc[j][e] = fmaf(sc[j][e], sl2, madd[j][e]);
        sc[j][2 + e] = fmaf(sc[j][2 + e], sl2, madd[j][e]);
        m0 = fmaxf(m0, sc[j][e]);
        m1 = fmaxf(m1, sc[j][2 + e]);
      }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float l0 = 0.f, l1 = 0.f;
    uint32_t pa[2][4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const float p00 = exp2f(sc[j][0] - m0), p01 = exp2f(sc[j][1] - m0);
      const float p10 = exp2f(sc[j][2] - m1), p11 = exp2f(sc[j][3] - m1);
      l0 += p00 + p01; l1 += p10 + p11;
      pa[j >> 1][(j & 1) * 2 + 0] = pack_bf16(p00, p01);
      pa[j >> 1][(j & 1) * 2 + 1] = pack_bf16(p10, p11);
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    float o[8][4];
#pragma unroll
    for (int j = 0; j < 8; j++) { o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < 2; kk++) {
      const int vrow = kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
      const uint32_t rowaddr = sv_addr + (uint32_t)vrow * 128;
#pragma unroll
      for (int jp = 0; jp < 4; jp++) {
        uint32_t vb[4];
        ldmatrix_x4_trans(rowaddr + (uint32_t)(((2 * jp + (lane >> 4)) ^ (vrow & 7)) << 4), vb);
        mma_bf16_16816(o[2 * jp], pa[kk], vb[0], vb[1]);
        mma_bf16_16816(o[2 * jp + 1], pa[kk], vb[2], vb[3]);
      }
    }
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (v0) *reinterpret_cast<uint32_t*>(Ob + (int64_t)r0 * p.o_rs + j * 8 + 2 * t) = pack_bf16(o[j][0] * i0, o[j][1] * i0);
      if (v1) *reinterpret_cast<uint32_t*>(Ob + (int64_t)r1 * p.o_rs + j * 8 + 2 * t) = pack_bf16(o[j][2] * i1, o[j][3] * i1);
    }
  }
}

template <int NWARPS>
int launch_mma(cir_ctx* ctx, const cir_attn_args* a, int mt) {
  const int cpb = (mt + NWARPS - 1) / NWARPS;
  const unsigned gx = a->work ? (unsigned)a->num_work : (unsigned)(a->B * cpb);
  const size_t smem = FA_STAGES * FA_STAGE_BYTES;
  const unsigned bit = 1u << (NWARPS == 2 ? 0 : (NWARPS == 4 ? 1 : 2));     // per context: the attribute is per device
  if (!(ctx->func_attr_mask & bit)) {
    CIR_CUDA(cudaFuncSetAttribute(attention_mma_kernel<NWARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->func_attr_mask |= bit;
  }
  attention_mma_kernel<NWARPS><<<dim3(gx, (unsigned)a->H), NWARPS * 32, smem, ctx->stream>>>(*a, mt);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

size_t simt_smem_bytes(int Lk) {
  const int lk_pad = (Lk + 3) & ~3;
  return sizeof(float) * (size_t)(QT * DH + KC * (DH + 1) + QT * (lk_pad + 1));
}

}  // namespace

extern "C" int cir_attention(cir_ctx* ctx, const cir_attn_args* a) {
  CIR_ENTER(ctx);
  if (a->B == 0 || a->Lq == 0) return CIR_OK;
  CIR_CHECK_ARG(a->Lk >= 1 && a->Lk <= 1024, "attention: Lk=%d out of range [1,1024]", a->Lk);
  CIR_CHECK_ARG(a->H >= 1 && a->H <= 65535, "attention: bad head count %d", a->H);
  if (ctx->dtype == CIR_DTYPE_BF16 && ctx->attn_impl == 0) {
    const int rc = cir_attention_tc(ctx, a);          // tcgen05/TMEM kernel where the shape is eligible
    if (rc != CIR_EUNSUPPORTED) return rc;
  }
  if (ctx->dtype == CIR_DTYPE_BF16 && ctx->attn_impl != 1) {
    // tensor-core path: needs 4-byte aligned rows for the packed loads/stores and 16 B aligned K/V rows
    CIR_CHECK_ARG((a->q_rs % 2) == 0 && (a->o_rs % 2) == 0 && (a->q_bs % 2) == 0 && (a->o_bs % 2) == 0 &&
                  (a->k_rs % 8) == 0 && (a->v_rs % 8) == 0 && (a->k_bs % 8) == 0 && (a->v_bs % 8) == 0 &&
                  ((uintptr_t)a->k & 15) == 0 && ((uintptr_t)a->v & 15) == 0 && ((uintptr_t)a->q & 3) == 0 && ((uintptr_t)a->o & 3) == 0,
                  "attention: operand strides/alignment not supported by the tensor-core kernel");
    const int mt = (a->Lq + 15) / 16;
    if (!a->work && a->Lq <= 32 && a->Lk <= 32 && a->Lq > 1 && ctx->attn_impl == 0) {      // masked text self-attention
      const int64_t warps = (int64_t)a->B * a->H;
      cir_prof_begin(ctx, CIR_PROF_ATTN_SELF, 4.0 * (double)a->B * a->H * (double)a->Lq * (double)a->Lk * 64.0);
      attention_small_kernel<<<(unsigned)((warps + SM_WARPS - 1) / SM_WARPS), SM_WARPS * 32, 0, ctx->stream>>>(*a);
      cir_prof_end(ctx);
      CIR_LAUNCH_CHECK(ctx);
      return CIR_OK;
    }
    if (a->work) { CIR_CHECK_ARG(a->num_work > 0, "attention: empty work list"); return launch_mma<8>(ctx, a, mt); }
    if (mt <= 2) return launch_mma<2>(ctx, a, mt);
    if (mt <= 4) return launch_mma<4>(ctx, a, mt);
    return launch_mma<8>(ctx, a, mt);
  }
  const size_t smem = simt_smem_bytes(a->Lk);
  dim3 grid((unsigned)a->B, (unsigned)a->H, (unsigned)((a->Lq + QT - 1) / QT));
  if (ctx->dtype == CIR_DTYPE_F32) {
    CIR_CUDA(cudaFuncSetAttribute(attention_simt_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attention_simt_kernel<float><<<grid, THREADS, smem, ctx->stream>>>(*a);
  } else {
    CIR_CUDA(cudaFuncSetAttribute(attention_simt_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attention_simt_kernel<bf16><<<grid, THREADS, smem, ctx->stream>>>(*a);
  }
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

// cir_attention for a tile list whose length the device wrote (a->tiles with at most a->num_tiles entries, the count at *ntiles_dev):
// the tcgen05 kernel reads the count itself; every other kernel ignores tile and work lists and runs each batch as its own run.
int cir_attention_counted(cir_ctx* ctx, const cir_attn_args* a, const int32_t* ntiles_dev) {
  CIR_ENTER(ctx);
  if (a->B == 0 || a->Lq == 0) return CIR_OK;
  if (ctx->dtype == CIR_DTYPE_BF16 && ctx->attn_impl == 0) {
    const int rc = cir_attention_tc_counted(ctx, a, ntiles_dev);
    if (rc != CIR_EUNSUPPORTED) return rc;
  }
  cir_attn_args b = *a;
  b.work = nullptr; b.num_work = 0;
  b.tiles = nullptr; b.num_tiles = 0;
  return cir_attention(ctx, &b);
}
