// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[b] = act(A[b] W[b]^T + bias[b]) (+ residual[b])
//
//   A [rows, K] bf16 K-major, W [N, K] bf16 K-major (PyTorch Linear layout) -> both operands are
//   "K-major" UMMA operands, loaded by TMA into 128B-swizzled shared-memory tiles.
//   One persistent CTA per SM, warp-specialised:
//     warp 0      TMA producer            (one elected lane)
//     warp 1      TMEM allocator + tcgen05.mma issuer (one elected lane)
//     warps 2..9  epilogue: tcgen05.ld TMEM -> registers -> bias/activation/residual -> global
//   Pipelines: smem ring full/empty mbarriers (TMA <-> MMA), 2 TMEM accumulator stages with
//   tmem_full/tmem_empty mbarriers (MMA <-> epilogue), static persistent tile scheduler.
//   Tile 128 x BN x 64 (BN = 256 or 128), UMMA 128 x BN x 16, fp32 accumulation in TMEM.
//
// Batched operands are folded into the row coordinate of 2-D tensor maps: batch b of A starts at
// row b*a_rows_per_batch (0 = shared A), of W at row b*w_rows_per_batch.  Tiles that cross a
// batch edge load neighbouring (or zero-filled OOB) rows and are masked in the epilogue.
#include "common.cuh"
#include "tcgen05_ptx.cuh"

namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;                 // 64 bf16 = 128 B = one SWIZZLE_128B atom row
constexpr int UMMA_K = 16;
constexpr int NUM_EPI_WARPS = 8;
constexpr int THREADS = 64 + NUM_EPI_WARPS * 32;   // 320
constexpr int ACC_STAGES = 2;

// PAIR = cta_group::2: two CTAs of a cluster compute one 256 x BN tile; each CTA stages its own 128 rows
// of A and HALF of the W tile (the tensor core reads the other half from the peer's shared memory), so
// L2->SM operand traffic per output drops 1.5x versus the single-CTA 128 x 256 tile.
template <int BN, bool PAIR = false> struct Cfg {
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;      // W rows staged by this CTA
  static constexpr int A_BYTES = BM * BK * 2;            // 16 KB
  static constexpr int B_BYTES = B_ROWS * BK * 2;        // 32 / 16 KB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_STAGING = NUM_EPI_WARPS * 4096;   // per-warp 32 x 128 B transpose tiles
  static constexpr int STAGES = (196608 - EPI_STAGING) / STAGE_BYTES;    // 5 (32 KB stages) or 3 (48 KB stages)
  static constexpr int TMEM_COLS = ACC_STAGES * BN;      // 512 / 256
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 192 /*barriers*/ + ACC_STAGES * BN * 4 /*bias*/ + EPI_STAGING;
};

struct Params {
  void* C; const float* bias; const void* residual;
  int64_t M, N, K;
  int64_t ldc, ldres;
  int64_t c_bstride, bias_bstride, res_bstride;
  int64_t a_rows_per_batch, w_rows_per_batch;
  int32_t batch, act, c_f32, res_f32;
  int32_t m_blocks, n_blocks, k_blocks, num_tiles;
  int32_t tma_store;       // 1: bf16 C tiles leave through cp.async.bulk.tensor stores (3-D map: N, M, batch)
  // threshold filter (FILT kernels, stage-I similarity tiles): nothing is stored; every accumulator >= thr[row] is appended
  // to the row's candidate list as (global column, value bits)
  cir_gemm_filter flt;
  int32_t n_major;         // 1: tiles ordered n-block major (all m-blocks of a W block side by side: W streams from HBM once)
  // tagged filter (TAGS kernels): column c may enter row r's list only if (flt_col_tags[c] & flt_row_masks[r]) != 0.
  // Last in the struct: the offsets of every other field, hence the untagged kernels, do not move.
  const uint32_t* flt_col_tags; const uint32_t* flt_row_masks;
};

// tile sequence of one worker: plain round-robin over tiles
__device__ __forceinline__ bool next_tile(const Params& p, int worker, int num_workers, int it, int& b, int& m_blk, int& n_blk) {
  const int tile = worker + it * num_workers;
  if (tile >= p.num_tiles) return false;
  const int tiles_per_batch = p.m_blocks * p.n_blocks;
  b = tile / tiles_per_batch;
  const int r = tile - b * tiles_per_batch;
  if (p.n_major) {
    n_blk = r / p.m_blocks;
    m_blk = r - n_blk * p.m_blocks;
    return true;
  }
  m_blk = r / p.n_blocks;
  n_blk = r - m_blk * p.n_blocks;
  return true;
}

// GELU in the bf16 epilogue: the tanh form with the hardware tanh.approx (one MUFU + 6 FMA-pipe ops per
// element; the erf form costs two MUFU + ~14 ops and made the FFN1 epilogue slower than its MMAs).
// |gelu_tanh - gelu_erf| <= 5e-4 and tanh.approx adds <= 2^-11 relative, both below the bf16 output
// rounding (2^-9 relative); the fp32 check mode uses the exact erff GELU (gemm_simt.cu).
__device__ __forceinline__ float gelu_fast(float x) {
  const float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f);     // sqrt(2/pi) * (x + 0.044715 x^3)
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

// packed fp32 pairs (sm_100 FADD2 / FMUL2 / FFMA2: one issue slot for two IEEE fp32 operations) for the epilogue math: the GEMMs run
// at the board's power cap, so every instruction the eight epilogue warps do not issue is energy for the tensor pipe
__device__ __forceinline__ uint64_t pk2(float lo, float hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
// gelu_fast on a pair: identical per-element arithmetic, five of the six FMA-pipe operations packed
__device__ __forceinline__ void gelu_fast2(float& x0, float& x1) {
  const uint64_t x = pk2(x0, x1);
  const uint64_t u = mul2(x, fma2(pk2(0.0356774081f, 0.0356774081f), mul2(x, x), pk2(0.7978845608f, 0.7978845608f)));
  float u0, u1, t0, t1;
  upk2(u, u0, u1);
  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(u0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(u1));
  const uint64_t hx = mul2(pk2(0.5f, 0.5f), x);
  upk2(fma2(hx, pk2(t0, t1), hx), x0, x1);
}

// ----------------------------------------------------------------------------- the kernel
// TAGS (FILT only): the threshold filter also tests the column's tag against the row's mask before a hit reserves a slot
template <int BN, bool PAIR, bool FILT, bool TAGS>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                    const __grid_constant__ CUtensorMap map_c, const Params p) {
  static_assert(FILT || !TAGS, "tags belong to the threshold filter");
  using C = Cfg<BN, PAIR>;
  constexpr int TILE_M = PAIR ? 2 * BM : BM;                 // rows of one scheduled tile
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;       // 0 = leader (issues the MMAs)
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int num_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B needs 1024 B alignment
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + C::STAGES * C::A_BYTES;
  const uint32_t bar_base = smem_base + C::STAGES * C::STAGE_BYTES + C::EPI_STAGING;   // [ring][epilogue staging][barriers][bias]
  // barrier layout: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], tmem_ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + ACC_STAGES + s); };
  const uint32_t tmem_ptr_smem = bar_base + 8u * (2 * C::STAGES + 2 * ACC_STAGES);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_ptr_gen = (volatile uint32_t*)(smem_gen + C::STAGES * C::STAGE_BYTES + C::EPI_STAGING + 8 * (2 * C::STAGES + 2 * ACC_STAGES));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < C::STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < ACC_STAGES; s++) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), NUM_EPI_WARPS * (PAIR ? 2 : 1)); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (PAIR) tmem_alloc_pair<C::TMEM_COLS>(tmem_ptr_smem);
    else tmem_alloc<C::TMEM_COLS>(tmem_ptr_smem);
  }
  tcgen05_fence_before();
  __syncwarp();
  if constexpr (PAIR) cluster_sync_all();      // the peer's barriers must exist before any remote arrive / multicast commit
  else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      int b, m_blk, n_blk;
      for (int it = 0; next_tile(p, worker, num_workers, it, b, m_blk, n_blk); ++it) {
        const int32_t a_row = (int32_t)(b * p.a_rows_per_batch + (int64_t)m_blk * TILE_M + rank * BM);
        const int32_t w_row = (int32_t)(b * p.w_rows_per_batch + (int64_t)n_blk * BN + rank * C::B_ROWS);
        for (int kb = 0; kb < p.k_blocks; kb++) {
          mbar_wait(empty_bar(stage), phase ^ 1);           // local: freed by the (multicast) MMA commit
          if constexpr (PAIR) {
            if (rank == 0) mbar_expect_tx(full_bar(stage), 2 * C::STAGE_BYTES);     // both CTAs' bytes land on the leader's barrier
            tma_load_2d_pair(smem_a + stage * C::A_BYTES, &map_a, full_bar(stage), kb * BK, a_row);
            tma_load_2d_pair(smem_b + stage * C::B_BYTES, &map_w, full_bar(stage), kb * BK, w_row);
          } else {
            mbar_expect_tx(full_bar(stage), C::STAGE_BYTES);
            tma_load_2d(smem_a + stage * C::A_BYTES, &map_a, full_bar(stage), kb * BK, a_row);
            tma_load_2d(smem_b + stage * C::B_BYTES, &map_w, full_bar(stage), kb * BK, w_row);
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (rank == 0 && elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(TILE_M, BN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      int b_, m_, n_;
      for (int it = 0; next_tile(p, worker, num_workers, it, b_, m_, n_); ++it) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);          // epilogue drained this accumulator
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < p.k_blocks; kb++) {
          mbar_wait(full_bar(stage), phase);                // TMA bytes landed
          tcgen05_fence_after();
          const uint64_t adesc = make_smem_desc_sw128(smem_a + stage * C::A_BYTES);
          const uint64_t bdesc = make_smem_desc_sw128(smem_b + stage * C::B_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; k++) {
            // advance 32 B (16 bf16) along K inside the 128 B swizzle atom: +2 in the >>4 address field
            if constexpr (PAIR) umma_bf16_pair(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (uint32_t)((kb | k) != 0));
            else umma_bf16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (uint32_t)((kb | k) != 0));
          }
          if constexpr (PAIR) umma_commit_pair(empty_bar(stage));   // frees the slot in BOTH CTAs when the MMAs retire
          else umma_commit(empty_bar(stage));
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (PAIR) umma_commit_pair(tfull_bar(acc));       // accumulator halves ready in both CTAs
        else umma_commit(tfull_bar(acc));
        if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (8 warps) =====================
    // Each warp owns 32 accumulator rows (its TMEM lane quarter) x BN/2 columns and walks them in spans of
    // 64 columns.  tcgen05.ld hands every thread one ROW (32 consecutive columns per load), which is the
    // worst possible shape for global memory (a warp-wide 16 B store would touch 32 different lines), so
    // rows are transposed through a warp-private, XOR-swizzled 4 KB shared-memory tile: global stores
    // (and bf16 residual loads) then move whole 128 B row segments, 4 rows per instruction.  The tile's
    // bias row is staged in shared memory before the accumulator is waited for, and residual segments
    // are fetched ahead of the TMEM load.
    const int ew = warp - 2;                 // 0..7
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access (warp_id % 4)
    const int half = ew >> 2;                // which half of the BN columns
    constexpr int COLS_PER_WARP = BN / 2;
    constexpr int NCH = COLS_PER_WARP / 32;  // 4 or 2 (even)
    float* sbias = reinterpret_cast<float*>(smem_gen + C::STAGES * C::STAGE_BYTES + C::EPI_STAGING + 192);   // [ACC_STAGES][BN]
    const uint32_t stg = smem_base + C::STAGES * C::STAGE_BYTES + (uint32_t)ew * 4096;                    // this warp's 32 x 128 B tile (4 KB aligned)
    const int etid = threadIdx.x - 64;       // 0..255
    const bool res_bf16_fast = p.residual && !p.res_f32 && (p.ldres & 7) == 0;
    const bool res_f32_fast = p.residual && p.res_f32 && (p.ldres & 3) == 0 && ((uintptr_t)p.residual & 15) == 0;
    const bool out_bf16_fast = !p.c_f32 && (p.ldc & 7) == 0;
    const bool out_f32_fast = p.c_f32 && (p.ldc & 3) == 0;
    const int lr = lane >> 3, lp = lane & 7; // coalesced mapping: 4 rows x 8 sixteen-byte pieces per instruction
    auto sts128 = [](uint32_t addr, const uint4& v) {
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds128 = [](uint32_t addr) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
      return v;
    };
    int acc = 0; uint32_t acc_phase = 0;
    bool tma_store_pending = false;
    int b, m_blk, n_blk;
    // FILT: slots reserved by the last atomicAdd of this lane and the (column, value) pairs that go there
    int pend_n = 0, pend_base = 0;
    uint32_t pend_col[2] = {0u, 0u}, pend_val[2] = {0u, 0u};
    int64_t pend_row = 0;
    auto flt_flush = [&]() {
      if (pend_n > 0) {
#pragma unroll
        for (int i = 0; i < 2; i++) {
          if (i < pend_n) {
            if (pend_base + i < p.flt.cap) p.flt.cand[pend_row * p.flt.cap + pend_base + i] = make_uint2(pend_col[i], pend_val[i]);
            else *p.flt.overflow = 1;
          }
        }
        pend_n = 0;
      }
    };
    for (int it = 0; next_tile(p, worker, num_workers, it, b, m_blk, n_blk); ++it) {
      const int64_t row_base = (int64_t)m_blk * TILE_M + rank * BM + quarter * 32;
      const int64_t row = row_base + lane;
      if constexpr (FILT) { flt_flush(); pend_row = row; }       // the row changes with the tile: write what the previous tile left pending
      const bool row_ok = row < p.M;
      const int64_t ntile0 = (int64_t)n_blk * BN;
      float flt_thr = INFINITY;
      if constexpr (FILT) { if (row_ok) flt_thr = __ldg(p.flt.thr + row); }
      uint32_t flt_mask = 0u;
      if constexpr (TAGS) { if (row_ok) flt_mask = __ldg(p.flt_row_masks + row); }
      if (!FILT && etid < BN) {
        const int64_t n = ntile0 + etid;
        sbias[acc * BN + etid] = (p.bias && n < p.N) ? __ldg(p.bias + b * p.bias_bstride + n) : 0.f;
      }
      if constexpr (!FILT) asm volatile("bar.sync 1, 256;" ::: "memory");       // epilogue warps only (bias row staged)
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();

#pragma unroll 1
      for (int c = 0; c < NCH; c += 2) {
        const int col0 = half * COLS_PER_WARP + c * 32;
        const int64_t n00 = ntile0 + col0;                 // first column of this 64-column span
        const bool span_full = n00 + 64 <= p.N;
        // ---- bf16 residual: coalesced fetch now (does not depend on the accumulator), transpose after the TMEM wait
        const bool res_fast = res_bf16_fast && span_full;
        uint4 rq[8];
        if (res_fast) {
          const bf16* rp = (const bf16*)p.residual + b * p.res_bstride + n00 + lp * 8;
#pragma unroll
          for (int it = 0; it < 8; it++) {
            const int64_t rg = row_base + it * 4 + lr;
            rq[it] = rg < p.M ? *reinterpret_cast<const uint4*>(rp + rg * p.ldres) : make_uint4(0, 0, 0, 0);
          }
        }
        // fp32 residual (the ViT's fp32 token stream): the same coalesced fetch, 32 columns (128 B per row) at a time
        const bool res32_fast = res_f32_fast && span_full;
        auto load_res32 = [&](int hh) {
          const float* rp = (const float*)p.residual + b * p.res_bstride + n00 + hh * 32 + lp * 4;
#pragma unroll
          for (int it = 0; it < 8; it++) {
            const int64_t rg = row_base + it * 4 + lr;
            rq[it] = rg < p.M ? *reinterpret_cast<const uint4*>(rp + rg * p.ldres) : make_uint4(0, 0, 0, 0);
          }
        };
        if (res32_fast) load_res32(0);
        uint32_t v0[32], v1[32];
        __syncwarp();                                      // tcgen05.ld is .sync.aligned: reconverge first
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + col0);
        tmem_ld_32x32b_x32(taddr, v0);
        tmem_ld_32x32b_x32(taddr + 32, v1);
        tmem_ld_wait();
        if (n00 >= p.N) continue;                          // whole span beyond N (warp-uniform)
        if constexpr (FILT) {
          // 2 x 32 similarities of this thread's row.  Fast path: max tree per 32 values.  A chunk that holds a candidate (rare once
          // the thresholds have warmed up) is parked in this lane's 128-byte row of the warp's staging tile so that the hits can be
          // fetched by (dynamic) bit index; the hit mask is built without branches.  ONE atomicAdd reserves the slots of all hits of
          // the chunk, and its result is not consumed here: up to two (column, value) pairs wait in registers and are written when
          // the lane next has a hit or at the end of the tile, so the ~1 us atomic round trip is off the warp's critical path (with
          // an atomic + dependent store per hit the epilogue, not the UMMAs, paced these K = 256 tiles: 17 % of the samples sat on
          // the returned slot).
          auto chunk = [&](const uint32_t (&v)[32], int64_t nbase) {
            // four independent 3-input max chains (5 deep) instead of one 31-deep chain
            float c0 = __uint_as_float(v[0]), c1 = __uint_as_float(v[8]), c2 = __uint_as_float(v[16]), c3 = __uint_as_float(v[24]);
#pragma unroll
            for (int j = 1; j < 8; j += 2) {
              c0 = fmaxf(fmaxf(c0, __uint_as_float(v[j])), __uint_as_float(v[j + 1 < 8 ? j + 1 : j]));
              c1 = fmaxf(fmaxf(c1, __uint_as_float(v[8 + j])), __uint_as_float(v[8 + (j + 1 < 8 ? j + 1 : j)]));
              c2 = fmaxf(fmaxf(c2, __uint_as_float(v[16 + j])), __uint_as_float(v[16 + (j + 1 < 8 ? j + 1 : j)]));
              c3 = fmaxf(fmaxf(c3, __uint_as_float(v[24 + j])), __uint_as_float(v[24 + (j + 1 < 8 ? j + 1 : j)]));
            }
            const float mx = fmaxf(fmaxf(c0, c1), fmaxf(c2, c3));
            // TAGS: the chunk's 32 column tags (one 128-byte load by the whole warp, only when some lane passed the max test) are
            // staged in this warp's slot of the (unused) bias area, where each hit lane reads them by index
            const uint32_t* stags = reinterpret_cast<const uint32_t*>(sbias) + ew * 32;
            if constexpr (TAGS) {
              if (__any_sync(0xffffffffu, mx >= flt_thr)) {
                const int64_t c = nbase + lane;
                const uint32_t t = c < p.N ? __ldg(p.flt_col_tags + c) : 0u;
                __syncwarp();                                                // the previous chunk's readers are done
                const_cast<uint32_t*>(stags)[lane] = t;
                __syncwarp();
              }
            }
            if (mx >= flt_thr) {
              uint32_t mask = 0u;
#pragma unroll
              for (int j = 0; j < 32; j++) mask |= (__uint_as_float(v[j]) >= flt_thr ? 1u : 0u) << j;
              if constexpr (TAGS) {                                          // eligibility before the atomicAdd reserves slots
                uint32_t elig = 0u;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const uint4 t = *reinterpret_cast<const uint4*>(stags + j);
                  elig |= ((t.x & flt_mask) ? 1u : 0u) << j | ((t.y & flt_mask) ? 1u : 0u) << (j + 1) |
                          ((t.z & flt_mask) ? 1u : 0u) << (j + 2) | ((t.w & flt_mask) ? 1u : 0u) << (j + 3);
                }
                mask &= elig;
              }
              const int64_t left = p.N - nbase;                              // columns of this chunk inside the matrix
              if (left < 32) mask &= left <= 0 ? 0u : ((1u << left) - 1u);
              const uint32_t mine = stg + (uint32_t)lane * 128;
#pragma unroll
              for (int j = 0; j < 8; j++) sts128(mine + (uint32_t)((j ^ (lane & 7)) << 4), make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
              auto value_at = [&](int j) {
                uint32_t bits;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(bits) : "r"(mine + (uint32_t)((((j >> 2) ^ (lane & 7)) << 4) + (j & 3) * 4)) : "memory");
                return bits;
              };
              flt_flush();                                                   // the previous reservation returned long ago
              const int n = __popc(mask);
              if (n > 0) {
                const int base = atomicAdd(p.flt.count + row, n);
                if (n <= 2) {
                  const int j0 = __ffs(mask) - 1;
                  pend_col[0] = (uint32_t)(p.flt.col_base + nbase + j0); pend_val[0] = value_at(j0);
                  if (n == 2) {
                    const int j1 = 31 - __clz(mask);
                    pend_col[1] = (uint32_t)(p.flt.col_base + nbase + j1); pend_val[1] = value_at(j1);
                  }
                  pend_base = base; pend_n = n;
                } else {                                                     // many hits (the first super-block: everything passes)
                  int slot = base;
                  while (mask) {
                    const int j = __ffs(mask) - 1;
                    mask &= mask - 1;
                    if (slot < p.flt.cap) p.flt.cand[row * p.flt.cap + slot] = make_uint2((uint32_t)(p.flt.col_base + nbase + j), value_at(j));
                    else *p.flt.overflow = 1;
                    slot++;
                  }
                }
              }
            }
          };
          chunk(v0, n00);
          chunk(v1, n00 + 32);
          continue;
        }
        float f[64];
        {
          const float4* sb = reinterpret_cast<const float4*>(sbias + acc * BN + col0);
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b0 = sb[j >> 2], b1 = sb[8 + (j >> 2)];
            upk2(add2(pk2(__uint_as_float(v0[j]), __uint_as_float(v0[j + 1])), pk2(b0.x, b0.y)), f[j], f[j + 1]);
            upk2(add2(pk2(__uint_as_float(v0[j + 2]), __uint_as_float(v0[j + 3])), pk2(b0.z, b0.w)), f[j + 2], f[j + 3]);
            upk2(add2(pk2(__uint_as_float(v1[j]), __uint_as_float(v1[j + 1])), pk2(b1.x, b1.y)), f[32 + j], f[32 + j + 1]);
            upk2(add2(pk2(__uint_as_float(v1[j + 2]), __uint_as_float(v1[j + 3])), pk2(b1.z, b1.w)), f[32 + j + 2], f[32 + j + 3]);
          }
        }
        if (p.act == CIR_ACT_GELU) {
#pragma unroll
          for (int j = 0; j < 64; j += 2) gelu_fast2(f[j], f[j + 1]);
        } else if (p.act == CIR_ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 64; j++) f[j] = fmaxf(f[j], 0.f);
        }
        if (p.residual) {
          if (res_fast) {
            if (tma_store_pending) {
              if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
              __syncwarp();
              tma_store_pending = false;
            }
#pragma unroll
            for (int it = 0; it < 8; it++) sts128(stg + (uint32_t)(it * 4 + lr) * 128 + (uint32_t)((lp ^ ((it * 4 + lr) & 7)) << 4), rq[it]);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const uint4 rv = lds128(stg + (uint32_t)lane * 128 + (uint32_t)((j ^ (lane & 7)) << 4));
              const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
              for (int q = 0; q < 4; q++) {
                const float2 t = __bfloat1622float2(h2[q]);
                upk2(add2(pk2(f[j * 8 + 2 * q], f[j * 8 + 2 * q + 1]), pk2(t.x, t.y)), f[j * 8 + 2 * q], f[j * 8 + 2 * q + 1]);
              }
            }
            __syncwarp();
          } else if (res32_fast) {
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
#pragma unroll
              for (int it = 0; it < 8; it++) sts128(stg + (uint32_t)(it * 4 + lr) * 128 + (uint32_t)((lp ^ ((it * 4 + lr) & 7)) << 4), rq[it]);
              __syncwarp();
              if (hh == 0) load_res32(1);                    // in flight while the first half is added
#pragma unroll
              for (int j = 0; j < 8; j++) {
                const uint4 rv = lds128(stg + (uint32_t)lane * 128 + (uint32_t)((j ^ (lane & 7)) << 4));
                f[hh * 32 + j * 4] += __uint_as_float(rv.x); f[hh * 32 + j * 4 + 1] += __uint_as_float(rv.y);
                f[hh * 32 + j * 4 + 2] += __uint_as_float(rv.z); f[hh * 32 + j * 4 + 3] += __uint_as_float(rv.w);
              }
              __syncwarp();
            }
          } else if (row_ok) {
            const int64_t ro = b * p.res_bstride + row * p.ldres + n00;
#pragma unroll
            for (int j = 0; j < 64; j++) {
              if (n00 + j < p.N) f[j] += p.res_f32 ? ((const float*)p.residual)[ro + j] : __bfloat162float(((const bf16*)p.residual)[ro + j]);
            }
          }
        }
        // ---- store
        if (tma_store_pending) {                             // the previous span's TMA store must have read the staging tile
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          __syncwarp();
          tma_store_pending = false;
        }
        if (out_bf16_fast && span_full) {
#pragma unroll
          for (int j = 0; j < 8; j++) {
            uint4 ov;
            __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&ov);
#pragma unroll
            for (int q = 0; q < 4; q++) h2[q] = __floats2bfloat162_rn(f[j * 8 + 2 * q], f[j * 8 + 2 * q + 1]);
            sts128(stg + (uint32_t)lane * 128 + (uint32_t)((j ^ (lane & 7)) << 4), ov);
          }
          if (p.tma_store) {
            // the staged 32 x 128 B tile already has the SWIZZLE_128B layout: hand it to the TMA engine (rows beyond M
            // are clipped by the tensor map) instead of spending 8 LDS + 8 STG per lane on it
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
              asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                           ::"l"(&map_c), "r"(stg), "r"((int32_t)n00), "r"((int32_t)row_base), "r"((int32_t)b) : "memory");
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            tma_store_pending = true;
          } else {
            __syncwarp();
            bf16* cp = (bf16*)p.C + b * p.c_bstride + n00 + lp * 8;
#pragma unroll
            for (int it = 0; it < 8; it++) {
              const int rr = it * 4 + lr;
              const uint4 ov = lds128(stg + (uint32_t)rr * 128 + (uint32_t)((lp ^ (rr & 7)) << 4));
              const int64_t rg = row_base + rr;
              if (rg < p.M) *reinterpret_cast<uint4*>(cp + rg * p.ldc) = ov;
            }
            __syncwarp();
          }
        } else if (out_f32_fast && span_full) {
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {                  // 32 fp32 columns = 128 B per row per pass
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const uint4 ov = make_uint4(__float_as_uint(f[hh * 32 + j * 4]), __float_as_uint(f[hh * 32 + j * 4 + 1]),
                                          __float_as_uint(f[hh * 32 + j * 4 + 2]), __float_as_uint(f[hh * 32 + j * 4 + 3]));
              sts128(stg + (uint32_t)lane * 128 + (uint32_t)((j ^ (lane & 7)) << 4), ov);
            }
            __syncwarp();
            float* cp = (float*)p.C + b * p.c_bstride + n00 + hh * 32 + lp * 4;
#pragma unroll
            for (int it = 0; it < 8; it++) {
              const int rr = it * 4 + lr;
              const uint4 ov = lds128(stg + (uint32_t)rr * 128 + (uint32_t)((lp ^ (rr & 7)) << 4));
              const int64_t rg = row_base + rr;
              if (rg < p.M) *reinterpret_cast<uint4*>(cp + rg * p.ldc) = ov;
            }
            __syncwarp();
          }
        } else if (row_ok) {                                // N tail / unaligned leading dimension: scalar path
          const int64_t co = b * p.c_bstride + row * p.ldc + n00;
#pragma unroll
          for (int j = 0; j < 64; j++) {
            if (n00 + j < p.N) {
              if (p.c_f32) ((float*)p.C)[co + j] = f[j];
              else ((bf16*)p.C)[co + j] = __float2bfloat16_rn(f[j]);
            }
          }
        }
      }
      // all TMEM reads of this warp are complete (wait::ld above): hand the accumulator back
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_leader(tempty_bar(acc));   // the leader's MMA thread waits for both CTAs' epilogues
        else mbar_arrive(tempty_bar(acc));
      }
      if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }

    }
    if constexpr (FILT) flt_flush();
  }

  if (warp >= 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // outstanding TMA stores
  tcgen05_fence_before();
  __syncwarp();
  if constexpr (PAIR) cluster_sync_all();      // no CTA may exit (or free TMEM) while its peer can still signal it
  else __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    if constexpr (PAIR) tmem_dealloc_pair<C::TMEM_COLS>(tmem_base);
    else tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

}  // namespace tc

// ----------------------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int get_encode_fn(cir_ctx* ctx, PFN_encodeTiled* fn) {
  if (!ctx->encode_tiled) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CIR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !p) {
      cir_set_error("cuTensorMapEncodeTiled not available from the driver");
      return CIR_EUNSUPPORTED;
    }
    ctx->encode_tiled = p;
  }
  *fn = (PFN_encodeTiled)ctx->encode_tiled;
  return CIR_OK;
}

// 2-D bf16 tensor map over a [rows, K] K-major matrix with row stride ld (elements); box = [box_rows, 64]
int cir_make_map_2d(cir_ctx* ctx, CUtensorMap* map, const void* base, int64_t rows, int64_t K, int64_t ld, int box_rows) {
  PFN_encodeTiled enc;
  CIR_TRY(get_encode_fn(ctx, &enc));
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)tc::BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    cir_set_error("cuTensorMapEncodeTiled failed (%d): base=%p rows=%lld K=%lld ld=%lld box_rows=%d", (int)r, base,
                  (long long)rows, (long long)K, (long long)ld, box_rows);
    return CIR_ECUDA;
  }
  return CIR_OK;
}

int cir_make_map_3d(cir_ctx* ctx, CUtensorMap* map, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t s1, int64_t s2,
                    int b0, int b1, int b2) {
  PFN_encodeTiled enc;
  CIR_TRY(get_encode_fn(ctx, &enc));
  cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t strides[2] = {(cuuint64_t)s1 * 2, (cuuint64_t)(d2 > 1 ? s2 : d1 * s1) * 2};
  cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, (cuuint32_t)b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    cir_set_error("cuTensorMapEncodeTiled (3-D) failed (%d): base=%p dims=(%lld,%lld,%lld) strides=(%lld,%lld) box=(%d,%d,%d)", (int)r, base,
                  (long long)d0, (long long)d1, (long long)d2, (long long)s1, (long long)s2, b0, b1, b2);
    return CIR_ECUDA;
  }
  return CIR_OK;
}

// C as (N, M, batch) with box [64 cols, 32 rows, 1]: one epilogue warp's staging tile
static int make_map_c(cir_ctx* ctx, CUtensorMap* map, const void* base, int64_t N, int64_t M, int64_t batch, int64_t ldc, int64_t c_bstride) {
  return cir_make_map_3d(ctx, map, base, N, M, batch, ldc, c_bstride, 64, 32, 1);
}

template <int BN, bool PAIR, bool FILT = false, bool TAGS = false>
static int launch_tc(cir_ctx* ctx, const tc::Params& p, const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& mc) {
  using C = tc::Cfg<BN, PAIR>;
  const auto kernel = tc::gemm_tcgen05_kernel<BN, PAIR, FILT, TAGS>;
  const unsigned bit = TAGS ? 1u << (12 + (PAIR ? 1 : 0))
                     : FILT ? 1u << (26 + (BN == 128 ? 0 : 1) + (PAIR ? 1 : 0))
                            : 1u << (8 + (BN == 128 ? 0 : 1) + (PAIR ? 2 : 0));   // per context: the attribute is per device
  if (!(ctx->func_attr_mask & bit)) {
    CIR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    ctx->func_attr_mask |= bit;
  }
  const int slots = PAIR ? ctx->num_sms / 2 : ctx->num_sms;
  const int workers = p.num_tiles < slots ? p.num_tiles : slots;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(PAIR ? 2 * workers : workers);
  cfg.blockDim = dim3(tc::THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cir_prof_gemm_begin(ctx, 2.0 * (double)p.M * (double)p.N * (double)p.K * (double)p.batch);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, ma, mw, mc, p);
  cir_prof_gemm_end(ctx);
  if (e != cudaSuccess) { cir_set_error("tcgen05 GEMM launch failed: %s", cudaGetErrorString(e)); return CIR_ECUDA; }
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_gemm_tcgen05(cir_ctx* ctx, const cir_gemm_args* a) {
  if (a->M == 0 || a->N == 0 || a->batch == 0) return CIR_OK;
  CIR_CHECK_ARG(ctx->dtype == CIR_DTYPE_BF16, "tcgen05 GEMM needs a bf16 context");
  CIR_CHECK_ARG(a->K % 8 == 0 && a->lda % 8 == 0 && a->ldw % 8 == 0, "tcgen05 GEMM: K, lda, ldw must be multiples of 8 (TMA 16 B strides)");
  CIR_CHECK_ARG(((uintptr_t)a->A & 15) == 0 && ((uintptr_t)a->W & 15) == 0, "tcgen05 GEMM: A and W must be 16 B aligned");
  CIR_CHECK_ARG(a->batch == 1 || (a->a_bstride % a->lda == 0 && a->w_bstride % a->ldw == 0),
                "tcgen05 GEMM: batch strides must be whole rows");
  tc::Params p{};
  p.C = a->C; p.bias = a->bias; p.residual = a->residual;
  p.M = a->M; p.N = a->N; p.K = a->K;
  p.ldc = a->ldc; p.ldres = a->ldres;
  p.c_bstride = a->c_bstride; p.bias_bstride = a->bias_bstride; p.res_bstride = a->res_bstride;
  p.batch = a->batch; p.act = a->act; p.c_f32 = a->c_f32; p.res_f32 = a->res_f32;
  p.a_rows_per_batch = a->batch > 1 ? a->a_bstride / a->lda : 0;
  p.w_rows_per_batch = a->batch > 1 ? a->w_bstride / a->ldw : 0;
  const int64_t a_rows = p.a_rows_per_batch * (a->batch - 1) + a->M;
  const int64_t w_rows = p.w_rows_per_batch * (a->batch - 1) + a->N;
  CIR_CHECK_ARG(a_rows < (1ll << 31) && w_rows < (1ll << 31), "tcgen05 GEMM: too many rows for a 32-bit TMA coordinate");
  // large problems: 256 x 256 CTA-pair tiles (cta_group::2); small ones: single-CTA tiles, narrower when
  // that is what it takes for the persistent grid to cover the SMs
  const int64_t tiles256 = ((a->M + tc::BM - 1) / tc::BM) * ((a->N + 255) / 256) * a->batch;
  const int64_t pair_tiles = ((a->M + 2 * tc::BM - 1) / (2 * tc::BM)) * ((a->N + 255) / 256) * a->batch;
  const bool use_pair = ctx->gemm_pair && (ctx->gemm_force_pair || pair_tiles >= ctx->num_sms / 2);
  const bool use128 = !use_pair && ((a->N <= 128) || (tiles256 < ctx->num_sms));
  const int BN = use128 ? 128 : 256;
  const int tile_m = use_pair ? 2 * tc::BM : tc::BM;
  p.m_blocks = (int32_t)((a->M + tile_m - 1) / tile_m);
  p.n_blocks = (int32_t)((a->N + BN - 1) / BN);
  p.k_blocks = (int32_t)((a->K + tc::BK - 1) / tc::BK);
  const int64_t nt = (int64_t)p.m_blocks * p.n_blocks * a->batch;
  CIR_CHECK_ARG(nt < (1ll << 31), "tcgen05 GEMM: too many tiles");
  p.num_tiles = (int32_t)nt;
  CUtensorMap ma, mw;
  CIR_TRY(cir_make_map_2d(ctx, &ma, a->A, a_rows, a->K, a->lda, tc::BM));
  CIR_TRY(cir_make_map_2d(ctx, &mw, a->W, w_rows, a->K, a->ldw, use_pair ? BN / 2 : BN));
  // bf16 outputs leave through TMA stores when the C layout is expressible as a tensor map (16 B aligned strides)
  CUtensorMap mc = ma;
  p.tma_store = 0;
  if (ctx->gemm_tma_store && !a->c_f32 && (a->ldc % 8) == 0 && (a->N % 64) == 0 && ((uintptr_t)a->C & 15) == 0 &&
      (a->batch == 1 || (a->c_bstride % 8) == 0) && a->M < (1ll << 31)) {
    CIR_TRY(make_map_c(ctx, &mc, a->C, a->N, a->M, a->batch, a->ldc, a->c_bstride));
    p.tma_store = 1;
  }
  if (use_pair) return launch_tc<256, true>(ctx, p, ma, mw, mc);
  if (use128) return launch_tc<128, false>(ctx, p, ma, mw, mc);
  return launch_tc<256, false>(ctx, p, ma, mw, mc);
}

// Similarity tiles with a threshold filter instead of an output matrix (stage-I top-K): S = A W^T is computed tile by tile on the
// tensor cores (bf16 operands, fp32 accumulation) and never stored; see cir_gemm_filter in common.cuh.
int cir_gemm_tcgen05_filter(cir_ctx* ctx, const void* A, const void* W, int64_t M, int64_t N, int64_t K, const cir_gemm_filter* f,
                            const uint32_t* col_tags, const uint32_t* row_masks) {
  if (M == 0 || N == 0) return CIR_OK;
  CIR_CHECK_ARG(ctx->dtype == CIR_DTYPE_BF16 && K % 64 == 0 && ((uintptr_t)A & 15) == 0 && ((uintptr_t)W & 15) == 0, "gemm_filter: bf16 context, K % 64 == 0, aligned operands");
  CIR_CHECK_ARG(M < (1ll << 31) && N < (1ll << 31) && f && f->thr && f->count && f->cand && f->overflow && f->cap > 0, "gemm_filter: bad argument");
  CIR_CHECK_ARG(!col_tags == !row_masks, "gemm_filter: column tags and row masks go together");
  tc::Params p{};
  p.M = M; p.N = N; p.K = K; p.batch = 1;
  p.flt = *f;
  p.n_major = 1;
  p.flt_col_tags = col_tags; p.flt_row_masks = row_masks;
  const int64_t pair_tiles = ((M + 2 * tc::BM - 1) / (2 * tc::BM)) * ((N + 255) / 256);
  const bool use_pair = ctx->gemm_pair && pair_tiles >= ctx->num_sms / 2;
  const int tile_m = use_pair ? 2 * tc::BM : tc::BM;
  p.m_blocks = (int32_t)((M + tile_m - 1) / tile_m);
  p.n_blocks = (int32_t)((N + 255) / 256);
  p.k_blocks = (int32_t)(K / tc::BK);
  const int64_t nt = (int64_t)p.m_blocks * p.n_blocks;
  CIR_CHECK_ARG(nt < (1ll << 31), "gemm_filter: too many tiles");
  p.num_tiles = (int32_t)nt;
  CUtensorMap ma, mw;
  CIR_TRY(cir_make_map_2d(ctx, &ma, A, M, K, K, tc::BM));
  CIR_TRY(cir_make_map_2d(ctx, &mw, W, N, K, K, use_pair ? 128 : 256));
  if (col_tags) return use_pair ? launch_tc<256, true, true, true>(ctx, p, ma, mw, ma) : launch_tc<256, false, true, true>(ctx, p, ma, mw, ma);
  return use_pair ? launch_tc<256, true, true>(ctx, p, ma, mw, ma) : launch_tc<256, false, true>(ctx, p, ma, mw, ma);
}
