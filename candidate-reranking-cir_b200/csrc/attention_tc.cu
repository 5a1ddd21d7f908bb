// tcgen05 / TMEM flash attention (bf16, head dim 64, no key mask): the cross-attention of the
// dual-stream encoder (32 text rows x 577 image keys per (triplet, stream, head),
// src/nlvr_encoder.py:175-217) and the ViT self-attention (src/vit.py:74-82).
//
// A work item = one 256-row query "double tile" of one head: two 128-row UMMA tiles A and B that attend the SAME
// K/V batch, so every K/V chunk is fetched once per 256 query rows.  A double tile is (256/RB) batches x RB rows
// (candidate-major triplets: 8 triplets x 32 rows share one candidate image), which fills the 128-row UMMA shape
// although a triplet has only 32 query rows.  One persistent CTA per SM walks the items with a stride of the grid
// size; rings, S/P buffers and mbarrier phases run on chunk counters that keep counting across items, so the next
// item's Q/K/V loads and first S products overlap the current item's tail.
//
//   warps 0-3   softmax of tile A, warps 4-7 softmax of tile B: thread r owns query row r == TMEM lane r.  Per
//               64-key chunk ONE tcgen05.ld sweep brings the row's scores into registers, row max -> exp2 -> packed bf16
//               P written straight back into TENSOR memory (tcgen05.st) over the first 32 columns of the S buffer it
//               came from; the PV product takes its A operand from TMEM, so P never touches shared memory.  S is
//               double-buffered per tile, so the tensor core computes S_{j+1}, S_{j+2} while the softmax works on
//               chunk j.  O accumulates in TMEM across chunks; the reference max moves lazily (only when the row
//               max grew by more than 2^8), so the O rescale (tcgen05.ld / tcgen05.st) is a rare path.
//   warp 8/9    one elected thread each: all tcgen05.mma issue of tile A / tile B:
//                 S_j = Q K_j^T  (A=Q smem, B=K_j smem, both K-major)
//                 O  += P_j V_j  (A=P in TMEM, B=V_j smem MN-major)
//               and the commits that hand the K / V ring stages back to the loader (2 arrivals per stage).
//   warp 10     one elected thread: TMA loads of Q tiles (3-D map, double-buffered per tile) and of the K / V
//               chunks into 6-deep rings -- deep enough that the L2 -> shared-memory latency under load
//               (> 1 us) never reaches the MMA issue loop.
//   TMEM: per tile S0/P0, S1/P1 (64 columns each) + O (64).  Scores and probabilities never leave the SM.
#include <algorithm>
#include <type_traits>
#include "common.cuh"
#include "tcgen05_ptx.cuh"

namespace fatc {

using namespace tc;

constexpr int KC = 64;                  // keys per chunk
constexpr int KS = 6;                   // K / V ring depth
constexpr int THREADS = 352;            // 8 softmax warps + 2 MMA-issue warps + 1 loader warp
constexpr int Q_BYTES = 128 * 128;      // 128 rows x 64 bf16
constexpr int KV_BYTES = KC * 128;      // 64 keys x 64 bf16
constexpr int P_BYTES = 128 * 128;      // O staging tile: [128 rows x 64 dims] bf16
constexpr int OFF_Q = 0;                               // [tile][item parity]
constexpr int OFF_P = OFF_Q + 4 * Q_BYTES;             // [tile]: staging of the O tile for its TMA store (P itself lives in TMEM)
constexpr int OFF_K = OFF_P + 2 * P_BYTES;
constexpr int OFF_V = OFF_K + KS * KV_BYTES;
constexpr int OFF_BAR = OFF_V + KS * KV_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 512;
constexpr int TMEM_COLS = 512;
constexpr int TILE_COLS = 256;          // TMEM columns per tile: S buffers at +0 and +64, O at +128
constexpr int S_COL = 0, O_COL = 128;
static_assert(SMEM_BYTES <= 232448, "attention_tc: shared memory budget");

// instruction descriptor with an MN-major B operand (V is [key][dh], dh contiguous): bit 16
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(int m, int n) { return make_idesc_bf16(m, n) | (1u << 16); }

__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {       // one MUFU.EX2; exp2(-inf) = 0, denormal results flush to 0
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// packed fp32 pairs (FFMA2 / FADD2 on sm_100: one issue slot for two IEEE fp32 operations)
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// O[row, 0:64] *= alpha in TMEM (whole warp, each lane its own row/alpha); rare path, kept out of line
__device__ __noinline__ void rescale_o(uint32_t o_addr, float alpha) {
#pragma unroll
  for (int hh = 0; hh < 2; hh++) {
    uint32_t ov[32];
    __syncwarp();
    tmem_ld_32x32b_x32(o_addr + hh * 32, ov);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; i++) ov[i] = __float_as_uint(__uint_as_float(ov[i]) * alpha);
    tmem_st_32x32b_x32(o_addr + hh * 32, ov);
  }
  tmem_st_wait();
}

struct Item { int batch0, nb, row0, kvrow0, h; };

// work item w = head * ntiles + tile (tile fastest: CTAs running side by side share one candidate's K/V head slice in L2)
__device__ __forceinline__ Item decode_item(const cir_attn_args& p, int w, int ntiles, int cpb, int RB) {
  Item it;
  it.h = w / ntiles;
  const int t = w - it.h * ntiles;
  if (p.tiles) {
    const int4 d = __ldg(reinterpret_cast<const int4*>(p.tiles) + t);
    it.batch0 = d.x; it.nb = d.y; it.row0 = d.z;
    if (d.w != RB) { printf("cir: attention tile %d built for RB=%d, kernel geometry RB=%d (see cir_attn_args.tiles)\n", t, d.w, RB); __trap(); }
  } else {
    it.batch0 = t / cpb; it.nb = 1; it.row0 = (t - it.batch0 * cpb) * 256;
  }
  const int kvb = p.kv_index ? __ldg(p.kv_index + it.batch0) : it.batch0;
  it.kvrow0 = kvb * p.Lk;
  return it;
}

// the softmax warps only need the row geometry of an item: one load, consumed an item later
__device__ __forceinline__ Item decode_rows(const cir_attn_args& p, int w, int ntiles, int cpb) {
  Item it;
  it.h = w / ntiles;
  const int t = w - it.h * ntiles;
  it.kvrow0 = 0;
  if (p.tiles) {
    const int4 d = __ldg(reinterpret_cast<const int4*>(p.tiles) + t);
    it.batch0 = d.x; it.nb = d.y; it.row0 = d.z;
  } else {
    it.batch0 = t / cpb; it.nb = 1; it.row0 = (t - it.batch0 * cpb) * 256;
  }
  return it;
}

// COUNTED: the tile count is read once from ntiles_dev (written on the device by an earlier kernel of the stream, e.g. the
// on-device planner of cir_stage2_rerank_cached); the grid was sized from the host bound `ntiles`, and CTAs past the device
// count have no items.  Every role derives its items from this one value.
template <bool COUNTED>
__global__ void __launch_bounds__(THREADS, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_o, const cir_attn_args p,
                    int cpb, int ntiles, int RB, int total, const int32_t* __restrict__ ntiles_dev) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (COUNTED) {
    ntiles = __ldg(ntiles_dev);
    total = ntiles * p.H;
  }
  const int nch = (p.Lk + KC - 1) / KC;
  const int n_my = (int)blockIdx.x < total ? (total - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int total_g = n_my * nch;

  // barriers: kfull[KS] vfull[KS] kempty[KS] vempty[KS] | per tile: sfull[2] pfull[2] pvdone[2] qfull[2] | tmem_ptr
  // (S / P / pvdone indexed by chunk parity, Q by item parity, so a waiter is never more than one phase behind)
  const uint32_t bar = sbase + OFF_BAR;
  auto kfull = [&](int s) { return bar + 8u * s; };
  auto vfull = [&](int s) { return bar + 8u * (KS + s); };
  auto kempty = [&](int s) { return bar + 8u * (2 * KS + s); };
  auto vempty = [&](int s) { return bar + 8u * (3 * KS + s); };
  auto sfull = [&](int t, int b) { return bar + 8u * (4 * KS + t * 8 + b); };
  auto pfull = [&](int t, int b) { return bar + 8u * (4 * KS + t * 8 + 2 + b); };
  auto pvdone = [&](int t, int b) { return bar + 8u * (4 * KS + t * 8 + 4 + b); };
  auto qfull = [&](int t, int b) { return bar + 8u * (4 * KS + t * 8 + 6 + b); };
  const uint32_t tmem_ptr_smem = bar + 8u * (4 * KS + 16);
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem + OFF_BAR + 8 * (4 * KS + 16));

  if ((sbase & 1023u) != 0) { if (tid == 0) printf("cir: attention_tc smem misaligned\n"); __trap(); }
  if (warp == 8) {
    if (elect_one()) {
      tma_prefetch_desc(&map_q);
      tma_prefetch_desc(&map_k);
      tma_prefetch_desc(&map_v);
      for (int s = 0; s < KS; s++) { mbar_init(kfull(s), 1); mbar_init(vfull(s), 1); mbar_init(kempty(s), 2); mbar_init(vempty(s), 2); }
      for (int t = 0; t < 2; t++)
        for (int b = 0; b < 2; b++) { mbar_init(sfull(t, b), 1); mbar_init(pfull(t, b), 4); mbar_init(pvdone(t, b), 1); mbar_init(qfull(t, b), 1); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc<TMEM_COLS>(tmem_ptr_smem);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  auto n_pad_of = [&](int j) {
    const int keys = (p.Lk - j * KC) < KC ? (p.Lk - j * KC) : KC;
    return (keys + 15) & ~15;                                // UMMA N (multiple of 16); padded keys are masked in the softmax
  };

  if (warp == 10) {
    // ===================== loader: TMA for Q tiles and the K / V rings =====================
    if (elect_one() && total_g > 0) {
      auto dec = [&](int i) { return i < n_my ? decode_item(p, (int)blockIdx.x + i * (int)gridDim.x, ntiles, cpb, RB) : Item{}; };
      // items i_cur .. i_cur+2 decoded ahead: the two dependent global loads of a decode never stall the ring
      Item it0 = dec(0), it1 = dec(1), it2 = dec(2);
      int i_cur = 0;
      auto item_at = [&](int i) -> Item { return i == i_cur ? it0 : (i == i_cur + 1 ? it1 : (i == i_cur + 2 ? it2 : dec(i))); };
      const int rbq = RB < 128 ? RB : 128;                   // rows per batch inside one 128-row tile
      auto issue_q = [&](int i) {                           // both tiles of item i; rows / batches out of bounds arrive as zeros
        const Item it = item_at(i);
#pragma unroll
        for (int t = 0; t < 2; t++) {
          mbar_expect_tx(qfull(t, i & 1), Q_BYTES);
          const int row = RB > 128 ? it.row0 + t * 128 : it.row0;
          const int bat = RB > 128 ? it.batch0 : it.batch0 + t * (128 / rbq);
          tma_load_3d(sbase + OFF_Q + (t * 2 + (i & 1)) * Q_BYTES, &map_q, qfull(t, i & 1), it.h * 64, row, bat);
        }
      };
      int q_next = 0;
      for (; q_next < 2 && q_next < n_my; q_next++) issue_q(q_next);
      int i = 0, j = 0;
      for (int g = 0; g < total_g; g++) {
        const int s = g % KS;
        const uint32_t ph = (uint32_t)((g / KS) & 1);
        const Item it = item_at(i);
        if (g >= KS) mbar_wait(kempty(s), ph ^ 1u);          // both tiles' S_{g-KS} retired
        mbar_expect_tx(kfull(s), KV_BYTES);
        tma_load_2d(sbase + OFF_K + s * KV_BYTES, &map_k, kfull(s), it.h * 64, it.kvrow0 + j * KC);
        if (g >= KS) mbar_wait(vempty(s), ph ^ 1u);          // both tiles' PV_{g-KS} retired
        mbar_expect_tx(vfull(s), KV_BYTES);
        tma_load_2d(sbase + OFF_V + s * KV_BYTES, &map_v, vfull(s), it.h * 64, it.kvrow0 + j * KC);
        // Q buffers of item q_next were last read by the S products of item q_next-2, whose last chunk is
        // (q_next-1)*nch - 1: its kempty has been observed once this loop has passed g = that + KS
        while (q_next < n_my && (q_next - 1) * nch - 1 + KS <= g) issue_q(q_next++);
        if (++j == nch) { j = 0; i++; i_cur = i; it0 = it1; it1 = it2; it2 = dec(i + 2); }
      }
      while (q_next < n_my) {                                // only reachable when nch < KS / 2: the ring never wrapped that far
        const int need = (q_next - 1) * nch - 1;             // chunk whose S products must have retired
        mbar_wait(kempty(need % KS), (uint32_t)((need / KS) & 1));
        issue_q(q_next++);
      }
    }
  } else if (warp >= 8) {
    // ===================== MMA issue for tile t =====================
    const int t = warp - 8;
    if (elect_one() && total_g > 0) {
      const uint32_t tm = tmem_base + t * TILE_COLS;
      auto issue_s = [&](int g) {                           // S[g&1] = Q_i K_j^T
        const int i = g / nch, j = g - i * nch, s = g % KS;
        if (j == 0) mbar_wait(qfull(t, i & 1), (uint32_t)((i >> 1) & 1));
        mbar_wait(kfull(s), (uint32_t)((g / KS) & 1));
        tcgen05_fence_after();
        const uint64_t qdesc = make_smem_desc_sw128(sbase + OFF_Q + (t * 2 + (i & 1)) * Q_BYTES);
        const uint64_t kdesc = make_smem_desc_sw128(sbase + OFF_K + s * KV_BYTES);
        const uint32_t idesc = make_idesc_bf16(128, n_pad_of(j));
#pragma unroll
        for (int k = 0; k < 4; k++)
          umma_bf16(tm + S_COL + (g & 1) * 64, qdesc + (uint64_t)(k * 2), kdesc + (uint64_t)(k * 2), idesc, (uint32_t)(k != 0));
        umma_commit(sfull(t, g & 1));
        umma_commit(kempty(s));                              // this tile is done with K stage s
      };
      issue_s(0);
      if (total_g > 1) issue_s(1);
      int j = 0;
      for (int g = 0; g < total_g; g++) {
        const int s = g % KS;
        mbar_wait(pfull(t, g & 1), (uint32_t)((g >> 1) & 1));    // P_g in shared memory, S_g consumed, O rescaled if needed
        mbar_wait(vfull(s), (uint32_t)((g / KS) & 1));
        tcgen05_fence_after();
        {                                                    // O (+)= P_g V_g, accumulating in TMEM across the item's chunks
          const uint32_t idesc = make_idesc_bf16_bmn(128, 64);
          const int ksteps = n_pad_of(j) >> 4;
          for (int k = 0; k < ksteps; k++) {
            const uint32_t p_tmem = tm + S_COL + (g & 1) * 64 + k * 8;     // P_g overwrote S_g: 16 keys = 8 packed columns per K step
            const uint64_t vdesc = make_smem_desc_sw128(sbase + OFF_V + s * KV_BYTES + k * 2048);                          // 16 key rows x 128 B
            umma_bf16_ts(tm + O_COL, p_tmem, vdesc, idesc, (uint32_t)((j | k) != 0));
          }
          umma_commit(pvdone(t, g & 1));
          umma_commit(vempty(s));                            // this tile is done with V stage s
        }
        if (g + 2 < total_g) issue_s(g + 2);                 // S buffer g&1 was drained before pfull(g)
        if (++j == nch) j = 0;
      }
    }
  } else {
    // ===================== softmax warps: thread = query row = TMEM lane =====================
    const int t = warp >> 2;                                 // tile A (warps 0-3) or B (warps 4-7)
    const int r = tid & 127;                                 // row inside the tile == TMEM lane
    const int rr = t * 128 + r;                              // row inside the double tile
    const uint32_t lane_addr = tmem_base + t * TILE_COLS + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t o_addr = lane_addr + O_COL;
    const float sl2 = p.scale * 1.4426950408889634f;
    // Warp w of tile A and warp w of tile B sit on the same scheduler and share its MUFU.  Left alone they fall into
    // lock-step: both exp2 phases collide, and the unit idles while both do max / waits / tcgen05.ld.  Two named
    // barriers per warp pair make the exp2 phases strictly alternate, so one tile's exp2 runs under the other's
    // non-MUFU work.
    const int wq = warp & 3;
    auto turn_wait = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(t == 0 ? 5 + wq : 1 + wq) : "memory"); };
    auto turn_pass = [&]() { asm volatile("bar.arrive %0, 64;" ::"r"(t == 0 ? 1 + wq : 5 + wq) : "memory"); };
    int g = 0;
    Item nxt = n_my > 0 ? decode_rows(p, (int)blockIdx.x, ntiles, cpb) : Item{};
    bool o_pending = false;                                  // a TMA store of this warp may still be reading its staging slice
    for (int it_i = 0; it_i < n_my; it_i++) {
      const Item it = nxt;
      if (it_i + 1 < n_my) nxt = decode_rows(p, (int)blockIdx.x + (it_i + 1) * (int)gridDim.x, ntiles, cpb);   // off the critical path
      const int bi = rr / RB, qi = it.row0 + rr % RB;
      const bool valid = bi < it.nb && qi < p.Lq;
      const int b = it.batch0 + (bi < it.nb ? bi : 0);
      float m = -INFINITY, l = 0.f;                          // m: lazily updated reference max (scaled log2 domain)
      for (int j = 0; j < nch; j++, g++) {
        const int pb = g & 1;
        const int keys = (p.Lk - j * KC) < KC ? (p.Lk - j * KC) : KC;
        const bool full_chunk = keys == KC;
        const bool two = keys > 32;                          // second 32-column piece needed?
        mbar_wait(sfull(t, pb), (uint32_t)((g >> 1) & 1));
        tcgen05_fence_after();
        // ---- the row's 64 scores -> registers in one sweep
        uint32_t v0[32], v1[32];
        __syncwarp();
        tmem_ld_32x32b_x32(lane_addr + S_COL + pb * 64, v0);
        if (two) tmem_ld_32x32b_x32(lane_addr + S_COL + pb * 64 + 32, v1);
        else {
#pragma unroll
          for (int x = 0; x < 32; x++) v1[x] = 0u;
        }
        tmem_ld_wait();
        // ---- row max of the chunk
        float cmax = -INFINITY;
        if (full_chunk) {                                    // four independent FMNMX3 chains (8 deep instead of 32)
          float c0 = -INFINITY, c1 = -INFINITY, c2 = -INFINITY, c3 = -INFINITY;
#pragma unroll
          for (int x = 0; x < 16; x += 2) {
            c0 = max3(c0, __uint_as_float(v0[x]), __uint_as_float(v0[x + 1]));
            c1 = max3(c1, __uint_as_float(v0[16 + x]), __uint_as_float(v0[17 + x]));
            c2 = max3(c2, __uint_as_float(v1[x]), __uint_as_float(v1[x + 1]));
            c3 = max3(c3, __uint_as_float(v1[16 + x]), __uint_as_float(v1[17 + x]));
          }
          cmax = fmaxf(max3(c0, c1, c2), c3);
        } else {
#pragma unroll
          for (int x = 0; x < 32; x++) if (x < keys) cmax = fmaxf(cmax, __uint_as_float(v0[x]));
          if (two) {
#pragma unroll
            for (int x = 0; x < 32; x++) if (32 + x < keys) cmax = fmaxf(cmax, __uint_as_float(v1[x]));
          }
        }
        cmax *= sl2;                                         // scale > 0: max commutes with the scaling
        // ---- lazy reference max: move it only when the row max grew by more than 2^8; the (rare) move rescales
        //      l and the O accumulator in TMEM.  Otherwise exp2(s - m) <= 256: harmless in fp32 / bf16.
        const bool grow = cmax > m + 8.0f;
        if (j == 0) {
          m = cmax;
        } else if (__any_sync(0xffffffffu, grow)) {
          mbar_wait(pvdone(t, (g - 1) & 1), (uint32_t)(((g - 1) >> 1) & 1));   // every PV issued so far has retired
          tcgen05_fence_after();
          const float m_new = grow ? cmax : m;
          const float alpha = ex2_approx(m - m_new);         // 1 for rows that keep their reference
          l *= alpha;
          m = m_new;
          rescale_o(o_addr, alpha);
        }
        // ---- P = exp2(S*c - m) as packed bf16 back into TENSOR memory, over the first 32 columns of the S buffer it was
        //      read from (the A operand of the PV product comes from TMEM: no shared-memory round trip, no proxy fence).
        //      PV_{g-2}, the last reader of these columns, retired before S_g was written (in-order pipe), so no wait.
        //      Two instantiations: full chunks carry no per-element masking; the tail chunk zero-fills the padded keys.
        auto exp_pack = [&](auto full_tag) {
          constexpr bool FULL = decltype(full_tag)::value;
          const uint64_t sl2_2 = pack_f32x2(sl2, sl2), negm_2 = pack_f32x2(-m, -m);
          uint64_t lsum = pack_f32x2(0.f, 0.f);              // two partial row sums (even / odd keys)
#pragma unroll
          for (int c = 0; c < 8; c++) {
            float e[8];
#pragma unroll
            for (int q = 0; q < 8; q += 2) {
              const int x = c * 8 + q;
              const uint32_t s0 = x < 32 ? v0[x & 31] : v1[x & 31], s1 = x < 32 ? v0[(x + 1) & 31] : v1[(x + 1) & 31];
              float a0, a1;
              unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(s0), __uint_as_float(s1)), sl2_2, negm_2), a0, a1);   // one FFMA2 per key pair
              e[q] = ex2_approx(a0);
              e[q + 1] = ex2_approx(a1);
              if (!FULL && x >= keys) e[q] = 0.f;
              if (!FULL && x + 1 >= keys) e[q + 1] = 0.f;
            }
            lsum = add_f32x2(lsum, add_f32x2(add_f32x2(pack_f32x2(e[0], e[1]), pack_f32x2(e[2], e[3])),
                                             add_f32x2(pack_f32x2(e[4], e[5]), pack_f32x2(e[6], e[7]))));
#pragma unroll
            for (int q = 0; q < 4; q++) {
              const __nv_bfloat162 h2 = __floats2bfloat162_rn(e[2 * q], e[2 * q + 1]);
              v0[c * 4 + q] = *reinterpret_cast<const uint32_t*>(&h2);       // in place: scores 8c.. of v0 / v1 are consumed by now
            }
          }
          float la, lb;
          unpack_f32x2(lsum, la, lb);
          l += la + lb;
        };
        if (t == 1 || g > 0) turn_wait();
        if (full_chunk) exp_pack(std::true_type{}); else exp_pack(std::false_type{});
        turn_pass();
        __syncwarp();
        tmem_st_32x32b_x32(lane_addr + S_COL + pb * 64, v0);
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pfull(t, pb));
      }
      // ---- O, normalise, store.  The next item's first PV (accumulate = 0) is issued only after these warps signal
      //      its pfull, i.e. after this read of O: one O accumulator per tile suffices.
      mbar_wait(pvdone(t, (g - 1) & 1), (uint32_t)(((g - 1) >> 1) & 1));
      tcgen05_fence_after();
      if (o_pending) {                                       // the previous item's O tile may still be read from the staging slice
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
        o_pending = false;
      }
      const float inv = 1.0f / l;
      // A warp's 32 rows are one batch when RB >= 32: the tile then leaves as ONE TMA store (rows >= Lq clipped by the
      // map) staged in this warp's 4 KB slice of the tile's staging buffer.  Otherwise per-row stores.
      const int rr0 = t * 128 + (warp & 3) * 32;
      const bool warp_tma = RB >= 32 && (rr0 / RB) < it.nb;
      const bool warp_skip = RB >= 32 && !warp_tma;          // the warp's batch does not exist in this tile
      uint8_t* stage = smem + OFF_P + t * P_BYTES + (warp & 3) * 4096 + lane * 128;
      uint4* dst = reinterpret_cast<uint4*>((bf16*)p.o + (int64_t)b * p.o_bs + (int64_t)qi * p.o_rs + it.h * 64);
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
        uint32_t ov[32];
        __syncwarp();
        tmem_ld_32x32b_x32(o_addr + hh * 32, ov);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 4; c++) {
          uint4 w;
          __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&w);
#pragma unroll
          for (int q = 0; q < 4; q++)
            h2[q] = __floats2bfloat162_rn(__uint_as_float(ov[c * 8 + 2 * q]) * inv, __uint_as_float(ov[c * 8 + 2 * q + 1]) * inv);
          if (warp_tma) *reinterpret_cast<uint4*>(stage + (((hh * 4 + c) ^ (lane & 7)) << 4)) = w;
          else if (valid && !warp_skip) dst[hh * 4 + c] = w;
        }
      }
      if (warp_tma) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          const int bw = it.batch0 + rr0 / RB, qw = it.row0 + rr0 % RB;
          asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                       ::"l"(&map_o), "r"(smem_u32(stage)), "r"(it.h * 64), "r"(qw), "r"(bw) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        o_pending = true;
      }
      tcgen05_fence_before();                                // O reads ordered before the pfull arrive that releases the next PV
    }
  }
  if (warp < 4 && total_g > 0) asm volatile("bar.sync %0, 64;" ::"r"(5 + (warp & 3)) : "memory");   // tile B's last turn_pass
  if (warp < 8 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // outstanding O stores
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 8) {
    tcgen05_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

}  // namespace fatc

// ntiles_dev == NULL: the tile count is a->num_tiles (or one tile per 256-row slice of every batch without a tile list).
// Otherwise a->tiles is required, a->num_tiles bounds the count the kernel reads from ntiles_dev, and the grid is sized from that bound.
static int attention_tc_launch(cir_ctx* ctx, const cir_attn_args* a, const int32_t* ntiles_dev) {
  // eligibility (the caller falls back to the mma.sync kernel on CIR_EUNSUPPORTED)
  if (ctx->dtype != CIR_DTYPE_BF16 || a->key_mask != nullptr || a->Lk < 16 || a->kv_batches <= 0 || a->H * 64 > 65536 ||
      a->k_bs != (int64_t)a->Lk * a->k_rs || a->v_bs != (int64_t)a->Lk * a->v_rs || (a->k_rs % 8) || (a->v_rs % 8) ||
      ((uintptr_t)a->k & 15) || ((uintptr_t)a->v & 15) || ((uintptr_t)a->q & 15) || ((uintptr_t)a->o & 15) ||
      (a->q_rs % 8) || (a->q_bs % 8) || (a->o_rs % 8) || (a->o_bs % 8))
    return CIR_EUNSUPPORTED;
  if (!a->tiles && a->Lq <= 64 && a->B > 1) return CIR_EUNSUPPORTED;      // unshared short queries would waste most of every tile
  const int64_t kv_rows = (int64_t)a->kv_batches * a->Lk;
  if (kv_rows >= (1ll << 31)) return CIR_EUNSUPPORTED;
  // double-tile geometry: RB rows per batch (schedule.build_attn_tiles: smallest power of two >= Lq, at most 256)
  int RB = 256;
  if (a->tiles) { RB = 1; while (RB < a->Lq && RB < 256) RB <<= 1; }
  const int rbq = RB < 128 ? RB : 128;
  CUtensorMap mq, mk, mv, mo;
  CIR_TRY(cir_make_map_3d(ctx, &mq, a->q, (int64_t)a->H * 64, a->Lq, a->B, a->q_rs, a->q_bs, 64, rbq, 128 / rbq));
  CIR_TRY(cir_make_map_3d(ctx, &mo, a->o, (int64_t)a->H * 64, a->Lq, a->B, a->o_rs, a->o_bs, 64, 32, 1));
  CIR_TRY(cir_make_map_2d(ctx, &mk, a->k, kv_rows, (int64_t)a->H * 64, a->k_rs, fatc::KC));
  CIR_TRY(cir_make_map_2d(ctx, &mv, a->v, kv_rows, (int64_t)a->H * 64, a->v_rs, fatc::KC));
  const unsigned bit = ntiles_dev ? 1u << 4 : 1u << 3;       // per context: the attribute is per device
  if (!(ctx->func_attr_mask & bit)) {
    CIR_CUDA(cudaFuncSetAttribute(ntiles_dev ? (const void*)fatc::attention_tc_kernel<true> : (const void*)fatc::attention_tc_kernel<false>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, fatc::SMEM_BYTES));
    ctx->func_attr_mask |= bit;
  }
  const int cpb = (a->Lq + 255) / 256;
  const int64_t ntiles = a->tiles ? (int64_t)a->num_tiles : (int64_t)a->B * cpb;
  const int64_t total = ntiles * a->H;
  if (total == 0) return CIR_OK;
  if (total >= (1ll << 31)) return CIR_EUNSUPPORTED;
  const unsigned gx = (unsigned)std::min<int64_t>(total, (int64_t)ctx->num_sms);      // persistent: one CTA per SM
  cir_prof_begin(ctx, CIR_PROF_ATTN_TC, 4.0 * (double)a->B * a->H * (double)a->Lq * (double)a->Lk * 64.0);
  if (ntiles_dev)
    fatc::attention_tc_kernel<true><<<gx, fatc::THREADS, fatc::SMEM_BYTES, ctx->stream>>>(mq, mk, mv, mo, *a, 1, 0, RB, 0, ntiles_dev);
  else
    fatc::attention_tc_kernel<false><<<gx, fatc::THREADS, fatc::SMEM_BYTES, ctx->stream>>>(mq, mk, mv, mo, *a, cpb, (int)ntiles, RB, (int)total,
                                                                                          nullptr);
  cir_prof_end(ctx);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

int cir_attention_tc(cir_ctx* ctx, const cir_attn_args* a) { return attention_tc_launch(ctx, a, nullptr); }

int cir_attention_tc_counted(cir_ctx* ctx, const cir_attn_args* a, const int32_t* ntiles_dev) {
  CIR_CHECK_ARG(a->tiles && ntiles_dev, "attention_tc_counted: needs a tile list and its device count");
  return attention_tc_launch(ctx, a, ntiles_dev);
}
