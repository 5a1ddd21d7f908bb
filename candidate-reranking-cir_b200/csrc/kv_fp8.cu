// MXFP8 K/V gallery (CIR_KV_MXFP8, include/cir_b200.h): e4m3 elements with one E8M0 power-of-two scale per 32 channels.
//   quantise kernel   bf16 K/V rows of the fill GEMM -> elements + scales (one thread per 32-channel block)
//   dequant kernel    the K/V rows of a chunk's unique candidates -> bf16 [C][N][3072] in the workspace, the layout the
//                     uncached path's K/V GEMM writes; bandwidth-bound, 16-byte loads and stores
// Both conversions are exact where the format says so: x * 2^-k is exact in fp32 (a power-of-two product of a bf16 value, at
// most 448), and float(e) * 2^k fits bf16 for every k >= -127 the quantiser emits, so dequantisation reproduces bf16 bits.
#include "common.cuh"
#include <cuda_fp8.h>

namespace {

constexpr int KV_COLS = 4 * CIR_HIDDEN;          // K0|V0|K1|V1
constexpr int KV_BLOCK = 32;                     // channels per scale
constexpr int KV_SCALES = KV_COLS / KV_BLOCK;    // 96 per row
constexpr int DQ_THREADS = 256;
constexpr int DQ_UNROLL = 4;                     // 16-byte units per thread and item

// 2^(b - 127) as a float for a scale byte b in [0, 254]; b = 0 is the fp32 subnormal 2^-127
__device__ __forceinline__ float e8m0_to_f32(uint32_t b) { return b ? __uint_as_float(b << 23) : __uint_as_float(1u << 22); }

// One thread per block of 32 channels.  amax from the bf16 bit patterns (|x| orders like its bits for finite x).  With
// amax = (1 + M/128) 2^(E-127) (E >= 1): the smallest k with amax <= 448 2^k = 1.75 2^(k+8) is E - 135 when M <= 96 (mantissa
// <= 1.75), else E - 134; clamped at -127, which also covers E = 0 (zero and subnormal amax).  Scale byte = k + 127.
__global__ void __launch_bounds__(256) kv_mxfp8_quantize_kernel(const uint4* __restrict__ src, int64_t blocks, uint4* __restrict__ elems,
                                                                uint8_t* __restrict__ scales) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= blocks) return;
  uint4 v[4];
#pragma unroll
  for (int j = 0; j < 4; j++) v[j] = src[b * 4 + j];
  const uint32_t* w = reinterpret_cast<const uint32_t*>(v);
  uint32_t amax = 0;
#pragma unroll
  for (int j = 0; j < 16; j++) amax = max(amax, max(w[j] & 0x7FFFu, (w[j] >> 16) & 0x7FFFu));
  const int E = (int)(amax >> 7), M = (int)(amax & 0x7F);
  const int sb = max(0, M <= 96 ? E - 8 : E - 7);                    // k + 127
  const float inv = __uint_as_float((uint32_t)(254 - sb) << 23);    // 2^-k: 127 - k = 254 - sb in [7, 254]
  uint32_t o[8];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const float x0 = __uint_as_float(w[2 * j] << 16) * inv, x1 = __uint_as_float(w[2 * j] & 0xFFFF0000u) * inv;
    const float x2 = __uint_as_float(w[2 * j + 1] << 16) * inv, x3 = __uint_as_float(w[2 * j + 1] & 0xFFFF0000u) * inv;
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(x0, x1), __NV_SATFINITE, __NV_E4M3);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(x2, x3), __NV_SATFINITE, __NV_E4M3);
    o[j] = lo | (hi << 16);
  }
  elems[b * 2] = make_uint4(o[0], o[1], o[2], o[3]);
  elems[b * 2 + 1] = make_uint4(o[4], o[5], o[6], o[7]);
  scales[b] = (uint8_t)sb;
}

// 4 e4m3 bytes * 2^k -> 4 bf16 (two words); e4m3 -> f16 -> f32 are exact, the product is exact, so is its bf16 rounding
__device__ __forceinline__ uint2 dequant4(uint32_t q, float s) {
  const __half2_raw h0 = __nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(q & 0xFFFF), __NV_E4M3);
  const __half2_raw h1 = __nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(q >> 16), __NV_E4M3);
  const float2 f0 = __half22float2(__half2(h0)), f1 = __half22float2(__half2(h1));
  const __nv_bfloat162 b0 = __floats2bfloat162_rn(f0.x * s, f0.y * s), b1 = __floats2bfloat162_rn(f1.x * s, f1.y * s);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&b0), *reinterpret_cast<const uint32_t*>(&b1));
}

// Work item = (candidate c, slice xb of DQ_THREADS * DQ_UNROLL 16-byte units of its N * 192 units); CTAs stride over the items
// of the first n = *count (device count, may be NULL) or C candidates.  Cache row of candidate c: cand_list[c] - row0.
__global__ void __launch_bounds__(DQ_THREADS) kv_mxfp8_dequant_kernel(const uint8_t* __restrict__ elems, const uint8_t* __restrict__ scales,
                                                                      const int32_t* __restrict__ cand_list, int64_t row0, int64_t C,
                                                                      const int32_t* __restrict__ count, int64_t units, int xblocks,
                                                                      uint4* __restrict__ dst) {
  const int64_t n = count ? min((int64_t)*count, C) : C;
  for (int64_t item = blockIdx.x; item < n * xblocks; item += gridDim.x) {
    const int64_t c = item / xblocks, xb = item - c * xblocks;
    const int64_t row = cand_list[c] - row0;
    const uint4* src = reinterpret_cast<const uint4*>(elems) + row * units;
    const uint8_t* sc = scales + row * (units / 2);
    uint4* out = dst + c * units * 2;
    const int64_t u0 = xb * (DQ_THREADS * DQ_UNROLL) + threadIdx.x;
    uint4 v[DQ_UNROLL];
    uint32_t s[DQ_UNROLL];
#pragma unroll
    for (int j = 0; j < DQ_UNROLL; j++) {
      const int64_t u = u0 + j * DQ_THREADS;
      if (u < units) { v[j] = __ldg(src + u); s[j] = __ldg(sc + (u >> 1)); }
    }
#pragma unroll
    for (int j = 0; j < DQ_UNROLL; j++) {
      const int64_t u = u0 + j * DQ_THREADS;
      if (u < units) {
        const float f = e8m0_to_f32(s[j]);
        const uint2 a = dequant4(v[j].x, f), b = dequant4(v[j].y, f), c2 = dequant4(v[j].z, f), d = dequant4(v[j].w, f);
        out[u * 2] = make_uint4(a.x, a.y, b.x, b.y);
        out[u * 2 + 1] = make_uint4(c2.x, c2.y, d.x, d.y);
      }
    }
  }
}

}  // namespace

// bf16 src [rows][3072] -> e4m3 elems [rows][3072] + E8M0 scales [rows][96]
int cir_kv_mxfp8_quantize(cir_ctx* ctx, const void* src, int64_t rows, void* elems, uint8_t* scales) {
  const int64_t blocks = rows * KV_SCALES;
  if (blocks == 0) return CIR_OK;
  kv_mxfp8_quantize_kernel<<<(unsigned)((blocks + 255) / 256), 256, 0, ctx->stream>>>(
      reinterpret_cast<const uint4*>(src), blocks, reinterpret_cast<uint4*>(elems), scales);
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}

// layer i of an MXFP8 cache, candidates cand_list[0 .. C) (gallery rows; only the first *count when count is not NULL) ->
// dst bf16 [C][N][3072]
int cir_kv_mxfp8_dequant(cir_ctx* ctx, const cir_stage2_kv_cache* cache, int i, const int32_t* cand_list, int64_t C,
                         const int32_t* count, void* dst) {
  const int64_t rn = cache->rows * cache->num_tokens;
  const uint8_t* elems = (const uint8_t*)cache->kv + (int64_t)i * rn * KV_COLS;
  const uint8_t* scales = (const uint8_t*)cache->kv + (int64_t)CIR_LAYERS * rn * KV_COLS + (int64_t)i * rn * KV_SCALES;
  const int64_t units = cache->num_tokens * (KV_COLS / 16);
  const int xblocks = (int)((units + DQ_THREADS * DQ_UNROLL - 1) / (DQ_THREADS * DQ_UNROLL));
  const int64_t items = C * xblocks, cap = (int64_t)ctx->num_sms * 8, grid = items < cap ? items : cap;
  kv_mxfp8_dequant_kernel<<<(unsigned)grid, DQ_THREADS, 0, ctx->stream>>>(elems, scales, cand_list, cache->row0, C, count, units, xblocks,
                                                                          reinterpret_cast<uint4*>(dst));
  CIR_LAUNCH_CHECK(ctx);
  return CIR_OK;
}
