// common.cuh — shared device helpers of the b2f engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace b2f {

constexpr int kD = 768;            // reference drivers/run_convdr_inference.py:353
constexpr int kRowF4 = kD / 4;     // float4 chunks per row (192)
constexpr int kF4PerLane = kRowF4 / 32;  // 6 float4 per lane per row

// ---------------------------------------------------------------------------------------------
// Layout of the bf16 shadow copy streamed by the tensor engine: "K-block-major tiles".
// Rows are grouped in tiles of 32; inside a tile the 12 K-blocks (64 columns = 128 bytes each)
// are stored one after the other, each as 32 rows x 128 bytes.  One TMA stage (32 rows of four
// consecutive K-blocks) is therefore ONE contiguous 16 KB read instead of 128-byte granules strided
// by the 1536-byte row pitch, and a CTA's whole tile is one contiguous 48 KB region.
// Element (row, col) lives at shadow_index(row, col) (in bf16 elements).
// ---------------------------------------------------------------------------------------------
constexpr int kShadowTileRows = 32;
constexpr int kShadowKBlock = 64;
__host__ __device__ __forceinline__ int64_t shadow_index(int64_t row, int col) {
  const int64_t tile = row / kShadowTileRows;
  const int r = static_cast<int>(row % kShadowTileRows);
  const int kb = col / kShadowKBlock, c = col % kShadowKBlock;
  return ((tile * (kD / kShadowKBlock) + kb) * kShadowTileRows + r) * kShadowKBlock + c;
}
__host__ __device__ __forceinline__ int64_t shadow_rows_padded(int64_t rows) {
  return (rows + kShadowTileRows - 1) / kShadowTileRows * kShadowTileRows;
}
// The int8 shadow keeps the same byte geometry: K-blocks of 128 int8 values (128 bytes, the same swizzle span),
// 6 of them per row, so a 32-row K-block piece is still 4 KB.  Each 32-row tile has one fp32 scale st; the
// shadow row is p8 with p - mu ~= st * p8 (element (row, col) at shadow8_index, in bytes).
constexpr int kShadow8KBlock = 128;
constexpr int kShadow8KBlocks = kD / kShadow8KBlock;   // 6
__host__ __device__ __forceinline__ int64_t shadow8_index(int64_t row, int col) {
  const int64_t tile = row / kShadowTileRows;
  const int r = static_cast<int>(row % kShadowTileRows);
  const int kb = col / kShadow8KBlock, c = col % kShadow8KBlock;
  return ((tile * kShadow8KBlocks + kb) * kShadowTileRows + r) * kShadow8KBlock + c;
}

// Shadow formats of a shard (option "shadow"; 3 = AUTO picks 1 or 2 per shard at its first ingest).
enum ShadowFormat { kShadowNone = 0, kShadowBf16 = 1, kShadowInt8 = 2, kShadowAuto = 3 };

// ---------------------------------------------------------------------------------------------
// Candidate records.  A candidate is one 64-bit word:
//   hi 32 bits: order-preserving key of the fp32 score (larger key <=> larger score)
//   lo 32 bits: ~row  (so that, for equal scores, the LOWER row compares larger)
// Comparing two records as unsigned integers therefore orders them by
// (score desc, row asc) — the engine's total order.  0 is the "empty slot" sentinel
// (every real record is > 0 because fkey(-inf) = 0x007fffff).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t fkey(float s) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(s);
#else
  union { float f; uint32_t u; } c; c.f = s; uint32_t u = c.u;
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float key2f(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ uint64_t pack_cand(float s, uint32_t row) {
  return (static_cast<uint64_t>(fkey(s)) << 32) | static_cast<uint64_t>(~row);
}
__host__ __device__ __forceinline__ uint32_t cand_row(uint64_t c) { return ~static_cast<uint32_t>(c); }
__host__ __device__ __forceinline__ float cand_score(uint64_t c) { return key2f(static_cast<uint32_t>(c >> 32)); }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), restated from the published algorithm.
// ---------------------------------------------------------------------------------------------
struct U4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
  uint64_t p = static_cast<uint64_t>(a) * static_cast<uint64_t>(b);
  hi = static_cast<uint32_t>(p >> 32);
  lo = static_cast<uint32_t>(p);
}

__host__ __device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    mulhilo32(M0, c.x, hi0, lo0);
    mulhilo32(M1, c.z, hi1, lo1);
    U4 n;
    n.x = hi1 ^ c.y ^ k0;
    n.y = lo1;
    n.z = hi0 ^ c.w ^ k1;
    n.w = lo0;
    c = n;
    k0 += W0;
    k1 += W1;
  }
  return c;
}

// One synthetic component from one 32-bit word: sum of its four bytes minus 510
// (Irwin-Hall(4) on bytes; integer, so CPU and GPU agree bit for bit).
__host__ __device__ __forceinline__ int synth_component(uint32_t w) {
  return static_cast<int>((w & 0xffu) + ((w >> 8) & 0xffu) + ((w >> 16) & 0xffu) + (w >> 24)) - 510;
}

#ifdef __CUDACC__
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// Exact score of one (query, passage) pair, evaluated by one full warp.
// Products are exact in fp64; each lane sums its 24 products in index order, then the
// xor-butterfly (16,8,4,2,1) combines lanes; one final rounding to fp32.  Every path of
// the engine reports scores produced by this function, so results are path-independent.
__device__ __forceinline__ double lane_partial_f64(const float4* __restrict__ q4 /*smem or global, 192 f4*/,
                                                   const float4* __restrict__ p4, int lane) {
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    float4 q = q4[lane + 32 * i];
    float4 p = __ldg(p4 + lane + 32 * i);
    acc = fma(static_cast<double>(q.x), static_cast<double>(p.x), acc);
    acc = fma(static_cast<double>(q.y), static_cast<double>(p.y), acc);
    acc = fma(static_cast<double>(q.z), static_cast<double>(p.z), acc);
    acc = fma(static_cast<double>(q.w), static_cast<double>(p.w), acc);
  }
  return acc;
}
__device__ __forceinline__ double warp_butterfly_sum(double v) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}
__device__ __forceinline__ float exact_dot_warp(const float4* q4, const float4* p4, int lane) {
  return static_cast<float>(warp_butterfly_sum(lane_partial_f64(q4, p4, lane)));
}
#endif

}  // namespace b2f
