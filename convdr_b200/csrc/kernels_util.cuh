// kernels_util.cuh — ingest-side kernels: bf16 shadow + norm bound, synthetic rows, query prep.
#pragma once
#include <climits>
#include "common.cuh"

namespace b2f {

// Sums of squares are accumulated in fp64 and turned into an fp32 upper bound here, so that every bound is one
// for all finite inputs (DESIGN.md section 4): the square of an fp32 value is exact and normal in fp64 (the
// smallest, (2^-149)^2 = 2^-298, is far above 2^-1022), so only the additions round.  768 non-negative terms in any
// order are then within 767 * 2^-53 < 2^-43 of their sum, relative; 1 + 2^-40 covers that and the conversion
// rounds up.  The result is 0 only for an all-zero vector and +inf above FLT_MAX.  An fp32 sum instead flushes
// squares below 2^-149 to zero and overflows at FLT_MAX, where no relative factor can recover the bound.
__device__ __forceinline__ float sumsq_upper(double s) { return __double2float_ru(__dmul_ru(s, 1.0 + 0x1p-40)); }
__device__ __forceinline__ double sumsq4(double acc, float4 v) {
  acc = fma(static_cast<double>(v.x), static_cast<double>(v.x), acc);
  acc = fma(static_cast<double>(v.y), static_cast<double>(v.y), acc);
  acc = fma(static_cast<double>(v.z), static_cast<double>(v.z), acc);
  return fma(static_cast<double>(v.w), static_cast<double>(v.w), acc);
}
// An fp32 operation (subtraction, fma) rounds to within 2^-24 of its result, or to within 2^-150 of it when the
// result is subnormal.  Over 768 components the absolute part is at most sqrt(768) * 2^-150 < 2^-145 in norm.
constexpr float kSubnormalNorm = 0x1p-145f;
// Upper bound of ||(x - mu) - shadow|| from the computed error vector e~ (sum of its squares s) and the computed
// centred row d (norm bound cn): the error components may carry one rounding each (rel_round: the fma of the
// int8 shadow) and d carries the rounding of the fp32 subtraction x - mu, each 2^-24 relative + 2^-145 in norm.
__device__ __forceinline__ float shadow_err_upper(double s, float cn, bool rel_round) {
  float e = __fsqrt_ru(sumsq_upper(s));
  if (rel_round) e = __fadd_ru(__fmul_ru(e, 1.0000001f), kSubnormalNorm);
  return __fadd_ru(__fadd_ru(e, __fmul_ru(cn, 6.0e-8f)), kSubnormalNorm);
}
// Upper bound of ||x - mu||^2 from cn >= ||d||, d = fl32(x - mu): ||x - mu|| <= (1 + 2^-24) ||d|| + 2^-145.
__device__ __forceinline__ float centred_norm2_upper(float cn) {
  const float c = __fadd_ru(__fmul_ru(cn, 1.0000001f), kSubnormalNorm);
  return __fmul_ru(c, c);
}

// acc + the squared bf16 rounding error of four components: (x - bf16_rn(x)) is exact in fp32 (the difference
// of two floats within half a bf16 ulp of each other), and so are its squares in fp64.
__device__ __forceinline__ double bf16_err2(double acc, float4 v) {
  float4 d;
  d.x = v.x - __bfloat162float(__float2bfloat16_rn(v.x));
  d.y = v.y - __bfloat162float(__float2bfloat16_rn(v.y));
  d.z = v.z - __bfloat162float(__float2bfloat16_rn(v.z));
  d.w = v.w - __bfloat162float(__float2bfloat16_rn(v.w));
  return sumsq4(acc, d);
}

__device__ __forceinline__ uint2 pack_bf16x4(float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  return r;
}

// Column means of rows [row0, row0 + n_rows) in two deterministic steps (fixed summation order, so the
// same rows always give the same centre and therefore the same shadow bits):
//   col_sum_partial_kernel : block b sums rows b, b + gridDim.x, ... (192 threads, one float4 column chunk each)
//   col_mean_final_kernel  : sums the partials in block order and divides by n_rows
__global__ void __launch_bounds__(kRowF4) col_sum_partial_kernel(const float* __restrict__ x32, int64_t row0,
                                                                 int64_t n_rows, float* __restrict__ partial) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
    const float4 v = ldg_stream_f4(reinterpret_cast<const float4*>(x32 + (row0 + r) * kD) + threadIdx.x);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  reinterpret_cast<float4*>(partial + static_cast<int64_t>(blockIdx.x) * kD)[threadIdx.x] = acc;
}
__global__ void __launch_bounds__(256) col_mean_final_kernel(const float* __restrict__ partial, int n_partials,
                                                             int64_t n_rows, float* __restrict__ mu) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= kD) return;
  float acc = 0.f;
  for (int b = 0; b < n_partials; ++b) acc += partial[static_cast<int64_t>(b) * kD + c];
  mu[c] = acc / static_cast<float>(n_rows);
}

// One warp per row: write the bf16 shadow row of the CENTRED vector d = fl32(x - mu) (round-to-nearest,
// K-block-major tiled layout — 16 lanes fill one 128-byte K-block segment) and fold into maxnorm2_bits
// (float bits; valid because the values are non-negative):
//   [0] an upper bound of max ||x||^2            (uncentred: the fp32 scan engine's margin)
//   [1] an upper bound of max ||(x - mu) - bf16(d)||^2, the rounding error of the shadow row INCLUDING the
//       rounding of the fp32 subtraction (|d - (x - mu)| <= 2^-24 |d| per component): what makes the
//       prefilter margin data-dependent and ~2x tighter than the worst case 2^-8 * ||d|| (DESIGN.md §4)
//   [2] an upper bound of max ||x - mu||^2
// mu is the shard's centre (all zeros when centring is off: d = x exactly, the bounds are the uncentred
// ones).  Inner products against centred rows differ from the true ones by the per-query constant q.mu,
// so every threshold comparison of a pass can live in centred space; the exact rescoring reads x32.
// HBM traffic per row: 3072 B read + 1536 B written.
__global__ void __launch_bounds__(256) convert_rows_kernel(const float* __restrict__ x32,
                                                           __nv_bfloat16* __restrict__ x16,
                                                           int64_t row0, int64_t n_rows,
                                                           unsigned int* __restrict__ maxnorm2_bits,
                                                           const float* __restrict__ mu) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  float4 m4[kF4PerLane];
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) m4[i] = __ldg(reinterpret_cast<const float4*>(mu) + lane + 32 * i);
  float wmax = 0.f, emax = 0.f, cmax = 0.f;
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const float4* src = reinterpret_cast<const float4*>(x32 + (row0 + r) * kD);
    double ss = 0.0, es = 0.0, cs = 0.0;
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) {
      const float4 v = ldg_stream_f4(src + lane + 32 * i);
      ss = sumsq4(ss, v);
      float4 d;
      d.x = __fsub_rn(v.x, m4[i].x); d.y = __fsub_rn(v.y, m4[i].y); d.z = __fsub_rn(v.z, m4[i].z); d.w = __fsub_rn(v.w, m4[i].w);
      cs = sumsq4(cs, d);
      es = bf16_err2(es, d);
      if (x16) *reinterpret_cast<uint2*>(x16 + shadow_index(row0 + r, 4 * (lane + 32 * i))) = pack_bf16x4(d);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
      ss += __shfl_xor_sync(0xffffffffu, ss, s);
      es += __shfl_xor_sync(0xffffffffu, es, s);
      cs += __shfl_xor_sync(0xffffffffu, cs, s);
    }
    const float cn = __fsqrt_ru(sumsq_upper(cs));                        // >= ||d||
    const float e = shadow_err_upper(es, cn, false);
    wmax = fmaxf(wmax, sumsq_upper(ss));
    emax = fmaxf(emax, __fmul_ru(e, e));
    cmax = fmaxf(cmax, centred_norm2_upper(cn));
  }
  if (lane == 0 && wmax > 0.f) atomicMax(maxnorm2_bits, __float_as_uint(wmax));
  if (lane == 0 && emax > 0.f) atomicMax(maxnorm2_bits + 1, __float_as_uint(emax));
  if (lane == 0 && cmax > 0.f) atomicMax(maxnorm2_bits + 2, __float_as_uint(cmax));
}

// Symmetric int8 code of v for the scale 1/inv (inv = 127 / max|v| over the scale's group; 0 for an all-zero group).
__device__ __forceinline__ int quant8(float v, float inv) {
  return max(-127, min(127, __float2int_rn(v * inv)));
}
// fl(v - sq * q8(v)) per component (one fma rounding each) and the upper bound of ||q - sq q8|| built from the
// sum of their squares: 2^-24 relative + 2^-145 in norm for the fma roundings.
__device__ __forceinline__ float4 i8_residual(float4 v, float sq, float inv) {
  return make_float4(fmaf(-sq, static_cast<float>(quant8(v.x, inv)), v.x), fmaf(-sq, static_cast<float>(quant8(v.y, inv)), v.y),
                     fmaf(-sq, static_cast<float>(quant8(v.z, inv)), v.z), fmaf(-sq, static_cast<float>(quant8(v.w, inv)), v.w));
}
// Entry of the int8 shard's per-tile scale array: {st, RD(1/st), RU(1/st), 0}; the reciprocals are the tile
// factors of the integer threshold (i8_threshold).
__device__ __forceinline__ float4 i8_tile_scale(float st) {
  return make_float4(st, __frcp_rd(st), __frcp_ru(st), 0.f);
}
__device__ __forceinline__ float i8_query_err_upper(double s) {
  return __fadd_ru(__fmul_ru(__fsqrt_ru(sumsq_upper(s)), 1.0000001f), kSubnormalNorm);
}

// int8 shadow (DESIGN.md section 4): one warp per 32-row tile of rows [tile_row0, row0 + n_rows), where tile_row0 is
// row0 rounded down to the tile — a tile that an earlier add left partly filled is re-quantised with the scale of
// all its rows.  Pass 1: st = max|d| / 127 over the tile (d = fl32(x - mu)); pass 2: p8 = rint(d / st), the
// K-block-major int8 row (common.cuh shadow8_index) and the same three bounds as convert_rows_kernel, with slot [1]
// an upper bound of max ||(x - mu) - st * p8||^2: fma(-st, p8, d) rounds the exact difference once, plus the
// rounding of the fp32 subtraction (shadow_err_upper).  Any p8 is valid — the bound
// measures the error that was made.  x8 == nullptr: bounds only (used by the format choice).
__global__ void __launch_bounds__(256) convert_rows_i8_kernel(const float* __restrict__ x32, int8_t* __restrict__ x8,
                                                              float4* __restrict__ tscale, int64_t row0, int64_t n_rows,
                                                              unsigned int* __restrict__ maxnorm2_bits,
                                                              const float* __restrict__ mu) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t end = row0 + n_rows;
  const int64_t t_begin = row0 / kShadowTileRows, t_end = (end + kShadowTileRows - 1) / kShadowTileRows;
  float4 m4[kF4PerLane];
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) m4[i] = __ldg(reinterpret_cast<const float4*>(mu) + lane + 32 * i);
  float wmax = 0.f, emax = 0.f, cmax = 0.f;
  for (int64_t t = t_begin + warp; t < t_end; t += nwarps) {
    const int64_t r0 = t * kShadowTileRows, r1 = min(end, r0 + kShadowTileRows);
    float amax = 0.f;
    for (int64_t r = r0; r < r1; ++r) {
      const float4* src = reinterpret_cast<const float4*>(x32 + r * kD);
#pragma unroll
      for (int i = 0; i < kF4PerLane; ++i) {
        const float4 v = __ldg(src + lane + 32 * i);
        amax = fmaxf(amax, fmaxf(fmaxf(fabsf(__fsub_rn(v.x, m4[i].x)), fabsf(__fsub_rn(v.y, m4[i].y))),
                                 fmaxf(fabsf(__fsub_rn(v.z, m4[i].z)), fabsf(__fsub_rn(v.w, m4[i].w)))));
      }
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, s));
    const float st = amax / 127.f;
    const float inv = amax > 0.f ? 127.f / amax : 0.f;
    if (x8 && lane == 0) tscale[t] = i8_tile_scale(st);
    for (int64_t r = r0; r < r1; ++r) {
      const float4* src = reinterpret_cast<const float4*>(x32 + r * kD);
      double ss = 0.0, es = 0.0, cs = 0.0;
#pragma unroll
      for (int i = 0; i < kF4PerLane; ++i) {
        const float4 v = __ldg(src + lane + 32 * i);
        ss = sumsq4(ss, v);
        float4 d;
        d.x = __fsub_rn(v.x, m4[i].x); d.y = __fsub_rn(v.y, m4[i].y); d.z = __fsub_rn(v.z, m4[i].z); d.w = __fsub_rn(v.w, m4[i].w);
        cs = sumsq4(cs, d);
        const int a = quant8(d.x, inv), b = quant8(d.y, inv), c = quant8(d.z, inv), e = quant8(d.w, inv);
        es = sumsq4(es, make_float4(fmaf(-st, static_cast<float>(a), d.x), fmaf(-st, static_cast<float>(b), d.y),
                                    fmaf(-st, static_cast<float>(c), d.z), fmaf(-st, static_cast<float>(e), d.w)));
        if (x8) {
          const uint32_t packed = (static_cast<uint32_t>(a) & 0xffu) | ((static_cast<uint32_t>(b) & 0xffu) << 8) |
                                  ((static_cast<uint32_t>(c) & 0xffu) << 16) | (static_cast<uint32_t>(e) << 24);
          *reinterpret_cast<uint32_t*>(x8 + shadow8_index(r, 4 * (lane + 32 * i))) = packed;
        }
      }
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) {
        ss += __shfl_xor_sync(0xffffffffu, ss, s);
        es += __shfl_xor_sync(0xffffffffu, es, s);
        cs += __shfl_xor_sync(0xffffffffu, cs, s);
      }
      const float cn = __fsqrt_ru(sumsq_upper(cs));
      const float e = shadow_err_upper(es, cn, true);
      wmax = fmaxf(wmax, sumsq_upper(ss));
      emax = fmaxf(emax, __fmul_ru(e, e));
      cmax = fmaxf(cmax, centred_norm2_upper(cn));
    }
  }
  if (lane == 0 && wmax > 0.f) atomicMax(maxnorm2_bits, __float_as_uint(wmax));
  if (lane == 0 && emax > 0.f) atomicMax(maxnorm2_bits + 1, __float_as_uint(emax));
  if (lane == 0 && cmax > 0.f) atomicMax(maxnorm2_bits + 2, __float_as_uint(cmax));
}

// Format choice (AUTO): 64 of the first m rows act as pseudo-queries q_j (uncentred, like real queries).  For every
// j this kernel accumulates, over `n_s` evenly spaced sample rows, the sum and the sum of squares of the centred
// scores q_j . (p - mu) in fp64 (stat[2j], stat[2j+1]) and writes ||q_j|| and ||q_j - sq q8_j|| (qstat[2j], +1).
// One warp per (j, sample row); blocks of 8 warps share j.
__global__ void __launch_bounds__(256) shadow_probe_kernel(const float* __restrict__ x32, int64_t m, int n_s,
                                                           const float* __restrict__ mu, double* __restrict__ stat,
                                                           float* __restrict__ qstat) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int j = blockIdx.y;
  const float4* q4 = reinterpret_cast<const float4*>(x32 + (m * j / 64) * kD);
  float4 q[kF4PerLane];
  float amax = 0.f;
  double qq = 0.0;
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    q[i] = __ldg(q4 + lane + 32 * i);
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(q[i].x), fabsf(q[i].y)), fmaxf(fabsf(q[i].z), fabsf(q[i].w))));
    qq = sumsq4(qq, q[i]);
  }
  double s1 = 0.0, s2 = 0.0;
  for (int r = blockIdx.x * 8 + w; r < n_s; r += gridDim.x * 8) {
    const float4* p4 = reinterpret_cast<const float4*>(x32 + (m * r / n_s) * kD);
    const float4* m4 = reinterpret_cast<const float4*>(mu);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) {
      const float4 p = __ldg(p4 + lane + 32 * i), c = __ldg(m4 + lane + 32 * i);
      acc += q[i].x * (p.x - c.x) + q[i].y * (p.y - c.y) + q[i].z * (p.z - c.z) + q[i].w * (p.w - c.w);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    s1 += acc;
    s2 += static_cast<double>(acc) * acc;
  }
  if (lane == 0) {
    atomicAdd(stat + 2 * j, s1);
    atomicAdd(stat + 2 * j + 1, s2);
  }
  if (blockIdx.x == 0 && w == 0) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, s));
    const float sq = amax / 127.f, inv = amax > 0.f ? 127.f / amax : 0.f;
    double es = 0.0;
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i)
      es = sumsq4(es, i8_residual(q[i], sq, inv));
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
      es += __shfl_xor_sync(0xffffffffu, es, s);
      qq += __shfl_xor_sync(0xffffffffu, qq, s);
    }
    if (lane == 0) {
      qstat[2 * j] = __fsqrt_ru(sumsq_upper(qq));
      qstat[2 * j + 1] = amax > 0.f ? i8_query_err_upper(es) : 0.f;
    }
  }
}

// Synthetic rows (see include/b2f.h b2f_add_synthetic).  One warp per row; lane l produces
// float4 chunks l, l+32, ..., l+160; chunk c of row r is Philox4x32-10(counter = (r_lo, r_hi, c, 0),
// key = (seed_lo ^ stream_lo, seed_hi ^ stream_hi ^ 0x5eed)).  With mean_shift = M > 0 every component t
// is shifted by sign_t * M before the normalisation, sign_t = +-1 from the low bit of word t of
// Philox(counter = (0xffffffff, 0xffffffff, c, 0x6d65616e), key = (seed_lo, seed_hi ^ 0x5eed)) — one fixed
// direction per seed, shared by every stream (passages and queries), which gives LayerNorm-like
// embeddings with a common mean (cos(p, p') ~ M^2 / (M^2 + 148^2); M = 443 -> 0.9).  Integer arithmetic up
// to the final scale, so CPU and GPU agree bit for bit.  Writes the fp32 rows only; the shadow and the
// norm bounds come from the same ingest pass as for real rows (convert_rows_kernel).
__global__ void __launch_bounds__(256) synth_rows_kernel(float* __restrict__ x32,
                                                         int64_t dst_row0, int64_t first_row,
                                                         int64_t n_rows, uint32_t k0, uint32_t k1,
                                                         float norm, int mean_shift, uint32_t km0, uint32_t km1) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  int shift[kF4PerLane][4];
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    shift[i][0] = shift[i][1] = shift[i][2] = shift[i][3] = 0;
    if (mean_shift) {
      U4 c;
      c.x = 0xffffffffu; c.y = 0xffffffffu; c.z = static_cast<uint32_t>(lane + 32 * i); c.w = 0x6d65616eu;
      const U4 o = philox4x32_10(c, km0, km1);
      shift[i][0] = (o.x & 1u) ? mean_shift : -mean_shift;
      shift[i][1] = (o.y & 1u) ? mean_shift : -mean_shift;
      shift[i][2] = (o.z & 1u) ? mean_shift : -mean_shift;
      shift[i][3] = (o.w & 1u) ? mean_shift : -mean_shift;
    }
  }
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const uint64_t row = static_cast<uint64_t>(first_row + r);
    int comp[kF4PerLane][4];
    long long ss = 0;
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) {
      U4 c;
      c.x = static_cast<uint32_t>(row);
      c.y = static_cast<uint32_t>(row >> 32);
      c.z = static_cast<uint32_t>(lane + 32 * i);
      c.w = 0u;
      U4 o = philox4x32_10(c, k0, k1);
      comp[i][0] = synth_component(o.x) + shift[i][0];
      comp[i][1] = synth_component(o.y) + shift[i][1];
      comp[i][2] = synth_component(o.z) + shift[i][2];
      comp[i][3] = synth_component(o.w) + shift[i][3];
      ss += static_cast<long long>(comp[i][0] * comp[i][0] + comp[i][1] * comp[i][1]) +
            static_cast<long long>(comp[i][2] * comp[i][2] + comp[i][3] * comp[i][3]);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, s);
    // ss <= 768 * (510 + 4096)^2 < 2^34: converted to fp32 with one rounding, like the host restatement.
    // IEEE sqrt and division: bit-identical to the host restatement.
    const float inv = (ss > 0) ? __fdiv_rn(norm, __fsqrt_rn(static_cast<float>(ss))) : 0.f;
    float4* dst32 = reinterpret_cast<float4*>(x32 + (dst_row0 + r) * kD);
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) {
      float4 v;
      v.x = __fmul_rn(static_cast<float>(comp[i][0]), inv);
      v.y = __fmul_rn(static_cast<float>(comp[i][1]), inv);
      v.z = __fmul_rn(static_cast<float>(comp[i][2]), inv);
      v.w = __fmul_rn(static_cast<float>(comp[i][3]), inv);
      dst32[lane + 32 * i] = v;
    }
  }
}

// Query preparation: one warp per (padded) query row.  Writes the bf16 copy used by the tensor
// path (zero rows for q >= nq), an upper bound of ||q|| and one of ||q - bf16(q)||.
__global__ void __launch_bounds__(128) prep_queries_kernel(const float* __restrict__ q32, int nq,
                                                           int nq_pad,
                                                           __nv_bfloat16* __restrict__ q16,
                                                           float* __restrict__ qnorm,
                                                           float* __restrict__ qerr) {
  const int lane = threadIdx.x & 31;
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (q >= nq_pad) return;
  uint2* dst = reinterpret_cast<uint2*>(q16 + static_cast<int64_t>(q) * kD);
  if (q >= nq) {
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) dst[lane + 32 * i] = make_uint2(0u, 0u);
    return;
  }
  const float4* src = reinterpret_cast<const float4*>(q32 + static_cast<int64_t>(q) * kD);
  double ss = 0.0, es = 0.0;
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    float4 v = __ldg(src + lane + 32 * i);
    ss = sumsq4(ss, v);
    es = bf16_err2(es, v);
    dst[lane + 32 * i] = pack_bf16x4(v);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, s);
    es += __shfl_xor_sync(0xffffffffu, es, s);
  }
  if (lane == 0) {
    qnorm[q] = __fsqrt_ru(sumsq_upper(ss));
    qerr[q] = __fsqrt_ru(sumsq_upper(es));   // the bf16 errors are exact: only their sum rounds
  }
}

// Query preparation for an int8 shadow: per query the scale sq = max|q| / 127, the row-major int8 code q8
// (zero rows and sq = 0 for q >= nq), an upper bound of ||q|| and one of ||q - sq q8||.
__global__ void __launch_bounds__(128) prep_queries_i8_kernel(const float* __restrict__ q32, int nq, int nq_pad,
                                                              int8_t* __restrict__ q8, float* __restrict__ qscale,
                                                              float* __restrict__ qnorm, float* __restrict__ qerr) {
  const int lane = threadIdx.x & 31;
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (q >= nq_pad) return;
  uint32_t* dst = reinterpret_cast<uint32_t*>(q8 + static_cast<int64_t>(q) * kD);
  if (q >= nq) {
#pragma unroll
    for (int i = 0; i < kF4PerLane; ++i) dst[lane + 32 * i] = 0u;
    if (lane == 0) qscale[q] = 0.f;
    return;
  }
  const float4* src = reinterpret_cast<const float4*>(q32 + static_cast<int64_t>(q) * kD);
  float4 v[kF4PerLane];
  float amax = 0.f;
  double ss = 0.0, es = 0.0;
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    v[i] = __ldg(src + lane + 32 * i);
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v[i].x), fabsf(v[i].y)), fmaxf(fabsf(v[i].z), fabsf(v[i].w))));
    ss = sumsq4(ss, v[i]);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, s));
  const float sq = amax / 127.f, inv = amax > 0.f ? 127.f / amax : 0.f;
#pragma unroll
  for (int i = 0; i < kF4PerLane; ++i) {
    const int a = quant8(v[i].x, inv), b = quant8(v[i].y, inv), c = quant8(v[i].z, inv), e = quant8(v[i].w, inv);
    es = sumsq4(es, i8_residual(v[i], sq, inv));
    dst[lane + 32 * i] = (static_cast<uint32_t>(a) & 0xffu) | ((static_cast<uint32_t>(b) & 0xffu) << 8) |
                         ((static_cast<uint32_t>(c) & 0xffu) << 16) | (static_cast<uint32_t>(e) << 24);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, s);
    es += __shfl_xor_sync(0xffffffffu, es, s);
  }
  if (lane == 0) {
    qscale[q] = sq;
    qnorm[q] = __fsqrt_ru(sumsq_upper(ss));
    qerr[q] = amax > 0.f ? i8_query_err_upper(es) : 0.f;   // a zero query is coded exactly
  }
}

// Integer threshold of the int8 tensor engine (DESIGN.md section 4).  A prefilter score is s~ = acc * sq * st with
// acc the exact int32 dot product of the codes, sq the query scale and st the tile scale.  The threshold T satisfies
// "acc * sq * st >= tau  =>  acc >= T" for every integer acc, and is formed from two factors so that the per-tile
// step needs no division:
//   per query (on a threshold change):  u = RD(tau / sq)                               (i8_tau_over_sq)
//   per tile (at ingest):               r_lo = RD(1 / st), r_hi = RU(1 / st)            (i8_tile_scale)
//   per (query, tile):                  x = RD(u * (u >= 0 ? r_lo : r_hi)),  T = floor(x), saturated; NaN -> INT_MIN
// u <= tau/sq and r_lo <= 1/st <= r_hi, so x <= tau / (sq st) in every sign case, and acc >= tau/(sq st) >= x gives
// acc >= floor(x).  The zero and infinite cases are what the IEEE operations give: st = 0 -> r = +inf (x = +-inf, or
// NaN for u = 0: every row passes, and every score of a zero tile is 0); sq = 0 -> u = +-inf for tau != 0 (NaN for
// tau = 0); tau = -inf -> u = -inf; a padded query column (tau = +inf, sq = 0) -> u = +inf; a subnormal st whose
// reciprocal overflows -> r_lo = FLT_MAX, r_hi = +inf.  Saturation: |acc| <= 768 * 127^2 < 2^24.
__device__ __forceinline__ float i8_tau_over_sq(float tau, float sq) { return __fdiv_rd(tau, sq); }
__device__ __forceinline__ int i8_threshold(float u, float4 ts) {
  const float x = __fmul_rd(u, u >= 0.f ? ts.y : ts.z);
  if (x >= 2147483520.f) return INT_MAX;
  if (!(x >= -2147483520.f)) return INT_MIN;   // and NaN
  return static_cast<int>(floorf(x));
}
// The score recorded for a hit: fl(fl(acc) * fl(sq * st)); |acc| <= 768 * 127^2 < 2^24, so fl(acc) is exact and the
// recorded value is within 2^-23 |s~| of s~ (covered by the relative term of the int8 margin, pass_init_kernel).
__device__ __forceinline__ float i8_score(int acc, float sq, float st) {
  return __fmul_rn(static_cast<float>(acc), __fmul_rn(sq, st));
}

}  // namespace b2f
