// kernels_scan.cuh — the SIMT scoring engine: 128-bit streaming fp32 loads, register-tiled dot
// products, warp-shuffle (transposing) reductions, threshold filter, candidate append.
//
// It is the engine for small query batches (HBM-bound up to ~16 queries) and, in its kExact
// instantiation (fp64 accumulation, total-order threshold), the robust fallback for any query the
// tensor path could not finish within its candidate capacity.
//
// Replaces the arithmetic of `index.search` (reference drivers/run_convdr_inference.py:182) —
// FAISS's `nq < 20` branch: per-query SIMD dot + heap (upstream utils/distances.cpp).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace b2f {

constexpr int kScanThreads = 256;
constexpr int kScanRows = 4;      // rows register-tiled per warp iteration
constexpr int kScanMaxQ = 32;     // queries per pass (smem: 32 * 3 KB = 96 KB)

struct ScanArgs {
  const float* x32;        // shard rows [*, 768]
  int64_t row_begin, row_end;  // rows scored by this launch
  const float* q32;        // pass queries [nq_pass, 768]
  int nq_pass;
  int dense;               // 1: write every score at slot (row - dense_row0); 0: threshold + append
  int64_t dense_row0;
  uint64_t* cand;          // [nq_pass][C]
  int* cnt;                // [nq_pass]
  int C;
  const float* tau;        // [nq_pass] approx-mode threshold
  const uint64_t* tauP;    // [nq_pass] exact-mode threshold record
  int* ovf;                // [nq_pass] set when a candidate did not fit
  const uint32_t* sel_bits;  // SEL instances: the shard's row bitmap (bit r & 31 of word r >> 5: row r is selected)
};

template <typename T, int V>
__device__ __forceinline__ T reduce_transpose(T (&a)[V], int lane) {
  // After the call lane l holds the all-lane sum of element (l & (V-1)).  The combination tree is
  // the xor butterfly 16,8,4,2,1 for every element (same as warp_butterfly_sum).
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    if (s >= V) {
#pragma unroll
      for (int i = 0; i < V; ++i) a[i] += __shfl_xor_sync(0xffffffffu, a[i], s);
    } else {
      const bool hi = (lane & s) != 0;
#pragma unroll
      for (int i = 0; i < s; ++i) {
        const T keep = hi ? a[i + s] : a[i];
        const T send = hi ? a[i] : a[i + s];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
      }
    }
  }
  return a[0];
}

// SEL: filtered search.  Unselected rows never pass; the dense phase stores empty records (0) for them, and outside
// it a row group without a selected row is not loaded at all.
template <bool kExact, bool SEL>
__global__ void __launch_bounds__(kScanThreads, 1) scan_kernel(const ScanArgs a) {
  using acc_t = typename std::conditional<kExact, double, float>::type;
  constexpr int R = kScanRows;
  constexpr int QB = kExact ? 4 : 8;
  constexpr int V = R * QB;
  extern __shared__ __align__(16) unsigned char scan_smem[];
  const int nqp = (a.nq_pass + QB - 1) / QB * QB;
  float4* Qs4 = reinterpret_cast<float4*>(scan_smem);
  float* tau_s = reinterpret_cast<float*>(Qs4 + static_cast<size_t>(nqp) * kRowF4);
  uint64_t* tauP_s = reinterpret_cast<uint64_t*>(tau_s + kScanMaxQ);

  for (int idx = threadIdx.x; idx < nqp * kRowF4; idx += kScanThreads) {
    const int qi = idx / kRowF4;
    Qs4[idx] = (qi < a.nq_pass) ? __ldg(reinterpret_cast<const float4*>(a.q32) + idx)
                                : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int qi = threadIdx.x; qi < nqp; qi += kScanThreads) {
    tau_s[qi] = (qi < a.nq_pass && !a.dense) ? a.tau[qi] : -INFINITY;
    tauP_s[qi] = (qi < a.nq_pass && !a.dense) ? a.tauP[qi] : 0ull;
  }
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const int64_t gwarp = (static_cast<int64_t>(blockIdx.x) * kScanThreads + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kScanThreads) >> 5;
  const int64_t ngroups = (a.row_end - a.row_begin + R - 1) / R;
  const int my_r = (lane & (V - 1)) / QB;   // (row-in-group, query-in-block) this lane tests
  const int my_qq = (lane & (V - 1)) % QB;

  for (int64_t g = gwarp; g < ngroups; g += nwarps) {
    const int64_t r0 = a.row_begin + g * R;
    if constexpr (SEL) {
      bool any_sel = false;
#pragma unroll
      for (int r = 0; r < R; ++r)
        any_sel = any_sel || (r0 + r < a.row_end && ((__ldg(a.sel_bits + ((r0 + r) >> 5)) >> ((r0 + r) & 31)) & 1u));
      if (!any_sel && !a.dense) continue;   // warp-uniform
    }
    float4 p[R][kF4PerLane];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const bool valid = (r0 + r) < a.row_end;
      const float4* src = reinterpret_cast<const float4*>(a.x32 + (valid ? (r0 + r) : r0) * kD);
#pragma unroll
      for (int i = 0; i < kF4PerLane; ++i) {
        p[r][i] = ldg_stream_f4(src + lane + 32 * i);
        if (!valid) p[r][i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    for (int qb = 0; qb < nqp; qb += QB) {
      acc_t acc[V];
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] = acc_t(0);
#pragma unroll
      for (int i = 0; i < kF4PerLane; ++i) {
#pragma unroll
        for (int qq = 0; qq < QB; ++qq) {
          const float4 q = Qs4[(qb + qq) * kRowF4 + lane + 32 * i];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            acc_t s = acc[r * QB + qq];
            if constexpr (kExact) {
              s = fma(static_cast<double>(q.x), static_cast<double>(p[r][i].x), s);
              s = fma(static_cast<double>(q.y), static_cast<double>(p[r][i].y), s);
              s = fma(static_cast<double>(q.z), static_cast<double>(p[r][i].z), s);
              s = fma(static_cast<double>(q.w), static_cast<double>(p[r][i].w), s);
            } else {
              s = fmaf(q.x, p[r][i].x, s);
              s = fmaf(q.y, p[r][i].y, s);
              s = fmaf(q.z, p[r][i].z, s);
              s = fmaf(q.w, p[r][i].w, s);
            }
            acc[r * QB + qq] = s;
          }
        }
      }
      const float score = static_cast<float>(reduce_transpose<acc_t, V>(acc, lane));
      const int64_t row = r0 + my_r;
      const int qi = qb + my_qq;
      if (lane < V && row < a.row_end && qi < a.nq_pass) {
        bool sel_ok = true;
        if constexpr (SEL) sel_ok = (__ldg(a.sel_bits + (row >> 5)) >> (row & 31)) & 1u;
        const uint64_t rec = pack_cand(score, static_cast<uint32_t>(row));
        if (a.dense) {
          a.cand[static_cast<int64_t>(qi) * a.C + (row - a.dense_row0)] = sel_ok ? rec : 0ull;
        } else {
          const bool pass = sel_ok && (kExact ? (rec > tauP_s[qi]) : (score >= tau_s[qi]));
          if (pass) {
            const int slot = atomicAdd(a.cnt + qi, 1);
            if (slot < a.C) a.cand[static_cast<int64_t>(qi) * a.C + slot] = rec;
            else a.ovf[qi] = 1;
          }
        }
      }
    }
  }
}

inline size_t scan_smem_bytes(int nq_pass, bool exact) {
  const int QB = exact ? 4 : 8;
  const int nqp = (nq_pass + QB - 1) / QB * QB;
  return static_cast<size_t>(nqp) * kD * sizeof(float) + kScanMaxQ * sizeof(float) +
         kScanMaxQ * sizeof(uint64_t);
}

}  // namespace b2f
