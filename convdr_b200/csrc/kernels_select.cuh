// kernels_select.cuh — candidate-list maintenance: threshold refresh (radix select + compaction),
// exact rescoring + final sort, and the cross-shard merge.
//
// Replaces, on device, what the reference does in interpreted Python after every block:
// `passage_embedding2id[I]`, tuple building and the 2-way sorted merge
// (drivers/run_convdr_inference.py:190-229), and what FAISS does inside search
// (heap / BlockSelect top-k, IndexShards CPU merge).
#pragma once
#include "common.cuh"

namespace b2f {

constexpr int kSelThreads = 256;
constexpr int kXchgMaxWorldMerge = 64;   // lists one merge handles (ranks of the exchange / shards of an index)
constexpr int kSortCap = 2048;  // == B2F_MAX_K

struct Seg {  // rows [local_start, local_start+count) of a shard carry ids global_start + i
  int64_t local_start, count, global_start;
};

struct SelectSmem {
  unsigned int hist[256];   // radix buckets
  unsigned int warp_tot[kSelThreads / 32];
  unsigned int digit, remaining, count, nvalid;
};

// Inclusive prefix sum over the block (256 threads), value per thread.
__device__ __forceinline__ unsigned int block_inclusive_scan(unsigned int v, SelectSmem& sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 1; s < 32; s <<= 1) {
    unsigned int t = __shfl_up_sync(0xffffffffu, v, s);
    if (lane >= s) v += t;
  }
  if (lane == 31) sm.warp_tot[warp] = v;
  __syncthreads();
  unsigned int base = 0;
  for (int w = 0; w < warp; ++w) base += sm.warp_tot[w];
  __syncthreads();
  return v + base;
}

// Top (8*passes) bits of the k-th largest record of in[0..n).  Requires >= k non-zero records.
__device__ uint64_t block_kth_prefix(const uint64_t* __restrict__ in, int n, int k, int passes,
                                     SelectSmem& sm) {
  uint64_t prefix = 0, mask = 0;
  unsigned int remaining = static_cast<unsigned int>(k);
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = 56 - 8 * pass;
    sm.hist[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += kSelThreads) {
      const uint64_t key = in[i];
      if ((key & mask) == prefix) atomicAdd(&sm.hist[static_cast<unsigned int>(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    const unsigned int h = sm.hist[255 - threadIdx.x];  // thread t owns bucket 255-t (descending)
    const unsigned int cum = block_inclusive_scan(h, sm);
    if (cum >= remaining && cum - h < remaining) {
      sm.digit = 255u - threadIdx.x;
      sm.remaining = remaining - (cum - h);
    }
    __syncthreads();
    prefix |= static_cast<uint64_t>(sm.digit) << shift;
    mask |= 0xffull << shift;
    remaining = sm.remaining;
    __syncthreads();
  }
  return prefix;
}

__device__ int block_count_valid(const uint64_t* __restrict__ in, int n, SelectSmem& sm) {
  if (threadIdx.x == 0) sm.nvalid = 0;
  __syncthreads();
  unsigned int c = 0;
  for (int i = threadIdx.x; i < n; i += kSelThreads) c += (in[i] != 0ull);
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&sm.nvalid, c);
  __syncthreads();
  const int r = static_cast<int>(sm.nvalid);
  __syncthreads();
  return r;
}

// Copy every non-empty record >= T from in[0..n) to out[0..limit); returns how many qualified
// (which may exceed `limit`: the caller flags the overflow).  Order arbitrary.
__device__ int block_compact(const uint64_t* __restrict__ in, int n, uint64_t T,
                             uint64_t* __restrict__ out, int limit, SelectSmem& sm) {
  if (threadIdx.x == 0) sm.count = 0;
  __syncthreads();
  for (int i0 = 0; i0 < n; i0 += kSelThreads) {
    const int i = i0 + threadIdx.x;
    const uint64_t key = (i < n) ? in[i] : 0ull;
    const bool keep = key != 0ull && key >= T;
    const unsigned int b = __ballot_sync(0xffffffffu, keep);
    if (b) {
      const int lane = threadIdx.x & 31;
      unsigned int base = 0;
      if (lane == 0) base = atomicAdd(&sm.count, __popc(b));
      base = __shfl_sync(0xffffffffu, base, 0);
      const unsigned int pos = base + __popc(b & ((1u << lane) - 1u));
      if (keep && pos < static_cast<unsigned int>(limit)) out[pos] = key;
    }
  }
  __syncthreads();
  const int m = static_cast<int>(sm.count);
  __syncthreads();
  return m;
}

// Threshold refresh between the phases of the SIMT scans, one block per query of the pass.
//   approx mode (exact == 0): tau = (k-th largest approximate score) - margin[q], rounded down;
//       survivors are the records with score >= tau.  Any true top-k row has an approximate score
//       within margin/2 of its exact score, so it survives (DESIGN.md "exactness argument").
//   exact mode: scores are final; tauP = the k-th largest record, survivors are exactly the top k.
// With fewer than k valid records nothing can be rejected yet (tau = -inf / tauP = 0).
__global__ void __launch_bounds__(kSelThreads) refresh_kernel(
    const uint64_t* __restrict__ cand_in, uint64_t* __restrict__ cand_out, int* __restrict__ cnt, int C, int k,
    int exact, const float* __restrict__ margin, float* __restrict__ tau, uint64_t* __restrict__ tauP,
    int n_override, int* __restrict__ ovf) {
  __shared__ SelectSmem sm;
  const int q = blockIdx.x;
  const uint64_t* in = cand_in + static_cast<int64_t>(q) * C;
  uint64_t* out = cand_out + static_cast<int64_t>(q) * C;
  int n = n_override >= 0 ? n_override : cnt[q];
  if (n > C) n = C;
  const int nvalid = block_count_valid(in, n, sm);
  uint64_t T = 0ull;
  float t = -INFINITY;
  if (nvalid >= k) {
    const uint64_t prefix = block_kth_prefix(in, n, k, exact ? 8 : 4, sm);
    if (exact) {
      T = prefix;
      t = key2f(static_cast<uint32_t>(prefix >> 32));
    } else {
      t = __fsub_rd(key2f(static_cast<uint32_t>(prefix >> 32)), margin[q]);
      T = static_cast<uint64_t>(fkey(t)) << 32;
    }
  }
  const int m = block_compact(in, n, T, out, C, sm);
  if (threadIdx.x == 0) {
    cnt[q] = min(m, C);
    tau[q] = t;
    tauP[q] = T;
    if (m > C) ovf[q] = 1;   // more rows within the error margin of the k-th score than the list holds
  }
}

__device__ __forceinline__ int64_t row_to_id(uint32_t row, const Seg* __restrict__ segs, int nseg,
                                             const int64_t* __restrict__ idmap) {
  if (idmap) return idmap[row];
  int lo = 0, hi = nseg - 1;
  while (lo < hi) {  // last segment with local_start <= row
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].local_start <= static_cast<int64_t>(row)) lo = mid; else hi = mid - 1;
  }
  return segs[lo].global_start + (static_cast<int64_t>(row) - segs[lo].local_start);
}

// Exact rescoring of the surviving candidates of a pass: fp64-accumulated dot, one warp per
// candidate, grid (queries, kRescoreSplit) so the ~2k random 3 KB row gathers per query are spread
// over the whole GPU.  Writes pack(exact score, row) to cand_out at the same position.
constexpr int kRescoreSplit = 8;
__global__ void __launch_bounds__(kSelThreads) rescore_kernel(
    const uint64_t* __restrict__ cand_in, uint64_t* __restrict__ cand_out, const int* __restrict__ cnt, int C,
    const float* __restrict__ q32 /* pass queries [nq_pass, 768] */, const float* __restrict__ x32) {
  __shared__ __align__(16) float Qs[kD];
  const int q = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int n = cnt[q];
  if (n > C) n = C;
  if (static_cast<int>(blockIdx.y) * (kSelThreads / 32) >= n) return;
  for (int i = threadIdx.x; i < kD; i += kSelThreads) Qs[i] = q32[static_cast<int64_t>(q) * kD + i];
  __syncthreads();
  const float4* q4 = reinterpret_cast<const float4*>(Qs);
  const uint64_t* src = cand_in + static_cast<int64_t>(q) * C;
  uint64_t* dst = cand_out + static_cast<int64_t>(q) * C;
  for (int c = blockIdx.y * (kSelThreads / 32) + warp; c < n; c += kRescoreSplit * (kSelThreads / 32)) {
    const uint64_t rec = src[c];
    uint64_t o = 0ull;
    if (rec != 0ull) {  // warp-uniform
      const uint32_t row = cand_row(rec);
      const float s = exact_dot_warp(q4, reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(row) * kD), lane);
      o = pack_cand(s, row);
    }
    if (lane == 0) dst[c] = o;
  }
}

// Final step of a pass, one block per query: top-k of the (exactly scored) candidates by the total
// order (score desc, row asc), sorted output, row -> id translation.
//   D_out / I_out: row stride `out_stride`, k entries written per query.
__global__ void __launch_bounds__(kSelThreads) final_kernel(
    uint64_t* __restrict__ cand_cur, uint64_t* __restrict__ cand_other, const int* __restrict__ cnt,
    int C, int k, const Seg* __restrict__ segs, int nseg, const int64_t* __restrict__ idmap,
    float* __restrict__ D_out, int64_t* __restrict__ I_out, int64_t out_stride, const int* __restrict__ ovf) {
  __shared__ SelectSmem sm;
  __shared__ uint64_t sortbuf[kSortCap];
  const int q = blockIdx.x;
  int n = cnt[q];
  if (n > C) n = C;
  uint64_t* src = cand_cur + static_cast<int64_t>(q) * C;
  uint64_t* dst = cand_other + static_cast<int64_t>(q) * C;
  if (n > kSortCap) {
    const int nvalid = block_count_valid(src, n, sm);
    uint64_t T = 0ull;
    if (nvalid >= k) T = block_kth_prefix(src, n, k, 8, sm);
    n = min(block_compact(src, n, T, dst, kSortCap, sm), kSortCap);  // == min(nvalid, k)
    uint64_t* t = src; src = dst; dst = t;
  }
  int P = 32;
  while (P < n) P <<= 1;
  for (int i = threadIdx.x; i < P; i += kSelThreads) sortbuf[i] = (i < n) ? src[i] : 0ull;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < (P >> 1); i += kSelThreads) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = sortbuf[lo], b = sortbuf[hi];
        if ((a < b) == desc) { sortbuf[lo] = b; sortbuf[hi] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < k; i += kSelThreads) {
    const uint64_t rec = (i < P) ? sortbuf[i] : 0ull;
    float s = -3.402823466e+38f;
    int64_t id = -1;
    if (rec != 0ull) {
      s = cand_score(rec);
      id = row_to_id(cand_row(rec), segs, nseg, idmap);
    }
    D_out[static_cast<int64_t>(q) * out_stride + i] = s;
    I_out[static_cast<int64_t>(q) * out_stride + i] = id;
  }
  __syncthreads();
  if (threadIdx.x == 0 && ovf != nullptr && ovf[q] != 0) I_out[static_cast<int64_t>(q) * out_stride] = -2;  // see finalize_kernel
}

// ---------------------------------------------------------------------------------------------
// Fused last step of a tensor-engine pass (both variants), one kFinThreads-thread block per query:
//   gather (every CTA's or CTA pair's private area)  ->  radix-select the k-th best
//   approximate score  ->  keep everything within the error margin of it  ->  exact fp64-accumulated
//   rescoring (one warp per survivor, two rows in flight per warp)  ->  bitonic sort by the total
//   order  ->  row -> id translation, (D, I) rows and the overflow flag.
// Replaces refresh_kernel + rescore_kernel + final_kernel (three launches and two trips of the
// lists through L2) at the end of the pass.  The lists stay in shared memory throughout
// (2 x P records of dynamic smem; lists longer than P are gathered to `gath` in global memory).
// ---------------------------------------------------------------------------------------------
constexpr int kFinThreads = 512;   // two blocks per SM: 173 queries fit one wave on 148 SMs

struct FinSmem {
  unsigned int hist[256];   // radix buckets
  unsigned int warp_tot[kFinThreads / 32];
  unsigned int digit, remaining, count, nvalid;
};

__device__ __forceinline__ unsigned int fin_scan256(unsigned int v, FinSmem& sm) {
  // inclusive scan of one value per thread over threads [0,256); every thread of the block calls it
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 1; s < 32; s <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, v, s);
    if (lane >= s) v += t;
  }
  if (lane == 31) sm.warp_tot[warp] = v;
  __syncthreads();
  unsigned int base = 0;
  if (warp < 8)
    for (int w = 0; w < warp; ++w) base += sm.warp_tot[w];
  __syncthreads();
  return v + base;
}

// Front part of finalize_kernel (all kFinThreads threads call it):
// gather the segmented list of query q ([0,m) + one private area per CTA or CTA pair) into `bufA`
// (shared memory, P records; longer lists go to `gath_q` in global memory), radix-select the key of
// the k-th best approximate score, derive the survivor threshold T = fkey(kth - margin) << 32.
struct FinFront {
  uint64_t* in;        // gathered list
  int n;               // its length
  int nvalid;          // non-empty records in it
  uint32_t kth_key;    // key of the k-th best approximate score (0xffffffff: fewer than k records)
  float tau;           // kth - margin (rounded down), -inf if fewer than k records
  uint64_t T;          // record threshold of tau (0: keep everything)
};

// histogram update with the increments of one warp pre-combined per bucket: in the first radix passes
// nearly all keys share their digit, and 32 same-address shared-memory atomics serialise
__device__ __forceinline__ void hist_add_aggregated(unsigned int* hist, bool active, unsigned int digit) {
  const unsigned int d = active ? digit : 0xffffffffu;
  const unsigned int peers = __match_any_sync(0xffffffffu, d);
  if (active && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[digit], static_cast<unsigned int>(__popc(peers)));
}

__device__ __forceinline__ FinFront fin_front(const uint64_t* __restrict__ list, uint64_t* __restrict__ gath_q, int m,
                                              int S, int cap_p, int max_pairs, const int* __restrict__ cnt2q, int k,
                                              float margin_q, uint64_t Tlow, uint64_t* bufA, int P, FinSmem& sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  FinFront f;
  // ---- 1. upper bound of the list length decides where it is gathered ----
  if (tid == 0) { sm.nvalid = 0; sm.count = 0; }
  __syncthreads();
  {
    int c = 0;
    if (tid < max_pairs) c = min(cnt2q[tid], cap_p);
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
    if (lane == 0 && c) atomicAdd(&sm.nvalid, static_cast<unsigned int>(c));
    __syncthreads();
  }
  int upper = m + static_cast<int>(sm.nvalid);
  if (upper > P && Tlow != 0ull) {
    // The raw list does not fit the shared-memory buffer, but most of it predates the thresholds (the
    // first tile of every CTA passes unfiltered: 148 x 128 records per query in the QS variant) and falls
    // to the Tlow filter below: count what survives it before sending the list through global memory.
    __syncthreads();
    int c = 0;
    for (int i = tid; i < m; i += kFinThreads) c += (list[i] != 0ull && list[i] >= Tlow);
    for (int p = warp; p < max_pairs; p += kFinThreads / 32) {
      const int cp = min(cnt2q[p], cap_p);
      const uint64_t* src = list + S + static_cast<int64_t>(p) * cap_p;
      for (int e = lane; e < cp; e += 32) c += (src[e] >= Tlow);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
    if (lane == 0 && c) atomicAdd(&sm.count, static_cast<unsigned int>(c));
    __syncthreads();
    upper = static_cast<int>(sm.count);
    __syncthreads();
    if (tid == 0) sm.count = 0;
    __syncthreads();
  }
  uint64_t* in = (upper <= P) ? bufA : gath_q;

  // ---- 2. gather + filter: keep the non-empty records >= Tlow.  Tlow is any lower bound of the final
  // survivor threshold (the last tau the in-kernel refresher published; 0 = keep all): everything at or
  // above the k-th score minus the margin passes it, so neither the k-th score nor the survivor set
  // changes, but the bulk of the early, loosely filtered appends never enters the select. ----
  auto append = [&](uint64_t rec) {
    const bool keep = rec != 0ull && rec >= Tlow;
    const unsigned int b = __ballot_sync(0xffffffffu, keep);
    if (b) {
      unsigned int base = 0;
      if (lane == 0) base = atomicAdd(&sm.count, __popc(b));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (keep) in[base + __popc(b & ((1u << lane) - 1u))] = rec;
    }
  };
  for (int i0 = 0; i0 < m; i0 += kFinThreads) {
    const int i = i0 + tid;
    append(i < m ? list[i] : 0ull);
  }
  for (int p = warp; p < max_pairs; p += kFinThreads / 32) {
    const int c = min(cnt2q[p], cap_p);
    const uint64_t* src = list + S + static_cast<int64_t>(p) * cap_p;
    for (int e0 = 0; e0 < c; e0 += 32) {
      const int e = e0 + lane;
      append(e < c ? src[e] : 0ull);
    }
  }
  __syncthreads();
  const int n = static_cast<int>(sm.count);
  __syncthreads();
  if (tid == 0) { sm.nvalid = static_cast<unsigned int>(n); sm.count = 0; }
  __syncthreads();

  // ---- 3. k-th best approximate score (radix select on the 32-bit score key) ----
  f.in = in;
  f.n = n;
  f.nvalid = static_cast<int>(sm.nvalid);
  f.kth_key = 0xffffffffu;
  f.tau = -INFINITY;
  f.T = 0ull;
  if (f.nvalid >= k) {
    uint32_t prefix = 0, mask = 0;
    unsigned int remaining = static_cast<unsigned int>(k);
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      if (tid < 256) sm.hist[tid] = 0;
      __syncthreads();
      for (int i0 = 0; i0 < n; i0 += kFinThreads) {
        const int i = i0 + tid;
        const uint32_t key = (i < n) ? static_cast<uint32_t>(in[i] >> 32) : 0u;
        hist_add_aggregated(sm.hist, key != 0u && (key & mask) == prefix, (key >> shift) & 255u);
      }
      __syncthreads();
      const unsigned int h = (tid < 256) ? sm.hist[255 - tid] : 0u;   // thread t owns bucket 255-t (descending)
      const unsigned int cum = fin_scan256(h, sm);
      if (tid < 256 && cum >= remaining && cum - h < remaining) {
        sm.digit = 255u - tid;
        sm.remaining = remaining - (cum - h);
      }
      __syncthreads();
      prefix |= sm.digit << shift;
      mask |= 0xffu << shift;
      remaining = sm.remaining;
      __syncthreads();
    }
    f.kth_key = prefix;
    f.tau = __fsub_rd(key2f(prefix), margin_q);
    f.T = static_cast<uint64_t>(fkey(f.tau)) << 32;
  }
  return f;
}

__global__ void __launch_bounds__(kFinThreads, 2) finalize_kernel(
    const uint64_t* __restrict__ cand, uint64_t* __restrict__ gath, const int* __restrict__ cnt, int C, int k,
    const float* __restrict__ margin, int S, int cap_p, int max_pairs, const int* __restrict__ cnt2,
    const int* __restrict__ ovf, int* __restrict__ ovf_out, const float* __restrict__ q32,
    const float* __restrict__ x32, const Seg* __restrict__ segs, int nseg, const int64_t* __restrict__ idmap,
    float* __restrict__ D_out, int64_t* __restrict__ I_out, int64_t out_stride, int P,
    const float* __restrict__ tau_low /* [nq] lower bounds of the survivor thresholds, or null */,
    const float* __restrict__ mu /* [768] centre of the shard: approximate scores are q.(p - mu) */) {
  extern __shared__ __align__(16) uint64_t fin_buf[];   // [P] gathered list, then the survivors
  __shared__ FinSmem sm;
  __shared__ __align__(16) float Qs[kD];
  __shared__ double q_dot_mu;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t* bufB = fin_buf + P;
  for (int i = tid; i < kD; i += kFinThreads) Qs[i] = q32[static_cast<int64_t>(q) * kD + i];
  const FinFront f = fin_front(cand + static_cast<int64_t>(q) * C, gath + static_cast<int64_t>(q) * C, min(cnt[q], S), S, cap_p,
                               max_pairs, cnt2 + q * max_pairs, k, margin[q],
                               tau_low ? static_cast<uint64_t>(fkey(tau_low[q])) << 32 : 0ull, fin_buf, P, sm);
  const uint64_t* in = f.in;
  const int n = f.n;
  const uint64_t T = f.T;

  // ---- 4./5. survivors and exact rescoring, in two rounds ----
  // Round A: the records at or above the k-th best APPROXIMATE score (>= k of them) are rescored exactly.
  //   Their smallest exact score T is a lower bound of the true k-th best score (k real rows reach it).
  // Round B: a true top-k row r has s_r >= T and an approximate score s~_r >= s_r - eps >= T - eps, so only
  //   the records in [T - eps, k-th approximate score) remain to be rescored.  Each of the round-A rows has
  //   s >= (k-th approximate) - eps, hence T - eps >= (k-th approximate) - 2 eps: never more rows than the
  //   one-round window [k-th approximate - 2 eps, ...), and about half the margin in practice (the real
  //   errors are far below their worst-case bound, so T sits next to the k-th approximate score).  Fewer 3 KB
  //   random row gathers is what this buys: ~140 instead of ~200 per query on isotropic rows, ~3x fewer on
  //   rows with a common mean.
  const float4* q4 = reinterpret_cast<const float4*>(Qs);
  auto collect = [&](uint64_t lo, uint64_t hi_excl, int base0) {   // records in [lo, hi_excl) -> bufB[base0 ...)
    if (tid == 0) sm.count = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += kFinThreads) {
      const int i = i0 + tid;
      const uint64_t rec = (i < n) ? in[i] : 0ull;
      const bool keep = rec != 0ull && rec >= lo && rec < hi_excl;
      const unsigned int b = __ballot_sync(0xffffffffu, keep);
      if (b) {
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(&sm.count, __popc(b));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned int pos = static_cast<unsigned int>(base0) + base + __popc(b & ((1u << lane) - 1u));
        if (keep && pos < static_cast<unsigned int>(S)) bufB[pos] = rec;
      }
    }
    __syncthreads();
    const int c = static_cast<int>(sm.count);
    __syncthreads();
    return c;
  };
  auto rescore = [&](int c_begin, int c_end) {   // exact scores in place, two rows in flight per warp
    uint32_t kmin = 0xffffffffu;
    for (int c = c_begin + warp; c < c_end; c += 2 * (kFinThreads / 32)) {
      const int c2 = c + kFinThreads / 32;
      const uint32_t rowA = cand_row(bufB[c]);
      const uint32_t rowB = (c2 < c_end) ? cand_row(bufB[c2]) : rowA;
      const double a = lane_partial_f64(q4, reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(rowA) * kD), lane);
      const double b = lane_partial_f64(q4, reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(rowB) * kD), lane);
      const float sa = static_cast<float>(warp_butterfly_sum(a));
      const float sb = static_cast<float>(warp_butterfly_sum(b));
      kmin = min(kmin, min(fkey(sa), fkey(sb)));
      if (lane == 0) {
        bufB[c] = pack_cand(sa, rowA);
        if (c2 < c_end) bufB[c2] = pack_cand(sb, rowB);
      }
    }
    return kmin;   // order-preserving key of the smallest exact score this warp produced
  };
  // The approximate scores live in CENTRED space (s~ ~ q.p - q.mu, DESIGN.md section 4), the exact ones do
  // not: T is moved into centred space with c = q.mu, evaluated in fp64 (products of fp32 values are exact,
  // the 768-term sum is good to ~1e-13 relative; 1e-9 |c| of slack covers it many times over).
  if (warp == 0) {
    const double c = warp_butterfly_sum(lane_partial_f64(q4, reinterpret_cast<const float4*>(mu), lane));
    if (lane == 0) q_dot_mu = c;
  }
  const bool two_rounds = f.kth_key != 0xffffffffu && margin[q] > 0.f;
  const uint64_t recA = two_rounds ? (static_cast<uint64_t>(f.kth_key) << 32) : T;   // T == 0 with fewer than k records
  const int mA_all = collect(recA, ~0ull, 0);
  const int mA = min(mA_all, S);
  if (tid == 0) sm.digit = 0xffffffffu;
  __syncthreads();
  const uint32_t kmin = rescore(0, mA);
  if (lane == 0 && kmin != 0xffffffffu) atomicMin(&sm.digit, kmin);
  __syncthreads();
  int m2_all = mA_all;
  if (two_rounds && mA_all <= S) {
    const double t_exact = static_cast<double>(key2f(sm.digit));         // min exact score of round A (uncentred)
    const double c = q_dot_mu;
    const float lowB = __double2float_rd(t_exact - c - static_cast<double>(__fmul_ru(margin[q], 0.5f)) - 1e-9 * fabs(c));   // (T - q.mu) - eps
    const uint64_t recB = max(T, static_cast<uint64_t>(fkey(lowB)) << 32);   // never below the one-round window
    __syncthreads();
    const int mB_all = collect(recB, recA, mA);
    m2_all = mA_all + mB_all;
    (void)rescore(mA, min(m2_all, S));
  }
  const int m2 = min(m2_all, S);
  int P2 = 32;
  while (P2 < m2) P2 <<= 1;
  for (int i = m2 + tid; i < P2; i += kFinThreads) bufB[i] = 0ull;
  __syncthreads();

  // ---- 6. bitonic sort, descending by (score, row asc) ----
  for (int size = 2; size <= P2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (P2 >> 1); i += kFinThreads) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = bufB[lo], b = bufB[hi];
        if ((a < b) == desc) { bufB[lo] = b; bufB[hi] = a; }
      }
      __syncthreads();
    }
  }

  // ---- 7. output ----
  for (int i = tid; i < k; i += kFinThreads) {
    const uint64_t rec = (i < P2) ? bufB[i] : 0ull;
    float s = -3.402823466e+38f;
    int64_t id = -1;
    if (rec != 0ull) {
      s = cand_score(rec);
      id = row_to_id(cand_row(rec), segs, nseg, idmap);
    }
    D_out[static_cast<int64_t>(q) * out_stride + i] = s;
    I_out[static_cast<int64_t>(q) * out_stride + i] = id;
  }
  if (tid == 0) {
    // flag bits: 1 = a private area was too small (thresholds came late), 2 = more rows within the error
    // margin of the k-th score than the survivor buffer holds (ties / unresolvable score distribution)
    const int kind = (ovf[q] != 0 ? 1 : 0) | (m2_all > S ? 2 : 0);
    const bool bad = kind != 0;
    if (ovf_out) ovf_out[q] = kind;
    // in-band marker for the sharded layout: a row whose list overflowed carries id -2 in its first
    // slot until the exact engine has re-run it; merge_kernel reports it to every rank
    if (bad) I_out[static_cast<int64_t>(q) * out_stride] = -2;
  }
}

// Marker mode of the merges (the asynchronous search of a multi-shard index): when some part's list overflowed
// (id -2 in its slot 0, see finalize_kernel) the merged row is not final either, so it carries -2 in its slot 0 too,
// exactly like the row of a single-shard search, until the re-run shard's parts are merged again.
__device__ __forceinline__ void mark_pending_row(const int64_t* Ip, int G, int64_t q, int k, int64_t strideI,
                                                 int64_t* __restrict__ I) {
  for (int g = 0; g < G; ++g)
    if (__ldcg(Ip + static_cast<int64_t>(g) * strideI + q * k) == -2) {
      I[q * k] = -2;
      return;
    }
}

// Cross-shard merge: parts [G][nq][k] (each sorted by score desc, padded with id = -1) -> [nq][k].
// Rank-by-counting: an element's output position is its position in its own list plus, for every
// other list, the number of elements that precede it; ties go to the earlier part, then the earlier
// position (the reference's merge keeps the earlier block on `>=`, :218).
// Part g starts at Dp + g*strideD floats / Ip + g*strideI int64s (nq*k for two dense arrays; the
// packed [D | I] records of the exchange use the packed part size).  Parts are read with ld.global.cg:
// in the peer-memory exchange they are written by OTHER GPUs while this kernel is already resident.
// The G lists of the query are first staged in shared memory (G*k*12 bytes; `staged` = 0 when that does
// not fit): the G-1 binary searches per element would otherwise be ~100 dependent L2 round trips per
// thread (measured 0.15-0.25 ms per merge at G = 8 before staging).
// Sort-mode merge (the default whenever the padded G*k records fit shared memory as 8-byte keys): every
// valid (score, part, position) becomes one key  fkey(score) << 32 | ~(g*k + i),  so a descending sort orders
// by (score desc, part asc, position asc) — the reference's `>=` merge rule — and the first k keys are the
// result; ids are fetched for those k only.  One bitonic sort of <= 8192 keys replaces (G-1) binary searches
// per record (measured 41 -> 18 us per launch at G = 8, k = 100; two lists stay on rank-by-counting: 7 vs 8 us).
__device__ __forceinline__ void merge_sort_body(const float* Dp, const int64_t* Ip, int G, int64_t q, int k,
                                                float* __restrict__ D, int64_t* __restrict__ I, int64_t strideD,
                                                int64_t strideI, int* saw_overflow, int mark_pending,
                                                unsigned char* stage_smem) {
  uint64_t* keys = reinterpret_cast<uint64_t*>(stage_smem);
  const int E = G * k;
  int P2 = 32;
  while (P2 < E) P2 <<= 1;
  for (int e = threadIdx.x; e < P2; e += blockDim.x) {
    uint64_t key = 0ull;
    if (e < E) {
      const int g = e / k, i = e - g * k;
      const int64_t id = __ldcg(Ip + static_cast<int64_t>(g) * strideI + q * k + i);
      if (id == -2 && saw_overflow != nullptr) *saw_overflow = 1;   // a shard's list overflowed: result pending its re-run
      if (id >= 0) {
        const float sc = __ldcg(Dp + static_cast<int64_t>(g) * strideD + q * k + i);
        key = (static_cast<uint64_t>(fkey(sc)) << 32) | static_cast<uint64_t>(0xffffffffu - static_cast<uint32_t>(e));
      }
    }
    keys[e] = key;
  }
  __syncthreads();
  for (int size = 2; size <= P2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < (P2 >> 1); i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a < b) == desc) { keys[lo] = b; keys[hi] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const uint64_t key = (i < P2) ? keys[i] : 0ull;
    float sc = -3.402823466e+38f;
    int64_t id = -1;
    if (key != 0ull) {
      const int e = static_cast<int>(0xffffffffu - static_cast<uint32_t>(key));
      const int g = e / k, ii = e - g * k;
      sc = key2f(static_cast<uint32_t>(key >> 32));
      id = __ldcg(Ip + static_cast<int64_t>(g) * strideI + q * k + ii);
    }
    D[q * k + i] = sc;
    I[q * k + i] = id;
  }
  if (mark_pending && threadIdx.x == 0) mark_pending_row(Ip, G, q, k, strideI, I);   // after this thread's slot-0 store
}

__device__ __forceinline__ void merge_body(const float* Dp, const int64_t* Ip, int G, int64_t q,
                                           int k, float* __restrict__ D, int64_t* __restrict__ I,
                                           int64_t strideD, int64_t strideI, int* saw_overflow, int* total_valid_s,
                                           int staged, int mark_pending, unsigned char* stage_smem) {
  const int E = G * k;
  int64_t* sI = reinterpret_cast<int64_t*>(stage_smem);            // [G][k]
  float* sD = reinterpret_cast<float*>(stage_smem + static_cast<size_t>(E) * sizeof(int64_t));   // [G][k]
  if (threadIdx.x == 0) *total_valid_s = 0;
  if (staged) {
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
      const int g = e / k, i = e - g * k;
      sI[e] = __ldcg(Ip + static_cast<int64_t>(g) * strideI + q * k + i);
      sD[e] = __ldcg(Dp + static_cast<int64_t>(g) * strideD + q * k + i);
    }
  }
  __syncthreads();
  auto ld_id = [&](int g, int i) -> int64_t {
    return staged ? sI[g * k + i] : __ldcg(Ip + static_cast<int64_t>(g) * strideI + q * k + i);
  };
  auto ld_score = [&](int g, int i) -> float {
    return staged ? sD[g * k + i] : __ldcg(Dp + static_cast<int64_t>(g) * strideD + q * k + i);
  };
  // valid prefix of every list (lists are padded at the END with id = -1, or id = -2 in slot 0 for a pending
  // re-run): the binary searches below then only ever read scores
  __shared__ int n_valid_s[kXchgMaxWorldMerge];
  if (threadIdx.x < G) {
    const int g = threadIdx.x;
    int lo = 0, hi = k;
    while (lo < hi) {                       // first index whose id is negative
      const int mid = (lo + hi) >> 1;
      if (ld_id(g, mid) >= 0) lo = mid + 1; else hi = mid;
    }
    n_valid_s[g] = lo;
    if (ld_id(g, 0) == -2 && saw_overflow != nullptr) *saw_overflow = 1;   // a shard's list overflowed: result pending its re-run
  }
  __syncthreads();
  for (int e = threadIdx.x; e < E; e += blockDim.x) {
    const int g = e / k, i = e - g * k;
    if (i >= n_valid_s[g]) continue;
    const int64_t id = ld_id(g, i);
    if (id < 0) continue;                   // the marker row of a pending re-run
    atomicAdd(total_valid_s, 1);
    const float s = ld_score(g, i);
    int rank = i;
    for (int g2 = 0; g2 < G; ++g2) {
      if (g2 == g) continue;
      // count valid elements of list g2 that precede (s): score > s, or == s when g2 < g
      int lo = 0, hi = n_valid_s[g2];
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float s2 = ld_score(g2, mid);
        const bool before = s2 > s || (s2 == s && g2 < g);
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      D[q * k + rank] = s;
      I[q * k + rank] = id;
    }
  }
  __syncthreads();
  for (int i = *total_valid_s + threadIdx.x; i < k; i += blockDim.x) {
    D[q * k + i] = -3.402823466e+38f;
    I[q * k + i] = -1;
  }
  // the ranked stores are behind the barrier above; the padding store of slot 0, if any, is this thread's own
  if (mark_pending && threadIdx.x == 0) mark_pending_row(Ip, G, q, k, strideI, I);
}

constexpr int kMergeStageMaxBytes = 96 * 1024;
// threads of a merge block: lists of a few hundred entries take 256; k = 1000 over 8 ranks is 8000 entries per query
inline int merge_threads(int G, int k) { return static_cast<int64_t>(G) * k > 2048 ? 1024 : 256; }
// How a merge of G lists of k runs: mode 2 = sort the keys in shared memory (padded count * 8 bytes), mode 1 =
// rank-by-counting over lists staged in shared memory (G*k*12 bytes), mode 0 = rank-by-counting out of L2.
inline int merge_mode(int G, int k) {
  int64_t p2 = 32;
  while (p2 < static_cast<int64_t>(G) * k) p2 <<= 1;
  if (G >= 4 && p2 * 8 <= kMergeStageMaxBytes) return 2;   // rank-by-counting costs (G-1) searches per record: fine for 2-3 lists
  return static_cast<int64_t>(G) * k * 12 <= kMergeStageMaxBytes ? 1 : 0;
}
inline int merge_stage_bytes(int G, int k) {   // dynamic shared memory of the merge kernels
  const int mode = merge_mode(G, k);
  if (mode == 2) {
    int64_t p2 = 32;
    while (p2 < static_cast<int64_t>(G) * k) p2 <<= 1;
    return static_cast<int>(p2 * 8);
  }
  return mode == 1 ? G * k * 12 : 0;
}

__global__ void __launch_bounds__(1024) merge_kernel(const float* Dp, const int64_t* Ip, int G, int64_t nq,
                                                    int k, float* __restrict__ D, int64_t* __restrict__ I,
                                                    int64_t strideD, int64_t strideI,
                                                    int* __restrict__ saw_overflow /* mapped host int or null */,
                                                    int staged, int mark_pending) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  __shared__ int total_valid;
  if (staged == 2) merge_sort_body(Dp, Ip, G, blockIdx.x, k, D, I, strideD, strideI, saw_overflow, mark_pending, merge_smem);
  else merge_body(Dp, Ip, G, blockIdx.x, k, D, I, strideD, strideI, saw_overflow, &total_valid, staged, mark_pending, merge_smem);
}

// ---------------------------------------------------------------------------------------------
// Peer-memory exchange of the one-process-per-GPU layout (replaces ncclAllGather + merge).
//
// Every rank owns an exchange buffer  [4 slots][world parts][part_cap bytes] + flags[4][world]
// that all peers have mapped (CUDA IPC, NVLink).  Step `seq` (parity seq & 1):
//   xchg_push_kernel : copies this rank's packed [D | I] part into slot `rank` of EVERY rank's buffer
//                      with 16-byte stores over NVLink; the last block to finish publishes
//                      flags[parity][rank] = seq on every rank (fence.sys + release store);
//   xchg_merge_kernel: waits until the `world` flags of its own buffer reach seq (acquire loads),
//                      then merges the parts exactly like merge_kernel.
// No host round trip, no NCCL kernel, no proxy thread.  The merge of step s is enqueued behind the push
// of step s+1 (deferred by one search; b2f_search_finish flushes the last one), so a rank never idles
// waiting for the momentarily slowest GPU.  Slot reuse four steps later is safe: a rank pushes step
// s+4 only after its merge of step s+2, which needs every peer's push of s+2, which each peer enqueues
// after its own merge of step s.
// ---------------------------------------------------------------------------------------------
constexpr int kXchgMaxWorld = 16;
constexpr int kXchgSlots = 4;       // exchange steps in flight per rank (deferred merge needs >= 3)
struct XchgPeers {
  char* part[kXchgMaxWorld];        // peer r: address of slot [parity][my rank] in r's buffer
  unsigned int* flag[kXchgMaxWorld];  // peer r: address of flags[parity][my rank] in r's buffer
  int world;
};

__global__ void __launch_bounds__(256) xchg_push_kernel(const uint4* __restrict__ stage, int64_t n_vec /* 16-byte units */,
                                                        XchgPeers peers, unsigned int seq, int* __restrict__ counter) {
  const int r = blockIdx.x;   // destination rank
  uint4* dst = reinterpret_cast<uint4*>(peers.part[r]);
  for (int64_t i = static_cast<int64_t>(blockIdx.y) * blockDim.x + threadIdx.x; i < n_vec;
       i += static_cast<int64_t>(gridDim.y) * blockDim.x)
    dst[i] = stage[i];
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();                                    // this block's stores, system-wide
    const int total = static_cast<int>(gridDim.x * gridDim.y);
    if (atomicAdd(counter, 1) == total - 1) {                  // last block of the launch
      __threadfence_system();
      *counter = 0;
      for (int p = 0; p < peers.world; ++p)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(peers.flag[p]), "r"(seq) : "memory");
    }
  }
}

__global__ void __launch_bounds__(1024) xchg_merge_kernel(const char* __restrict__ parts /* [world][part_cap] of this parity */,
                                                         const unsigned int* flags /* [world] of this parity */,
                                                         unsigned int seq, int world, int64_t part_cap, int64_t i_off,
                                                         int64_t nq, int k, float* __restrict__ D, int64_t* __restrict__ I,
                                                         int* __restrict__ saw_overflow, int* __restrict__ err, int staged) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  __shared__ int total_valid;
  if (threadIdx.x < world) {
    long long t0 = 0;
    for (unsigned int spin = 0;; ++spin) {
      unsigned int v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
      if (static_cast<int>(v - seq) >= 0) break;             // sequence numbers only grow (wrap-safe compare)
      if ((spin & 255u) == 255u) {
        const long long now = clock64();
        if (t0 == 0) t0 = now;
        else if (now - t0 > 8000000000ll) { if (err) *err = 1; break; }   // ~4 s: a peer died; report, never hang
        __nanosleep(200);
      }
    }
  }
  __syncthreads();
  if (staged == 2)
    merge_sort_body(reinterpret_cast<const float*>(parts), reinterpret_cast<const int64_t*>(parts + i_off), world, blockIdx.x,
                    k, D, I, part_cap / 4, part_cap / 8, saw_overflow, 0, merge_smem);
  else
    merge_body(reinterpret_cast<const float*>(parts), reinterpret_cast<const int64_t*>(parts + i_off), world, blockIdx.x, k,
               D, I, part_cap / 4, part_cap / 8, saw_overflow, &total_valid, staged, 0, merge_smem);
}

// ---------------------------------------------------------------------------------------------
// EvalDevQuery's id handling on device (reference drivers/run_convdr_inference.py:43-69): for every query,
// the first topN entries of the merged ranking (passage offsets, best first) are translated with
// pid = offset2pid[offset]; a pid that already appeared at a better rank is dropped; the survivors keep their
// order and move to the front; unfilled tail slots hold (pid 0, score 0) exactly like the reference's
// pre-filled `[(0, 0)] * topN`.  A negative offset indexes from the end (Python semantics: the reference's
// `-1` wrap of a short block, :190).  One block per query; the pids of the row live in shared memory and
// position i looks for an equal pid among positions < i.
// ---------------------------------------------------------------------------------------------
constexpr int kDedupThreads = 256;
__global__ void __launch_bounds__(kDedupThreads) rank_dedup_kernel(
    const int64_t* __restrict__ I, const float* __restrict__ D32, const double* __restrict__ D64, int64_t in_stride,
    int topN, const int64_t* __restrict__ offset2pid, int64_t n_offsets, int64_t* __restrict__ pid_out,
    double* __restrict__ score_out, int* __restrict__ count_out) {
  extern __shared__ __align__(16) unsigned char dd_smem[];
  int64_t* pid_s = reinterpret_cast<int64_t*>(dd_smem);                        // [topN]
  int* keep_s = reinterpret_cast<int*>(dd_smem + sizeof(int64_t) * topN);      // [topN] then exclusive ranks
  __shared__ int warp_tot[kDedupThreads / 32];
  __shared__ int running;
  const int64_t q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < topN; i += kDedupThreads) {
    int64_t off = I[q * in_stride + i];
    if (off < 0) off += n_offsets;
    pid_s[i] = (off >= 0 && off < n_offsets) ? offset2pid[off] : -1;           // out of range: never equal to a real pid
  }
  if (tid == 0) running = 0;
  __syncthreads();
  for (int i = tid; i < topN; i += kDedupThreads) {
    const int64_t p = pid_s[i];
    int first = 1;
    for (int j = 0; j < i; ++j) first &= (pid_s[j] != p);
    keep_s[i] = first;
  }
  __syncthreads();
  // compaction: ranks in position order, chunk by chunk
  for (int i0 = 0; i0 < topN; i0 += kDedupThreads) {
    const int i = i0 + tid;
    const int kp = (i < topN) ? keep_s[i] : 0;
    int v = kp;
#pragma unroll
    for (int sft = 1; sft < 32; sft <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, sft);
      if (lane >= sft) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int base = running;
    for (int w = 0; w < warp; ++w) base += warp_tot[w];
    if (kp) {
      const int r = base + v - 1;
      pid_out[q * topN + r] = pid_s[i];
      score_out[q * topN + r] = D64 ? D64[q * in_stride + i] : static_cast<double>(D32[q * in_stride + i]);
    }
    __syncthreads();
    if (tid == kDedupThreads - 1) running = base + v;
    __syncthreads();
  }
  const int n_kept = running;
  for (int i = n_kept + tid; i < topN; i += kDedupThreads) {
    pid_out[q * topN + i] = 0;
    score_out[q * topN + i] = 0.0;
  }
  if (tid == 0) count_out[q] = n_kept;
}

}  // namespace b2f
