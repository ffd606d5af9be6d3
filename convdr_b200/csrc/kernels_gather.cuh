// kernels_gather.cuh — rows by label: the label -> row lookup of a shard and the row gather behind faiss's
// reconstruct / reconstruct_batch / search_and_reconstruct.  Off the search path: no scoring, selection or merge
// kernel reads anything defined here.
//
// A shard's labels take one of three forms (the host picks one per index generation, DESIGN.md section 2):
//   1. segment labels (add / add_synthetic): rows [local_start, local_start + count) carry global_start + i.  The
//      segments, sorted by global_start, and end_max[i] = max(global_start + count) over segments 0..i are the
//      whole index;
//   2. explicit labels in ascending (non-decreasing) order: the label map itself is searched, row = position;
//   3. any other explicit labels: a sorted copy, keys [n] and their rows [n] (12 bytes per row).
// A lookup reports how many rows hold the label (0, 1, or 2 for "two or more"), so a label held by several rows is
// detected from overlapping segments (form 1) or equal neighbours (forms 2 and 3).
#pragma once
#include "common.cuh"
#include "kernels_select.cuh"

namespace b2f {

constexpr int kGatherThreads = 256;   // 8 warps, one label each per iteration

struct LabelIndex {
  const Seg* segs;             // form 1: sorted by global_start
  const int64_t* end_max;      // form 1: prefix maximum of global_start + count
  int nseg;
  const int64_t* keys;         // forms 2 and 3: ascending labels [n] (form 2: the label map)
  const uint32_t* rows;        // form 3: row of keys[i]; null in form 2 (row = i)
  int64_t n;
};

// Warp-uniform lookup: every lane returns the same count and row.
__device__ __forceinline__ int label_lookup(const LabelIndex& L, int64_t label, uint32_t* row) {
  const int lane = threadIdx.x & 31;
  int found = 0;
  if (L.segs) {
    int lo = 0, hi = L.nseg;   // segments [0, lo) start at or below the label
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(&L.segs[mid].global_start) <= label) lo = mid + 1; else hi = mid;
    }
    // walk back 32 segments at a time while some segment at or before `base` still reaches past the label: one step
    // when the segments do not overlap
    for (int base = lo - 1; base >= 0 && found < 2 && __ldg(L.end_max + base) > label; base -= 32) {
      const int j = base - lane;
      const bool hit = j >= 0 && label < __ldg(&L.segs[j].global_start) + __ldg(&L.segs[j].count);
      const unsigned int b = __ballot_sync(0xffffffffu, hit);
      if (b && found == 0) {
        const int s = base - (__ffs(b) - 1);
        *row = static_cast<uint32_t>(__ldg(&L.segs[s].local_start) + (label - __ldg(&L.segs[s].global_start)));
      }
      found += __popc(b);
    }
  } else {
    int64_t lo = 0, hi = L.n;   // first key >= label
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(L.keys + mid) < label) lo = mid + 1; else hi = mid;
    }
    if (lo < L.n && __ldg(L.keys + lo) == label) {
      found = (lo + 1 < L.n && __ldg(L.keys + lo + 1) == label) ? 2 : 1;
      *row = L.rows ? __ldg(L.rows + lo) : static_cast<uint32_t>(lo);
    }
  }
  return min(found, 2);
}

// One warp per requested label labels[i], i < n: when this shard holds the label, found[i] grows by the rows that
// hold it and one of them is copied (3 KB, 128-bit non-coherent loads, 128-bit stores) to
//   out + i * 768            when out is set (the output itself: this shard can store there), or
//   stage + slot * 768       otherwise, with stage_pos[slot] = i and slot taken from *stage_count.
// A negative label (search padding) is written as 0xFF bytes, by the shard with pad_owner only.
__global__ void __launch_bounds__(kGatherThreads) gather_rows_kernel(
    LabelIndex L, const float* __restrict__ x32, const int64_t* __restrict__ labels, int64_t n, int pad_owner,
    float* __restrict__ out, int* __restrict__ found, float* __restrict__ stage, uint32_t* __restrict__ stage_pos,
    unsigned int* __restrict__ stage_count) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t i = warp0; i < n; i += nwarps) {
    const int64_t label = __ldg(labels + i);
    if (label < 0) {
      if (pad_owner) {
        float4* dst = reinterpret_cast<float4*>(out + i * kD);
        const float4 ff = make_float4(__uint_as_float(0xffffffffu), __uint_as_float(0xffffffffu),
                                      __uint_as_float(0xffffffffu), __uint_as_float(0xffffffffu));
#pragma unroll
        for (int j = 0; j < kF4PerLane; ++j) dst[lane + 32 * j] = ff;
      }
      continue;
    }
    uint32_t row = 0;
    const int c = label_lookup(L, label, &row);
    if (c == 0) continue;
    float* dst_row;
    if (out) {
      dst_row = out + i * kD;
    } else {
      unsigned int slot = 0;
      if (lane == 0) {
        slot = atomicAdd(stage_count, 1u);
        stage_pos[slot] = static_cast<uint32_t>(i);
      }
      slot = __shfl_sync(0xffffffffu, slot, 0);
      dst_row = stage + static_cast<int64_t>(slot) * kD;
    }
    if (lane == 0) atomicAdd(found + i, c);
    const float4* src = reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(row) * kD);
    float4 v[kF4PerLane];
#pragma unroll
    for (int j = 0; j < kF4PerLane; ++j) v[j] = __ldg(src + lane + 32 * j);
    float4* dst = reinterpret_cast<float4*>(dst_row);
#pragma unroll
    for (int j = 0; j < kF4PerLane; ++j) dst[lane + 32 * j] = v[j];
  }
}

// First shard, after the staging shards' rows arrived: row r of `rows` goes to out + pos[r] * 768 (one warp per
// row), and the per-label counts of the n_parts staging shards ([n_parts][n]) are added to found.
__global__ void __launch_bounds__(kGatherThreads) scatter_rows_kernel(
    const float* __restrict__ rows, const uint32_t* __restrict__ pos, int64_t n_rows, float* __restrict__ out,
    const int* __restrict__ parts, int n_parts, int64_t n, int* __restrict__ found) {
  const int lane = threadIdx.x & 31;
  const int64_t t0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = t0 >> 5; r < n_rows; r += nthreads >> 5) {
    const float4* src = reinterpret_cast<const float4*>(rows + r * kD);
    float4* dst = reinterpret_cast<float4*>(out + static_cast<int64_t>(__ldg(pos + r)) * kD);
    float4 v[kF4PerLane];
#pragma unroll
    for (int j = 0; j < kF4PerLane; ++j) v[j] = __ldg(src + lane + 32 * j);
#pragma unroll
    for (int j = 0; j < kF4PerLane; ++j) dst[lane + 32 * j] = v[j];
  }
  for (int64_t i = t0; i < n; i += nthreads) {
    int c = 0;
    for (int p = 0; p < n_parts; ++p) c += parts[static_cast<int64_t>(p) * n + i];
    if (c) found[i] += c;
  }
}

// Form 2 test: *descending = 1 when some label is smaller than the one before it (must be 0 on entry).
__global__ void labels_descend_kernel(const int64_t* __restrict__ ids, int64_t n, int* __restrict__ descending) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  bool d = false;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i + 1 < n; i += stride)
    d = d || __ldg(ids + i) > __ldg(ids + i + 1);
  if (__syncthreads_or(d) && threadIdx.x == 0) *descending = 1;
}

__global__ void iota_rows_kernel(uint32_t* __restrict__ rows, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    rows[i] = static_cast<uint32_t>(i);
}

}  // namespace b2f
