// kernels_selector.cuh — build of a filtered-search selector (faiss IDSelector semantics), off the search path.
//
// A selector is evaluated once per shard against the labels search returns (explicit ids or the implicit
// positions of the segments, row_to_id) and stored as
//   - a row bitmap over shard-local rows, one 32-bit word per 32 rows: the unit of a QS epilogue warp, of a TS
//     epilogue thread and of an int8 shadow tile, so every role that decides hits reads ONE word;
//   - per-tile "any selected row" flags of the QS tiles (256 rows) and TS tiles (64 rows), which the host compacts
//     into the tile lists the scoring launches walk.
#pragma once
#include "common.cuh"
#include "kernels_select.cuh"

namespace b2f {

enum SelKind { kSelRange = 1, kSelBatch = 2, kSelBitmap = 3 };

struct SelDesc {
  int kind, invert;
  int64_t imin, imax;        // range: imin <= id < imax
  const int64_t* ids;        // batch: sorted, unique
  int64_t n_ids;
  const uint8_t* bitmap;     // bitmap: id selected iff (bitmap[id >> 3] >> (id & 7)) & 1, ids >= 8 n_bytes never
  int64_t n_bytes;
};

__device__ __forceinline__ bool sel_member(const SelDesc& d, int64_t id) {
  bool m;
  if (d.kind == kSelRange) {
    m = id >= d.imin && id < d.imax;
  } else if (d.kind == kSelBatch) {
    int64_t lo = 0, hi = d.n_ids;   // first index with ids[i] >= id
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(d.ids + mid) < id) lo = mid + 1; else hi = mid;
    }
    m = lo < d.n_ids && __ldg(d.ids + lo) == id;
  } else {
    const uint64_t u = static_cast<uint64_t>(id);   // negative ids wrap to huge values: never selected
    m = (u >> 3) < static_cast<uint64_t>(d.n_bytes) && ((__ldg(d.bitmap + (u >> 3)) >> (u & 7)) & 1);
  }
  return m != (d.invert != 0);
}

// One warp per bitmap word: lane l decides row 32 w + l.  n_words covers the shard rounded up to whole QS tiles, so
// the scoring kernels may read the word of any row of a listed tile; rows >= n are never selected.  qs_flag / ts_flag
// must be zero on entry.
__global__ void selector_bits_kernel(SelDesc d, int64_t n, int64_t n_words, const Seg* __restrict__ segs, int nseg,
                                     const int64_t* __restrict__ idmap, uint32_t* __restrict__ bits,
                                     unsigned char* __restrict__ qs_flag, unsigned char* __restrict__ ts_flag,
                                     unsigned long long* __restrict__ count) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  unsigned long long mine = 0;
  for (int64_t w = warp0; w < n_words; w += nwarps) {
    const int64_t row = w * 32 + lane;
    const bool m = row < n && sel_member(d, row_to_id(static_cast<uint32_t>(row), segs, nseg, idmap));
    const uint32_t word = __ballot_sync(0xffffffffu, m);
    if (lane == 0) {
      bits[w] = word;
      if (word) {
        qs_flag[w >> 3] = 1;   // 8 words per QS tile of 256 rows
        ts_flag[w >> 1] = 1;   // 2 words per TS tile of 64 rows
        mine += __popc(word);
      }
    }
  }
  if (lane == 0 && mine) atomicAdd(count, mine);
}

}  // namespace b2f
