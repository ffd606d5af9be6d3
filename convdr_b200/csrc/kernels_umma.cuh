// kernels_umma.cuh — the tensor-core scoring engine (sm_100a): a fused score + select kernel.
//
//   queries  : bf16, loaded ONCE per launch into TMEM (tcgen05.st) — the A operand of every MMA
//   passages : bf16 shadow tiles  HBM --TMA (contiguous 16 KB, 128B swizzle)--> 14-stage smem ring
//   scores   : tcgen05.mma cta_group::2 (A from TMEM, B from smem) --> TMEM accumulator
//   select   : tcgen05.ld --> one (QUERY, half tile) per epilogue thread (8 epilogue warps), threshold in a
//              register, one predicate-chained compare per score; survivors appended to a private area of
//              the candidate list per (query, CTA pair, half tile): no atomics, no shared memory, no
//              cross-thread traffic
//
// TS variant of the tensor engine: the kernel of passes with 209..256 queries (the full passes of large
// batches); smaller passes take the QS variant (kernels_umma_qs.cuh), whose MMA shape follows the batch.
//
// One CTA pair (2 SMs) holds up to 256 queries (128 TMEM lanes per CTA, the MMA M dimension) and
// walks tiles of 64 passage rows (32 per CTA, the MMA N dimension; two accumulator stages of 64
// TMEM columns, so the epilogue of tile i overlaps the MMAs of tile i+1).  Keeping the queries in TMEM
// instead of shared memory leaves the whole 227 KB of smem to the passage ring: ~224 KB in flight
// per SM is what lets a latency-bound HBM stream reach the roofline (with the queries in smem only
// 80 KB fit and the kernel stalled at ~75 % — profiles/r01).  K = 768 is walked in 3 stages of four
// 64-column K-blocks.  The [queries x rows] score tile never leaves the SM.
//
// Replaces the arithmetic of `index.search` (reference drivers/run_convdr_inference.py:182) —
// FAISS's `nq >= 20` branch: blocked sgemm + per-row heap (upstream utils/distances.cpp), and
// FAISS-GPU's cuBLAS GEMM + BlockSelect that materialise score tiles in HBM.
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "kernels_util.cuh"

namespace b2f {

constexpr int kUmmaThreads = 416;                // 4 service warps + 8 epilogue warps (two per TMEM lane quarter) + refresher
constexpr int kUmmaEpiWarps = 8;
constexpr int kUmmaRefresherWarp = 12;           // highest warp id: scheduled ahead of the epilogue warps of its quarter
constexpr int kBlockK = 64;                    // bf16 per K-block = 128 bytes (one swizzle span)
constexpr int kNumKBlocks = kD / kBlockK;      // 12
constexpr int kTileRowsCta = kShadowTileRows;  // passage rows per CTA per tile (32)
constexpr int kTileRows = 2 * kTileRowsCta;    // per CTA pair = MMA N (64)
constexpr int kStageBytes = 16384;             // one TMA box, contiguous in HBM
constexpr int kSubTileBytes = kTileRowsCta * 128;                   // one K-block of a CTA tile
constexpr int kKBlocksPerStage = kStageBytes / kSubTileBytes;       // 4
constexpr int kStagesPerTile = kNumKBlocks / kKBlocksPerStage;      // 3
constexpr int kNumStages = 14;
constexpr int kUmmaMaxQ = 256;                 // queries per pass = MMA M (both CTAs)
constexpr int kTmemCols = 512;
constexpr int kTmemColsA = kD / 2;             // 384 columns: 128 lanes x 768 bf16
constexpr int kTmemColD = kTmemColsA;          // accumulators: columns [384, 512)
constexpr int kAccStages = (kTmemCols - kTmemColsA) / kTileRows;    // 2 (double-buffered)
constexpr int kUmmaTailBytes = 2048;           // barriers, tmem pointer
constexpr int kHistBuckets = 512;              // tightening histogram: 16 buckets per refresher lane
constexpr int kHistCoarse = kHistBuckets / 16; // + one coarse counter per lane (sum of its 16 buckets)
constexpr int kHistStride = kHistBuckets + kHistCoarse;   // uints per query: [512 fine][32 coarse]
constexpr int kUmmaSmemBytes = kNumStages * kStageBytes + kUmmaTailBytes + 1024;  // + alignment slack
static_assert(kUmmaSmemBytes <= 232448, "exceeds the 227 KB opt-in shared memory of sm_100");
static_assert(kAccStages >= 1 && kAccStages <= 2, "TMEM budget: 384 query columns + accumulators in 128 columns");
static_assert(kTileRows % 32 == 0 && kNumKBlocks % kKBlocksPerStage == 0, "tile shape");

struct UmmaArgs {
  int64_t n_rows;             // valid rows of the shard
  int tile_begin, tile_end;   // pair tiles of 128 rows
  int nq;                     // valid queries of the pass (<= 256)
  const __nv_bfloat16* q16;   // pass queries, row-major [>= nq, 768] bf16
  int dense;                  // 1: store every score (bootstrap phase), 0: threshold filter
  // Candidate list of query q: cand[q*C .. q*C+C).  [0, S) holds the survivors of earlier phases
  // (written by refresh_kernel); the rest is split in `max_pairs` private areas of `cap_p` slots,
  // TWO per CTA pair (one per half of a tile's 64 rows), so the thread that owns (query, pair, half)
  // appends without any atomic.
  uint64_t* cand;
  int C, S, cap_p, max_pairs; // max_pairs = number of areas = 2 x CTA pairs of the largest grid
  int* cnt2;                  // [nq][max_pairs] entries written to each area in this launch
  float* tau;                 // [nq] thresholds (raised in-kernel when tighten != 0)
  int* ovf;                   // [nq] set when a private area was too small
  int* err;                   // device error flag (barrier timeout)
  // In-kernel threshold tightening (see the refresher role below).  Every hit is also counted in a
  // per-query histogram over the score-key range above the bootstrap's k-th score:
  //   bucket(key) = min(kHistBuckets-1, (key - hkey0[q]) >> hshift[q])   for key >= hkey0[q]
  // so "k rows seen so far score at least edge(b)" is one suffix sum away.  Two ways to place the
  // buckets (host option "bootstrap"):
  //   0 (default): no bootstrap at all.  hkey0 = ((fkey(R) >> 17) - 511) << 17, hshift = 17 with
  //      R >= any |score| of the query (Cauchy-Schwarz): 64 buckets per binade (1.6 % of the score)
  //      over the eight binades below R.  tau starts at -inf, the first tile of every pair passes
  //      entirely, and the thresholds rise from there — ONE launch streams the whole shard.
  //   1: a dense bootstrap launch + bootstrap_select_kernel place 512 linear buckets above the k-th
  //      best score of the first rows.
  int tighten;                // >0: the idle warp of each CTA keeps raising tau[q] while the stream runs;
                              //     the value is the minimum pause between its rounds in ns
  int tighten_adaptive;       // 1: the pause grows with the time since the kernel started (elapsed / 4, capped at
                              //     50 us): the pass rate falls like k / rows_seen, so a threshold of bounded
                              //     relative age costs a bounded fraction of extra hits whatever the moment,
                              //     and a launch needs ~50 polling rounds instead of thousands
  int k;
  int count_exact_lower_bound; // 1 (one-launch schedule): hits are counted at s~ - eps, a lower bound of the EXACT score,
                              //   so "k hits at or above edge e" bounds the k-th exact score itself and tau = e - eps;
                              // 0 (phased schedules, whose histogram is seeded with raw approximate keys): count at
                              //   s~, tau = e - 2 eps
  int first_wait_cycles;      // one-launch schedule: after its first tile an epilogue thread waits this long at most
                              // for its query's first threshold (0: no wait)
  const float* margin;        // [nq] 2*eps of the prefilter
  unsigned int* hist;         // [nq][kHistStride], initialised by pass_init_kernel / bootstrap_select_kernel
  const uint32_t* hkey0;      // [nq] key of the bootstrap's k-th best approximate score (0xffffffff: none yet)
  const int* hshift;          // [nq] log2(keys per bucket)
  const float* qscale;        // int8 shadow: [nq] query scales sq (q16 then points at the int8 codes)
  const float4* tscale;       // int8 shadow: [row tiles of 32] tile scales {st, RD(1/st), RU(1/st), 0}
  // Filtered search (SEL instances only): the launch walks tile_list[tile_begin .. tile_end) (pair tiles that hold
  // at least one selected row) instead of the tiles themselves; sel_bits is the shard's row bitmap (bit r & 31 of
  // word r >> 5: row r is selected).
  const uint32_t* sel_bits;
  const int* tile_list;
};

// Tile of iteration i: the listed tile of a filtered launch, i itself otherwise.  Every role that walks tiles calls
// it with the same i, so they stay in lockstep.
template <bool SEL>
__device__ __forceinline__ int tile_at(const int* tile_list, int i) {
  if constexpr (SEL) return __ldg(tile_list + i);
  else return i;
}

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Remote arrive on a barrier of the peer CTA.  Deliberately the plain form (default .release.cta):
// `.release.cluster` compiles to MEMBAR.ALL.GPU + ERRBAR, which cost ~1300 cycles per TMA stage
// when the peer's producer executed it (profiles/r01: the whole pipeline ran at that pace).  The
// data these barriers guard travels through the async proxy (TMA complete_tx) or is ordered by
// tcgen05.fence::before_thread_sync, not by this arrive.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// Bounded wait: a protocol bug must end in a trap (reported as a CUDA error), never in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if ((spin & 1023u) == 1023u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 6000000000ll) {  // ~3 s at 2 GHz
        if (err) atomicExch(err, 1);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* tmap,
                                                uint32_t leader_bar_cluster, int c0, int c1,
                                                uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar_cluster), "r"(c0), "r"(c1),
        "l"(hint)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once) on the barrier at this smem offset in BOTH CTAs of the pair when all previously
// issued MMAs have completed.
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(static_cast<uint16_t>(3))
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ uint32_t tmem_ld_x1(uint32_t taddr) {
  uint32_t v;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr));
  return v;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand descriptor (PTX ISA "tcgen05 shared memory descriptor"):
// start address >> 4 in bits [0,14); stride-dimension byte offset (8 rows * 128 B = 1024) >> 4 in
// bits [32,46); descriptor version 1 in bits [46,48); swizzle mode 2 (128B) in bits [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu) | (static_cast<uint64_t>(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
// Instruction descriptor, kind::f16: D = fp32 (bits [4,6) = 1), A = B = bf16 (bits [7,10), [10,13)
// = 1), both K-major (bits 15, 16 = 0), N >> 3 in bits [17,23), M >> 4 in bits [24,29).
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// kind::i8: D = s32 (bits [4,6) = 2), A = B = signed 8-bit (bits [7,10), [10,13) = 1); the rest as for bf16.
__host__ __device__ __forceinline__ uint32_t umma_idesc_i8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void umma_i8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

constexpr uint64_t kHintEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kHintEvictLast = 0x14F0000000000000ull;

// D[tmem] (+)= A[tmem] * B[smem]^T : the queries (A) stay resident in tensor memory.
__device__ __forceinline__ void umma_bf16_2sm_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc,
                                                 uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_i8_2sm_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// "does any of these 32 scores reach the threshold?" as two interleaved predicate chains (setp.ge.or
// accumulates into its predicate): one instruction per score instead of compare + select + or, and the mask
// of WHICH scores hit is only built when some lane of the warp reports a hit.  The epilogue runs with one
// warp per scheduler, so every instruction it saves is exposed latency saved (profiles/r02: the round-1
// epilogue, not the tensor pipe, paced this kernel at full clocks).
__device__ __forceinline__ bool any_ge32(const uint32_t* v, float tau) {
  uint32_t r;
  asm("{\n\t.reg .pred p, q;\n\t"
      "setp.ge.f32 p, %1, %33;\n\t"
      "setp.ge.f32 q, %2, %33;\n\t"
      "setp.ge.or.f32 p, %3, %33, p;\n\t"
      "setp.ge.or.f32 q, %4, %33, q;\n\t"
      "setp.ge.or.f32 p, %5, %33, p;\n\t"
      "setp.ge.or.f32 q, %6, %33, q;\n\t"
      "setp.ge.or.f32 p, %7, %33, p;\n\t"
      "setp.ge.or.f32 q, %8, %33, q;\n\t"
      "setp.ge.or.f32 p, %9, %33, p;\n\t"
      "setp.ge.or.f32 q, %10, %33, q;\n\t"
      "setp.ge.or.f32 p, %11, %33, p;\n\t"
      "setp.ge.or.f32 q, %12, %33, q;\n\t"
      "setp.ge.or.f32 p, %13, %33, p;\n\t"
      "setp.ge.or.f32 q, %14, %33, q;\n\t"
      "setp.ge.or.f32 p, %15, %33, p;\n\t"
      "setp.ge.or.f32 q, %16, %33, q;\n\t"
      "setp.ge.or.f32 p, %17, %33, p;\n\t"
      "setp.ge.or.f32 q, %18, %33, q;\n\t"
      "setp.ge.or.f32 p, %19, %33, p;\n\t"
      "setp.ge.or.f32 q, %20, %33, q;\n\t"
      "setp.ge.or.f32 p, %21, %33, p;\n\t"
      "setp.ge.or.f32 q, %22, %33, q;\n\t"
      "setp.ge.or.f32 p, %23, %33, p;\n\t"
      "setp.ge.or.f32 q, %24, %33, q;\n\t"
      "setp.ge.or.f32 p, %25, %33, p;\n\t"
      "setp.ge.or.f32 q, %26, %33, q;\n\t"
      "setp.ge.or.f32 p, %27, %33, p;\n\t"
      "setp.ge.or.f32 q, %28, %33, q;\n\t"
      "setp.ge.or.f32 p, %29, %33, p;\n\t"
      "setp.ge.or.f32 q, %30, %33, q;\n\t"
      "setp.ge.or.f32 p, %31, %33, p;\n\t"
      "setp.ge.or.f32 q, %32, %33, q;\n\t"
      "or.pred p, p, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r)
      : "f"(__uint_as_float(v[0])), "f"(__uint_as_float(v[1])), "f"(__uint_as_float(v[2])), "f"(__uint_as_float(v[3])), "f"(__uint_as_float(v[4])), "f"(__uint_as_float(v[5])), "f"(__uint_as_float(v[6])), "f"(__uint_as_float(v[7])), "f"(__uint_as_float(v[8])), "f"(__uint_as_float(v[9])), "f"(__uint_as_float(v[10])), "f"(__uint_as_float(v[11])), "f"(__uint_as_float(v[12])), "f"(__uint_as_float(v[13])), "f"(__uint_as_float(v[14])), "f"(__uint_as_float(v[15])), "f"(__uint_as_float(v[16])), "f"(__uint_as_float(v[17])), "f"(__uint_as_float(v[18])), "f"(__uint_as_float(v[19])), "f"(__uint_as_float(v[20])), "f"(__uint_as_float(v[21])), "f"(__uint_as_float(v[22])), "f"(__uint_as_float(v[23])), "f"(__uint_as_float(v[24])), "f"(__uint_as_float(v[25])), "f"(__uint_as_float(v[26])), "f"(__uint_as_float(v[27])), "f"(__uint_as_float(v[28])), "f"(__uint_as_float(v[29])), "f"(__uint_as_float(v[30])), "f"(__uint_as_float(v[31])), "f"(tau));
  return r != 0u;
}

// The same chains on int32 accumulators against an integer threshold (int8 shadow, i8_threshold).
__device__ __forceinline__ bool any_ge32_s32(const uint32_t* v, int tau) {
  uint32_t r;
  asm("{\n\t.reg .pred p, q;\n\t"
      "setp.ge.s32 p, %1, %33;\n\t"
      "setp.ge.s32 q, %2, %33;\n\t"
      "setp.ge.or.s32 p, %3, %33, p;\n\t"
      "setp.ge.or.s32 q, %4, %33, q;\n\t"
      "setp.ge.or.s32 p, %5, %33, p;\n\t"
      "setp.ge.or.s32 q, %6, %33, q;\n\t"
      "setp.ge.or.s32 p, %7, %33, p;\n\t"
      "setp.ge.or.s32 q, %8, %33, q;\n\t"
      "setp.ge.or.s32 p, %9, %33, p;\n\t"
      "setp.ge.or.s32 q, %10, %33, q;\n\t"
      "setp.ge.or.s32 p, %11, %33, p;\n\t"
      "setp.ge.or.s32 q, %12, %33, q;\n\t"
      "setp.ge.or.s32 p, %13, %33, p;\n\t"
      "setp.ge.or.s32 q, %14, %33, q;\n\t"
      "setp.ge.or.s32 p, %15, %33, p;\n\t"
      "setp.ge.or.s32 q, %16, %33, q;\n\t"
      "setp.ge.or.s32 p, %17, %33, p;\n\t"
      "setp.ge.or.s32 q, %18, %33, q;\n\t"
      "setp.ge.or.s32 p, %19, %33, p;\n\t"
      "setp.ge.or.s32 q, %20, %33, q;\n\t"
      "setp.ge.or.s32 p, %21, %33, p;\n\t"
      "setp.ge.or.s32 q, %22, %33, q;\n\t"
      "setp.ge.or.s32 p, %23, %33, p;\n\t"
      "setp.ge.or.s32 q, %24, %33, q;\n\t"
      "setp.ge.or.s32 p, %25, %33, p;\n\t"
      "setp.ge.or.s32 q, %26, %33, q;\n\t"
      "setp.ge.or.s32 p, %27, %33, p;\n\t"
      "setp.ge.or.s32 q, %28, %33, q;\n\t"
      "setp.ge.or.s32 p, %29, %33, p;\n\t"
      "setp.ge.or.s32 q, %30, %33, q;\n\t"
      "setp.ge.or.s32 p, %31, %33, p;\n\t"
      "setp.ge.or.s32 q, %32, %33, q;\n\t"
      "or.pred p, p, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r)
      : "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]), "r"(tau));
  return r != 0u;
}

// ------------------------------------------------------------------------------------------
// The kernel.  Grid = 2 * (number of CTA pairs), cluster (2,1,1), 384 threads:
//   warp 0 lane 0 : TMA producer (both CTAs stream their own 32 rows of every tile)
//   warp 1 lane 0 : MMA issuer (leader CTA only)
//   warp 2        : TMEM allocation / release
//   warp 3        : idle
//   warps 4..11   : load the queries into TMEM, then epilogue — thread (rank, lane) of warp w owns query
//                   128*rank + 32*(w%4) + lane and, of every 64-row tile, the 32 rows of half (w-4)/4: two
//                   threads per query, each with its own private list area (hit handling is per-thread
//                   instruction overhead in a warp that the scheduler cannot hide: two warps per TMEM lane
//                   quarter halve it and overlap each other's latencies)
//   warp 12       : refresher (in-kernel threshold tightening)
// I8: int8 shadow and queries (kind::i8, s32 accumulators).  A 32-row tile is 6 K-blocks of 128 bytes, walked in 2
// stages of 3 K-blocks (12 KB boxes, 18 of them in the ring); the queries take 192 TMEM columns (4 codes per
// column, so a K-step of 32 codes is still 8 columns).  Each epilogue thread's 32 rows are one shadow tile: its
// float threshold becomes ONE integer threshold per tile (i8_threshold: one product of the thread's tau / sq and
// the tile's reciprocal scale), the compare chain stays one instruction
// per score, and the float score is only formed for a hit.
// SEL: filtered search.  The roles walk the listed tiles only; the epilogue ANDs the row bitmap word of its 32 rows
// into the hit mask (and stores empty records for unselected rows in the dense phase), so only selected rows are
// ever appended or counted in the tightening histogram.
// ------------------------------------------------------------------------------------------
template <bool I8, bool SEL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kUmmaThreads, 1)
    umma_score_select_kernel(const __grid_constant__ CUtensorMap tmap_p, const UmmaArgs a) {
  constexpr int NKB = I8 ? kShadow8KBlocks : kNumKBlocks;        // K-blocks of 128 bytes per row
  constexpr int KBPS = I8 ? 3 : kKBlocksPerStage;                // K-blocks per ring stage
  constexpr int STAGE_BYTES = KBPS * kSubTileBytes;
  constexpr int STAGES_PER_TILE = NKB / KBPS;
  constexpr int NST = I8 ? 18 : kNumStages;
  constexpr int COLS_A = I8 ? kD / 4 : kTmemColsA;                // query columns in TMEM
  static_assert(NST * STAGE_BYTES <= kNumStages * kStageBytes, "ring fits the bf16 layout's shared memory");
  extern __shared__ unsigned char umma_smem_raw[];
  const uint32_t raw = smem_u32(umma_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // 1024-byte alignment for the 128B swizzle atoms
  unsigned char* base_ptr = umma_smem_raw + (base - raw);
  const uint32_t smem_b = base;                                   // [NST][STAGE_BYTES]
  const uint32_t tail = smem_b + NST * STAGE_BYTES;
  const uint32_t bar_full = tail;                                 // [NST]
  const uint32_t bar_empty = tail + 8 * NST;                      // [NST]
  const uint32_t bar_qready = tail + 16 * NST;
  const uint32_t bar_tfull = bar_qready + 8;                      // [2]
  const uint32_t bar_tempty = bar_tfull + 16;                     // [2]
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(base_ptr + NST * STAGE_BYTES + 16 * NST + 40);
  volatile int* epi_done_s = reinterpret_cast<volatile int*>(tmem_ptr_s + 1);     // epilogue warps that finished

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) prefetch_tmap(&tmap_p);
  if (warp == 3 && lane == 0) *epi_done_s = 0;
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(bar_full + 8 * s, 2);   // leader's expect_tx arrive + peer's remote arrive
      mbar_init(bar_empty + 8 * s, 1);  // one multicast commit
    }
    mbar_init(bar_qready, 2 * kUmmaEpiWarps);           // query-loading warps x 2 CTAs
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_tfull + 8 * s, 1);   // one multicast commit
      mbar_init(bar_tempty + 8 * s, 2 * kUmmaEpiWarps);  // epilogue warps x 2 CTAs (leader's copy is the one used)
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_ptr_s)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_s);

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    uint32_t stage = 0, phase = 0;
    for (int ti = a.tile_begin + pair; ti < a.tile_end; ti += npairs) {
      const int tile = tile_at<SEL>(a.tile_list, ti);
      // shadow layout (common.cuh): CTA tile = 2*tile + rank; kKBlocksPerStage consecutive K-blocks
      // of it are 128 consecutive 128-byte rows = one contiguous 16 KB box
      const int row0 = (tile * 2 + static_cast<int>(cta_rank)) * NKB * kTileRowsCta;
      for (int st = 0; st < STAGES_PER_TILE; ++st) {
        mbar_wait(bar_empty + 8 * stage, phase ^ 1u, a.err);
        const uint32_t full_leader = mapa_u32(bar_full + 8 * stage, 0);
        if (leader) mbar_arrive_expect_tx(bar_full + 8 * stage, 2u * STAGE_BYTES);
        else mbar_arrive_cluster(full_leader);
        tma_load_2d_2sm(smem_b + stage * STAGE_BYTES, &tmap_p, full_leader, 0,
                        row0 + st * (KBPS * kTileRowsCta), kHintEvictFirst);
        if (++stage == NST) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1 && leader) {
    // ===================== MMA issuer (leader CTA; the whole warp waits, one elected lane issues) =====
    const uint32_t idesc = I8 ? umma_idesc_i8(256, kTileRows) : umma_idesc_bf16(256, kTileRows);
    const bool elected = elect_one();
    mbar_wait(bar_qready, 0, a.err);   // both CTAs have their queries in TMEM
    tc_fence_after();
    uint32_t stage = 0, phase = 0;
    int it = 0;
    for (int tile = a.tile_begin + pair; tile < a.tile_end; tile += npairs, ++it) {
      const uint32_t as = static_cast<uint32_t>(it) % kAccStages, aph = (static_cast<uint32_t>(it) / kAccStages) & 1u;
      mbar_wait(bar_tempty + 8 * as, aph ^ 1u, a.err);   // epilogue has drained this accumulator stage
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + kTmemColD + as * kTileRows;
      for (int st = 0; st < STAGES_PER_TILE; ++st) {
        mbar_wait(bar_full + 8 * stage, phase, a.err);
        tc_fence_after();
        if (elected) {
#pragma unroll
          for (int j = 0; j < KBPS; ++j) {
            const uint64_t bdesc = umma_desc_sw128(smem_b + stage * STAGE_BYTES + j * kSubTileBytes);
#pragma unroll
            for (int k = 0; k < 4; ++k) {   // UMMA K = 16 bf16 / 32 int8: 8 TMEM columns of A, 32 bytes of B
              const int kstep = (st * KBPS + j) * 4 + k;
              if (I8) umma_i8_2sm_ts(tmem_d, tmem_base + 8 * kstep, bdesc + 2 * k, idesc, kstep != 0);
              else umma_bf16_2sm_ts(tmem_d, tmem_base + 8 * kstep, bdesc + 2 * k, idesc, kstep != 0);
            }
          }
          umma_commit_pair(bar_empty + 8 * stage);                             // frees this smem stage in both CTAs
          if (st == STAGES_PER_TILE - 1) umma_commit_pair(bar_tfull + 8 * as); // accumulator ready
        }
        __syncwarp();
        if (++stage == NST) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp >= 4 && warp < 4 + kUmmaEpiWarps) {
    // ===================== queries -> TMEM, then epilogue =====================
    const int ew = warp & 3;
    const int half = (warp - 4) >> 2;      // which 32 rows of every 64-row tile / which half of the query columns to load
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16);
    const int q = static_cast<int>(cta_rank) * 128 + ew * 32 + lane;
    const bool q_ok = q < a.nq;
    {
      const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(a.q16) +
                                                        static_cast<int64_t>(q_ok ? q : 0) * kD * (I8 ? 1 : 2));
      // three 128-byte chunks (3 x 8 independent 16-byte loads) in flight per round: 4 L2 round trips
      // for the whole 1536-byte query row instead of 12
      constexpr int kQChunk = 3;
      static_assert((COLS_A / 32) % kQChunk == 0, "query row = whole rounds");
#pragma unroll 1
      static_assert((COLS_A / 64) % kQChunk == 0, "each of the two warps of a quarter loads whole rounds");
      for (int c0 = half * (COLS_A / 64); c0 < (half + 1) * (COLS_A / 64); c0 += kQChunk) {   // 32 columns = 128 bytes per chunk
        uint32_t w[kQChunk][32];
#pragma unroll
        for (int u = 0; u < kQChunk; ++u)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint4 t = q_ok ? __ldg(src + (c0 + u) * 8 + i) : make_uint4(0u, 0u, 0u, 0u);
            w[u][4 * i] = t.x; w[u][4 * i + 1] = t.y; w[u][4 * i + 2] = t.z; w[u][4 * i + 3] = t.w;
          }
#pragma unroll
        for (int u = 0; u < kQChunk; ++u) tmem_st_x32(lane_addr + 32 * (c0 + u), w[u]);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(bar_qready, 0));
    }
    float tau = (q_ok && !a.dense) ? a.tau[q] : INFINITY;
    volatile float* tau_g = a.tau + (q_ok ? q : 0);
    const int area = 2 * pair + half;
    int* my_cnt = a.cnt2 + (q_ok ? q : 0) * a.max_pairs + area;
    const bool live = a.tighten && q_ok && !a.dense;
    const uint32_t hkey0 = live ? a.hkey0[q] : 0xffffffffu;
    const int hshift = live ? a.hshift[q] : 0;
    unsigned int* my_hist = a.hist + static_cast<int64_t>(q_ok ? q : 0) * kHistStride;
    uint64_t* my_list = a.cand + static_cast<int64_t>(q_ok ? q : 0) * a.C + a.S + static_cast<int64_t>(area) * a.cap_p;
    int n_mine = 0;   // entries this thread appended for (query q, this pair)
    // count a hit in the tightening histogram (fire-and-forget RED; hits are rare)
    const float eps_cnt = (live && a.count_exact_lower_bound) ? __fmul_ru(a.margin[q], 0.5f) : 0.f;
    auto count_hit = [&](uint32_t bits) {
      const uint32_t key = fkey(__fsub_rd(__uint_as_float(bits), eps_cnt));
      if (key >= hkey0) {
        const uint32_t b = min(static_cast<uint32_t>(kHistBuckets - 1), (key - hkey0) >> hshift);
        atomicAdd(my_hist + b, 1u);
        atomicAdd(my_hist + kHistBuckets + (b >> 4), 1u);
      }
    };
    const uint32_t tempty_leader = mapa_u32(bar_tempty, 0);
    const float sq = I8 ? a.qscale[q_ok ? q : 0] : 0.f;
    float u = I8 ? i8_tau_over_sq(tau, sq) : 0.f;   // query factor of the integer threshold, redone when tau rises
    int it = 0;
    for (int ti = a.tile_begin + pair; ti < a.tile_end; ti += npairs, ++it) {
      const int tile = tile_at<SEL>(a.tile_list, ti);
      const uint32_t as = static_cast<uint32_t>(it) % kAccStages, aph = (static_cast<uint32_t>(it) / kAccStages) & 1u;
      if (it == 1 && live && a.first_wait_cycles > 0) {
        // The first tile of every pair passed unfiltered (thresholds start at -inf): together those rows place
        // every query's first threshold.  Waiting for it here (bounded) instead of streaming on keeps the
        // private areas from filling with rows the final selection would throw away — at full clocks a pair
        // finishes a tile every ~0.8 us, the first threshold takes a few us to travel.
        const long long t0 = clock64();
        while (*tau_g == -INFINITY && clock64() - t0 < a.first_wait_cycles) __nanosleep(256);
      }
      float tau_new = tau;
      if (live) tau_new = *tau_g;            // issued before the wait: the L2 latency hides behind it
      mbar_wait(bar_tfull + 8 * as, aph, a.err);
      tc_fence_after();
      if (I8 && tau_new > tau) u = i8_tau_over_sq(tau_new, sq);
      tau = fmaxf(tau, tau_new);             // thresholds only rise
      constexpr int kHalfRows = kTileRows / 2;   // 32: this thread's rows of the tile
      uint32_t v[kHalfRows];
      const uint32_t col0 = lane_addr + kTmemColD + as * kTileRows + kHalfRows * half;
      tmem_ld_x32(col0, v);
      tmem_ld_wait();
      const int64_t row0 = static_cast<int64_t>(tile) * kTileRows + kHalfRows * half;
      const int n_valid = static_cast<int>(max(static_cast<int64_t>(0), min(static_cast<int64_t>(kHalfRows), a.n_rows - row0)));
      uint32_t sel_word = 0xffffffffu;       // this thread's 32 rows are one bitmap word
      if constexpr (SEL) sel_word = __ldg(a.sel_bits + (row0 >> 5));
      if constexpr (I8) {
        // one integer threshold for this (query, shadow tile); scores as floats only where they are stored
        const float4 ts = n_valid > 0 ? __ldg(a.tscale + (row0 >> 5)) : make_float4(0.f, INFINITY, INFINITY, 0.f);
        const float st = ts.x;
        if (a.dense) {
          if (q_ok && n_mine + kHalfRows <= a.cap_p) {
            uint64_t* dst = my_list + n_mine;
#pragma unroll
            for (int c = 0; c < kHalfRows; c += 2) {
              ulonglong2 o;
              o.x = (c < n_valid && ((sel_word >> c) & 1u)) ? pack_cand(i8_score(static_cast<int>(v[c]), sq, st), static_cast<uint32_t>(row0 + c)) : 0ull;
              o.y = (c + 1 < n_valid && ((sel_word >> (c + 1)) & 1u)) ? pack_cand(i8_score(static_cast<int>(v[c + 1]), sq, st), static_cast<uint32_t>(row0 + c + 1)) : 0ull;
              *reinterpret_cast<ulonglong2*>(dst + c) = o;
            }
          }
          n_mine += kHalfRows;
        } else {
          const int T = i8_threshold(u, ts);
          if (__any_sync(0xffffffffu, any_ge32_s32(v, T))) {
            uint32_t m = 0;
#pragma unroll
            for (int c = 0; c < kHalfRows; ++c) m |= (static_cast<int>(v[c]) >= T) ? (1u << c) : 0u;
            if (n_valid < kHalfRows) m &= (n_valid > 0) ? ((1u << n_valid) - 1u) : 0u;   // shard tail
            if constexpr (SEL) m &= sel_word;
            uint32_t any = __reduce_or_sync(0xffffffffu, m);
            if (__popc(any) > 6) {   // busy word: unrolled predicated stores, v[] stays in registers
              if (m) {
#pragma unroll
                for (int c = 0; c < kHalfRows; ++c) {
                  if ((m >> c) & 1u) {
                    const uint32_t bits = __float_as_uint(i8_score(static_cast<int>(v[c]), sq, st));
                    const int slot = n_mine + __popc(m & ((1u << c) - 1u));
                    if (slot < a.cap_p) my_list[slot] = pack_cand(__uint_as_float(bits), static_cast<uint32_t>(row0 + c));
                    count_hit(bits);
                  }
                }
                n_mine += __popc(m);
              }
              any = 0;
            }
            while (any) {
              const int c = __ffs(any) - 1;
              any &= any - 1;
              const uint32_t acc = tmem_ld_x1(col0 + c);
              tmem_ld_wait();
              if ((m >> c) & 1u) {
                const uint32_t bits = __float_as_uint(i8_score(static_cast<int>(acc), sq, st));
                if (n_mine < a.cap_p) my_list[n_mine] = pack_cand(__uint_as_float(bits), static_cast<uint32_t>(row0 + c));
                ++n_mine;
                count_hit(bits);
              }
            }
          }
        }
      } else if (a.dense) {
        // bootstrap: every score of this half tile goes to the private area (zeros for rows past the end)
        if (q_ok && n_mine + kHalfRows <= a.cap_p) {
          uint64_t* dst = my_list + n_mine;
#pragma unroll
          for (int c = 0; c < kHalfRows; c += 2) {
            ulonglong2 o;
            o.x = (c < n_valid && ((sel_word >> c) & 1u)) ? pack_cand(__uint_as_float(v[c]), static_cast<uint32_t>(row0 + c)) : 0ull;
            o.y = (c + 1 < n_valid && ((sel_word >> (c + 1)) & 1u)) ? pack_cand(__uint_as_float(v[c + 1]), static_cast<uint32_t>(row0 + c + 1)) : 0ull;
            *reinterpret_cast<ulonglong2*>(dst + c) = o;
          }
        }
        n_mine += kHalfRows;
      } else if (__any_sync(0xffffffffu, any_ge32(v, tau))) {     // the common case is: no lane hits
        // One predicate bit per score; hits are handled in a warp-uniform loop over the columns any lane
        // flagged, re-reading that single column from TMEM (a dynamic register index would demote v[] to
        // local memory) — or, for a busy word (loose thresholds early in a pass), by unrolled predicated stores.
        uint32_t m = 0;
#pragma unroll
        for (int c = 0; c < kHalfRows; ++c) m |= (__uint_as_float(v[c]) >= tau) ? (1u << c) : 0u;
        if (n_valid < kHalfRows) m &= (n_valid > 0) ? ((1u << n_valid) - 1u) : 0u;   // shard tail
        if constexpr (SEL) m &= sel_word;
        uint32_t any = __reduce_or_sync(0xffffffffu, m);
        if (__popc(any) > 6) {
          if (m) {
#pragma unroll
            for (int c = 0; c < kHalfRows; ++c) {
              if ((m >> c) & 1u) {
                const int slot = n_mine + __popc(m & ((1u << c) - 1u));
                if (slot < a.cap_p) my_list[slot] = pack_cand(__uint_as_float(v[c]), static_cast<uint32_t>(row0 + c));
                count_hit(v[c]);
              }
            }
            n_mine += __popc(m);
          }
        } else {
          while (any) {
            const int c = __ffs(any) - 1;
            any &= any - 1;
            const uint32_t bits = tmem_ld_x1(col0 + c);
            tmem_ld_wait();
            if ((m >> c) & 1u) {   // no atomics: the area is private to this thread
              if (n_mine < a.cap_p) my_list[n_mine] = pack_cand(__uint_as_float(bits), static_cast<uint32_t>(row0 + c));
              ++n_mine;
              count_hit(bits);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader + 8 * as);   // this accumulator stage is free again
    }
    if (q_ok) {
      *my_cnt = min(n_mine, a.cap_p);
      if (n_mine > a.cap_p) a.ovf[q] = 1;
    }
    __syncwarp();
    if (lane == 0) atomicAdd(const_cast<int*>(epi_done_s), 1);
  } else if (warp == kUmmaRefresherWarp && a.tighten && !a.dense) {
    // ===================== refresher: in-kernel threshold tightening =====================
    // While the stream runs, this otherwise idle warp keeps reading, for the queries assigned to
    // this CTA (q = blockIdx.x, + gridDim.x, ...), the histogram of hits above the bootstrap's k-th
    // score and raises tau[q] to (lower edge of the highest bucket b with >= k hits in buckets >= b)
    // - 2*eps.  At least k rows seen so far have an approximate score >= that edge, so the k-th best
    // approximate score of any superset is >= it: the bound of DESIGN.md section 4 holds for every
    // intermediate value, whatever the interleaving (counts only grow; a stale read is a smaller
    // suffix sum, i.e. a lower, still valid, threshold).  Every hit with key >= hkey0 is counted by
    // every pair because all thresholds in use are <= the current one.  Effect: the pass rate
    // follows k/rows_seen continuously, so ONE launch streams the whole shard after the bootstrap.
    float last[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    const long long t_start = clock64();
    while (*epi_done_s < kUmmaEpiWarps) {
      int qi = 0;
      for (int q = blockIdx.x; q < a.nq; q += gridDim.x, ++qi) {
        const uint32_t key0 = a.hkey0[q];
        if (key0 == 0xffffffffu) continue;     // fewer than k rows seen by the bootstrap: nothing to reject
        // lane l owns buckets [16l, 16l+16).  One 128-byte read of the 32 coarse counters per round; only
        // the lane where the suffix sum crosses k reads its 16 fine buckets (192 B per query and round
        // instead of 2 KB: the polling shares the L2 -> SM path with the 6 TB/s passage stream).
        const unsigned int* hq = a.hist + static_cast<int64_t>(q) * kHistStride;
        const unsigned int mine = __ldcv(hq + kHistBuckets + lane);
        unsigned int suf = mine;               // hits in the buckets of lanes >= this one
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned int t = __shfl_down_sync(0xffffffffu, suf, o);
          if (lane + o < 32) suf += t;
        }
        const unsigned int kk = static_cast<unsigned int>(a.k);
        unsigned int above = suf - mine;
        int b = -1;
        if (suf >= kk && above < kk) {         // exactly one lane: walk its 16 fine buckets from the top
          const uint4* hp = reinterpret_cast<const uint4*>(hq) + 4 * lane;
#pragma unroll
          for (int u = 3; u >= 0; --u) {
            const uint4 h4 = __ldcv(hp + u);
            const unsigned int c4[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
            for (int j = 3; j >= 0; --j) {
              if (b < 0) {
                above += c4[j];
                if (above >= kk) b = 16 * lane + 4 * u + j;
              }
            }
          }
        }
        const unsigned int who = __ballot_sync(0xffffffffu, b >= 0);
        if (who == 0u) continue;
        b = __shfl_sync(0xffffffffu, b, __ffs(who) - 1);
        if (lane == 0) {
          const uint64_t edge = static_cast<uint64_t>(key0) + (static_cast<uint64_t>(b) << a.hshift[q]);
          if (edge <= 0xff7fffffull) {         // a finite score key
            const float t = __fsub_rd(key2f(static_cast<uint32_t>(edge)),
                                      a.count_exact_lower_bound ? __fmul_ru(a.margin[q], 0.5f) : a.margin[q]);
            const float prev = (qi < 4) ? last[qi] : *reinterpret_cast<volatile float*>(a.tau + q);
            if (t > prev) {
              *reinterpret_cast<volatile float*>(a.tau + q) = t;
              if (qi < 4) last[qi] = t;
            }
          }
        }
      }
      unsigned int pause = static_cast<unsigned int>(a.tighten);
      const long long age_ns = (clock64() - t_start) >> 1;       // cycles -> ns at ~2 GHz; only a pacing hint
      if (age_ns < 30000) pause = min(pause, 500u);              // start of the pass: epilogue threads wait for the first thresholds
      else if (a.tighten_adaptive) {
        pause = static_cast<unsigned int>(min(max(static_cast<long long>(pause), age_ns >> 2), 50000ll));
      }
      __nanosleep(pause);
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

}  // namespace b2f
