// kernels_umma_qs.cuh — tensor-core scoring engine, QS variant: the queries on the MMA N side (sm_100a).
//
//   passages : bf16 shadow tiles  HBM --TMA (128B swizzle)--> shared-memory ring of 16 KB stages   : A operand
//   queries  : bf16, N = batch rounded up to 16 (176 for 173 queries: no padded lanes); the first R
//              K-blocks (default: all 12) stay resident in shared memory, the others are re-read from L2
//              for every passage tile through their own shallow ring                               : B operand
//   scores   : tcgen05.mma cta_group::2, M = 256 passage rows per CTA pair, fp32 accumulators in TMEM (x2)
//   select   : tcgen05.ld --> one PASSAGE ROW per epilogue thread, 8 epilogue warps; per-query thresholds in
//              shared memory, ONE predicate-chained compare per score; hits appended to a (query, CTA)-private
//              list area (shared-memory counters, no global atomics) and counted in the tightening histogram;
//              a dedicated warp keeps raising the thresholds while the stream runs (ONE launch per pass)
//
// Why this variant exists (VERDICT r1 weak #2): with the queries as the A operand in TMEM
// (kernels_umma.cuh) every MMA issues M = 256 query lanes, so 173 queries pay for 256 and the kernel is
// tensor-bound at 0.75-0.80 of HBM once the board's power cap pulls the SM clock to ~1.1-1.3 GHz.  With
// the queries on the N side the MMA shape follows the batch (N = 176: 31 % fewer tensor cycles and joules),
// but the B operand must live in shared memory: 135 KB per CTA for 173 queries, which leaves a 5-stage
// passage ring (80 KB in flight per SM).  Streaming the query K-blocks from L2 instead (R < 12) buys a ring of
// up to 11 stages at the price of 11 KB of L2->SM traffic per 16 KB passage stage; measured (DESIGN.md
// section 3) every split lands within 2 % at 173 queries and the fully resident layout wins in sustained,
// power-capped runs, so R = 12 is the default and the streamed path serves batches too large to stay
// resident.  What made this orientation pay at all was the epilogue: see any_ge16 below.
//
// Replaces the arithmetic of `index.search` (reference drivers/run_convdr_inference.py:182).
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "kernels_umma.cuh"

namespace b2f {

constexpr int kQsTileRowsCta = 128;
constexpr int kQsTileRows = 256;                 // per CTA pair = MMA M
constexpr int kQsStageBytes = kQsTileRowsCta * kBlockK * 2;  // 16 KB: 128 rows of one K-block
constexpr int kQsMaxAStages = 12;
constexpr int kQsMaxQStages = 4;
constexpr int kQsMaxCols = 256;                  // MMA N limit; two accumulators of 256 TMEM columns
constexpr int kQsAccStride = 256;
constexpr int kQsTailBytes = 4096;               // barriers, thresholds, counters, histogram bases
constexpr int kQsSmemLimit = 232448;
constexpr int kQsThreads = 416;                  // 4 service warps + 8 epilogue warps (two per TMEM lane quarter) + refresher
constexpr int kQsEpiWarps = 8;
constexpr int kQsEpiWarpsI8Scratch = 8 * 128 * 4;   // [8 epilogue warps][<= 128 query columns] int thresholds
constexpr int kQsTailBytesI8 = kQsTailBytes + kQsEpiWarpsI8Scratch + kQsMaxCols * 4;   // int8: tail + that scratch + u_s
constexpr int kQsRefresherWarp = 12;             // the highest warp id: the scheduler prefers it over the epilogue
                                                 // warps of its quarter, so thresholds never wait behind appends

struct UmmaQsArgs {
  int64_t n_rows;             // valid rows of the shard
  int tile_begin, tile_end;   // pair tiles of 256 rows
  int n_cols;                 // MMA N: padded query count, multiple of 16, 16..256
  int nq;                     // valid queries (<= n_cols)
  int a_stages, q_stages;     // ring depths
  int resident_kb;            // K-blocks [0, resident_kb) of the queries stay in shared memory
  const __nv_bfloat16* q16;   // unused by the kernel (the tensor map carries it); kept for debugging
  // Candidate list of query q: cand[q*C .. q*C+C): [0,S) unused by this variant, then one private area
  // of cap_p slots per CTA (n_areas of them), so appends need no global atomic.
  uint64_t* cand;
  int C, S, cap_p, n_areas;
  int* cnt2;                  // [nq][n_areas] entries appended by each CTA
  float* tau;                 // [nq] thresholds, raised in-kernel
  int* ovf;                   // [nq] set when a private area was too small
  int* err;
  int tighten;                // minimum pause of the refresher between rounds, ns
  int tighten_adaptive;
  int k;
  const float* margin;        // [nq] 2*eps of the prefilter
  unsigned int* hist;         // [nq][kHistStride]
  const uint32_t* hkey0;      // [nq]
  const int* hshift;          // [nq]
  const unsigned char* x16_bytes;   // base of the shadow (for the L2 prefetch)
  int64_t pf_limit_bytes;     // prefetches stay below this offset (end of the padded shadow rows)
  int prefetch;               // D > 0: warp 3 keeps an L2 prefetch (LSU path) D tiles ahead of the producer; 0: off
  int half_stage;             // 1: ring stages are 8 KB half K-blocks (64B swizzle), 2 MMAs per stage; 0: 16 KB, 4 MMAs
  int dense_quarters;         // first tile of a CTA: lane quarters [0, dense_quarters) pass unfiltered
  int first_wait_cycles;      // the other quarters wait this long at most for every threshold to exist (0: no wait)
  const float* qscale;        // int8 shadow: [n_cols] query scales sq (0 for padded columns)
  const float4* tscale;       // int8 shadow: [row tiles of 32] tile scales {st, RD(1/st), RU(1/st), 0}
  // Filtered search (SEL instances only): the launch walks tile_list[tile_begin .. tile_end) (pair tiles of 256 rows
  // that hold at least one selected row); sel_bits is the shard's row bitmap (bit r & 31 of word r >> 5: row r).
  const uint32_t* sel_bits;
  const int* tile_list;
};

struct QsPlan { int a_stages, q_stages, resident_kb, smem_bytes, half_stage; };

// Shared-memory budget: [resident query K-blocks][query ring][passage ring][tail].
// half_stage_mode: 0 never, 1 = use 8 KB half stages (128 rows x 32 K-elements, 64B swizzle) when the queries are
// fully resident and only <= 5 full 16 KB stages fit (161..176+ queries): 11 half stages keep 88 KB in flight
// instead of 80 KB and recycle ring slots at twice the granularity.
// n_kb: K-blocks of 128 bytes per row (12 for bf16, 6 for int8 rows and queries: half the query bytes, so the int8
// layout keeps every query resident next to a 9-stage ring at 173 queries).
inline QsPlan umma_qs_plan(int n_cols, int resident_kb, int q_stages, int half_stage_mode = 0, int n_kb = kNumKBlocks) {
  const int qkb = (n_cols / 2) * 128;
  if (resident_kb < 0) resident_kb = 0;
  if (resident_kb > n_kb) resident_kb = n_kb;
  if (q_stages < 2) q_stages = 2;
  if (q_stages > kQsMaxQStages) q_stages = kQsMaxQStages;
  const int tail_bytes = n_kb == kNumKBlocks ? kQsTailBytes : kQsTailBytesI8;
  QsPlan p;
  for (;;) {
    const int qs = resident_kb == n_kb ? 0 : q_stages;
    const int avail = kQsSmemLimit - 1024 - tail_bytes - (resident_kb + qs) * qkb;
    int a = avail / kQsStageBytes;
    if (a > kQsMaxAStages) a = kQsMaxAStages;
    if (a >= 4 || resident_kb == 0) {
      p.a_stages = a; p.q_stages = qs; p.resident_kb = resident_kb; p.half_stage = 0;
      if (half_stage_mode && resident_kb == n_kb && a <= 5) {
        int ah = avail / (kQsStageBytes / 2);
        if (ah > kQsMaxAStages) ah = kQsMaxAStages;
        if (ah * (kQsStageBytes / 2) > a * kQsStageBytes) { p.half_stage = 1; p.a_stages = ah; }
      }
      p.smem_bytes = (resident_kb + qs) * qkb + (p.half_stage ? p.a_stages * (kQsStageBytes / 2) : a * kQsStageBytes) +
                     tail_bytes + 1024;
      return p;
    }
    --resident_kb;   // too many resident K-blocks for this batch size: stream more of them
  }
}

// K-major, 64-byte-swizzled operand descriptor: rows of 64 bytes (32 bf16), 8-row groups 512 bytes apart,
// swizzle mode 4 (64B) in bits [61,64) — the layout TMA writes with CU_TENSOR_MAP_SWIZZLE_64B.
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu) | (static_cast<uint64_t>(512 >> 4) << 32) |
         (1ull << 46) | (4ull << 61);
}

__device__ __forceinline__ float4 lds_volatile_f4(uint32_t addr) {
  float4 r;
  asm volatile("ld.volatile.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
  return r;
}

// "does any of these 16 scores reach its threshold?" as ONE predicate chain: setp.ge.or accumulates into the
// same predicate, one instruction per score (the mask of WHICH scores hit is only built on the rare path).
// With one or two warps per scheduler every instruction of the epilogue is exposed latency; the round-1
// form (FSETP + SEL + IADD per score, then a warp reduction) made the epilogue — not the tensor pipe or
// HBM — the bottleneck of this kernel (profiles/r02_ncu_qs_epilogue_bound.md).
__device__ __forceinline__ bool any_ge16(const uint32_t (&v)[16], const float (&t)[16]) {
  uint32_t r;
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ge.f32 p, %1, %17;\n\t"
      "setp.ge.or.f32 p, %2, %18, p;\n\t"
      "setp.ge.or.f32 p, %3, %19, p;\n\t"
      "setp.ge.or.f32 p, %4, %20, p;\n\t"
      "setp.ge.or.f32 p, %5, %21, p;\n\t"
      "setp.ge.or.f32 p, %6, %22, p;\n\t"
      "setp.ge.or.f32 p, %7, %23, p;\n\t"
      "setp.ge.or.f32 p, %8, %24, p;\n\t"
      "setp.ge.or.f32 p, %9, %25, p;\n\t"
      "setp.ge.or.f32 p, %10, %26, p;\n\t"
      "setp.ge.or.f32 p, %11, %27, p;\n\t"
      "setp.ge.or.f32 p, %12, %28, p;\n\t"
      "setp.ge.or.f32 p, %13, %29, p;\n\t"
      "setp.ge.or.f32 p, %14, %30, p;\n\t"
      "setp.ge.or.f32 p, %15, %31, p;\n\t"
      "setp.ge.or.f32 p, %16, %32, p;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r)
      : "f"(__uint_as_float(v[0])), "f"(__uint_as_float(v[1])), "f"(__uint_as_float(v[2])), "f"(__uint_as_float(v[3])),
        "f"(__uint_as_float(v[4])), "f"(__uint_as_float(v[5])), "f"(__uint_as_float(v[6])), "f"(__uint_as_float(v[7])),
        "f"(__uint_as_float(v[8])), "f"(__uint_as_float(v[9])), "f"(__uint_as_float(v[10])), "f"(__uint_as_float(v[11])),
        "f"(__uint_as_float(v[12])), "f"(__uint_as_float(v[13])), "f"(__uint_as_float(v[14])), "f"(__uint_as_float(v[15])),
        "f"(t[0]), "f"(t[1]), "f"(t[2]), "f"(t[3]), "f"(t[4]), "f"(t[5]), "f"(t[6]), "f"(t[7]),
        "f"(t[8]), "f"(t[9]), "f"(t[10]), "f"(t[11]), "f"(t[12]), "f"(t[13]), "f"(t[14]), "f"(t[15]));
  return r != 0u;
}

// The same chain on the int32 accumulators of the int8 engine against integer thresholds (i8_threshold).
__device__ __forceinline__ bool any_ge16_s32(const uint32_t (&v)[16], const int (&t)[16]) {
  uint32_t r;
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ge.s32 p, %1, %17;\n\t"
      "setp.ge.or.s32 p, %2, %18, p;\n\t"
      "setp.ge.or.s32 p, %3, %19, p;\n\t"
      "setp.ge.or.s32 p, %4, %20, p;\n\t"
      "setp.ge.or.s32 p, %5, %21, p;\n\t"
      "setp.ge.or.s32 p, %6, %22, p;\n\t"
      "setp.ge.or.s32 p, %7, %23, p;\n\t"
      "setp.ge.or.s32 p, %8, %24, p;\n\t"
      "setp.ge.or.s32 p, %9, %25, p;\n\t"
      "setp.ge.or.s32 p, %10, %26, p;\n\t"
      "setp.ge.or.s32 p, %11, %27, p;\n\t"
      "setp.ge.or.s32 p, %12, %28, p;\n\t"
      "setp.ge.or.s32 p, %13, %29, p;\n\t"
      "setp.ge.or.s32 p, %14, %30, p;\n\t"
      "setp.ge.or.s32 p, %15, %31, p;\n\t"
      "setp.ge.or.s32 p, %16, %32, p;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r)
      : "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7]),
        "r"(t[8]), "r"(t[9]), "r"(t[10]), "r"(t[11]), "r"(t[12]), "r"(t[13]), "r"(t[14]), "r"(t[15]));
  return r != 0u;
}

// ------------------------------------------------------------------------------------------
// Grid = 2 * (number of CTA pairs), cluster (2,1,1), 384 threads:
//   warp 0 lane 0 : passage producer (TMA; both CTAs stream their own 128 rows of every tile)
//   warp 1        : MMA issuer (leader CTA only; one elected lane)
//   warp 2        : TMEM allocation, then lane 0 = query producer (TMA from L2)
//   warp 3        : optional L2 prefetcher (LSU path), else idle
//   warps 4..11   : epilogue — TMEM lane quarter (warp % 4), one passage row per thread; the two warps of a
//                   quarter take alternate 16-query chunks of the row
//   warp 12       : refresher — raises the global thresholds from the hit histogram and refreshes the
//                   CTA's shared-memory copy of all thresholds
// I8: int8 shadow and queries (kind::i8, s32 accumulators, 6 K-blocks of 128 bytes; the byte geometry of every
// stage, box and K-step is the bf16 one).  The epilogue compares the raw int32 accumulators with integer
// thresholds (i8_threshold): the refresher keeps u = RD(tau / sq) of every query in shared memory next to tau, and
// once per tile, before the accumulator is ready, the warp's lanes multiply the u of its query columns by the
// reciprocal tile scale (one 32-row shadow tile per warp; no division) into a per-warp shared-memory scratch, which
// every lane reads per 16-query chunk with 4 LDS.128 — the same cost as the float thresholds of the bf16 path.
// SEL: filtered search.  Every role walks the listed tiles only (tile_at); an epilogue warp's 32 rows are one word
// of the row bitmap, ANDed into row_ok, and a warp whose word is 0 skips the threshold snapshot and the chunks.
// ------------------------------------------------------------------------------------------
template <bool I8, bool SEL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kQsThreads, 1)
    umma_qs_score_select_kernel(const __grid_constant__ CUtensorMap tmap_p,
                                const __grid_constant__ CUtensorMap tmap_ph /* 32-column boxes, 64B swizzle */,
                                const __grid_constant__ CUtensorMap tmap_q, const UmmaQsArgs a) {
  extern __shared__ unsigned char umma_smem_raw[];
  const uint32_t raw = smem_u32(umma_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // 1024-byte alignment for the 128B swizzle atoms
  unsigned char* base_ptr = umma_smem_raw + (base - raw);

  const int n_half = a.n_cols >> 1;
  const uint32_t qkb_bytes = static_cast<uint32_t>(n_half) * 128u;   // one K-block of this CTA's query half
  const int R = a.resident_kb;
  const uint32_t smem_qres = base;
  const uint32_t smem_qring = base + static_cast<uint32_t>(R) * qkb_bytes;
  const uint32_t smem_a = smem_qring + static_cast<uint32_t>(a.q_stages) * qkb_bytes;
  const uint32_t a_stage_bytes = a.half_stage ? kQsStageBytes / 2 : kQsStageBytes;
  const int n_sub = a.half_stage ? 2 : 1;          // ring stages per K-block
  const uint32_t tail_off = static_cast<uint32_t>(R + a.q_stages) * qkb_bytes + static_cast<uint32_t>(a.a_stages) * a_stage_bytes;
  const uint32_t tail = base + tail_off;
  const uint32_t bar_afull = tail;                               // [kQsMaxAStages]
  const uint32_t bar_aempty = tail + 8 * kQsMaxAStages;          // [kQsMaxAStages]
  const uint32_t bar_qfull = tail + 16 * kQsMaxAStages;          // [kQsMaxQStages]
  const uint32_t bar_qempty = bar_qfull + 8 * kQsMaxQStages;     // [kQsMaxQStages]
  const uint32_t bar_qres = bar_qempty + 8 * kQsMaxQStages;
  const uint32_t bar_tfull = bar_qres + 8;                       // [2]
  const uint32_t bar_tempty = bar_tfull + 16;                    // [2]
  unsigned char* tail_ptr = base_ptr + tail_off;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tail_ptr + 16 * kQsMaxAStages + 16 * kQsMaxQStages + 8 + 32);
  volatile int* epi_done_s = reinterpret_cast<volatile int*>(tmem_ptr_s + 1);
  volatile int* tau_ready_s = reinterpret_cast<volatile int*>(tmem_ptr_s + 2);   // every query has a finite threshold
  volatile int* prod_it_s = reinterpret_cast<volatile int*>(tmem_ptr_s + 3);     // tile iteration the passage producer is at
  float* tau_s = reinterpret_cast<float*>(tail_ptr + 512);               // [kQsMaxCols]
  int* cnt_s = reinterpret_cast<int*>(tail_ptr + 512 + 1024);            // [kQsMaxCols]
  uint32_t* hkey0_s = reinterpret_cast<uint32_t*>(tail_ptr + 512 + 2048);  // [kQsMaxCols]
  const uint32_t tau_s_addr = tail + 512;
  int* thr_s = reinterpret_cast<int*>(tail_ptr + kQsTailBytes);          // int8: [kQsEpiWarps][128] integer thresholds
  float* u_s = reinterpret_cast<float*>(tail_ptr + kQsTailBytes + kQsEpiWarpsI8Scratch);   // int8: [kQsMaxCols] tau / sq
  constexpr int NKB = I8 ? kShadow8KBlocks : kNumKBlocks;                 // K-blocks of 128 bytes per row

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_p);
    prefetch_tmap(&tmap_ph);
    prefetch_tmap(&tmap_q);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kQsMaxAStages; ++s) {
      mbar_init(bar_afull + 8 * s, 2);   // leader's expect_tx arrive + peer's remote arrive
      mbar_init(bar_aempty + 8 * s, 1);  // one multicast commit
    }
    for (int s = 0; s < kQsMaxQStages; ++s) {
      mbar_init(bar_qfull + 8 * s, 2);
      mbar_init(bar_qempty + 8 * s, 1);
    }
    mbar_init(bar_qres, 2);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_tfull + 8 * s, 1);   // one multicast commit
      mbar_init(bar_tempty + 8 * s, 2 * kQsEpiWarps);  // epilogue warps x 2 CTAs (leader's copy is the one used)
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_ptr_s)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x == 0) { *epi_done_s = 0; *tau_ready_s = 0; *prod_it_s = 0; }
  for (int i = threadIdx.x; i < kQsMaxCols; i += kQsThreads) {
    tau_s[i] = (i < a.nq) ? a.tau[i] : INFINITY;     // padded query columns never hit
    if constexpr (I8) u_s[i] = (i < a.nq) ? i8_tau_over_sq(tau_s[i], __ldg(a.qscale + i)) : INFINITY;
    cnt_s[i] = 0;
    hkey0_s[i] = (i < a.nq) ? a.hkey0[i] : 0xffffffffu;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_s);

  if (warp == 0 && lane == 0) {
    // ===================== passage producer =====================
    uint32_t stage = 0, phase = 0;
    int prod_it = 0;
    for (int ti = a.tile_begin + pair; ti < a.tile_end; ti += npairs, ++prod_it) {
      const int tile = tile_at<SEL>(a.tile_list, ti);
      *prod_it_s = prod_it;       // progress mark for the L2 prefetch warp
      // shadow layout (common.cuh): this CTA's 128 rows are 4 consecutive 32-row tiles; K-block kb of
      // each is a contiguous 4 KB piece -> 4 TMA boxes per 16 KB stage (rows past the end: zero fill)
      const int t32 = (tile * 2 + static_cast<int>(cta_rank)) * (kQsTileRowsCta / kShadowTileRows);
      for (int kb = 0; kb < NKB; ++kb) {
        for (int h = 0; h < n_sub; ++h) {
          mbar_wait(bar_aempty + 8 * stage, phase ^ 1u, a.err);
          const uint32_t full_leader = mapa_u32(bar_afull + 8 * stage, 0);
          if (leader) mbar_arrive_expect_tx(bar_afull + 8 * stage, 2u * a_stage_bytes);
          else mbar_arrive_cluster(full_leader);
          if (a.half_stage) {
#pragma unroll
            for (int j = 0; j < kQsTileRowsCta / kShadowTileRows; ++j)
              tma_load_2d_2sm(smem_a + stage * a_stage_bytes + j * (kShadowTileRows * 64), &tmap_ph, full_leader, 32 * h,
                              ((t32 + j) * NKB + kb) * kShadowTileRows, kHintEvictFirst);
          } else {
#pragma unroll
            for (int j = 0; j < kQsTileRowsCta / kShadowTileRows; ++j)
              tma_load_2d_2sm(smem_a + stage * a_stage_bytes + j * (kShadowTileRows * 128), &tmap_p, full_leader, 0,
                              ((t32 + j) * NKB + kb) * kShadowTileRows, kHintEvictFirst);
          }
          if (++stage == static_cast<uint32_t>(a.a_stages)) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 2 && lane == 0) {
    // ===================== query producer (L2 -> smem) =====================
    if (R > 0) {
      const uint32_t qres_leader = mapa_u32(bar_qres, 0);
      if (leader) mbar_arrive_expect_tx(bar_qres, 2u * static_cast<uint32_t>(R) * qkb_bytes);
      else mbar_arrive_cluster(qres_leader);
      for (int kb = 0; kb < R; ++kb)
        tma_load_2d_2sm(smem_qres + kb * qkb_bytes, &tmap_q, qres_leader, kb * kBlockK,
                        static_cast<int>(cta_rank) * n_half, kHintEvictLast);
    }
    if (R < NKB) {
      uint32_t stage = 0, phase = 0;
      for (int tile = a.tile_begin + pair; tile < a.tile_end; tile += npairs) {
        for (int kb = R; kb < NKB; ++kb) {
          mbar_wait(bar_qempty + 8 * stage, phase ^ 1u, a.err);
          const uint32_t full_leader = mapa_u32(bar_qfull + 8 * stage, 0);
          if (leader) mbar_arrive_expect_tx(bar_qfull + 8 * stage, 2u * qkb_bytes);
          else mbar_arrive_cluster(full_leader);
          tma_load_2d_2sm(smem_qring + stage * qkb_bytes, &tmap_q, full_leader, kb * kBlockK,
                          static_cast<int>(cta_rank) * n_half, kHintEvictLast);
          if (++stage == static_cast<uint32_t>(a.q_stages)) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 3 && a.prefetch > 0) {
    // ===================== L2 prefetcher (optional) =====================
    // With the queries resident, 80 KB of ring per SM are too few bytes in flight to cover HBM latency at
    // full bandwidth (5 stages: 5.9 TB/s, 7 stages: 6.7).  Prefetching through the TMA unit (cp.async.bulk.
    // prefetch) made things worse both times it was tried — the requests queue in front of the demand loads
    // of the same unit.  This warp uses the LSU path instead: one `prefetch.global.L2` per 128-byte line of
    // the CTA's tile `prefetch` rounds ahead (a tile is ONE contiguous 192 KB region of the shadow: 4
    // consecutive 32-row tiles x 12 K-blocks x 4 KB), paced by the producer's progress mark.
    constexpr int64_t kTileBytesCta = static_cast<int64_t>(kQsTileRowsCta) * kD * (I8 ? 1 : 2);     // 196,608 (bf16)
    int it_pf = 0;
    for (int ti = a.tile_begin + pair; ti < a.tile_end; ti += npairs, ++it_pf) {
      const int tile = tile_at<SEL>(a.tile_list, ti);
      while (it_pf > *prod_it_s + a.prefetch) __nanosleep(400);
      if (it_pf <= *prod_it_s) continue;          // the producer is already there
      const int64_t off = (static_cast<int64_t>(tile) * 2 + cta_rank) * kTileBytesCta;
      if (off + kTileBytesCta > a.pf_limit_bytes) continue;
      const unsigned char* base_g = a.x16_bytes + off;
      for (int i = lane; i < static_cast<int>(kTileBytesCta / 128); i += 32)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base_g + static_cast<int64_t>(i) * 128));
    }
  } else if (warp == 1 && leader) {
    // ===================== MMA issuer (leader CTA; the whole warp waits, one elected lane issues) =====
    const uint32_t idesc = I8 ? umma_idesc_i8(256, a.n_cols) : umma_idesc_bf16(256, a.n_cols);
    const bool elected = elect_one();
    if (R > 0) {
      mbar_wait(bar_qres, 0, a.err);
      tc_fence_after();
    }
    uint32_t sa = 0, pa = 0, sq = 0, pq = 0;
    int it = 0;
    for (int tile = a.tile_begin + pair; tile < a.tile_end; tile += npairs, ++it) {
      const uint32_t as = it & 1, aph = (it >> 1) & 1;
      mbar_wait(bar_tempty + 8 * as, aph ^ 1u, a.err);   // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * kQsAccStride;
      for (int kb = 0; kb < NKB; ++kb) {
        const bool streamed = kb >= R;
        if (streamed) mbar_wait(bar_qfull + 8 * sq, pq, a.err);
        for (int h = 0; h < n_sub; ++h) {
          mbar_wait(bar_afull + 8 * sa, pa, a.err);
          tc_fence_after();
          if (elected) {
            const uint32_t a_addr = smem_a + sa * a_stage_bytes;
            const uint64_t adesc = a.half_stage ? umma_desc_sw64(a_addr) : umma_desc_sw128(a_addr);
            const uint64_t bdesc = umma_desc_sw128(streamed ? smem_qring + sq * qkb_bytes : smem_qres + kb * qkb_bytes);
            const int k_steps = a.half_stage ? 2 : 4;     // UMMA K = 16 bf16 / 32 int8 = 32 bytes = 2 descriptor units
            for (int k = 0; k < k_steps; ++k) {
              const int kq = a.half_stage ? 2 * h + k : k;   // position of this K-step inside the query K-block
              if (I8) umma_i8_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * kq, idesc, (kb | h | k) != 0);
              else umma_bf16_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * kq, idesc, (kb | h | k) != 0);
            }
            umma_commit_pair(bar_aempty + 8 * sa);                 // frees the passage stage in both CTAs
            if (h == n_sub - 1) {
              if (streamed) umma_commit_pair(bar_qempty + 8 * sq);   // and the query stage
              if (kb == NKB - 1) umma_commit_pair(bar_tfull + 8 * as);  // accumulator ready
            }
          }
          __syncwarp();
          if (++sa == static_cast<uint32_t>(a.a_stages)) { sa = 0; pa ^= 1u; }
        }
        if (streamed && ++sq == static_cast<uint32_t>(a.q_stages)) { sq = 0; pq ^= 1u; }
      }
    }
  } else if (warp >= 4 && warp < 4 + kQsEpiWarps) {
    // ===================== epilogue: filter + append =====================
    const int ew = warp & 3;                 // TMEM lane quarter this warp may read
    const int half = (warp - 4) >> 2;        // which of the alternating 16-query chunks
    const uint32_t tempty_leader0 = mapa_u32(bar_tempty, 0);
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int area = static_cast<int>(blockIdx.x);    // this CTA's private area in every query's list
    uint64_t* area0 = a.cand + a.S + static_cast<int64_t>(area) * a.cap_p;
    // one hit of query column qc: reserve a slot in the CTA's area (shared-memory counter, one atomic per
    // warp), write the record, count it in the tightening histogram
    auto hit = [&](int qc, bool pass, uint32_t bits, uint32_t row) {
      const uint32_t b = __ballot_sync(0xffffffffu, pass);
      if (b == 0u) return;
      const int first = __ffs(b) - 1;
      int s0 = 0;
      if (lane == first) s0 = atomicAdd(cnt_s + qc, __popc(b));
      s0 = __shfl_sync(0xffffffffu, s0, first);
      if (pass) {
        const int slot = s0 + __popc(b & lt_mask);
        if (slot < a.cap_p) area0[static_cast<int64_t>(qc) * a.C + slot] = pack_cand(__uint_as_float(bits), row);
        // counted at s~ - eps: a lower bound of the row's EXACT (centred) score, so that "k hits at or above
        // bucket edge e" bounds the k-th best exact score itself and the threshold is e - eps, not e - 2 eps
        const uint32_t key = fkey(__fsub_rd(__uint_as_float(bits), __fmul_ru(__ldg(a.margin + qc), 0.5f)));
        const uint32_t k0 = hkey0_s[qc];
        if (key >= k0) {
          const uint32_t hb = min(static_cast<uint32_t>(kHistBuckets - 1), (key - k0) >> __ldg(a.hshift + qc));
          unsigned int* hq = a.hist + static_cast<int64_t>(qc) * kHistStride;
          atomicAdd(hq + hb, 1u);
          atomicAdd(hq + kHistBuckets + (hb >> 4), 1u);
        }
      }
    };
    // int8: this warp's query columns are 16 * half + 32 * i + j (i-th chunk, j < 16); their integer thresholds for
    // the warp's shadow tile (one scale: the warp's 32 rows are one shadow tile) go to the warp's scratch.  Thresholds
    // only rise, so a snapshot taken before the accumulator is ready keeps every filter valid.
    auto snap_thresholds = [&](float4 ts, int* thr_w) {
      const int n_own = 16 * ((a.n_cols - 16 * half + 31) / 32);
      for (int x = lane; x < n_own; x += 32) {
        const int col = 16 * half + 32 * (x >> 4) + (x & 15);
        thr_w[x] = i8_threshold(*reinterpret_cast<volatile float*>(u_s + col), ts);
      }
      __syncwarp();
    };
    int it = 0;
    for (int ti = a.tile_begin + pair; ti < a.tile_end; ti += npairs, ++it) {
      const int tile = tile_at<SEL>(a.tile_list, ti);
      const uint32_t as = it & 1, aph = (it >> 1) & 1;
      const int64_t row64 = static_cast<int64_t>(tile) * kQsTileRows + cta_rank * kQsTileRowsCta + ew * 32 + lane;
      bool row_ok = row64 < a.n_rows;
      uint32_t sel_word = 0xffffffffu;
      if constexpr (SEL) {
        sel_word = __ldg(a.sel_bits + ((row64 - lane) >> 5));
        row_ok = row_ok && ((sel_word >> lane) & 1u);
      }
      const uint32_t row = static_cast<uint32_t>(row64);
      const float4 ts = (I8 && row64 - lane < a.n_rows) ? __ldg(a.tscale + ((row64 - lane) >> 5))
                                                         : make_float4(0.f, INFINITY, INFINITY, 0.f);
      const float st = ts.x;
      int* thr_w = thr_s + (warp - 4) * 128;
      // the conversion overlaps the MMA of this tile; the first tile converts after the wait for the first thresholds
      if (I8 && it > 0 && sel_word != 0u) snap_thresholds(ts, thr_w);
      mbar_wait(bar_tfull + 8 * as, aph, a.err);
      tc_fence_after();
      if (it == 0 && ew >= a.dense_quarters && a.first_wait_cycles > 0) {
        // Thresholds start at -inf.  Only the first quarter(s) of a CTA's first tile pass unfiltered — enough
        // rows over all CTAs to place every query's threshold; the other quarters wait for the refresher's
        // "every query has a threshold" flag instead of appending 96 more rows x all queries that the final
        // selection would throw away again.  Bounded wait: a query whose scores never reach the histogram
        // keeps tau = -inf, which is slow (its lists overflow and the query is re-run) but never wrong.
        const long long t0 = clock64();
        while (*tau_ready_s == 0 && clock64() - t0 < a.first_wait_cycles) __nanosleep(256);
      }
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + as * kQsAccStride;
      if (sel_word != 0u) {   // warp-uniform; always true without a filter
        if (I8 && it == 0) snap_thresholds(ts, thr_w);
        for (int c0 = 16 * half; c0 < a.n_cols; c0 += 32) {
          uint32_t v[16];
          tmem_ld_x16(taddr + c0, v);
          if constexpr (I8) {
            const int* thr = thr_w + 16 * ((c0 - 16 * half) >> 5);
            int t[16];
  #pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int4 f = *reinterpret_cast<const int4*>(thr + 4 * u);
              t[4 * u] = f.x; t[4 * u + 1] = f.y; t[4 * u + 2] = f.z; t[4 * u + 3] = f.w;
            }
            tmem_ld_wait();
            const bool mine = row_ok && any_ge16_s32(v, t);
            if (__any_sync(0xffffffffu, mine)) {
              uint32_t m = 0;
  #pragma unroll
              for (int j = 0; j < 16; ++j) m |= (static_cast<int>(v[j]) >= t[j]) ? (1u << j) : 0u;
              if (!row_ok) m = 0;
              uint32_t any = __reduce_or_sync(0xffffffffu, m);
              if (__popc(any) > 4) {
                // busy chunk (loose thresholds early in a pass): unrolled, v[] stays in registers
  #pragma unroll
                for (int j = 0; j < 16; ++j)
                  if ((any >> j) & 1u)
                    hit(c0 + j, (m >> j) & 1u, __float_as_uint(i8_score(static_cast<int>(v[j]), __ldg(a.qscale + c0 + j), st)), row);
                any = 0;
              }
              while (any) {   // the recorded score is formed on this rare path only
                const int j = __ffs(any) - 1;
                any &= any - 1;
                const uint32_t acc = tmem_ld_x1(taddr + c0 + j);
                tmem_ld_wait();
                hit(c0 + j, (m >> j) & 1u, __float_as_uint(i8_score(static_cast<int>(acc), __ldg(a.qscale + c0 + j), st)), row);
              }
            }
            continue;
          }
          // thresholds of these 16 queries (volatile: the refresher warp rewrites them while we run)
          float t[16];
  #pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float4 f = lds_volatile_f4(tau_s_addr + 4u * static_cast<uint32_t>(c0 + 4 * u));
            t[4 * u] = f.x; t[4 * u + 1] = f.y; t[4 * u + 2] = f.z; t[4 * u + 3] = f.w;
          }
          tmem_ld_wait();
          const bool mine = row_ok && any_ge16(v, t);
          if (__any_sync(0xffffffffu, mine)) {
            // some row of this warp reached a threshold of this chunk: now build the per-lane hit mask
            uint32_t m = 0;
  #pragma unroll
            for (int j = 0; j < 16; ++j) m |= (__uint_as_float(v[j]) >= t[j]) ? (1u << j) : 0u;
            if (!row_ok) m = 0;
            uint32_t any = __reduce_or_sync(0xffffffffu, m);
            if (__popc(any) > 4) {
              // busy chunk (loose thresholds, the first tiles of a pass): unrolled, v[] stays in registers
  #pragma unroll
              for (int j = 0; j < 16; ++j)
                if ((any >> j) & 1u) hit(c0 + j, (m >> j) & 1u, v[j], row);
            } else {
              while (any) {   // rare: re-read the flagged column from TMEM (a dynamic index would spill v[])
                const int j = __ffs(any) - 1;
                any &= any - 1;
                const uint32_t bits = tmem_ld_x1(taddr + c0 + j);
                tmem_ld_wait();
                hit(c0 + j, (m >> j) & 1u, bits, row);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader0 + 8 * as);
    }
    // all epilogue warps are done appending: publish the per-area counts
    asm volatile("bar.sync 1, 256;" ::: "memory");
    for (int q = threadIdx.x - 128; q < a.nq; q += 32 * kQsEpiWarps) {
      const int c = cnt_s[q];
      a.cnt2[q * a.n_areas + area] = min(c, a.cap_p);
      if (c > a.cap_p) a.ovf[q] = 1;
    }
    __syncwarp();
    if (lane == 0) atomicAdd(const_cast<int*>(epi_done_s), 1);
  } else if (warp == kQsRefresherWarp) {
    // ===================== refresher: in-kernel threshold tightening =====================
    // Same rule as the TS variant (refresh_threshold) for the queries assigned to this CTA; additionally copy
    // ALL current thresholds into this CTA's shared memory, where the epilogue threads (one passage row each,
    // all queries) read them.
    float last[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    const long long t_start = clock64();
    while (*epi_done_s < kQsEpiWarps) {
      int qi = 0;
      for (int q = blockIdx.x; q < a.nq; q += gridDim.x, ++qi)
        refresh_threshold(a.hist, hkey0_s[q], a.hshift, a.margin, a.tau, a.k, q, qi, lane, last);
      // thresholds published by every CTA -> this CTA's shared memory (they only rise)
      bool all_finite = true;
      for (int i = lane; i < a.nq; i += 32) {
        const float t = *reinterpret_cast<volatile float*>(a.tau + i);
        if (t > tau_s[i]) {
          *reinterpret_cast<volatile float*>(tau_s + i) = t;
          // int8: the query factor of the integer thresholds; the divisions stay off the epilogue warps
          if constexpr (I8) *reinterpret_cast<volatile float*>(u_s + i) = i8_tau_over_sq(t, __ldg(a.qscale + i));
        }
        all_finite = all_finite && (t > -INFINITY);
      }
      if (__all_sync(0xffffffffu, all_finite) && lane == 0) *tau_ready_s = 1;
      unsigned int pause = static_cast<unsigned int>(a.tighten);
      if (*tau_ready_s == 0) pause = 500;     // start of the pass: epilogue warps are waiting for the first thresholds
      else if (a.tighten_adaptive) {
        const long long age_ns = (clock64() - t_start) >> 1;     // cycles -> ns at ~2 GHz; only a pacing hint
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
