// b2f_api.cu — host side of the engine behind the C ABI declared in include/b2f.h.
//
// One b2f_index owns one shard per device: the fp32 rows (for exact rescoring and the SIMT
// engine), the shard's centre, the bf16 shadow of the centred rows (streamed by the tensor engine),
// the norm bounds of the shard, and a per-shard workspace.  A search is a fixed sequence of kernels:
//
//   prep_queries -> per pass of <= 256 queries: pass_init -> score+select (ONE launch) -> finalize
//
// where score+select is umma_qs_score_select_kernel (<= 208 queries) or umma_score_select_kernel
// (tcgen05, both), with the phased schedules (dense bootstrap / refresh between phases) kept for the
// SIMT scan_kernel and as A/B options.  There is no CPU arithmetic anywhere on this path; without a
// CUDA device every entry point fails.
#include "../../include/b2f.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <type_traits>
#include <atomic>
#include <chrono>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <vector>

#include "common.cuh"
#include "kernels_scan.cuh"
#include "kernels_select.cuh"
#include "kernels_selector.cuh"
#include "kernels_umma.cuh"
#include "kernels_umma_qs.cuh"
#include "kernels_util.cuh"

using namespace b2f;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU_TRY(call)                                                                           \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      (void)cudaGetLastError();                                                                \
      return fail(e_ == cudaErrorMemoryAllocation ? B2F_ERR_OOM : B2F_ERR_CUDA,                \
                  std::string(#call) + ": " + cudaGetErrorString(e_) + " (" __FILE__ ":" +     \
                      std::to_string(__LINE__) + ")");                                         \
    }                                                                                          \
  } while (0)

#define B2F_TRY(call)        \
  do {                       \
    int rc_ = (call);        \
    if (rc_ != B2F_OK) return rc_; \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 tensor [rows, cols] with row pitch cols*2 bytes, box = 64 columns (128 bytes) x box_rows,
// 128-byte swizzle.  Queries: cols = 768 (row-major).  Shadow: cols = 64 — the K-block-major tiled
// layout (common.cuh) is a [tiles*12*128, 64] matrix of 128-byte rows.
// `half_box`: boxes of 32 columns (64 bytes) with the 64-byte swizzle instead (the QS kernel's half stages).
int make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint32_t cols, uint32_t box_rows, bool half_box = false) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(B2F_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), rows};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(cols) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(half_box ? kBlockK / 2 : kBlockK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, half_box ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B2F_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return B2F_OK;
}

constexpr int kMaxPending = 16;
constexpr int kLoadBufs = 6;            // pinned staging buffers of the flat-file loader
constexpr int64_t kLoadPieceRows = 8192; // rows per staged piece (24 MB)
constexpr int kMuBlocks = 256;          // partial column sums of the centre
constexpr int64_t kMuRows = 65536;      // the centre is the mean of (up to) the first 65536 rows of the first add   // asynchronous device searches in flight (one overflow-flag slot each)

struct Workspace {
  // candidate state of one pass
  int qp_cap = 0, C = 0;
  uint64_t* cand[2] = {nullptr, nullptr};
  int* cnt = nullptr;
  float* tau = nullptr;
  uint64_t* tauP = nullptr;
  int* ovf = nullptr;
  float* margin = nullptr;
  int* err = nullptr;
  bool areas_clean = false;   // tensor-engine invariant: private areas of both cand buffers are all-zero
  uint64_t* gath = nullptr;   // refresh scratch: dense copy of a segmented list
  int* cnt2 = nullptr;        // [qp][max_pairs] per-pair append counts of the tensor engine
  unsigned int* hist = nullptr;   // [qp][kHistBuckets] tightening histogram of the tensor engine
  uint32_t* hkey0 = nullptr;      // [qp] its base key
  int* hshift = nullptr;          // [qp] log2(keys per bucket)
  // queries of one search
  int64_t nq_cap = 0;
  float* q32 = nullptr;
  __nv_bfloat16* q16 = nullptr;
  float* qnorm = nullptr;
  float* qerr = nullptr;      // [nq] upper bound of ||q - bf16(q)|| (int8 shadow: of ||q - sq q8||)
  float* qscale = nullptr;    // [nq] int8 shadow: query scales sq (the int8 codes live in q16's buffer)
  int* ovf_all = nullptr;
  int* ovf_host = nullptr;  // pinned
  // per-shard results of one search
  int64_t out_cap = 0;
  float* D = nullptr;
  int64_t* I = nullptr;
  // merge staging (shard 0 only): the parts [G][nq][k] of a multi-shard search, one area per pending slot (a
  // search owns its slot's parts until it is settled: a re-run shard's part is merged again then)
  int64_t parts_cap[kMaxPending] = {};
  float* Dp[kMaxPending] = {};
  int64_t* Ip[kMaxPending] = {};
  // fallback staging
  float* fbq = nullptr;   // [kScanMaxQ, 768]
  float* fbD = nullptr;   // [kScanMaxQ, B2F_MAX_K]
  int64_t* fbI = nullptr;
  // pinned host staging for query upload / result download
  size_t pin_bytes = 0;
  void* pin = nullptr;
};

struct Stats {
  double launches = 0, phases = 0, candidates = 0, fallback_queries = 0, path = 0, passes = 0, qs_passes = 0;
  double ovf_area = 0, ovf_survivors = 0;   // why queries fell back: private area too small / too many rows within the margin
  double score_ms = 0, score_launches = 0, score_rows = 0, select_ms = 0, xchg_ms = 0;
};

// Optional per-launch device timing ("profile" option): CUDA events on the shard stream around
// every scoring launch (kind 0) and every refresh/final launch (kind 1).
struct Prof {
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  struct Span { int kind; size_t b, e; };
  std::vector<Span> spans;
  cudaEvent_t get() {
    if (used == pool.size()) {
      cudaEvent_t ev;
      cudaEventCreate(&ev);
      pool.push_back(ev);
    }
    return pool[used++];
  }
};

struct Shard {
  int dev = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev = nullptr;
  int sm_count = 148;
  int max_pairs = 74;
  float* x32 = nullptr;
  __nv_bfloat16* x16 = nullptr;     // bf16 shadow (format 1)
  int8_t* x8 = nullptr;              // int8 shadow (format 2) ...
  float4* tscale = nullptr;          // ... and its per-32-row-tile scales {st, RD(1/st), RU(1/st), 0} (i8_tile_scale)
  int fmt = 0;                       // shadow format of the buffers: 0 none / not chosen yet, 1 bf16, 2 int8
  double rho = 0;                    // AUTO: median 2 eps8 / sigma of the probe (0: not measured)
  int64_t n = 0, cap = 0;
  unsigned int* maxnorm2 = nullptr;  // device, float bits: [0] max ||p||^2, [1] max ||(p - mu) - shadow||^2, [2] max ||p - mu||^2
  float* mu = nullptr;               // device [768]: the shard's centre (zeros until set / when centring is off)
  float* mu_part = nullptr;          // device [kMuBlocks][768]: partial column sums
  bool mu_set = false;
  char* load_bufs[kLoadBufs] = {nullptr};       // pinned staging ring of b2f_add_flat_file (allocated on first use)
  cudaEvent_t load_evs[kLoadBufs] = {nullptr};
  int64_t* idmap = nullptr;          // optional explicit labels [cap]
  bool has_ids = false;
  std::vector<Seg> segs;
  Seg* segs_d = nullptr;
  int segs_d_cap = 0;
  bool segs_dirty = true;            // host segment list changed since it was last uploaded
  Workspace ws;
  Prof prof;
  Stats stats;
  bool peer_to_first = false;   // this device can store into shard 0's device memory (in-process result gather)
};

}  // namespace

// One persistent host thread per shard beyond the first: a multi-device search is enqueued on all
// devices at the same time (FAISS IndexShards runs one host thread per GPU shard too) instead of
// paying the launch sequence of every device one after the other.
struct ShardWorker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<int()> task;
  bool has_task = false, done = false, stop = false;
  int rc = 0;
  std::string err;
  void loop() {
    std::unique_lock<std::mutex> lk(m);
    for (;;) {
      cv.wait(lk, [&] { return has_task || stop; });
      if (stop) return;
      lk.unlock();
      const int r = task();
      lk.lock();
      rc = r;
      err = g_err;            // the worker's thread-local error text travels back with the code
      has_task = false;
      done = true;
      cv.notify_all();
    }
  }
  void submit(std::function<int()> f) {
    std::lock_guard<std::mutex> lk(m);
    task = std::move(f);
    has_task = true;
    done = false;
    cv.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [&] { return done; });
    done = false;
    if (rc != B2F_OK) g_err = err;
    return rc;
  }
  ~ShardWorker() {
    if (th.joinable()) {
      { std::lock_guard<std::mutex> lk(m); stop = true; cv.notify_all(); }
      th.join();
    }
  }
};

struct Pending {
  const float* q; int64_t nq; int k; float* D; int64_t* I; int slot;
  const b2f_selector* sel;   // the overflow re-run filters with it too
};

namespace {
// One shard's part of a selector (kernels_selector.cuh): the row bitmap and the lists of the tiles that hold a
// selected row, in ascending order.
struct SelShard {
  int dev = 0;
  int64_t count = 0;                 // selected rows
  uint32_t* bits = nullptr;          // [round_up(n, kQsTileRows) / 32]
  int* qs_tiles = nullptr;           // QS tiles (kQsTileRows rows)
  int* ts_tiles = nullptr;           // TS tiles (kTileRows rows)
  int n_qs = 0, n_ts = 0;
  std::vector<int> ts_host;          // host copy: the phased TS schedules walk a sub-range per phase
};
}  // namespace

struct b2f_selector {
  b2f_index* idx = nullptr;
  uint64_t generation = 0;           // the index generation it was built against
  int64_t count = 0;
  std::vector<SelShard> parts;       // one per shard
};

struct b2f_index {
  int d = kD;
  std::vector<Shard> shards;
  std::vector<Pending> pending;   // enqueued by b2f_search_device_async, settled by b2f_search_finish
  std::vector<std::unique_ptr<ShardWorker>> workers;   // [shards - 1], created by the first multi-shard search
  int (*xchg_flush)(b2f_index*) = nullptr;   // set by b2f_xchg_connect (enqueues a deferred exchange merge)
  int* merge_flag_host = nullptr; // mapped host ints: [0] a merge saw a part whose list had overflowed,
  int* merge_flag_dev = nullptr;  //                   [1] the peer exchange timed out waiting for a rank
  // peer-memory exchange (one process per GPU; see kernels_select.cuh)
  struct Xchg {
    int rank = -1, world = 0;
    int64_t max_nq = 0;
    int max_k = 0;
    size_t part_cap = 0, flags_off = 0, bytes = 0;
    char* local = nullptr;                 // this rank's buffer [2][world][part_cap] + flags[2][world]
    char* peer[kXchgMaxWorld] = {nullptr}; // the same buffer of every rank (peer[rank] == local)
    char* stage = nullptr;                 // local packed part [D | I] written by the search
    int* counter = nullptr;
    unsigned int seq = 0;
    bool connected = false;
    // deferred merge: the merge of exchange step s is enqueued behind the push of step s+1 (or by
    // b2f_search_finish), when every rank's part has long arrived, so the ranks are coupled with one
    // step of slack instead of a barrier per search (they all wait for the momentarily slowest GPU otherwise)
    int defer = 1;
    struct Deferred { bool valid = false; unsigned int seq = 0; int64_t nq = 0; int k = 0; float* D = nullptr; int64_t* I = nullptr; } deferred;
  } xchg;
  int64_t ntotal = 0;
  std::atomic<uint64_t> generation{0};   // bumped by every add and reset: a selector built before is stale
  std::mutex ntotal_mutex;     // b2f_add_flat_file may run on several shards at once (one host thread each)
  // options
  int path = B2F_PATH_AUTO;
  int shadow = kShadowAuto;   // 0 none, 1 bf16, 2 int8, 3 AUTO (per shard, from its first rows; DESIGN.md section 4)
  int growth = 32;
  int64_t margin_ppm = 1000000;
  int keep_on_reset = 1;
  int scan_max_auto = 0;  // AUTO: batches up to this size use the SIMT scan (0: the tensor engine streams half the
                          // bytes and wins from one query on — profiles/r01s2_sweep_8p8M_*.json)
  int profile = 0;
  int umma_variant = 0;   // 0 auto (QS up to qs_max_q queries per pass, TS above), 1 QS with every query K-block
                          // resident in shared memory (the round-1 "SS" layout), 2 TS (queries in TMEM), 3 QS
  int qs_max_q = 208;     // AUTO: passes of up to this many queries take the QS variant (MMA N = nq rounded to 16)
  int qs_resident_kb = 12; // QS: query K-blocks kept resident in shared memory (0..12; lowered automatically when the
                          // batch is too large to leave a passage ring of 4 stages); the rest streams from L2.  Measured
                          // (profiles/r02): fully resident wins for <= 208 queries — the re-read query bytes cost more
                          // L2->SM bandwidth and power than the deeper passage ring gains
  int qs_q_stages = 3;    // QS: depth of the query ring
  int qs_half_stage = 0;  // QS: 1 = 8 KB half stages when only <= 5 full stages fit next to the resident queries
  int center = 1;         // subtract the collection mean (first rows of the first add) before the bf16 rounding
  int synth_mean_shift = 0;  // b2f_add_synthetic: integer shift of every component along a fixed sign vector
  int l2_prefetch = 0;    // QS: distance (tiles) of the optional L2 prefetch warp; 0 = off (default: measured slower)
  int worst_case_margin = 0;  // 1: bf16 margin from the data-independent worst case (A/B only)
  int tighten_adaptive = 1;  // refresher pause grows with the elapsed kernel time (see UmmaArgs)
  int bootstrap = 0;      // TS engine with tightening: 1 = dense bootstrap launch + bootstrap_select_kernel before the
                          // main launch, 0 = none (thresholds start at -inf inside the single launch)
  int tighten = 2000;      // TS engine: in-kernel threshold tightening through a global hit histogram (one
                          // launch after the bootstrap); pause of the refresher between rounds in ns,
                          // 0 = off (geometric phases with a refresh kernel between them).
  Stats stats;
};

namespace {

template <typename T>
int dev_alloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) return B2F_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(B2F_ERR_OOM, "cudaMalloc of " + std::to_string(count * sizeof(T)) + " bytes failed: " +
                                 cudaGetErrorString(e));
  }
  return B2F_OK;
}
template <typename T>
void dev_free(T*& p) {
  if (p) cudaFree(p);
  p = nullptr;
}

int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

int ensure_capacity(b2f_index* idx, Shard& S, int64_t need) {
  if (need <= S.cap) return B2F_OK;
  CU_TRY(cudaSetDevice(S.dev));
  int64_t ncap = std::max<int64_t>(need, S.cap + S.cap / 2);
  if (S.n == 0) {   // nothing to keep: release first, so that regrowing a large empty shard never holds both copies
    dev_free(S.x32); dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale); dev_free(S.idmap);
    S.cap = 0;
    ncap = need;
  }
  float* n32 = nullptr;
  __nv_bfloat16* n16 = nullptr;
  int8_t* n8 = nullptr;
  float4* nts = nullptr;
  int64_t* nid = nullptr;
  B2F_TRY(dev_alloc(&n32, static_cast<size_t>(ncap) * kD));
  // the shadow in the shard's format; under AUTO an empty shard has none yet (ingest_rows allocates it once the
  // first rows have decided the format, so a reserve() never commits bf16-sized memory for an int8 shard)
  int rc = B2F_OK;
  if (S.fmt == kShadowBf16) rc = dev_alloc(&n16, static_cast<size_t>(shadow_rows_padded(ncap)) * kD);
  if (S.fmt == kShadowInt8) {
    rc = dev_alloc(&n8, static_cast<size_t>(shadow_rows_padded(ncap)) * kD);
    if (rc == B2F_OK) rc = dev_alloc(&nts, static_cast<size_t>(shadow_rows_padded(ncap) / kShadowTileRows + 16));
  }
  if (rc == B2F_OK && S.has_ids) rc = dev_alloc(&nid, static_cast<size_t>(ncap));
  if (rc != B2F_OK) { dev_free(n32); dev_free(n16); dev_free(n8); dev_free(nts); return rc; }
  if (S.n > 0) {
    CU_TRY(cudaMemcpyAsync(n32, S.x32, static_cast<size_t>(S.n) * kD * 4, cudaMemcpyDeviceToDevice, S.stream));
    if (n16 && S.x16)
      CU_TRY(cudaMemcpyAsync(n16, S.x16, static_cast<size_t>(shadow_rows_padded(S.n)) * kD * 2,
                             cudaMemcpyDeviceToDevice, S.stream));  // tiles are stored in row order
    if (n8 && S.x8) {
      CU_TRY(cudaMemcpyAsync(n8, S.x8, static_cast<size_t>(shadow_rows_padded(S.n)) * kD, cudaMemcpyDeviceToDevice, S.stream));
      CU_TRY(cudaMemcpyAsync(nts, S.tscale, static_cast<size_t>(shadow_rows_padded(S.n) / kShadowTileRows) * sizeof(float4),
                             cudaMemcpyDeviceToDevice, S.stream));
    }
    if (nid && S.idmap)
      CU_TRY(cudaMemcpyAsync(nid, S.idmap, static_cast<size_t>(S.n) * 8, cudaMemcpyDeviceToDevice, S.stream));
    CU_TRY(cudaStreamSynchronize(S.stream));
  }
  dev_free(S.x32); dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale); dev_free(S.idmap);
  S.x32 = n32; S.x16 = n16; S.x8 = n8; S.tscale = nts; S.idmap = nid; S.cap = ncap;
  return B2F_OK;
}

int upload_segs(Shard& S) {
  if (!S.segs_dirty) return B2F_OK;   // one small H2D copy less on the stream of every search
  S.segs_dirty = false;
  const int n = static_cast<int>(S.segs.size());
  if (n > S.segs_d_cap) {
    dev_free(S.segs_d);
    S.segs_d_cap = std::max(16, 2 * n);
    B2F_TRY(dev_alloc(&S.segs_d, static_cast<size_t>(S.segs_d_cap)));
  }
  if (n) CU_TRY(cudaMemcpyAsync(S.segs_d, S.segs.data(), sizeof(Seg) * n, cudaMemcpyHostToDevice, S.stream));
  return B2F_OK;
}

void push_seg(Shard& S, int64_t local_start, int64_t count, int64_t global_start) {
  S.segs_dirty = true;
  if (!S.segs.empty()) {
    Seg& b = S.segs.back();
    if (b.local_start + b.count == local_start && b.global_start + b.count == global_start) {
      b.count += count;
      return;
    }
  }
  S.segs.push_back(Seg{local_start, count, global_start});
}

int launch_grid_rows(const Shard& S, int64_t rows) {
  int64_t blocks = (rows + 7) / 8;  // 8 warps per 256-thread block, one row per warp iteration
  return static_cast<int>(std::min<int64_t>(std::max<int64_t>(blocks, 1), static_cast<int64_t>(S.sm_count) * 8));
}

bool has_shadow(const Shard& S) { return S.x16 != nullptr || S.x8 != nullptr; }

// AUTO format choice at the first ingest of a shard (DESIGN.md section 4): 64 evenly spaced rows among the first
// m <= 65,536 act as pseudo-queries; with sigma_j the spread of their centred scores over 4096 sample rows and
// eps8_j the int8 margin from the sample's own bounds (int8 tiles of the first m rows, not stored), int8 is chosen
// when the median of 2 eps8_j / sigma_j is <= 1.2 (tools/margin_model.py: ~0.8 for isotropic rows, ~1.9 for rows
// with a common mean, where the int8 margin would let tens of thousands of rows per query through).  Fewer than
// 4096 rows or no spread (all-equal rows): bf16.  Only speed depends on this choice, never the results.
int choose_format(Shard& S, int64_t n, int* fmt) {
  const int64_t m = std::min<int64_t>(n, kMuRows);
  S.rho = 0;
  *fmt = kShadowBf16;
  if (m < 4096) return B2F_OK;
  constexpr int kProbeQ = 64, kProbeRows = 4096;
  // scratch: the partial column sums of the centre are consumed by now (stream order)
  unsigned char* scratch = reinterpret_cast<unsigned char*>(S.mu_part);
  unsigned int* bounds = reinterpret_cast<unsigned int*>(scratch);
  double* stat = reinterpret_cast<double*>(scratch + 64);
  float* qstat = reinterpret_cast<float*>(scratch + 64 + 16 * kProbeQ);
  CU_TRY(cudaMemsetAsync(scratch, 0, 64 + 24 * kProbeQ, S.stream));
  convert_rows_i8_kernel<<<launch_grid_rows(S, m / kShadowTileRows), 256, 0, S.stream>>>(S.x32, nullptr, nullptr, 0, m,
                                                                                              bounds, S.mu);
  shadow_probe_kernel<<<dim3(16, kProbeQ), 256, 0, S.stream>>>(S.x32, m, kProbeRows, S.mu, stat, qstat);
  CU_TRY(cudaGetLastError());
  unsigned char host[64 + 24 * kProbeQ];
  CU_TRY(cudaMemcpyAsync(host, scratch, sizeof(host), cudaMemcpyDeviceToHost, S.stream));
  CU_TRY(cudaStreamSynchronize(S.stream));
  unsigned int hb[3];
  std::memcpy(hb, host, sizeof(hb));
  auto bits2f = [](unsigned int u) { float f; std::memcpy(&f, &u, 4); return static_cast<double>(f); };
  const double E8 = std::sqrt(bits2f(hb[1])), P = std::sqrt(bits2f(hb[2]));
  std::vector<double> rho(kProbeQ);
  for (int j = 0; j < kProbeQ; ++j) {
    double s1, s2;
    float qn, qe;
    std::memcpy(&s1, host + 64 + 16 * j, 8);
    std::memcpy(&s2, host + 64 + 16 * j + 8, 8);
    std::memcpy(&qn, host + 64 + 16 * kProbeQ + 8 * j, 4);
    std::memcpy(&qe, host + 64 + 16 * kProbeQ + 8 * j + 4, 4);
    const double mean = s1 / kProbeRows, var = std::max(0.0, s2 / kProbeRows - mean * mean);
    const double eps = (qn + qe) * E8 + qe * P;
    rho[j] = var > 0 ? 2 * eps / std::sqrt(var) : HUGE_VAL;
  }
  std::nth_element(rho.begin(), rho.begin() + kProbeQ / 2, rho.end());
  S.rho = rho[kProbeQ / 2];
  if (std::isfinite(S.rho) && S.rho <= 1.2) *fmt = kShadowInt8;
  return B2F_OK;
}

// Append rows already resident at x32[S.n .. S.n+n): build shadow + norm bound.
int ingest_rows(b2f_index* idx, Shard& S, int64_t n) {
  if (!S.mu_set) {
    // First rows of an empty shard: fix the centre.  Any vector is a valid centre (correctness never depends
    // on it); the mean of the first rows is what shrinks ||p - mu|| — and with it the prefilter margin — for
    // embeddings that share a large common component (LayerNorm outputs; reference model/models.py:136-145).
    if (idx->center && idx->shadow && S.n == 0) {
      const int64_t m = std::min<int64_t>(n, kMuRows);
      const int blocks = static_cast<int>(std::min<int64_t>(m, kMuBlocks));
      col_sum_partial_kernel<<<blocks, kRowF4, 0, S.stream>>>(S.x32, 0, m, S.mu_part);
      col_mean_final_kernel<<<(kD + 255) / 256, 256, 0, S.stream>>>(S.mu_part, blocks, m, S.mu);
      CU_TRY(cudaGetLastError());
    }
    if (S.n == 0) {
      // the shadow format of these rows (AUTO: from the rows themselves); buffers of another format are replaced
      int fmt = idx->shadow;
      if (fmt == kShadowAuto) B2F_TRY(choose_format(S, n, &fmt));
      if (fmt != S.fmt || (fmt == kShadowBf16 && !S.x16) || (fmt == kShadowInt8 && !S.x8)) {
        dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale);
        S.fmt = fmt;
        if (fmt == kShadowBf16) B2F_TRY(dev_alloc(&S.x16, static_cast<size_t>(shadow_rows_padded(S.cap)) * kD));
        if (fmt == kShadowInt8) {
          B2F_TRY(dev_alloc(&S.x8, static_cast<size_t>(shadow_rows_padded(S.cap)) * kD));
          B2F_TRY(dev_alloc(&S.tscale, static_cast<size_t>(shadow_rows_padded(S.cap) / kShadowTileRows + 16)));
        }
      }
    }
    S.mu_set = true;
  }
  if (S.fmt == kShadowInt8) {
    const int64_t tiles = (S.n + n + kShadowTileRows - 1) / kShadowTileRows - S.n / kShadowTileRows;
    convert_rows_i8_kernel<<<launch_grid_rows(S, tiles), 256, 0, S.stream>>>(S.x32, S.x8, S.tscale, S.n, n,
                                                                                S.maxnorm2, S.mu);
  } else {
    convert_rows_kernel<<<launch_grid_rows(S, n), 256, 0, S.stream>>>(S.x32, S.x16, S.n, n, S.maxnorm2, S.mu);
  }
  CU_TRY(cudaGetLastError());
  return B2F_OK;
}

int ensure_query_ws(Shard& S, int64_t nq, int k) {
  Workspace& W = S.ws;
  if (nq > W.nq_cap) {
    dev_free(W.q32); dev_free(W.q16); dev_free(W.qnorm); dev_free(W.qerr); dev_free(W.qscale);
    if (W.ovf_host) { cudaFreeHost(W.ovf_host); W.ovf_host = nullptr; W.ovf_all = nullptr; }
    const int64_t cap = std::max<int64_t>(nq, 256);
    B2F_TRY(dev_alloc(&W.q32, static_cast<size_t>(cap) * kD));
    B2F_TRY(dev_alloc(&W.q16, static_cast<size_t>(cap + kUmmaMaxQ + 16) * kD));
    B2F_TRY(dev_alloc(&W.qnorm, static_cast<size_t>(cap + kUmmaMaxQ + 16)));
    B2F_TRY(dev_alloc(&W.qerr, static_cast<size_t>(cap + kUmmaMaxQ + 16)));
    B2F_TRY(dev_alloc(&W.qscale, static_cast<size_t>(cap + kUmmaMaxQ + 16)));
    // per-query overflow flags live in mapped pinned host memory: the last kernel of a pass writes them
    // straight to the host (no copy operation on the stream), the host reads them after the sync
    CU_TRY(cudaHostAlloc(reinterpret_cast<void**>(&W.ovf_host), static_cast<size_t>(cap) * kMaxPending * sizeof(int),
                         cudaHostAllocMapped));
    CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&W.ovf_all), W.ovf_host, 0));
    W.nq_cap = cap;
  }
  const int64_t need_out = nq * k;
  if (need_out > W.out_cap) {
    dev_free(W.D); dev_free(W.I);
    B2F_TRY(dev_alloc(&W.D, static_cast<size_t>(need_out)));
    B2F_TRY(dev_alloc(&W.I, static_cast<size_t>(need_out)));
    W.out_cap = need_out;
  }
  if (!W.fbq) {
    B2F_TRY(dev_alloc(&W.fbq, static_cast<size_t>(kScanMaxQ) * kD));
    B2F_TRY(dev_alloc(&W.fbD, static_cast<size_t>(kScanMaxQ) * B2F_MAX_K));
    B2F_TRY(dev_alloc(&W.fbI, static_cast<size_t>(kScanMaxQ) * B2F_MAX_K));
  }
  return B2F_OK;
}

int ensure_pass_ws(Shard& S, int qp, int C) {
  Workspace& W = S.ws;
  if (qp <= W.qp_cap && C <= W.C) return B2F_OK;
  qp = std::max(qp, W.qp_cap);
  C = std::max(C, W.C);
  dev_free(W.cand[0]); dev_free(W.cand[1]); dev_free(W.cnt); dev_free(W.tau); dev_free(W.tauP);
  dev_free(W.ovf); dev_free(W.margin); dev_free(W.gath); dev_free(W.cnt2);
  dev_free(W.hist); dev_free(W.hkey0); dev_free(W.hshift);
  B2F_TRY(dev_alloc(&W.gath, static_cast<size_t>(qp) * C));
  B2F_TRY(dev_alloc(&W.cnt2, static_cast<size_t>(qp) * 256));   // per (query, area): <= 128 pairs / 256 CTAs
  B2F_TRY(dev_alloc(&W.hist, static_cast<size_t>(qp) * kHistStride));
  B2F_TRY(dev_alloc(&W.hkey0, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.hshift, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.cand[0], static_cast<size_t>(qp) * C));
  B2F_TRY(dev_alloc(&W.cand[1], static_cast<size_t>(qp) * C));
  B2F_TRY(dev_alloc(&W.cnt, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.tau, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.tauP, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.ovf, static_cast<size_t>(qp)));
  B2F_TRY(dev_alloc(&W.margin, static_cast<size_t>(qp)));
  if (!W.err) {
    B2F_TRY(dev_alloc(&W.err, 1));
    CU_TRY(cudaMemsetAsync(W.err, 0, sizeof(int), S.stream));
  }
  W.qp_cap = qp;
  W.C = C;
  W.areas_clean = false;
  return B2F_OK;
}

int ensure_pin(Shard& S, size_t bytes) {
  Workspace& W = S.ws;
  if (bytes <= W.pin_bytes) return B2F_OK;
  if (W.pin) cudaFreeHost(W.pin);
  W.pin = nullptr;
  W.pin_bytes = 0;
  CU_TRY(cudaMallocHost(&W.pin, bytes));
  W.pin_bytes = bytes;
  return B2F_OK;
}

// Start of a pass, one block per query: the prefilter margin 2*eps_q = 2u * ||q|| * max||p|| (rounded
// up) and the zeroing of the pass state (one launch instead of three memsets and a kernel).
//   mode 0 (exact engine): margin 0.
//   mode 1 (fp32 scan):    eps = u_scan * ||q|| * P,  P = max ||p||   (Cauchy-Schwarz on sum |q_t p_t|).
//   mode 2 (bf16 tensor):  s~ = fl(sum q^_t p^_t) with q^ = bf16(q), p^ = bf16(p).  Then
//       |s~ - s| <= |sum q^ (p^ - p)| + |sum (q^ - q) p| + accumulation
//                <= (1 + 2^-8) ||q|| E + e_q P + g ||q|| P,
//     where p stands for the centred row p - mu and p^ for its bf16 shadow,
//     E = max ||p - p^|| and P = max ||p|| (kept per shard at add time), e_q = ||q - q^||, g = 1.1e-4 >= 768 * 2^-23
//     (fp32 accumulation of 768 exact products inside the tensor core, truncation allowed).
//   mode 4 (int8 tensor):  q^ = sq q8, p^ = st p8 (real products of the fp32 scales and the int8 codes); the tensor
//     core sums the 768 code products exactly in int32, so s~ = q^ . p^ exactly and
//       |s~ - s| <= |q^ . (p^ - p)| + |(q^ - q) . p| <= (||q|| + e_q) E8 + e_q P,
//     with E8 = max ||p - p^|| (slot [1] of an int8 shard, kept at add time), e_q = ||q - q^||, ||q^|| <= ||q|| + e_q.
//     No accumulation term.  What is compared and recorded are fp32 images of s~: the threshold test never rejects
//     a row with s~ >= tau (i8_threshold), the recorded score fl(fl(acc) fl(sq st)) is within 2^-23 |s~| of s~, and
//     |s~| <= ||q^|| ||p^|| <= (||q|| + e_q)(P + E8): the term 2^-21 (||q|| + e_q)(P + E8) covers it 4x over.
// Every factor is an upper bound and every operation rounds up; `scale` (margin_ppm) multiplies the result.
// Outside the normal fp32 range (DESIGN.md section 4):
//   - a product of bounds with a zero factor is an exactly-zero term (bound_mul): a zero bound means a zero vector,
//     so 0 * inf must not turn the margin into NaN;
//   - the relative bounds above assume normal arithmetic.  With subnormal values each fp32 rounding (scan FMA
//     chain, tensor-core accumulation) may add up to 2^-126 of absolute error, a flushed tensor-core product less
//     than 2^-126, and the recorded int8 score fl(acc) fl(sq st) less than 2^24 * 2^-150 + 2^-150 when the scale
//     product is subnormal.  At most 768 products and 768 additions: < 1536 * 2^-126 < 2^-115, added in every mode;
//   - a query whose margin or histogram top R is not finite (a norm bound overflowed) is flagged here and re-run
//     by the exact engine, like an overflowed list; it is never filtered with a NaN threshold.
__device__ __forceinline__ float bound_mul(float a, float b) { return (a == 0.f || b == 0.f) ? 0.f : __fmul_ru(a, b); }
constexpr float kSubnormalAbs = 0x1p-115f;

__global__ void pass_init_kernel(const float* __restrict__ qnorm, const float* __restrict__ qerr,
                                 const unsigned int* __restrict__ maxnorm2_bits, int mode, float scale, float u_scan,
                                 float* __restrict__ margin, int* __restrict__ cnt,
                                 int* __restrict__ ovf, int* __restrict__ cnt2, int max_pairs,
                                 unsigned int* __restrict__ hist, uint32_t* __restrict__ hkey0, int* __restrict__ hshift,
                                 float* __restrict__ tau) {
  const int q = blockIdx.x;
  bool finite = true;
  if (hist != nullptr) {
    // TS engine without a bootstrap launch: empty tightening histogram of 64 buckets per binade over
    // the eight binades below R = (1 + 2^-6) * ||q|| * max||p|| >= |any prefilter score of q|; tau = -inf.
    for (int b = threadIdx.x; b < kHistStride; b += blockDim.x) hist[static_cast<int64_t>(q) * kHistStride + b] = 0u;
    if (threadIdx.x == 0) {
      const float R = __fmul_ru(bound_mul(qnorm[q], __fsqrt_ru(__uint_as_float(maxnorm2_bits[2]))), 1.015625f);
      finite = isfinite(R);
      const uint32_t top = fkey(finite ? R : FLT_MAX) >> 17;
      hkey0[q] = (top >= static_cast<uint32_t>(kHistBuckets - 1) ? top - (kHistBuckets - 1) : 0u) << 17;
      hshift[q] = 17;
    }
  }
  if (threadIdx.x == 0) {
    // Every pass starts without a threshold: finalize_kernel filters on tau[q] whenever tightening is on,
    // and a pass that ends inside the dense phase (shard smaller than the bootstrap) never writes it.
    tau[q] = -INFINITY;
    // tensor engine: scores are taken against the CENTRED rows p - mu (constant shift q.mu per query), so its
    // bounds use Pc = max ||p - mu||; the fp32 scan reads the rows themselves: P = max ||p||
    const float P = __fsqrt_ru(__uint_as_float(maxnorm2_bits[mode == 1 ? 0 : 2]));
    const float qn = qnorm[q], qe = qerr[q];
    float eps = 0.f;
    if (mode == 1) {
      eps = bound_mul(bound_mul(qn, P), u_scan);
    } else if (mode == 3) {   // data-independent worst case (A/B reference for mode 2): bf16 round-to-nearest has
      // unit roundoff 2^-8, so E <= 2^-8 P, ||q^|| <= (1 + 2^-8) ||q||, e_q <= 2^-8 ||q||:
      // 2^-8 (1 + 2^-8) + 2^-8 + 1.1e-4 < 0.007954
      eps = bound_mul(bound_mul(qn, P), 0.007954f);
    } else if (mode == 2) {
      const float E = __fsqrt_ru(__uint_as_float(maxnorm2_bits[1]));
      const float a = bound_mul(bound_mul(qn, E), 1.00390625f);   // ||bf16(q)|| <= (1 + 2^-8) ||q||
      const float b = bound_mul(qe, P);
      const float c = bound_mul(bound_mul(qn, P), 1.1e-4f);
      eps = __fadd_ru(__fadd_ru(a, b), c);
    } else if (mode == 4) {
      const float E = __fsqrt_ru(__uint_as_float(maxnorm2_bits[1]));
      const float qh = __fadd_ru(qn, qe);
      const float a = bound_mul(qh, E);
      const float b = bound_mul(qe, P);
      const float c = bound_mul(bound_mul(qh, __fadd_ru(P, E)), 4.76837158203125e-7f);   // 2^-21
      eps = __fadd_ru(__fadd_ru(a, b), c);
    }
    if (mode != 0) eps = __fadd_ru(eps, kSubnormalAbs);
    const float m = __fmul_ru(__fmul_ru(eps, 2.0f), scale);
    const bool fallback = mode != 0 && !(finite && isfinite(m));
    margin[q] = fallback ? FLT_MAX : m;
    cnt[q] = 0;
    ovf[q] = fallback ? 1 : 0;
  }
  if (cnt2 != nullptr)
    for (int p = threadIdx.x; p < max_pairs; p += blockDim.x) cnt2[q * max_pairs + p] = 0;
}

__global__ void fill_pad_kernel(float* D, int64_t* I, int64_t n) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) { D[i] = -FLT_MAX; I[i] = -1; }
}

struct ProfScope {
  Prof* p;
  cudaStream_t s;
  size_t b = 0;
  int kind;
  ProfScope(b2f_index* idx, Shard& S, int kind_) : p(idx->profile ? &S.prof : nullptr), s(S.stream), kind(kind_) {
    if (p) { b = p->used; cudaEventRecord(p->get(), s); }
  }
  ~ProfScope() {
    if (p) { size_t e = p->used; cudaEventRecord(p->get(), s); p->spans.push_back({kind, b, e}); }
  }
};

void collect_prof(b2f_index* idx, Shard& S) {
  Prof& P = S.prof;
  for (const Prof::Span& sp : P.spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, P.pool[sp.b], P.pool[sp.e]) == cudaSuccess) {
      if (sp.kind == 0) { S.stats.score_ms += ms; S.stats.score_launches += 1; }
      else if (sp.kind == 2) S.stats.xchg_ms += ms;
      else S.stats.select_ms += ms;
    } else {
      (void)cudaGetLastError();
    }
  }
  P.spans.clear();
  P.used = 0;
}

// Rigorous error bounds of the prefilter scores (see pass_init_kernel for the bf16 tensor engine,
// whose bound is data-dependent: max ||p - bf16(p)|| is kept per shard at add time):
//   fp32 scan  : 24 sequential fma + 5 tree adds, one rounding each -> 29 * 2^-24 < 2^-19, relative to
//                ||q|| * ||p|| (Cauchy-Schwarz on sum |q_t p_t|)
constexpr double kUScan = 1.9073486328125e-06;

struct PassPlan {
  int path;     // resolved engine
  bool exact;   // total-order keys, zero margin, bounded phases
  int qp;       // max queries per pass
  int C;        // candidate capacity per query
  int64_t n0;   // rows of the dense (bootstrap) phase
  int S;        // tensor engine: survivor area [0, S) of a list
  int cap_p;    // TS variant: private slots per (query, CTA pair) and launch
  int cap_a;    // QS variant: private slots per (query, CTA)
  int variant;  // tensor engine variant: 0 = per pass (QS up to qs_max_q queries, TS above), 2 = TS, 3 = QS
};

PassPlan make_plan(const b2f_index* idx, const Shard& S, int path, int k, int64_t nq) {
  PassPlan p;
  p.path = path;
  p.exact = (path == B2F_PATH_SCAN_EXACT);
  p.S = 0;
  p.cap_p = 0;
  p.cap_a = 0;
  p.variant = 0;
  (void)nq;
  if (path == B2F_PATH_UMMA_BF16) {
    // Two kernels share one list layout (survivors [0,S) + private areas).  TS: queries in TMEM, MMA M is
    // always 256 query lanes, 256 queries per pass, areas per CTA pair.  QS: queries on the MMA N side
    // (N = nq rounded up to 16), streamed from L2 next to the passages, areas per CTA.  AUTO decides per
    // pass: QS while the batch leaves lanes unused in TS (profiles/r02: 173 queries -> N = 176, 31 % fewer
    // tensor cycles), TS for (nearly) full passes.
    p.variant = idx->umma_variant == 1 ? 3 : idx->umma_variant;
    p.qp = kUmmaMaxQ;
    // bootstrap (dense) phase of the phased TS schedules: whole tiles per CTA pair, at least 8k rows
    const int64_t wave = static_cast<int64_t>(S.max_pairs) * kTileRows;
    const int64_t t0 = (std::max<int64_t>(4096, 8ll * k) + wave - 1) / wave;
    p.n0 = t0 * wave;
    // survivors within the margin of the k-th score: ~k * (e^(z * 2eps / sigma) - 1) with z ~ 5 the tail slope
    // at rank 100 of 4e7: ~200 for isotropic unit rows, ~700 for LayerNorm-like rows with a common mean after
    // centring (DESIGN.md section 4) — 4096 leaves a factor of 5
    // int8 shadow: a margin ~4x wider (2 eps / sigma ~0.8 instead of ~0.2 on isotropic rows): the rescoring
    // window holds ~650 rows per query at k = 100 and ~4.5k at k = 1000 on 8.8 M rows, so S follows 8k (up to the
    // 8192 records finalize_kernel keeps in shared memory)
    const int s_k = S.fmt == kShadowInt8 ? std::max(4 * k, std::min(8 * k, 8192)) : 4 * k;
    p.S = static_cast<int>(round_up(std::max(4096, s_k), 256));
    // expected appends per (query, area) in a phase: 2 (margin) * (growth-1) * k / areas; x2 safety
    // (with in-kernel tightening the pass rate follows k/rows_seen, far fewer appends; keep the bound)
    const int64_t expect = 4ll * (std::max(2, idx->growth) - 1) * k / S.max_pairs;
    p.cap_p = static_cast<int>(round_up(std::max<int64_t>(std::max<int64_t>(512, t0 * kTileRows), expect), 64));   // per pair; half per (pair, half tile)
    p.cap_a = static_cast<int>(round_up(std::max<int64_t>(512, kQsTileRowsCta + expect / 2), 32));
    p.C = p.S + std::max(S.max_pairs * p.cap_p, 2 * S.max_pairs * p.cap_a);
  } else {
    p.qp = kScanMaxQ;
    p.n0 = 16384;
    // a phase of `growth` times the rows seen so far passes ~growth * k rows (plus the margin's share)
    p.C = static_cast<int>(round_up(std::max<int64_t>(p.n0, (std::max(2, idx->growth) + 4ll) * k * 5 / 4), 256));
  }
  return p;
}

// Which tensor kernel runs a pass of nqp queries.
int pass_variant(const b2f_index* idx, const PassPlan& plan, int nqp) {
  if (plan.variant == 2 || plan.variant == 3) return plan.variant;
  if (!idx->tighten || idx->bootstrap) return 2;      // the phased schedules exist for TS only
  return nqp <= idx->qs_max_q ? 3 : 2;
}

// Enqueue one pass (<= plan.qp queries) on the shard stream.  q32p: the pass's fp32 queries
// [nqp,768]; q16p: their bf16 copies padded with zero rows (tensor path).  Results go to
// D_out/I_out with row stride out_stride.
int enqueue_pass(b2f_index* idx, Shard& S, const PassPlan& plan, const float* q32p, const __nv_bfloat16* q16p,
                 const float* qnormp, const float* qerrp, int nqp, int k, float* D_out, int64_t* I_out, int64_t out_stride,
                 int* ovf_dst, const float* qscalep, const SelShard* sel) {
  Workspace& W = S.ws;
  Stats& st = S.stats;   // per shard: shards may be enqueued from different host threads
  const int64_t N = S.n;
  const int C = W.C;
  cudaStream_t s = S.stream;
  const int variant = plan.path == B2F_PATH_UMMA_BF16 ? pass_variant(idx, plan, nqp) : 0;
  const bool tensor = variant == 2;      // TS: queries in TMEM, areas per CTA pair
  const bool tensor_qs = variant == 3;   // QS: queries streamed on the N side, areas per CTA
  const bool one_launch = tensor_qs || (tensor && idx->tighten && !idx->bootstrap);   // ONE scoring launch per pass
  if (tensor && !one_launch) {
    if (!W.areas_clean) {   // phased TS schedules gather whole areas: they must be all-zero between launches
      CU_TRY(cudaMemsetAsync(W.cand[0], 0, sizeof(uint64_t) * static_cast<size_t>(W.qp_cap) * W.C, s));
      CU_TRY(cudaMemsetAsync(W.cand[1], 0, sizeof(uint64_t) * static_cast<size_t>(W.qp_cap) * W.C, s));
      W.areas_clean = true;
    }
  } else {
    W.areas_clean = false;  // flat lists / one-launch passes leave records behind in the areas
  }
  const int n_areas = 2 * S.max_pairs;   // TS: two per CTA pair (one per half tile); QS: one per CTA
  const int cap_h = plan.cap_p / 2;       // TS: slots per (query, pair, half tile)
  const bool i8 = S.fmt == kShadowInt8;
  const int margin_mode = plan.exact ? 0 : (plan.path == B2F_PATH_UMMA_BF16 ? (i8 ? 4 : (idx->worst_case_margin ? 3 : 2)) : 1);
  pass_init_kernel<<<nqp, 128, 0, s>>>(qnormp, qerrp, S.maxnorm2, margin_mode,
                                       static_cast<float>(idx->margin_ppm * 1e-6 * 1.0000001), static_cast<float>(kUScan),
                                       W.margin, W.cnt, W.ovf, (tensor || tensor_qs) ? W.cnt2 : nullptr, n_areas,
                                       one_launch ? W.hist : nullptr, W.hkey0, W.hshift, W.tau);
  st.launches += 1;

  if (tensor_qs) {
    // ---- QS: one launch over the whole shard, then the fused last step ----
    const int n_cols = static_cast<int>(round_up(nqp, 16));
    // int8: 6 K-blocks of 128 bytes; the tensor maps only move bytes, so they describe the int8 rows as bf16 pairs
    const int n_kb = i8 ? kShadow8KBlocks : kNumKBlocks;
    const QsPlan qp = umma_qs_plan(n_cols, idx->umma_variant == 1 ? n_kb : std::min(idx->qs_resident_kb * n_kb / kNumKBlocks, n_kb),
                                   idx->qs_q_stages, i8 ? 0 : idx->qs_half_stage, n_kb);
    CUtensorMap tmap_p, tmap_ph, tmap_q;
    const void* shadow = i8 ? static_cast<const void*>(S.x8) : static_cast<const void*>(S.x16);
    const uint64_t srows = static_cast<uint64_t>(shadow_rows_padded(N)) * n_kb;
    B2F_TRY(make_tmap_bf16(&tmap_p, shadow, srows, kBlockK, kShadowTileRows));        // one K-block of a 32-row tile
    B2F_TRY(make_tmap_bf16(&tmap_ph, shadow, srows, kBlockK, kShadowTileRows, true)); // half a K-block of a 32-row tile
    B2F_TRY(make_tmap_bf16(&tmap_q, q16p, static_cast<uint64_t>(n_cols), i8 ? kD / 2 : kD, static_cast<uint32_t>(n_cols / 2)));
    // filtered: the launch walks the listed tiles only
    const int te = sel ? sel->n_qs : static_cast<int>((N + kQsTileRows - 1) / kQsTileRows);
    UmmaQsArgs a;
    a.sel_bits = sel ? sel->bits : nullptr; a.tile_list = sel ? sel->qs_tiles : nullptr;
    a.n_rows = N; a.tile_begin = 0; a.tile_end = te; a.n_cols = n_cols; a.nq = nqp;
    a.a_stages = qp.a_stages; a.q_stages = qp.q_stages; a.resident_kb = qp.resident_kb; a.q16 = q16p;
    a.half_stage = qp.half_stage;
    a.cand = W.cand[0]; a.C = C; a.S = plan.S; a.cap_p = plan.cap_a; a.n_areas = n_areas; a.cnt2 = W.cnt2;
    a.tau = W.tau; a.ovf = W.ovf; a.err = W.err; a.tighten = idx->tighten; a.tighten_adaptive = idx->tighten_adaptive;
    a.k = k; a.margin = W.margin; a.hist = W.hist; a.hkey0 = W.hkey0; a.hshift = W.hshift;
    const int pairs = std::min(S.max_pairs, te);
    // First tile of every CTA: `dense_quarters` of its four 32-row quarters pass unfiltered (they seed the
    // histogram: 2 * pairs * 32 rows per quarter, about half of which score above the histogram floor), the
    // other quarters wait until every query has a threshold (bounded: first_wait_cycles).  Shards too small
    // to fill the first tiles do not wait.
    a.x16_bytes = static_cast<const unsigned char*>(shadow);
    a.pf_limit_bytes = shadow_rows_padded(N) * static_cast<int64_t>(kD) * (i8 ? 1 : 2);
    a.qscale = qscalep; a.tscale = S.tscale;
    a.prefetch = sel ? 0 : idx->l2_prefetch;
    if (!sel) {
      a.dense_quarters = std::min(4, std::max(1, (4 * k + 2 * pairs * 32 - 1) / (2 * pairs * 32)));
      a.first_wait_cycles = (idx->tighten && N >= 4ll * pairs * kQsTileRows && a.dense_quarters < 4) ? 100000 : 0;
    } else {
      // the same protocol on the selected rows: a quarter of the first listed tiles holds about `density` x 32 of them
      const double rows_q = 2.0 * pairs * 32 * static_cast<double>(sel->count) / (static_cast<double>(te) * kQsTileRows);
      a.dense_quarters = static_cast<int>(std::min(4.0, std::max(1.0, std::ceil(4.0 * k / rows_q))));
      a.first_wait_cycles = (idx->tighten && te >= 4 * pairs && a.dense_quarters < 4) ? 100000 : 0;
    }
    {
      ProfScope ps(idx, S, 0);
      const dim3 g(2 * pairs);
      if (sel) {
        if (i8) umma_qs_score_select_kernel<true, true><<<g, kQsThreads, qp.smem_bytes, s>>>(tmap_p, tmap_ph, tmap_q, a);
        else umma_qs_score_select_kernel<false, true><<<g, kQsThreads, qp.smem_bytes, s>>>(tmap_p, tmap_ph, tmap_q, a);
      } else {
        if (i8) umma_qs_score_select_kernel<true, false><<<g, kQsThreads, qp.smem_bytes, s>>>(tmap_p, tmap_ph, tmap_q, a);
        else umma_qs_score_select_kernel<false, false><<<g, kQsThreads, qp.smem_bytes, s>>>(tmap_p, tmap_ph, tmap_q, a);
      }
    }
    CU_TRY(cudaGetLastError());
    st.score_rows += sel ? static_cast<double>(te) * kQsTileRows : static_cast<double>(N);
    st.launches += 1;
    st.phases += 1;
    st.qs_passes += 1;
    ProfScope ps(idx, S, 1);
    int PS = 1024;
    while (PS < plan.S) PS <<= 1;
    int P = 8192;
    while (P < PS) P <<= 1;
    finalize_kernel<<<nqp, kFinThreads, static_cast<size_t>(P + PS) * sizeof(uint64_t), s>>>(
        W.cand[0], W.gath, W.cnt, C, k, W.margin, plan.S, plan.cap_a, n_areas, W.cnt2, W.ovf, ovf_dst, q32p,
        S.x32, S.segs_d, static_cast<int>(S.segs.size()), S.has_ids ? S.idmap : nullptr, D_out, I_out, out_stride, P,
        W.tau, S.mu);
    CU_TRY(cudaGetLastError());
    st.launches += 1;
    st.passes += 1;
    return B2F_OK;
  }

  int cur = 0;
  CUtensorMap tmap_p;
  if (tensor) {
    // shadow = [row tiles x 12 K-blocks x tile rows, 64 columns] bf16; box = 128 x 128 B = 16 KB
    // (int8: 6 K-blocks of 128 bytes per tile, boxes of 3 K-blocks = 12 KB)
    if (i8) B2F_TRY(make_tmap_bf16(&tmap_p, S.x8, static_cast<uint64_t>(shadow_rows_padded(N)) * kShadow8KBlocks, kBlockK,
                                   3 * kTileRowsCta));
    else B2F_TRY(make_tmap_bf16(&tmap_p, S.x16, static_cast<uint64_t>(shadow_rows_padded(N)) * kNumKBlocks, kBlockK,
                                kKBlocksPerStage * kTileRowsCta));
  }

  // Phase boundaries in rows.  Dense phase first, then geometric growth (or, in exact mode,
  // fixed-size phases that cannot overflow the candidate capacity even if every row passes).
  int64_t begin = 0;
  int phase = 0;
  while (begin < N) {
    int64_t end;
    const bool dense = (phase == 0) && !one_launch;
    if (one_launch) end = N;
    else if (dense) end = std::min<int64_t>(N, plan.n0);
    else if (plan.exact) end = std::min<int64_t>(N, begin + (C - k));
    else if (tensor && idx->tighten) end = N;   // thresholds are tightened inside the kernel
    else end = std::min<int64_t>(N, begin * std::max(2, idx->growth));
    int n_override = -1;
    if (tensor) {
      const int tb = static_cast<int>(begin / kTileRows);
      const int te = static_cast<int>((end + kTileRows - 1) / kTileRows);
      if (end < N) end = static_cast<int64_t>(te) * kTileRows;  // phases end on tile boundaries
      // filtered: the listed tiles of [tb, te)
      int lb = tb, le = te;
      if (sel) {
        lb = static_cast<int>(std::lower_bound(sel->ts_host.begin(), sel->ts_host.end(), tb) - sel->ts_host.begin());
        le = static_cast<int>(std::lower_bound(sel->ts_host.begin(), sel->ts_host.end(), te) - sel->ts_host.begin());
      }
      UmmaArgs a;
      a.n_rows = N; a.tile_begin = lb; a.tile_end = le; a.nq = nqp; a.q16 = q16p;
      a.sel_bits = sel ? sel->bits : nullptr; a.tile_list = sel ? sel->ts_tiles : nullptr;
      a.qscale = qscalep; a.tscale = S.tscale;
      a.dense = dense ? 1 : 0; a.cand = W.cand[cur]; a.C = C; a.S = plan.S; a.cap_p = cap_h;
      a.max_pairs = n_areas; a.cnt2 = W.cnt2; a.tau = W.tau; a.ovf = W.ovf; a.err = W.err;
      a.tighten = idx->tighten; a.tighten_adaptive = idx->tighten_adaptive; a.k = k; a.margin = W.margin; a.hist = W.hist; a.hkey0 = W.hkey0; a.hshift = W.hshift;
      const int pairs = std::min(S.max_pairs, le - lb);
      // wait for the first thresholds after the first tile: only when that tile's rows can place them (about half of
      // pairs * 64 rows score above the histogram floor) and the shard is long enough to be worth it
      a.count_exact_lower_bound = one_launch ? 1 : 0;
      if (!sel) {
        a.first_wait_cycles = (one_launch && N >= 8ll * pairs * kTileRows && 4ll * k <= static_cast<int64_t>(pairs) * kTileRows) ? 100000 : 0;
      } else {   // the same rule on the selected rows of the listed tiles
        const double density = static_cast<double>(sel->count) / (static_cast<double>(sel->n_ts) * kTileRows);
        a.first_wait_cycles = (one_launch && le - lb >= 8 * pairs && 4.0 * k <= pairs * kTileRows * density) ? 100000 : 0;
      }
      if (pairs > 0) {   // a filtered phase may hold no listed tile
        ProfScope ps(idx, S, 0);
        const dim3 g(2 * pairs);
        if (sel) {
          if (i8) umma_score_select_kernel<true, true><<<g, kUmmaThreads, kUmmaSmemBytes, s>>>(tmap_p, a);
          else umma_score_select_kernel<false, true><<<g, kUmmaThreads, kUmmaSmemBytes, s>>>(tmap_p, a);
        } else {
          if (i8) umma_score_select_kernel<true, false><<<g, kUmmaThreads, kUmmaSmemBytes, s>>>(tmap_p, a);
          else umma_score_select_kernel<false, false><<<g, kUmmaThreads, kUmmaSmemBytes, s>>>(tmap_p, a);
        }
      }
      st.score_rows += sel ? static_cast<double>(le - lb) * kTileRows
                           : static_cast<double>(std::min<int64_t>(N, static_cast<int64_t>(te) * kTileRows) - begin);
    } else {
      ScanArgs a;
      a.x32 = S.x32; a.row_begin = begin; a.row_end = end; a.q32 = q32p; a.nq_pass = nqp;
      a.dense = dense ? 1 : 0; a.dense_row0 = 0; a.cand = W.cand[cur]; a.cnt = W.cnt; a.C = C;
      a.tau = W.tau; a.tauP = W.tauP; a.ovf = W.ovf; a.sel_bits = sel ? sel->bits : nullptr;
      const int64_t groups = (end - begin + kScanRows - 1) / kScanRows;
      const int blocks = static_cast<int>(std::min<int64_t>((groups + 7) / 8, static_cast<int64_t>(S.sm_count)));
      const size_t sm = scan_smem_bytes(nqp, plan.exact);
      {
        ProfScope ps(idx, S, 0);
        const dim3 g(std::max(blocks, 1));
        if (sel) {
          if (plan.exact) scan_kernel<true, true><<<g, kScanThreads, sm, s>>>(a);
          else scan_kernel<false, true><<<g, kScanThreads, sm, s>>>(a);
        } else {
          if (plan.exact) scan_kernel<true, false><<<g, kScanThreads, sm, s>>>(a);
          else scan_kernel<false, false><<<g, kScanThreads, sm, s>>>(a);
        }
      }
      st.score_rows += static_cast<double>(end - begin);
      if (dense) n_override = static_cast<int>(end - begin);
    }
    CU_TRY(cudaGetLastError());
    if (tensor && end >= N) {   // the last refresh of a TS pass is part of finalize_kernel
      st.launches += 1;
      st.phases += 1;
      begin = end;
      ++phase;
      break;
    }
    if (tensor && idx->tighten && phase == 0) {   // TS bootstrap: select in shared memory + histogram seed
      ProfScope ps(idx, S, 1);
      int P = 4096;
      while (P < plan.n0 + plan.S && P < 16384) P <<= 1;   // longer lists are gathered to global memory
      bootstrap_select_kernel<<<nqp, kFinThreads, static_cast<size_t>(P) * sizeof(uint64_t), s>>>(
          W.cand[cur], W.cand[cur ^ 1], W.gath, W.cnt, C, k, W.margin, W.tau, plan.S, cap_h, n_areas, W.cnt2,
          W.ovf, W.hist, W.hkey0, W.hshift, P);
    } else {
      ProfScope ps(idx, S, 1);
      refresh_kernel<<<nqp, kSelThreads, 0, s>>>(W.cand[cur], W.cand[cur ^ 1], W.gath, W.cnt, C, k, plan.exact ? 1 : 0,
                                                W.margin, W.tau, W.tauP, n_override, plan.S, cap_h,
                                                tensor ? n_areas : 0, W.cnt2, W.ovf,
                                                (tensor && idx->tighten && end < N) ? W.hist : nullptr, W.hkey0, W.hshift);
    }
    CU_TRY(cudaGetLastError());
    cur ^= 1;
    st.launches += 2;
    st.phases += 1;
    begin = end;
    ++phase;
  }
  if (tensor) {
    ProfScope ps(idx, S, 1);
    int PS = 1024;                       // survivors (bufB): >= S
    while (PS < plan.S) PS <<= 1;
    int P = 8192;                        // gathered list (bufA); longer lists go through global memory
    while (P < PS) P <<= 1;
    finalize_kernel<<<nqp, kFinThreads, static_cast<size_t>(P + PS) * sizeof(uint64_t), s>>>(
        W.cand[cur], W.gath, W.cnt, C, k, W.margin, plan.S, cap_h, n_areas, W.cnt2, W.ovf, ovf_dst, q32p,
        S.x32, S.segs_d, static_cast<int>(S.segs.size()), S.has_ids ? S.idmap : nullptr, D_out, I_out, out_stride, P,
        idx->tighten ? W.tau : nullptr, S.mu);
    CU_TRY(cudaGetLastError());
    st.launches += 1;
    st.passes += 1;
    return B2F_OK;
  }
  {
    ProfScope ps(idx, S, 1);
    if (!plan.exact) {   // approximate engines: replace the prefilter scores by exact ones first
      rescore_kernel<<<dim3(nqp, kRescoreSplit), kSelThreads, 0, s>>>(W.cand[cur], W.cand[cur ^ 1], W.cnt, C, q32p, S.x32);
      cur ^= 1;
      st.launches += 1;
    }
    final_kernel<<<nqp, kSelThreads, 0, s>>>(W.cand[cur], W.cand[cur ^ 1], W.cnt, C, k, S.segs_d,
                                            static_cast<int>(S.segs.size()), S.has_ids ? S.idmap : nullptr,
                                            D_out, I_out, out_stride, W.ovf);
  }
  CU_TRY(cudaGetLastError());
  st.launches += 1;
  st.passes += 1;
  if (ovf_dst) CU_TRY(cudaMemcpyAsync(ovf_dst, W.ovf, sizeof(int) * nqp, cudaMemcpyDefault, s));
  return B2F_OK;
}

int resolve_path(const b2f_index* idx, const Shard& S, int64_t nq) {
  int path = idx->path;
  if (path == B2F_PATH_AUTO) {
    if (!has_shadow(S)) path = B2F_PATH_SCAN_F32;
    else path = (nq <= idx->scan_max_auto) ? B2F_PATH_SCAN_F32 : B2F_PATH_UMMA_BF16;
  }
  if (path == B2F_PATH_UMMA_BF16 && !has_shadow(S)) path = B2F_PATH_SCAN_F32;
  return path;
}

// Enqueue the whole search of one shard.  q_d: fp32 queries on the shard's device.
// sel: this shard's part of a selector, or null (no filter).
int enqueue_search(b2f_index* idx, Shard& S, const float* q_d, int64_t nq, int k, float* D_d, int64_t* I_d,
                   int slot = 0, const SelShard* sel = nullptr) {
  CU_TRY(cudaSetDevice(S.dev));
  Workspace& W = S.ws;
  cudaStream_t s = S.stream;
  int* ovf_slot_host = W.ovf_host + static_cast<size_t>(slot) * W.nq_cap;
  int* ovf_slot = W.ovf_all + static_cast<size_t>(slot) * W.nq_cap;
  if (S.n == 0 || (sel && sel->count == 0)) {   // nothing to search: padding only
    fill_pad_kernel<<<static_cast<int>((nq * k + 255) / 256), 256, 0, s>>>(D_d, I_d, nq * k);
    CU_TRY(cudaGetLastError());
    std::memset(ovf_slot_host, 0, sizeof(int) * nq);   // no kernel writes the flags of an empty shard
    return B2F_OK;
  }
  const int path = resolve_path(idx, S, nq);
  S.stats.path = path;
  const PassPlan plan = make_plan(idx, S, path, k, nq);
  B2F_TRY(ensure_pass_ws(S, plan.qp, plan.C));
  B2F_TRY(upload_segs(S));
  const int64_t nq_pad = round_up(nq, 16) + kUmmaMaxQ;
  if (S.fmt == kShadowInt8)   // int8 codes in the bf16 query buffer (half its size)
    prep_queries_i8_kernel<<<static_cast<int>((nq_pad * 32 + 127) / 128), 128, 0, s>>>(
        q_d, static_cast<int>(nq), static_cast<int>(nq_pad), reinterpret_cast<int8_t*>(W.q16), W.qscale, W.qnorm, W.qerr);
  else
    prep_queries_kernel<<<static_cast<int>((nq_pad * 32 + 127) / 128), 128, 0, s>>>(
        q_d, static_cast<int>(nq), static_cast<int>(nq_pad), W.q16, W.qnorm, W.qerr);
  CU_TRY(cudaGetLastError());
  S.stats.launches += 1;
  if (plan.path == B2F_PATH_UMMA_BF16) {
    static bool attr_set[64] = {false};
    if (!attr_set[S.dev & 63]) {
      CU_TRY(cudaFuncSetAttribute(umma_score_select_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUmmaSmemBytes));
      CU_TRY(cudaFuncSetAttribute(umma_score_select_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUmmaSmemBytes));
      CU_TRY(cudaFuncSetAttribute(umma_score_select_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUmmaSmemBytes));
      CU_TRY(cudaFuncSetAttribute(umma_score_select_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUmmaSmemBytes));
      CU_TRY(cudaFuncSetAttribute(umma_qs_score_select_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kQsSmemLimit));
      CU_TRY(cudaFuncSetAttribute(umma_qs_score_select_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kQsSmemLimit));
      CU_TRY(cudaFuncSetAttribute(umma_qs_score_select_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kQsSmemLimit));
      CU_TRY(cudaFuncSetAttribute(umma_qs_score_select_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kQsSmemLimit));
      CU_TRY(cudaFuncSetAttribute(finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 8192 * 8));   // P + PS records
      CU_TRY(cudaFuncSetAttribute(bootstrap_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8));
      attr_set[S.dev & 63] = true;
    }
  } else {
    static bool attr_set2[64] = {false};
    if (!attr_set2[S.dev & 63]) {
      CU_TRY(cudaFuncSetAttribute(scan_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
      CU_TRY(cudaFuncSetAttribute(scan_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
      CU_TRY(cudaFuncSetAttribute(scan_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
      CU_TRY(cudaFuncSetAttribute(scan_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
      attr_set2[S.dev & 63] = true;
    }
  }
  for (int64_t q0 = 0; q0 < nq; q0 += plan.qp) {
    const int nqp = static_cast<int>(std::min<int64_t>(plan.qp, nq - q0));
    // the pass's queries: bf16 rows, or int8 rows (half the bytes) in the same buffer
    const __nv_bfloat16* q16p = S.fmt == kShadowInt8 ? reinterpret_cast<const __nv_bfloat16*>(reinterpret_cast<const int8_t*>(W.q16) + q0 * kD)
                                                     : W.q16 + q0 * kD;
    B2F_TRY(enqueue_pass(idx, S, plan, q_d + q0 * kD, q16p, W.qnorm + q0, W.qerr + q0, nqp, k, D_d + q0 * k,
                         I_d + q0 * k, k, ovf_slot + q0, W.qscale + q0, sel));
  }
  return B2F_OK;
}

// After the stream drained: re-run any query whose candidate list overflowed on the exact engine
// (bounded phases, cannot overflow).  Normally a no-op.
int finish_search(b2f_index* idx, Shard& S, const float* q_d, int64_t nq, int k, float* D_d, int64_t* I_d,
                  int slot = 0, bool* reran = nullptr, const SelShard* sel = nullptr) {
  CU_TRY(cudaSetDevice(S.dev));
  CU_TRY(cudaStreamSynchronize(S.stream));
  if (idx->profile) collect_prof(idx, S);
  if (reran) *reran = false;
  if (S.n == 0 || (sel && sel->count == 0)) return B2F_OK;
  Workspace& W = S.ws;
  const int* flags = W.ovf_host + static_cast<size_t>(slot) * W.nq_cap;
  std::vector<int64_t> bad;
  for (int64_t q = 0; q < nq; ++q)
    if (flags[q]) {
      bad.push_back(q);
      if (flags[q] & 1) S.stats.ovf_area += 1;
      if (flags[q] & 2) S.stats.ovf_survivors += 1;
    }
  if (bad.empty()) return B2F_OK;
  if (reran) *reran = true;
  S.stats.fallback_queries += static_cast<double>(bad.size());
  static bool attr_set3[64] = {false};
  if (!attr_set3[S.dev & 63]) {
    CU_TRY(cudaFuncSetAttribute(scan_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
    CU_TRY(cudaFuncSetAttribute(scan_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
    attr_set3[S.dev & 63] = true;
  }
  const PassPlan plan = make_plan(idx, S, B2F_PATH_SCAN_EXACT, k, 0);
  B2F_TRY(ensure_pass_ws(S, plan.qp, plan.C));
  cudaStream_t s = S.stream;
  for (size_t b0 = 0; b0 < bad.size(); b0 += kScanMaxQ) {
    const int nb = static_cast<int>(std::min<size_t>(kScanMaxQ, bad.size() - b0));
    for (int i = 0; i < nb; ++i)   // cudaMemcpyDefault: a multi-shard search re-runs from the first device's queries
      CU_TRY(cudaMemcpyAsync(W.fbq + static_cast<size_t>(i) * kD, q_d + bad[b0 + i] * kD, kD * 4,
                             cudaMemcpyDefault, s));
    B2F_TRY(enqueue_pass(idx, S, plan, W.fbq, nullptr, W.qnorm /*unused: exact*/, W.qerr, nb, k, W.fbD, W.fbI, k, nullptr,
                         nullptr, sel));
    for (int i = 0; i < nb; ++i) {
      // cudaMemcpyDefault: D_d / I_d may be mapped pinned host memory (b2f_search writes results there directly)
      // or a part on the first device
      CU_TRY(cudaMemcpyAsync(D_d + bad[b0 + i] * k, W.fbD + static_cast<size_t>(i) * k, sizeof(float) * k,
                             cudaMemcpyDefault, s));
      CU_TRY(cudaMemcpyAsync(I_d + bad[b0 + i] * k, W.fbI + static_cast<size_t>(i) * k, sizeof(int64_t) * k,
                             cudaMemcpyDefault, s));
    }
  }
  CU_TRY(cudaStreamSynchronize(s));
  if (idx->profile) collect_prof(idx, S);
  return B2F_OK;
}

// Run fn(g) for every shard: shard 0 on the calling thread, the others on their workers.  Returns the
// first failure (its error text becomes this thread's b2f_last_error()).
int run_on_shards(b2f_index* idx, const std::function<int(int)>& fn) {
  const int G = static_cast<int>(idx->shards.size());
  if (G == 1) return fn(0);
  if (idx->workers.empty()) {
    for (int g = 1; g < G; ++g) {
      idx->workers.emplace_back(new ShardWorker());
      ShardWorker* w = idx->workers.back().get();
      w->th = std::thread([w] { w->loop(); });
    }
  }
  for (int g = 1; g < G; ++g) idx->workers[g - 1]->submit([&fn, g] { return fn(g); });
  int rc = fn(0);
  std::string err0 = rc != B2F_OK ? g_err : std::string();
  for (int g = 1; g < G; ++g) {
    const int r = idx->workers[g - 1]->wait();
    if (rc == B2F_OK && r != B2F_OK) { rc = r; err0 = g_err; }
  }
  if (rc != B2F_OK) g_err = err0;
  return rc;
}

// The parts area of one slot on the first device.  Only the search that takes the slot uses it, so it can grow while
// the searches of lower slots are still in flight.
int ensure_parts(Shard& S0, int slot, int64_t need) {
  Workspace& W = S0.ws;
  if (need <= W.parts_cap[slot]) return B2F_OK;
  CU_TRY(cudaSetDevice(S0.dev));
  dev_free(W.Dp[slot]); dev_free(W.Ip[slot]);
  W.parts_cap[slot] = 0;
  B2F_TRY(dev_alloc(&W.Dp[slot], static_cast<size_t>(need)));
  B2F_TRY(dev_alloc(&W.Ip[slot], static_cast<size_t>(need)));
  W.parts_cap[slot] = need;
  return B2F_OK;
}

// Merge the parts of the slot's multi-shard search into D / I on shard 0's stream.
int enqueue_merge(b2f_index* idx, int slot, int64_t nq, int k, float* D, int64_t* I, bool mark_pending) {
  Shard& S0 = idx->shards[0];
  const int G = static_cast<int>(idx->shards.size());
  const int64_t per = nq * k;
  CU_TRY(cudaSetDevice(S0.dev));
  merge_kernel<<<static_cast<int>(nq), merge_threads(G, k), merge_stage_bytes(G, k), S0.stream>>>(
      S0.ws.Dp[slot], S0.ws.Ip[slot], G, nq, k, D, I, per, per, nullptr, merge_mode(G, k), mark_pending ? 1 : 0);
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  return B2F_OK;
}

// Enqueue one search of a multi-shard index, without a host wait: every shard searches (each device enqueued by its
// own host thread) into its part of the slot's parts area, and shard 0's stream merges the parts into D / I (on the
// first device, or mapped host memory) once every part is there.
//   q_host: host queries, uploaded by every shard.  Else q_dev, on the first device: shard 0 reads it in place, every
//   other shard copies it once shard 0's stream has reached this call (the caller orders q's producer before that).
//   A shard whose device can store into the first device's memory writes its part there directly (the last kernel of
//   its search pushes the rows over NVLink); any other searches into its own buffer and copies the part over on its
//   own stream, so that its next search cannot overwrite the buffer before the copy.
//   mark_pending: a merged row whose part overflowed on some shard carries id -2 in its slot 0 until finish_sharded.
int enqueue_sharded(b2f_index* idx, const b2f_selector* sel, const float* q_host, const float* q_dev, int64_t nq, int k,
                    float* D, int64_t* I, int slot, bool mark_pending) {
  const int G = static_cast<int>(idx->shards.size());
  Shard& S0 = idx->shards[0];
  const int64_t per = nq * k;
  const size_t qbytes = static_cast<size_t>(nq) * kD * 4;
  B2F_TRY(ensure_parts(S0, slot, per * G));
  float* Dp = S0.ws.Dp[slot];
  int64_t* Ip = S0.ws.Ip[slot];
  if (q_dev) CU_TRY(cudaEventRecord(S0.ev, S0.stream));
  B2F_TRY(run_on_shards(idx, [&](int g) -> int {
    Shard& S = idx->shards[g];
    CU_TRY(cudaSetDevice(S.dev));
    B2F_TRY(ensure_query_ws(S, nq, k));
    const float* q = S.ws.q32;
    if (!q_dev) {
      CU_TRY(cudaMemcpyAsync(S.ws.q32, q_host, qbytes, cudaMemcpyHostToDevice, S.stream));
    } else if (g == 0) {
      q = q_dev;
    } else {
      CU_TRY(cudaStreamWaitEvent(S.stream, S0.ev, 0));
      if (S.dev == S0.dev) CU_TRY(cudaMemcpyAsync(S.ws.q32, q_dev, qbytes, cudaMemcpyDeviceToDevice, S.stream));
      else CU_TRY(cudaMemcpyPeerAsync(S.ws.q32, S.dev, q_dev, S0.dev, qbytes, S.stream));
    }
    const bool direct = g == 0 || S.peer_to_first;
    B2F_TRY(enqueue_search(idx, S, q, nq, k, direct ? Dp + per * g : S.ws.D, direct ? Ip + per * g : S.ws.I, slot,
                           sel ? &sel->parts[g] : nullptr));
    if (g == 0) return B2F_OK;
    if (!direct) {
      CU_TRY(cudaMemcpyPeerAsync(Dp + per * g, S0.dev, S.ws.D, S.dev, sizeof(float) * per, S.stream));
      CU_TRY(cudaMemcpyPeerAsync(Ip + per * g, S0.dev, S.ws.I, S.dev, sizeof(int64_t) * per, S.stream));
    }
    CU_TRY(cudaEventRecord(S.ev, S.stream));
    return B2F_OK;
  }));
  CU_TRY(cudaSetDevice(S0.dev));
  for (int g = 1; g < G; ++g) CU_TRY(cudaStreamWaitEvent(S0.stream, idx->shards[g].ev, 0));
  return enqueue_merge(idx, slot, nq, k, D, I, mark_pending);
}

// Settle a search of enqueue_sharded: every shard waits for its stream and re-runs its overflowed queries (reading
// them from q0, on the first device) straight into its part of the slot; if any shard re-ran, the parts are merged
// again.  One host wait per shard, and one more only after a re-run.
int finish_sharded(b2f_index* idx, const b2f_selector* sel, const float* q0, int64_t nq, int k, float* D, int64_t* I,
                   int slot) {
  const int G = static_cast<int>(idx->shards.size());
  Shard& S0 = idx->shards[0];
  const int64_t per = nq * k;
  bool any = false;
  for (int g = 0; g < G; ++g) {
    bool reran = false;
    B2F_TRY(finish_search(idx, idx->shards[g], q0, nq, k, S0.ws.Dp[slot] + per * g, S0.ws.Ip[slot] + per * g, slot,
                          &reran, sel ? &sel->parts[g] : nullptr));
    any = any || reran;
  }
  if (!any) return B2F_OK;
  B2F_TRY(enqueue_merge(idx, slot, nq, k, D, I, false));
  CU_TRY(cudaStreamSynchronize(S0.stream));
  return B2F_OK;
}

// Settle every search enqueued by b2f_search_device_async: wait for the stream, then re-run (on the
// exact engine) the queries whose candidate lists overflowed.  Normally just the synchronisation.
int settle_pending(b2f_index* idx) {
  if (idx->xchg_flush) B2F_TRY(idx->xchg_flush(idx));   // a merge owed by the peer exchange joins the stream first
  if (idx->pending.empty()) return B2F_OK;
  Shard& S = idx->shards[0];
  std::vector<Pending> todo;
  todo.swap(idx->pending);
  for (const Pending& p : todo) {
    if (idx->shards.size() > 1)
      B2F_TRY(finish_sharded(idx, p.sel, p.q, p.nq, p.k, p.D, p.I, p.slot));
    else
      B2F_TRY(finish_search(idx, S, p.q, p.nq, p.k, p.D, p.I, p.slot, nullptr, p.sel ? &p.sel->parts[0] : nullptr));
  }
  return B2F_OK;
}

// True when enqueueing this search would (re)allocate a workspace of some shard that searches in flight still use.
bool search_would_realloc(const b2f_index* idx, int64_t nq, int k) {
  for (const Shard& S : idx->shards) {
    const Workspace& W = S.ws;
    if (nq > W.nq_cap || nq * k > W.out_cap || !W.fbq) return true;
    if (S.n == 0) continue;
    const PassPlan plan = make_plan(idx, S, resolve_path(idx, S, nq), k, nq);
    if (plan.qp > W.qp_cap || plan.C > W.C) return true;
  }
  return false;
}

// A selector filters only the index it was built for, and only while no row was added or removed since.
int check_selector(const b2f_index* idx, const b2f_selector* sel) {
  if (!sel) return B2F_OK;
  if (sel->idx != idx) return fail(B2F_ERR_INVALID, "selector was built for another index");
  if (sel->generation != idx->generation.load())
    return fail(B2F_ERR_INVALID, "stale selector: rows were added to or removed from the index after it was built");
  return B2F_OK;
}

int check_args_search(const b2f_index* idx, const void* q, int64_t nq, int k, const void* D, const void* I) {
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  if (nq < 0) return fail(B2F_ERR_INVALID, "negative query count");
  if (k < 1 || k > B2F_MAX_K) return fail(B2F_ERR_INVALID, "k must be in [1, " + std::to_string(B2F_MAX_K) + "], got " + std::to_string(k));
  if (nq > 0 && (!q || !D || !I)) return fail(B2F_ERR_INVALID, "null query or output pointer");
  return B2F_OK;
}

void reset_stats(b2f_index* idx) {
  idx->stats = Stats();
  for (Shard& S : idx->shards) S.stats = Stats();
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* b2f_last_error(void) { return g_err.c_str(); }
const char* b2f_version(void) { return "b2f 0.1 sm_100a"; }

int b2f_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

int b2f_create(int d, const int* devices, int n_dev, b2f_index** out) {
  if (!out) return fail(B2F_ERR_INVALID, "null out pointer");
  *out = nullptr;
  if (d != kD) return fail(B2F_ERR_INVALID, "only d = 768 is supported (reference hard-codes IndexFlatIP(768)), got " + std::to_string(d));
  const int avail = b2f_device_count();
  if (avail <= 0) return fail(B2F_ERR_NO_DEVICE, "no CUDA device available; b2f has no CPU fallback");
  std::vector<int> devs;
  if (!devices || n_dev <= 0) devs.push_back(0);
  else devs.assign(devices, devices + n_dev);
  for (int dv : devs)
    if (dv < 0 || dv >= avail) return fail(B2F_ERR_INVALID, "device " + std::to_string(dv) + " out of range");
  b2f_index* idx = new b2f_index();
  idx->shards.resize(devs.size());
  for (size_t i = 0; i < devs.size(); ++i) {
    Shard& S = idx->shards[i];
    S.dev = devs[i];
    cudaDeviceProp prop;
    cudaError_t e = cudaSetDevice(S.dev);
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, S.dev);
    if (e == cudaSuccess && prop.major != 10) {
      b2f_destroy(idx);
      return fail(B2F_ERR_NO_DEVICE, "device " + std::to_string(S.dev) + " is sm_" + std::to_string(prop.major) +
                                         std::to_string(prop.minor) + "; b2f is built for sm_100a only");
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&S.ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&S.maxnorm2), 4 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(S.maxnorm2, 0, 4 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&S.mu), kD * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(S.mu, 0, kD * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&S.mu_part), static_cast<size_t>(kMuBlocks) * kD * sizeof(float));
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      std::string m = std::string("device setup failed: ") + cudaGetErrorString(e);
      b2f_destroy(idx);
      return fail(B2F_ERR_CUDA, m);
    }
    if (cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMergeStageMaxBytes) != cudaSuccess ||
        cudaFuncSetAttribute(xchg_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMergeStageMaxBytes) != cudaSuccess) {
      (void)cudaGetLastError();
      b2f_destroy(idx);
      return fail(B2F_ERR_CUDA, "cannot reserve shared memory for the merge kernels");
    }
    S.sm_count = prop.multiProcessorCount;
    S.max_pairs = std::min(128, std::max(1, S.sm_count / 2));
  }
  {
    cudaSetDevice(idx->shards[0].dev);
    if (cudaHostAlloc(reinterpret_cast<void**>(&idx->merge_flag_host), 2 * sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(reinterpret_cast<void**>(&idx->merge_flag_dev), idx->merge_flag_host, 0) != cudaSuccess) {
      (void)cudaGetLastError();
      b2f_destroy(idx);
      return fail(B2F_ERR_CUDA, "mapped host allocation failed");
    }
    idx->merge_flag_host[0] = idx->merge_flag_host[1] = 0;
  }
  // peer access between shard devices (direct NVLink copies for the result gather)
  for (size_t i = 0; i < devs.size(); ++i)
    for (size_t j = 0; j < devs.size(); ++j) {
      if (i == j) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, devs[i], devs[j]) == cudaSuccess && can) {
        cudaSetDevice(devs[i]);
        cudaError_t e = cudaDeviceEnablePeerAccess(devs[j], 0);
        if (e != cudaSuccess) (void)cudaGetLastError();
        if (j == 0 && (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled)) idx->shards[i].peer_to_first = true;
      }
    }
  (void)get_encode_fn();   // resolve the driver entry point before any worker thread needs it
  *out = idx;
  return B2F_OK;
}

void b2f_destroy(b2f_index* idx) {
  if (!idx) return;
  idx->pending.clear();
  idx->workers.clear();      // joins the shard threads
  for (Shard& S : idx->shards) {
    cudaSetDevice(S.dev);
    if (S.stream) cudaStreamSynchronize(S.stream);
    Workspace& W = S.ws;
    dev_free(S.x32); dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale); dev_free(S.idmap); dev_free(S.maxnorm2); dev_free(S.segs_d);
    dev_free(S.mu); dev_free(S.mu_part);
    for (int b = 0; b < kLoadBufs; ++b) {
      if (S.load_bufs[b]) cudaFreeHost(S.load_bufs[b]);
      if (S.load_evs[b]) cudaEventDestroy(S.load_evs[b]);
    }
    dev_free(W.cand[0]); dev_free(W.cand[1]); dev_free(W.cnt); dev_free(W.tau); dev_free(W.tauP);
    dev_free(W.ovf); dev_free(W.margin); dev_free(W.err); dev_free(W.q32); dev_free(W.q16);
    dev_free(W.gath); dev_free(W.cnt2); dev_free(W.hist); dev_free(W.hkey0); dev_free(W.hshift);
    dev_free(W.qnorm); dev_free(W.qerr); dev_free(W.D); dev_free(W.I);
    for (int s = 0; s < kMaxPending; ++s) { dev_free(W.Dp[s]); dev_free(W.Ip[s]); }
    dev_free(W.fbq); dev_free(W.fbD); dev_free(W.fbI);
    if (W.ovf_host) cudaFreeHost(W.ovf_host);
    if (W.pin) cudaFreeHost(W.pin);
    for (cudaEvent_t ev : S.prof.pool) cudaEventDestroy(ev);
    if (S.ev) cudaEventDestroy(S.ev);
    if (S.stream) cudaStreamDestroy(S.stream);
  }
  if (idx->merge_flag_host) cudaFreeHost(idx->merge_flag_host);
  if (idx->xchg.local) {
    cudaSetDevice(idx->shards[0].dev);
    for (int r = 0; r < idx->xchg.world; ++r)
      if (r != idx->xchg.rank && idx->xchg.peer[r]) cudaIpcCloseMemHandle(idx->xchg.peer[r]);
    cudaFree(idx->xchg.local);
    cudaFree(idx->xchg.stage);
    cudaFree(idx->xchg.counter);
  }
  (void)cudaGetLastError();
  delete idx;
}

int64_t b2f_ntotal(const b2f_index* idx) { return idx ? idx->ntotal : -1; }
int b2f_num_shards(const b2f_index* idx) { return idx ? static_cast<int>(idx->shards.size()) : 0; }
int64_t b2f_shard_rows(const b2f_index* idx, int shard) {
  if (!idx || shard < 0 || shard >= static_cast<int>(idx->shards.size())) return -1;
  return idx->shards[shard].n;
}
void* b2f_stream(b2f_index* idx, int shard) {
  if (!idx || shard < 0 || shard >= static_cast<int>(idx->shards.size())) return nullptr;
  return idx->shards[shard].stream;
}

int b2f_reserve(b2f_index* idx, int64_t n_per_shard) {
  if (!idx || n_per_shard < 0) return fail(B2F_ERR_INVALID, "bad reserve arguments");
  if (n_per_shard >= 0xfffffff0ll) return fail(B2F_ERR_INVALID, "a shard holds at most 2^32-16 rows");
  B2F_TRY(settle_pending(idx));
  for (Shard& S : idx->shards) B2F_TRY(ensure_capacity(idx, S, n_per_shard));
  return B2F_OK;
}

static int add_impl(b2f_index* idx, const float* x_host, const int64_t* ids_host, int64_t n) {
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  if (n < 0 || (n > 0 && !x_host)) return fail(B2F_ERR_INVALID, "bad add arguments");
  if (n == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  ++idx->generation;
  const int G = static_cast<int>(idx->shards.size());
  if (ids_host) {
    for (Shard& S : idx->shards)
      if (S.n > 0 && !S.has_ids) return fail(B2F_ERR_INVALID, "cannot mix add() and add_with_ids() on a non-empty index");
  } else {
    for (Shard& S : idx->shards)
      if (S.has_ids && S.n > 0) return fail(B2F_ERR_INVALID, "cannot mix add_with_ids() and add() on a non-empty index");
  }
  // contiguous split, like FAISS IndexShards with successive ids; every device copies and ingests its
  // slice from its own host thread, so the PCIe links of all GPUs run in parallel
  B2F_TRY(run_on_shards(idx, [&](int g) -> int {
    Shard& S = idx->shards[g];
    const int64_t lo = n * g / G, hi = n * (g + 1) / G, m = hi - lo;
    if (m == 0) return B2F_OK;
    CU_TRY(cudaSetDevice(S.dev));
    if (ids_host && !S.has_ids) {
      S.has_ids = true;
      if (S.cap > 0 && !S.idmap) B2F_TRY(dev_alloc(&S.idmap, static_cast<size_t>(S.cap)));
    }
    if (!ids_host) S.has_ids = false;
    if (S.n + m >= 0xfffffff0ll) return fail(B2F_ERR_INVALID, "a shard holds at most 2^32-16 rows");
    B2F_TRY(ensure_capacity(idx, S, S.n + m));
    CU_TRY(cudaMemcpyAsync(S.x32 + S.n * kD, x_host + lo * kD, static_cast<size_t>(m) * kD * 4,
                           cudaMemcpyHostToDevice, S.stream));
    if (ids_host)
      CU_TRY(cudaMemcpyAsync(S.idmap + S.n, ids_host + lo, static_cast<size_t>(m) * 8, cudaMemcpyHostToDevice, S.stream));
    B2F_TRY(ingest_rows(idx, S, m));
    push_seg(S, S.n, m, idx->ntotal + lo);
    S.n += m;
    CU_TRY(cudaStreamSynchronize(S.stream));  // FAISS add() is synchronous: the caller may free x now
    return B2F_OK;
  }));
  idx->ntotal += n;
  return B2F_OK;
}

int b2f_add(b2f_index* idx, const float* x_host, int64_t n) { return add_impl(idx, x_host, nullptr, n); }
int b2f_add_with_ids(b2f_index* idx, const float* x_host, const int64_t* ids_host, int64_t n) {
  if (n > 0 && !ids_host) return fail(B2F_ERR_INVALID, "null ids");
  return add_impl(idx, x_host, ids_host, n);
}

int b2f_add_device(b2f_index* idx, int shard, const float* x_dev, int64_t n) {
  if (!idx || shard < 0 || shard >= static_cast<int>(idx->shards.size()) || n < 0 || (n > 0 && !x_dev))
    return fail(B2F_ERR_INVALID, "bad add_device arguments");
  if (n == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  Shard& S = idx->shards[shard];
  if (S.has_ids && S.n > 0) return fail(B2F_ERR_INVALID, "index uses explicit ids");
  ++idx->generation;
  CU_TRY(cudaSetDevice(S.dev));
  B2F_TRY(ensure_capacity(idx, S, S.n + n));
  CU_TRY(cudaMemcpyAsync(S.x32 + S.n * kD, x_dev, static_cast<size_t>(n) * kD * 4, cudaMemcpyDeviceToDevice, S.stream));
  B2F_TRY(ingest_rows(idx, S, n));
  push_seg(S, S.n, n, idx->ntotal);
  S.n += n;
  idx->ntotal += n;
  CU_TRY(cudaStreamSynchronize(S.stream));
  return B2F_OK;
}

int b2f_add_synthetic(b2f_index* idx, int shard, int64_t first_row, int64_t n, uint64_t seed, uint64_t stream,
                      float norm, int64_t id_base) {
  if (!idx || shard < 0 || shard >= static_cast<int>(idx->shards.size()) || n < 0 || first_row < 0)
    return fail(B2F_ERR_INVALID, "bad add_synthetic arguments");
  if (n == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  Shard& S = idx->shards[shard];
  if (S.has_ids && S.n > 0) return fail(B2F_ERR_INVALID, "index uses explicit ids");
  ++idx->generation;
  CU_TRY(cudaSetDevice(S.dev));
  B2F_TRY(ensure_capacity(idx, S, S.n + n));
  const uint32_t k0 = static_cast<uint32_t>(seed) ^ static_cast<uint32_t>(stream);
  const uint32_t k1 = static_cast<uint32_t>(seed >> 32) ^ static_cast<uint32_t>(stream >> 32) ^ 0x5eedu;
  synth_rows_kernel<<<launch_grid_rows(S, n), 256, 0, S.stream>>>(S.x32, S.n, first_row, n, k0, k1, norm,
                                                                  idx->synth_mean_shift, static_cast<uint32_t>(seed),
                                                                  static_cast<uint32_t>(seed >> 32) ^ 0x5eedu);
  CU_TRY(cudaGetLastError());
  B2F_TRY(ingest_rows(idx, S, n));
  push_seg(S, S.n, n, id_base);
  S.n += n;
  idx->ntotal += n;
  CU_TRY(cudaStreamSynchronize(S.stream));
  return B2F_OK;
}

int b2f_reconstruct_n(b2f_index* idx, int shard, int64_t row0, int64_t n, float* out_host) {
  if (!idx || shard < 0 || shard >= static_cast<int>(idx->shards.size()) || row0 < 0 || n < 0 || (n > 0 && !out_host))
    return fail(B2F_ERR_INVALID, "bad reconstruct_n arguments");
  Shard& S = idx->shards[shard];
  if (row0 + n > S.n) return fail(B2F_ERR_INVALID, "reconstruct_n range exceeds the shard's rows");
  if (n == 0) return B2F_OK;
  CU_TRY(cudaSetDevice(S.dev));
  CU_TRY(cudaMemcpyAsync(out_host, S.x32 + row0 * kD, static_cast<size_t>(n) * kD * 4, cudaMemcpyDeviceToHost, S.stream));
  CU_TRY(cudaStreamSynchronize(S.stream));
  return B2F_OK;
}

int b2f_reset(b2f_index* idx) {
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  B2F_TRY(settle_pending(idx));
  ++idx->generation;
  for (Shard& S : idx->shards) {
    CU_TRY(cudaSetDevice(S.dev));
    CU_TRY(cudaStreamSynchronize(S.stream));
    S.n = 0;
    S.segs.clear();
    S.segs_dirty = true;
    S.has_ids = false;
    CU_TRY(cudaMemsetAsync(S.maxnorm2, 0, 4 * sizeof(unsigned int), S.stream));
    CU_TRY(cudaMemsetAsync(S.mu, 0, kD * sizeof(float), S.stream));
    S.mu_set = false;
    if (!idx->keep_on_reset) {
      dev_free(S.x32); dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale); dev_free(S.idmap);
      S.cap = 0;
    }
  }
  idx->ntotal = 0;
  return B2F_OK;
}

int b2f_search_device(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  B2F_TRY(check_args_search(idx, q_dev, nq, k, D_dev, I_dev));
  if (nq == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  reset_stats(idx);
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  if (idx->shards.size() > 1) {
    B2F_TRY(enqueue_sharded(idx, nullptr, nullptr, q_dev, nq, k, D_dev, I_dev, 0, false));
    return finish_sharded(idx, nullptr, q_dev, nq, k, D_dev, I_dev, 0);
  }
  B2F_TRY(ensure_query_ws(S, nq, k));
  B2F_TRY(enqueue_search(idx, S, q_dev, nq, k, D_dev, I_dev));
  B2F_TRY(finish_search(idx, S, q_dev, nq, k, D_dev, I_dev));
  return B2F_OK;
}

int b2f_search_device_async(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  return b2f_search_device_async_sel(idx, nullptr, q_dev, nq, k, D_dev, I_dev);
}

int b2f_search_device_async_sel(b2f_index* idx, const b2f_selector* sel, const float* q_dev, int64_t nq, int k,
                                float* D_dev, int64_t* I_dev) {
  B2F_TRY(check_args_search(idx, q_dev, nq, k, D_dev, I_dev));
  B2F_TRY(check_selector(idx, sel));
  if (nq == 0) return B2F_OK;
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  if (static_cast<int>(idx->pending.size()) >= kMaxPending || search_would_realloc(idx, nq, k))
    B2F_TRY(settle_pending(idx));
  const int slot = static_cast<int>(idx->pending.size());
  if (idx->shards.size() > 1) {
    B2F_TRY(enqueue_sharded(idx, sel, nullptr, q_dev, nq, k, D_dev, I_dev, slot, true));
  } else {
    B2F_TRY(ensure_query_ws(S, nq, k));
    B2F_TRY(enqueue_search(idx, S, q_dev, nq, k, D_dev, I_dev, slot, sel ? &sel->parts[0] : nullptr));
  }
  idx->pending.push_back(Pending{q_dev, nq, k, D_dev, I_dev, slot, sel});
  return B2F_OK;
}

int b2f_search_finish(b2f_index* idx) {
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  B2F_TRY(settle_pending(idx));
  // also wait for work queued behind the searches (exchange push / merge kernels, a re-push)
  for (Shard& S : idx->shards) {
    CU_TRY(cudaSetDevice(S.dev));
    CU_TRY(cudaStreamSynchronize(S.stream));
  }
  return B2F_OK;
}

int b2f_merge_device(b2f_index* idx, const float* D_parts_dev, const int64_t* I_parts_dev, int n_parts,
                     int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  if (!idx || n_parts < 1 || n_parts > kXchgMaxWorldMerge || nq < 0 || k < 1 || !D_parts_dev || !I_parts_dev || !D_dev || !I_dev)
    return fail(B2F_ERR_INVALID, "bad merge arguments (1..64 parts)");
  if (nq == 0) return B2F_OK;
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  const int msb = merge_stage_bytes(n_parts, k);
  merge_kernel<<<static_cast<int>(nq), merge_threads(n_parts, k), msb, S.stream>>>(D_parts_dev, I_parts_dev, n_parts, nq, k, D_dev, I_dev,
                                                             nq * k, nq * k, nullptr, merge_mode(n_parts, k), 0);
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  CU_TRY(cudaStreamSynchronize(S.stream));
  return B2F_OK;
}

int b2f_merge_packed_device_async(b2f_index* idx, const void* parts_dev, int n_parts, int64_t part_bytes,
                                  int64_t i_offset_bytes, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  if (!idx || n_parts < 1 || n_parts > kXchgMaxWorldMerge || nq < 0 || k < 1 || !parts_dev || !D_dev || !I_dev || part_bytes % 8 != 0 ||
      i_offset_bytes % 8 != 0 || i_offset_bytes < nq * k * 4 || part_bytes < i_offset_bytes + nq * k * 8)
    return fail(B2F_ERR_INVALID, "bad packed merge arguments");
  if (nq == 0) return B2F_OK;
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  const char* base = static_cast<const char*>(parts_dev);
  const int msb = merge_stage_bytes(n_parts, k);
  merge_kernel<<<static_cast<int>(nq), merge_threads(n_parts, k), msb, S.stream>>>(
      reinterpret_cast<const float*>(base), reinterpret_cast<const int64_t*>(base + i_offset_bytes), n_parts, nq, k,
      D_dev, I_dev, part_bytes / 4, part_bytes / 8, idx->merge_flag_dev, merge_mode(n_parts, k), 0);
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  return B2F_OK;
}

static int xchg_flush_deferred(b2f_index* idx);

int b2f_xchg_create(b2f_index* idx, int rank, int world, int64_t max_nq, int max_k, void* handle_out) {
  if (!idx || !handle_out || world < 2 || world > kXchgMaxWorld || rank < 0 || rank >= world || max_nq < 1 ||
      max_k < 1 || max_k > B2F_MAX_K)
    return fail(B2F_ERR_INVALID, "bad exchange arguments (2 <= world <= 16)");
  if (idx->shards.size() != 1) return fail(B2F_ERR_INVALID, "the peer exchange needs a single-shard index per process");
  if (idx->xchg.local) return fail(B2F_ERR_INVALID, "exchange already created");
  B2F_TRY(settle_pending(idx));
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  auto& X = idx->xchg;
  X.rank = rank; X.world = world; X.max_nq = max_nq; X.max_k = max_k;
  X.part_cap = static_cast<size_t>(round_up(round_up(max_nq * max_k * 4, 16) + max_nq * max_k * 8, 128));
  X.flags_off = kXchgSlots * static_cast<size_t>(world) * X.part_cap;
  X.bytes = X.flags_off + kXchgSlots * static_cast<size_t>(world) * sizeof(unsigned int);
  CU_TRY(cudaMalloc(reinterpret_cast<void**>(&X.local), X.bytes));
  CU_TRY(cudaMalloc(reinterpret_cast<void**>(&X.stage), X.part_cap));
  CU_TRY(cudaMalloc(reinterpret_cast<void**>(&X.counter), sizeof(int)));
  CU_TRY(cudaMemset(X.local, 0, X.bytes));
  CU_TRY(cudaMemset(X.counter, 0, sizeof(int)));
  CU_TRY(cudaDeviceSynchronize());
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
  cudaIpcMemHandle_t h;
  CU_TRY(cudaIpcGetMemHandle(&h, X.local));
  std::memcpy(handle_out, &h, sizeof(h));
  return B2F_OK;
}

int b2f_xchg_connect(b2f_index* idx, const void* handles) {
  if (!idx || !handles || !idx->xchg.local) return fail(B2F_ERR_INVALID, "exchange not created");
  auto& X = idx->xchg;
  CU_TRY(cudaSetDevice(idx->shards[0].dev));
  for (int r = 0; r < X.world; ++r) {
    if (r == X.rank) { X.peer[r] = X.local; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const char*>(handles) + 64 * r, sizeof(h));
    void* p = nullptr;
    CU_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    X.peer[r] = static_cast<char*>(p);
  }
  X.connected = true;
  idx->xchg_flush = &xchg_flush_deferred;
  return B2F_OK;
}

// enqueue the wait + merge of one exchange step on the index stream
static int xchg_launch_merge(b2f_index* idx, unsigned int seq, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  auto& X = idx->xchg;
  Shard& S = idx->shards[0];
  const int slot = static_cast<int>(seq % kXchgSlots);
  const int64_t i_off = round_up(nq * k * 4, 16);
  {
    ProfScope ps(idx, S, 2);
    const int msb = merge_stage_bytes(X.world, k);
    xchg_merge_kernel<<<static_cast<int>(nq), merge_threads(X.world, k), msb, S.stream>>>(
        X.local + static_cast<size_t>(slot) * X.world * X.part_cap,
        reinterpret_cast<const unsigned int*>(X.local + X.flags_off) + slot * X.world, seq, X.world,
        static_cast<int64_t>(X.part_cap), i_off, nq, k, D_dev, I_dev, idx->merge_flag_dev, idx->merge_flag_dev + 1,
        merge_mode(X.world, k));
  }
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  return B2F_OK;
}

// the merge of the previous exchange step, if it is still owed
static int xchg_flush_deferred(b2f_index* idx) {
  auto& X = idx->xchg;
  if (!X.deferred.valid) return B2F_OK;
  X.deferred.valid = false;
  CU_TRY(cudaSetDevice(idx->shards[0].dev));
  return xchg_launch_merge(idx, X.deferred.seq, X.deferred.nq, X.deferred.k, X.deferred.D, X.deferred.I);
}

// push the staged local part to every rank; merge what every rank pushed (now, or one step later)
static int xchg_push_and_merge(b2f_index* idx, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
  auto& X = idx->xchg;
  Shard& S = idx->shards[0];
  const unsigned int seq = ++X.seq;
  const int slot = static_cast<int>(seq % kXchgSlots);
  XchgPeers peers;
  peers.world = X.world;
  for (int r = 0; r < X.world; ++r) {
    peers.part[r] = X.peer[r] + (static_cast<size_t>(slot) * X.world + X.rank) * X.part_cap;
    peers.flag[r] = reinterpret_cast<unsigned int*>(X.peer[r] + X.flags_off) + slot * X.world + X.rank;
  }
  const int64_t i_off = round_up(nq * k * 4, 16);
  const int64_t n_vec = (i_off + nq * k * 8 + 15) / 16;
  // 4 blocks per destination for the headline part (208 KB); large batches (16,384 x 1000: 197 MB per part)
  // get one block per 64 KB, up to 128 per destination, so the push runs at NVLink speed
  const int gy = static_cast<int>(std::min<int64_t>(128, std::max<int64_t>(4, n_vec / 4096)));
  xchg_push_kernel<<<dim3(X.world, gy), 256, 0, S.stream>>>(reinterpret_cast<const uint4*>(X.stage), n_vec, peers, seq,
                                                            X.counter);
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  if (!X.defer) return xchg_launch_merge(idx, seq, nq, k, D_dev, I_dev);
  B2F_TRY(xchg_flush_deferred(idx));          // step seq-1: its parts arrived a whole search ago
  X.deferred.valid = true;
  X.deferred.seq = seq; X.deferred.nq = nq; X.deferred.k = k; X.deferred.D = D_dev; X.deferred.I = I_dev;
  return B2F_OK;
}

int b2f_search_xchg_async(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                          int repush_only) {
  return b2f_search_xchg_async_sel(idx, nullptr, q_dev, nq, k, D_dev, I_dev, repush_only);
}

int b2f_search_xchg_async_sel(b2f_index* idx, const b2f_selector* sel, const float* q_dev, int64_t nq, int k,
                              float* D_dev, int64_t* I_dev, int repush_only) {
  B2F_TRY(check_args_search(idx, q_dev, nq, k, D_dev, I_dev));
  B2F_TRY(check_selector(idx, sel));
  if (!idx->xchg.connected) return fail(B2F_ERR_INVALID, "exchange not connected (b2f_xchg_create / b2f_xchg_connect)");
  if (nq > idx->xchg.max_nq || k > idx->xchg.max_k || nq * static_cast<int64_t>(k) > idx->xchg.max_nq * idx->xchg.max_k)
    return fail(B2F_ERR_INVALID, "batch exceeds the exchange buffers");
  if (nq == 0) return B2F_OK;
  auto& X = idx->xchg;
  float* Dl = reinterpret_cast<float*>(X.stage);
  int64_t* Il = reinterpret_cast<int64_t*>(X.stage + round_up(nq * k * 4, 16));
  if (!repush_only) B2F_TRY(b2f_search_device_async_sel(idx, sel, q_dev, nq, k, Dl, Il));
  CU_TRY(cudaSetDevice(idx->shards[0].dev));
  return xchg_push_and_merge(idx, nq, k, D_dev, I_dev);
}

int b2f_xchg_flush(b2f_index* idx) {
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  return xchg_flush_deferred(idx);
}

// Page-locked host memory (cudaHostAlloc / cudaHostRegister / torch pin_memory) is addressable by the device
// under unified addressing: copies from it need no staging, and kernels can store results straight into it.
static bool is_pinned_host(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

int b2f_search(b2f_index* idx, const float* q_host, int64_t nq, int k, float* D_host, int64_t* I_host) {
  return b2f_search_sel(idx, nullptr, q_host, nq, k, D_host, I_host);
}

int b2f_search_sel(b2f_index* idx, const b2f_selector* sel, const float* q_host, int64_t nq, int k, float* D_host,
                   int64_t* I_host) {
  B2F_TRY(check_args_search(idx, q_host, nq, k, D_host, I_host));
  B2F_TRY(check_selector(idx, sel));
  if (nq == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  reset_stats(idx);
  const int G = static_cast<int>(idx->shards.size());
  const size_t qbytes = static_cast<size_t>(nq) * kD * 4;
  const size_t d_off = static_cast<size_t>(round_up(static_cast<int64_t>(nq) * k * 4, 16));
  const size_t obytes = d_off + static_cast<size_t>(nq) * k * sizeof(int64_t);  // pinned layout [D | pad | I]
  Shard& S0 = idx->shards[0];
  CU_TRY(cudaSetDevice(S0.dev));
  // Host side of the call (the e2e path): queries are uploaded from the caller's buffer when it is page-locked,
  // else through one pinned staging copy; results are written by the LAST kernel of the search (finalize /
  // merge) straight into page-locked host memory over PCIe — the caller's arrays when they are page-locked,
  // else the library's buffer followed by one memcpy — so no device-to-host copy operation is queued at all
  // and the host waits exactly once.
  const bool q_pinned = is_pinned_host(q_host);
  const bool out_pinned = is_pinned_host(D_host) && is_pinned_host(I_host);
  B2F_TRY(ensure_pin(S0, qbytes + obytes + 64));
  char* pin = static_cast<char*>(S0.ws.pin);
  const float* q_src = q_host;
  if (!q_pinned) {
    std::memcpy(pin, q_host, qbytes);
    q_src = reinterpret_cast<const float*>(pin);
  }
  char* out_base = pin + round_up(static_cast<int64_t>(qbytes), 64);
  float* outD = out_pinned ? D_host : reinterpret_cast<float*>(out_base);
  int64_t* outI = out_pinned ? I_host : reinterpret_cast<int64_t*>(out_base + d_off);
  if (G == 1) {
    B2F_TRY(ensure_query_ws(S0, nq, k));
    CU_TRY(cudaMemcpyAsync(S0.ws.q32, q_src, qbytes, cudaMemcpyHostToDevice, S0.stream));
    B2F_TRY(enqueue_search(idx, S0, S0.ws.q32, nq, k, outD, outI, 0, sel ? &sel->parts[0] : nullptr));
    // ONE synchronisation; only if a candidate list overflowed (rare) the affected queries are re-run,
    // their rows rewritten in place
    B2F_TRY(finish_search(idx, S0, S0.ws.q32, nq, k, outD, outI, 0, nullptr, sel ? &sel->parts[0] : nullptr));
  } else {
    // every device is enqueued by its own host thread; the merge stores the result rows into the output
    B2F_TRY(enqueue_sharded(idx, sel, q_src, nullptr, nq, k, outD, outI, 0, false));
    B2F_TRY(finish_sharded(idx, sel, S0.ws.q32, nq, k, outD, outI, 0));
  }
  if (!out_pinned) {
    std::memcpy(D_host, outD, sizeof(float) * nq * k);
    std::memcpy(I_host, outI, sizeof(int64_t) * nq * k);
  }
  return B2F_OK;
}

// The whole end-to-end call of the one-process-per-GPU layout in ONE entry point: stage / upload the queries,
// local search, NVLink push, wait + merge (storing the result straight into page-locked host memory), one
// host wait, overflow protocol.  Collective: every rank calls it with the same nq, k.  (The Python layer
// used to queue these pieces one ctypes / torch call at a time: ~0.25 ms of host time per search at a
// 1.4 ms step.)
int b2f_search_xchg_host(b2f_index* idx, const float* q_host, int64_t nq, int k, float* D_host, int64_t* I_host) {
  B2F_TRY(check_args_search(idx, q_host, nq, k, D_host, I_host));
  if (!idx->xchg.connected) return fail(B2F_ERR_INVALID, "exchange not connected (b2f_xchg_create / b2f_xchg_connect)");
  if (nq == 0) return B2F_OK;
  B2F_TRY(settle_pending(idx));
  reset_stats(idx);
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  const size_t qbytes = static_cast<size_t>(nq) * kD * 4;
  const size_t d_off = static_cast<size_t>(round_up(static_cast<int64_t>(nq) * k * 4, 16));
  const size_t obytes = d_off + static_cast<size_t>(nq) * k * sizeof(int64_t);
  const bool q_pinned = is_pinned_host(q_host);
  const bool out_pinned = is_pinned_host(D_host) && is_pinned_host(I_host);
  B2F_TRY(ensure_pin(S, qbytes + obytes + 64));
  B2F_TRY(ensure_query_ws(S, nq, k));
  char* pin = static_cast<char*>(S.ws.pin);
  const float* q_src = q_host;
  if (!q_pinned) {
    std::memcpy(pin, q_host, qbytes);
    q_src = reinterpret_cast<const float*>(pin);
  }
  char* out_base = pin + round_up(static_cast<int64_t>(qbytes), 64);
  float* outD = out_pinned ? D_host : reinterpret_cast<float*>(out_base);
  int64_t* outI = out_pinned ? I_host : reinterpret_cast<int64_t*>(out_base + d_off);
  CU_TRY(cudaMemcpyAsync(S.ws.q32, q_src, qbytes, cudaMemcpyHostToDevice, S.stream));
  *idx->merge_flag_host = 0;
  B2F_TRY(b2f_search_xchg_async(idx, S.ws.q32, nq, k, outD, outI, 0));
  B2F_TRY(xchg_flush_deferred(idx));          // the merge of THIS step joins the stream now
  B2F_TRY(b2f_search_finish(idx));            // the one host wait (+ local re-run of overflowed queries)
  if (idx->merge_flag_host[1]) return fail(B2F_ERR_INTERNAL, "peer exchange timed out: a rank's part never arrived");
  if (*idx->merge_flag_host) {
    // some rank's list had overflowed when its part travelled (in-band marker, seen by every rank's merge):
    // every rank pushes again — the owner with its re-run rows — and merges again
    *idx->merge_flag_host = 0;
    B2F_TRY(b2f_search_xchg_async(idx, S.ws.q32, nq, k, outD, outI, 1));
    B2F_TRY(xchg_flush_deferred(idx));
    B2F_TRY(b2f_search_finish(idx));
    *idx->merge_flag_host = 0;
  }
  if (!out_pinned) {
    std::memcpy(D_host, outD, sizeof(float) * nq * k);
    std::memcpy(I_host, outI, sizeof(int64_t) * nq * k);
  }
  return B2F_OK;
}

static void free_selector_parts(b2f_selector* sel) {
  for (SelShard& P : sel->parts) {
    if (!P.bits && !P.qs_tiles && !P.ts_tiles) continue;
    cudaSetDevice(P.dev);
    dev_free(P.bits); dev_free(P.qs_tiles); dev_free(P.ts_tiles);
  }
  (void)cudaGetLastError();
}

// Evaluate the selector on every row of one shard (selector_bits_kernel), then compact the tile flags into the
// tile lists on the host: the one synchronisation of the build.
static int build_selector_part(b2f_index* idx, Shard& S, const SelDesc& desc_host, const std::vector<int64_t>& ids,
                               const uint8_t* bitmap_host, SelShard& P) {
  P.dev = S.dev;
  if (S.n == 0) return B2F_OK;
  CU_TRY(cudaSetDevice(S.dev));
  B2F_TRY(upload_segs(S));
  const int64_t n_words = round_up(S.n, kQsTileRows) / 32;
  const int64_t n_qs = n_words / (kQsTileRows / 32), n_ts = n_words / (kTileRows / 32);
  B2F_TRY(dev_alloc(&P.bits, static_cast<size_t>(n_words)));
  // scratch: [count (8 bytes)][QS tile flags][TS tile flags], the sorted ids, the bitmap
  struct Scratch {
    unsigned char* flags = nullptr; int64_t* ids = nullptr; uint8_t* bitmap = nullptr;
    ~Scratch() { dev_free(flags); dev_free(ids); dev_free(bitmap); }
  } tmp;
  const size_t flag_bytes = 8 + static_cast<size_t>(n_qs + n_ts);
  B2F_TRY(dev_alloc(&tmp.flags, flag_bytes));
  SelDesc d = desc_host;
  if (d.kind == kSelBatch && !ids.empty()) {
    B2F_TRY(dev_alloc(&tmp.ids, ids.size()));
    CU_TRY(cudaMemcpyAsync(tmp.ids, ids.data(), ids.size() * 8, cudaMemcpyHostToDevice, S.stream));
  }
  if (d.kind == kSelBitmap && d.n_bytes > 0) {
    B2F_TRY(dev_alloc(&tmp.bitmap, static_cast<size_t>(d.n_bytes)));
    CU_TRY(cudaMemcpyAsync(tmp.bitmap, bitmap_host, static_cast<size_t>(d.n_bytes), cudaMemcpyHostToDevice, S.stream));
  }
  d.ids = tmp.ids;
  d.n_ids = static_cast<int64_t>(ids.size());
  d.bitmap = tmp.bitmap;
  CU_TRY(cudaMemsetAsync(tmp.flags, 0, flag_bytes, S.stream));
  const int blocks = static_cast<int>(std::min<int64_t>((n_words + 7) / 8, static_cast<int64_t>(S.sm_count) * 8));
  selector_bits_kernel<<<blocks, 256, 0, S.stream>>>(d, S.n, n_words, S.segs_d, static_cast<int>(S.segs.size()),
                                                     S.has_ids ? S.idmap : nullptr, P.bits, tmp.flags + 8,
                                                     tmp.flags + 8 + n_qs, reinterpret_cast<unsigned long long*>(tmp.flags));
  CU_TRY(cudaGetLastError());
  std::vector<unsigned char> flags(flag_bytes);
  CU_TRY(cudaMemcpyAsync(flags.data(), tmp.flags, flag_bytes, cudaMemcpyDeviceToHost, S.stream));
  CU_TRY(cudaStreamSynchronize(S.stream));
  unsigned long long count = 0;
  std::memcpy(&count, flags.data(), 8);
  P.count = static_cast<int64_t>(count);
  std::vector<int> qs;
  for (int64_t t = 0; t < n_qs; ++t)
    if (flags[8 + t]) qs.push_back(static_cast<int>(t));
  for (int64_t t = 0; t < n_ts; ++t)
    if (flags[8 + n_qs + t]) P.ts_host.push_back(static_cast<int>(t));
  P.n_qs = static_cast<int>(qs.size());
  P.n_ts = static_cast<int>(P.ts_host.size());
  B2F_TRY(dev_alloc(&P.qs_tiles, qs.size()));
  B2F_TRY(dev_alloc(&P.ts_tiles, P.ts_host.size()));
  if (!qs.empty()) CU_TRY(cudaMemcpy(P.qs_tiles, qs.data(), qs.size() * 4, cudaMemcpyHostToDevice));
  if (!P.ts_host.empty()) CU_TRY(cudaMemcpy(P.ts_tiles, P.ts_host.data(), P.ts_host.size() * 4, cudaMemcpyHostToDevice));
  return B2F_OK;
}

int b2f_selector_create(b2f_index* idx, int kind, int invert, int64_t imin, int64_t imax, const int64_t* ids_host,
                        int64_t n_ids, const uint8_t* bitmap_host, int64_t n_bytes, b2f_selector** out) {
  if (!out) return fail(B2F_ERR_INVALID, "null out pointer");
  *out = nullptr;
  if (!idx) return fail(B2F_ERR_INVALID, "null index");
  if (kind != kSelRange && kind != kSelBatch && kind != kSelBitmap)
    return fail(B2F_ERR_INVALID, "selector kind must be B2F_SEL_RANGE, B2F_SEL_BATCH or B2F_SEL_BITMAP");
  if (kind == kSelBatch && (n_ids < 0 || (n_ids > 0 && !ids_host))) return fail(B2F_ERR_INVALID, "bad batch selector ids");
  if (kind == kSelBitmap && (n_bytes < 0 || (n_bytes > 0 && !bitmap_host)))
    return fail(B2F_ERR_INVALID, "bad bitmap selector bytes");
  B2F_TRY(settle_pending(idx));
  SelDesc d{kind, invert ? 1 : 0, imin, imax, nullptr, 0, nullptr, kind == kSelBitmap ? n_bytes : 0};
  std::vector<int64_t> ids;
  if (kind == kSelBatch) {   // any order, duplicates allowed: sorted and unique for the per-row binary search
    ids.assign(ids_host, ids_host + n_ids);
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
  }
  std::unique_ptr<b2f_selector> sel(new b2f_selector());
  sel->idx = idx;
  sel->generation = idx->generation.load();
  sel->parts.resize(idx->shards.size());
  for (size_t g = 0; g < idx->shards.size(); ++g) {
    const int rc = build_selector_part(idx, idx->shards[g], d, ids, bitmap_host, sel->parts[g]);
    if (rc != B2F_OK) {
      const std::string msg = g_err;
      free_selector_parts(sel.get());
      return fail(rc, msg);
    }
    sel->count += sel->parts[g].count;
  }
  *out = sel.release();
  return B2F_OK;
}

int b2f_selector_count(const b2f_selector* sel, int64_t* selected_out) {
  if (!sel || !selected_out) return fail(B2F_ERR_INVALID, "null selector or output pointer");
  *selected_out = sel->count;
  return B2F_OK;
}

void b2f_selector_destroy(b2f_selector* sel) {
  if (!sel) return;
  (void)settle_pending(sel->idx);   // searches in flight may still read its bitmap and tile lists
  free_selector_parts(sel);
  delete sel;
}

int b2f_set_option(b2f_index* idx, const char* key, int64_t value) {
  if (!idx || !key) return fail(B2F_ERR_INVALID, "bad option arguments");
  B2F_TRY(settle_pending(idx));
  const std::string k(key);
  if (k == "reset_stats") { reset_stats(idx); return B2F_OK; }
  if (k == "path") {
    if (value < 0 || value > 3) return fail(B2F_ERR_INVALID, "path must be 0..3");
    idx->path = static_cast<int>(value);
  } else if (k == "shadow") {
    if (idx->ntotal > 0) return fail(B2F_ERR_INVALID, "shadow can only be changed on an empty index");
    if (value < 0 || value > 3) return fail(B2F_ERR_INVALID, "shadow must be 0 (none), 1 (bf16), 2 (int8) or 3 (auto)");
    idx->shadow = static_cast<int>(value);
    ++idx->generation;
    for (Shard& S : idx->shards) {
      cudaSetDevice(S.dev);
      dev_free(S.x32); dev_free(S.x16); dev_free(S.x8); dev_free(S.tscale); dev_free(S.idmap);
      S.cap = 0;
      S.fmt = idx->shadow == kShadowAuto ? 0 : idx->shadow;
      S.mu_set = false;
    }
  } else if (k == "growth") {
    if (value < 2 || value > 1024) return fail(B2F_ERR_INVALID, "growth must be in [2, 1024]");
    idx->growth = static_cast<int>(value);
  } else if (k == "margin_ppm") {
    if (value < 0) return fail(B2F_ERR_INVALID, "margin_ppm must be >= 0");
    idx->margin_ppm = value;
  } else if (k == "keep_on_reset") {
    idx->keep_on_reset = value ? 1 : 0;
  } else if (k == "umma_variant") {
    if (value < 0 || value > 3) return fail(B2F_ERR_INVALID, "umma_variant must be 0 (auto), 1 (QS, resident queries), 2 (TS) or 3 (QS)");
    idx->umma_variant = static_cast<int>(value);
  } else if (k == "qs_max_q") {
    if (value < 0 || value > kQsMaxCols) return fail(B2F_ERR_INVALID, "qs_max_q must be in [0, 256]");
    idx->qs_max_q = static_cast<int>(value);
  } else if (k == "qs_resident_kb") {
    if (value < 0 || value > kNumKBlocks) return fail(B2F_ERR_INVALID, "qs_resident_kb must be in [0, 12]");
    idx->qs_resident_kb = static_cast<int>(value);
  } else if (k == "qs_q_stages") {
    if (value < 2 || value > kQsMaxQStages) return fail(B2F_ERR_INVALID, "qs_q_stages must be in [2, 4]");
    idx->qs_q_stages = static_cast<int>(value);
  } else if (k == "qs_half_stage") {
    idx->qs_half_stage = value ? 1 : 0;
  } else if (k == "center") {
    if (idx->ntotal > 0) return fail(B2F_ERR_INVALID, "center can only be changed on an empty index");
    idx->center = value ? 1 : 0;
  } else if (k == "synth_mean_shift") {
    if (value < 0 || value > 4096) return fail(B2F_ERR_INVALID, "synth_mean_shift must be in [0, 4096]");
    idx->synth_mean_shift = static_cast<int>(value);
  } else if (k == "l2_prefetch") {
    if (value < 0 || value > 8) return fail(B2F_ERR_INVALID, "l2_prefetch must be 0 (off) or a distance of 1..8 tiles");
    idx->l2_prefetch = static_cast<int>(value);
  } else if (k == "tighten") {
    if (value < 0 || value > 1000000) return fail(B2F_ERR_INVALID, "tighten must be 0 (off) or a pause in ns <= 1e6");
    idx->tighten = static_cast<int>(value);
  } else if (k == "tighten_adaptive") {
    idx->tighten_adaptive = value ? 1 : 0;
  } else if (k == "xchg_defer") {
    idx->xchg.defer = value ? 1 : 0;
  } else if (k == "bootstrap") {
    idx->bootstrap = value ? 1 : 0;
  } else if (k == "worst_case_margin") {
    idx->worst_case_margin = value ? 1 : 0;
  } else if (k == "profile") {
    idx->profile = value ? 1 : 0;
  } else if (k == "scan_max_auto") {
    if (value < 0 || value > kScanMaxQ) return fail(B2F_ERR_INVALID, "scan_max_auto must be in [0, 32]");
    idx->scan_max_auto = static_cast<int>(value);
  } else {
    return fail(B2F_ERR_INVALID, "unknown option '" + k + "'");
  }
  return B2F_OK;
}

int b2f_get_stat(const b2f_index* idx, const char* key, double* out) {
  if (!idx || !key || !out) return fail(B2F_ERR_INVALID, "bad stat arguments");
  const std::string k(key);
  Stats s = idx->stats;          // index-level counters (merges, exchange) + the sum over shards
  for (const Shard& S : idx->shards) {
    s.launches += S.stats.launches; s.phases += S.stats.phases; s.candidates += S.stats.candidates;
    s.fallback_queries += S.stats.fallback_queries; s.passes += S.stats.passes; s.qs_passes += S.stats.qs_passes; s.score_ms += S.stats.score_ms;
    s.ovf_area += S.stats.ovf_area; s.ovf_survivors += S.stats.ovf_survivors;
    s.score_launches += S.stats.score_launches; s.score_rows += S.stats.score_rows; s.select_ms += S.stats.select_ms;
    s.xchg_ms += S.stats.xchg_ms;
  }
  if (!idx->shards.empty()) {
    s.path = idx->shards[0].stats.path;
    s.passes = idx->shards[0].stats.passes;   // passes / phases are per search, not per shard
    s.qs_passes = idx->shards[0].stats.qs_passes;
    s.phases = idx->shards[0].stats.phases;
  }
  if (k == "shadow_format") *out = idx->shards.empty() ? 0 : idx->shards[0].fmt;   // 0 none, 1 bf16, 2 int8
  else if (k == "generation") *out = static_cast<double>(idx->generation.load());   // bumped by every add and reset
  else if (k == "shadow_rho") *out = idx->shards.empty() ? 0 : idx->shards[0].rho;  // AUTO: median 2 eps8 / sigma
  else if (k == "launches") *out = s.launches;
  else if (k == "phases") *out = s.phases;
  else if (k == "candidates") *out = s.candidates;
  else if (k == "fallback_queries") *out = s.fallback_queries;
  else if (k == "path") *out = s.path;
  else if (k == "passes") *out = s.passes;
  else if (k == "qs_passes") *out = s.qs_passes;
  else if (k == "overflow_area") *out = s.ovf_area;
  else if (k == "overflow_survivors") *out = s.ovf_survivors;
  else if (k == "score_ms") *out = s.score_ms;
  else if (k == "score_launches") *out = s.score_launches;
  else if (k == "score_rows") *out = s.score_rows;
  else if (k == "select_ms") *out = s.select_ms;
  else if (k == "xchg_ms") *out = s.xchg_ms;
  else if (k == "xchg_timeout") {
    *out = idx->merge_flag_host ? static_cast<double>(idx->merge_flag_host[1]) : 0.0;
  }
  else if (k == "merge_saw_overflow") {   // read-and-clear; meaningful after the stream has been synchronised
    *out = idx->merge_flag_host ? static_cast<double>(*idx->merge_flag_host) : 0.0;
    if (idx->merge_flag_host) *idx->merge_flag_host = 0;
  }
  else return fail(B2F_ERR_INVALID, "unknown stat '" + k + "'");
  return B2F_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Resident load of a flat shard file (SURVEY.md §8 f1): what replaces `pickle.load` + `index.add` of the
// reference's block loop (drivers/run_convdr_inference.py:161-180), whose 118 GB of unpickling + pageable
// H2D per run is its real wall-clock cost.  Reader threads pread() fixed-size pieces of the row region into a
// ring of pinned staging buffers; the calling thread queues one cudaMemcpyAsync per piece as soon as it is
// filled, two copies in flight, so file reads (page cache or disk), PCIe and — at the end — the ingest kernel
// (bf16 shadow + bounds, ~1 ms per million rows) overlap.  One call per shard; calls for different shards may
// run concurrently from different host threads (every GPU has its own PCIe link).
// ---------------------------------------------------------------------------------------------------------
namespace {

#pragma pack(push, 1)
struct FlatHeader {              // convdr_b200/blocks.py `_HEADER` = "<8sIIQIQQ"
  char magic[8];
  uint32_t version, d;
  uint64_t n;
  uint32_t dtype;
  uint64_t rows_off, ids_off;
};
#pragma pack(pop)
static_assert(sizeof(FlatHeader) == 44, "header layout is part of the file format");

bool pread_all(int fd, void* dst, size_t bytes, off_t off) {
  char* p = static_cast<char*>(dst);
  while (bytes > 0) {
    const ssize_t r = pread(fd, p, bytes, off);
    if (r <= 0) return false;
    p += r; off += r; bytes -= static_cast<size_t>(r);
  }
  return true;
}

}  // namespace

extern "C" int b2f_add_flat_file(b2f_index* idx, int shard, const char* path, int n_threads, double* seconds_out,
                                 double* gbytes_out) {
  if (!idx || !path || shard < 0 || shard >= static_cast<int>(idx->shards.size()))
    return fail(B2F_ERR_INVALID, "bad add_flat_file arguments");
  B2F_TRY(settle_pending(idx));
  Shard& S = idx->shards[shard];
  if (S.n > 0 && !S.has_ids) return fail(B2F_ERR_INVALID, "cannot mix add() and labelled rows on a non-empty shard");
  const int fd = open(path, O_RDONLY);
  if (fd < 0) return fail(B2F_ERR_INVALID, std::string("cannot open ") + path);
  struct FdGuard { int fd; ~FdGuard() { close(fd); } } guard{fd};
  FlatHeader h;
  struct stat st;
  if (fstat(fd, &st) != 0 || !pread_all(fd, &h, sizeof(h), 0) || std::memcmp(h.magic, "B2FSHARD", 8) != 0)
    return fail(B2F_ERR_INVALID, std::string(path) + ": not a b2f flat shard");
  if (h.version != 1 || h.dtype != 0 || h.d != static_cast<uint32_t>(kD))
    return fail(B2F_ERR_INVALID, std::string(path) + ": unsupported version / dtype / dimension");
  const int64_t n = static_cast<int64_t>(h.n);
  if (h.rows_off + static_cast<uint64_t>(n) * kD * 4 > h.ids_off || h.ids_off + static_cast<uint64_t>(n) * 8 > static_cast<uint64_t>(st.st_size))
    return fail(B2F_ERR_INVALID, std::string(path) + ": file shorter than its header claims");
  if (seconds_out) *seconds_out = 0.0;
  if (gbytes_out) *gbytes_out = 0.0;
  if (n == 0) return B2F_OK;
  if (S.n + n >= 0xfffffff0ll) return fail(B2F_ERR_INVALID, "a shard holds at most 2^32-16 rows");
  ++idx->generation;
  CU_TRY(cudaSetDevice(S.dev));
  CU_TRY(cudaStreamSynchronize(S.stream));
  if (!S.has_ids) {
    S.has_ids = true;
    if (S.cap > 0 && !S.idmap) B2F_TRY(dev_alloc(&S.idmap, static_cast<size_t>(S.cap)));
  }
  B2F_TRY(ensure_capacity(idx, S, S.n + n));
  const auto t_begin = std::chrono::steady_clock::now();

  constexpr int64_t kPieceRows = kLoadPieceRows;
  constexpr int kBufs = kLoadBufs;
  const size_t piece_bytes = static_cast<size_t>(kPieceRows) * kD * 4;
  const int64_t n_pieces = (n + kPieceRows - 1) / kPieceRows;
  // reader threads: a pread from the page cache is a ~3 GB/s memcpy, a PCIe 5 x16 link takes ~50 GB/s: by
  // default the host's cores are shared out over the shards (each shard is loaded by its own caller thread)
  const int hw = static_cast<int>(std::max(1u, std::thread::hardware_concurrency()));
  const int T = n_threads > 0 ? std::min(n_threads, 32)
                              : std::max(2, std::min(12, hw / static_cast<int>(idx->shards.size())));
  char** bufs = S.load_bufs;
  cudaEvent_t* evs = S.load_evs;
  int rc = B2F_OK;
  for (int b = 0; b < kBufs && rc == B2F_OK; ++b) {   // pinned allocations are slow (~100 ms): kept for the next file
    if ((!bufs[b] && cudaMallocHost(reinterpret_cast<void**>(&bufs[b]), piece_bytes) != cudaSuccess) ||
        (!evs[b] && cudaEventCreateWithFlags(&evs[b], cudaEventDisableTiming) != cudaSuccess)) {
      (void)cudaGetLastError();
      rc = fail(B2F_ERR_OOM, "pinned staging allocation failed");
    }
  }
  // piece state: filled[i] set by its reader, released[i] set by this thread once the copy out of the buffer is done
  std::vector<std::atomic<int>> filled(static_cast<size_t>(n_pieces)), released(static_cast<size_t>(n_pieces));
  for (auto& a : filled) a.store(0);
  for (auto& a : released) a.store(0);
  std::atomic<int> failed{0};
  std::mutex m;
  std::condition_variable cv;
  std::vector<std::thread> readers;
  if (rc == B2F_OK) {
    for (int t = 0; t < T; ++t) {
      readers.emplace_back([&, t] {
        for (int64_t i = t; i < n_pieces && !failed.load(); i += T) {
          if (i >= kBufs) {   // the buffer is reused: wait until piece i - kBufs has left it
            std::unique_lock<std::mutex> lk(m);
            cv.wait(lk, [&] { return released[static_cast<size_t>(i - kBufs)].load() || failed.load(); });
            if (failed.load()) return;
          }
          const int64_t r0 = i * kPieceRows, rows = std::min<int64_t>(kPieceRows, n - r0);
          if (!pread_all(fd, bufs[i % kBufs], static_cast<size_t>(rows) * kD * 4,
                         static_cast<off_t>(h.rows_off + static_cast<uint64_t>(r0) * kD * 4)))
            failed.store(1);
          { std::lock_guard<std::mutex> lk(m); filled[static_cast<size_t>(i)].store(1); }
          cv.notify_all();
        }
      });
    }
    // labels: one read, one copy (8 bytes per row)
    std::vector<int64_t> ids(static_cast<size_t>(n));
    if (!pread_all(fd, ids.data(), static_cast<size_t>(n) * 8, static_cast<off_t>(h.ids_off))) failed.store(1);
    if (!failed.load() &&
        cudaMemcpyAsync(S.idmap + S.n, ids.data(), static_cast<size_t>(n) * 8, cudaMemcpyHostToDevice, S.stream) != cudaSuccess)
      failed.store(2);
    if (!failed.load() && cudaStreamSynchronize(S.stream) != cudaSuccess) failed.store(2);   // `ids` is pageable and local
    for (int64_t i = 0; i < n_pieces && !failed.load(); ++i) {
      {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return filled[static_cast<size_t>(i)].load() || failed.load(); });
      }
      if (failed.load()) break;
      const int64_t r0 = i * kPieceRows, rows = std::min<int64_t>(kPieceRows, n - r0);
      if (cudaMemcpyAsync(S.x32 + (S.n + r0) * kD, bufs[i % kBufs], static_cast<size_t>(rows) * kD * 4,
                          cudaMemcpyHostToDevice, S.stream) != cudaSuccess ||
          cudaEventRecord(evs[i % kBufs], S.stream) != cudaSuccess) {
        failed.store(2);
        break;
      }
      if (i >= 2) {   // two copies stay queued; the one before them has finished or is about to
        if (cudaEventSynchronize(evs[(i - 2) % kBufs]) != cudaSuccess) { failed.store(2); break; }
        { std::lock_guard<std::mutex> lk(m); released[static_cast<size_t>(i - 2)].store(1); }
        cv.notify_all();
      }
    }
    if (cudaStreamSynchronize(S.stream) != cudaSuccess && !failed.load()) failed.store(2);
    {
      std::lock_guard<std::mutex> lk(m);
      for (auto& a : released) a.store(1);
      if (failed.load() == 0) { /* nothing */ }
    }
    cv.notify_all();
    for (std::thread& th : readers) th.join();
    if (failed.load() == 1) rc = fail(B2F_ERR_INVALID, std::string(path) + ": read error");
    else if (failed.load() == 2) { (void)cudaGetLastError(); rc = fail(B2F_ERR_CUDA, "copy of a staged piece failed"); }
  }
  if (rc != B2F_OK) return rc;
  B2F_TRY(ingest_rows(idx, S, n));
  S.n += n;
  CU_TRY(cudaStreamSynchronize(S.stream));
  {
    std::lock_guard<std::mutex> lk(idx->ntotal_mutex);
    idx->ntotal += n;
  }
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
  if (seconds_out) *seconds_out = secs;
  if (gbytes_out) *gbytes_out = static_cast<double>(n) * (kD * 4 + 8) / 1e9;
  return B2F_OK;
}

// Writer side of the flat shard format (SURVEY.md §8 f4; what `gen_passage_embeddings.py:146-169` +
// `utils/util.py:105-111` do with pickles): dump the rows and labels of one device-resident shard to ONE flat
// shard file that b2f_add_flat_file (or numpy.memmap, convdr_b200/blocks.py) reads back.  Rows leave the device
// in 24 MB pieces through two pinned buffers, the copy of piece i+1 overlapping the write of piece i.
extern "C" int b2f_write_flat_file(b2f_index* idx, int shard, const char* path) {
  if (!idx || !path || shard < 0 || shard >= static_cast<int>(idx->shards.size()))
    return fail(B2F_ERR_INVALID, "bad write_flat_file arguments");
  B2F_TRY(settle_pending(idx));
  Shard& S = idx->shards[shard];
  CU_TRY(cudaSetDevice(S.dev));
  CU_TRY(cudaStreamSynchronize(S.stream));
  const int64_t n = S.n;
  const size_t piece_bytes = static_cast<size_t>(kLoadPieceRows) * kD * 4;
  for (int b = 0; b < 2; ++b) {
    if ((!S.load_bufs[b] && cudaMallocHost(reinterpret_cast<void**>(&S.load_bufs[b]), piece_bytes) != cudaSuccess) ||
        (!S.load_evs[b] && cudaEventCreateWithFlags(&S.load_evs[b], cudaEventDisableTiming) != cudaSuccess)) {
      (void)cudaGetLastError();
      return fail(B2F_ERR_OOM, "pinned staging allocation failed");
    }
  }
  // labels: the explicit ones, or the implicit ids of the segments
  std::vector<int64_t> ids(static_cast<size_t>(n));
  if (n > 0) {
    if (S.has_ids) {
      CU_TRY(cudaMemcpy(ids.data(), S.idmap, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToHost));
    } else {
      for (const Seg& sg : S.segs)
        for (int64_t i = 0; i < sg.count; ++i) ids[static_cast<size_t>(sg.local_start + i)] = sg.global_start + i;
    }
  }
  FlatHeader h;
  std::memcpy(h.magic, "B2FSHARD", 8);
  h.version = 1; h.d = kD; h.n = static_cast<uint64_t>(n); h.dtype = 0;
  h.rows_off = 64;
  h.ids_off = static_cast<uint64_t>(round_up(static_cast<int64_t>(h.rows_off) + n * kD * 4, 64));
  const std::string tmp = std::string(path) + ".tmp";
  FILE* f = std::fopen(tmp.c_str(), "wb");
  if (!f) return fail(B2F_ERR_INVALID, "cannot create " + tmp);
  auto bail = [&](int code, const std::string& msg) { std::fclose(f); std::remove(tmp.c_str()); return fail(code, msg); };
  char head[64] = {0};
  std::memcpy(head, &h, sizeof(h));
  if (std::fwrite(head, 1, 64, f) != 64) return bail(B2F_ERR_INVALID, "write error on " + tmp);
  const int64_t n_pieces = (n + kLoadPieceRows - 1) / kLoadPieceRows;
  auto piece_rows = [&](int64_t i) { return std::min<int64_t>(kLoadPieceRows, n - i * kLoadPieceRows); };
  for (int64_t i = 0; i <= n_pieces; ++i) {
    if (i < n_pieces) {   // queue the copy of piece i
      if (cudaMemcpyAsync(S.load_bufs[i & 1], S.x32 + i * kLoadPieceRows * kD, static_cast<size_t>(piece_rows(i)) * kD * 4,
                          cudaMemcpyDeviceToHost, S.stream) != cudaSuccess ||
          cudaEventRecord(S.load_evs[i & 1], S.stream) != cudaSuccess) {
        (void)cudaGetLastError();
        return bail(B2F_ERR_CUDA, "device-to-host copy failed");
      }
    }
    if (i >= 1) {         // ... while piece i-1 goes to the file
      if (cudaEventSynchronize(S.load_evs[(i - 1) & 1]) != cudaSuccess) { (void)cudaGetLastError(); return bail(B2F_ERR_CUDA, "device-to-host copy failed"); }
      const size_t bytes = static_cast<size_t>(piece_rows(i - 1)) * kD * 4;
      if (std::fwrite(S.load_bufs[(i - 1) & 1], 1, bytes, f) != bytes) return bail(B2F_ERR_INVALID, "write error on " + tmp);
    }
  }
  const size_t pad = static_cast<size_t>(h.ids_off - (h.rows_off + static_cast<uint64_t>(n) * kD * 4));
  const char zeros[64] = {0};
  if (pad && std::fwrite(zeros, 1, pad, f) != pad) return bail(B2F_ERR_INVALID, "write error on " + tmp);
  if (n && std::fwrite(ids.data(), 8, static_cast<size_t>(n), f) != static_cast<size_t>(n)) return bail(B2F_ERR_INVALID, "write error on " + tmp);
  if (std::fclose(f) != 0) { std::remove(tmp.c_str()); return fail(B2F_ERR_INVALID, "write error on " + tmp); }
  if (std::rename(tmp.c_str(), path) != 0) { std::remove(tmp.c_str()); return fail(B2F_ERR_INVALID, std::string("cannot rename to ") + path); }
  return B2F_OK;
}

extern "C" int b2f_rank_dedup_device(b2f_index* idx, const int64_t* I_dev, const float* D32_dev, const double* D64_dev,
                                     int64_t nq, int64_t in_stride, int topN, const int64_t* offset2pid_dev,
                                     int64_t n_offsets, int64_t* pid_out_dev, double* score_out_dev, int* count_out_dev) {
  if (!idx || nq < 0 || topN < 1 || topN > B2F_MAX_K || in_stride < topN || !I_dev || (!D32_dev && !D64_dev) ||
      !offset2pid_dev || n_offsets < 1 || !pid_out_dev || !score_out_dev || !count_out_dev)
    return fail(B2F_ERR_INVALID, "bad rank_dedup arguments");
  if (nq == 0) return B2F_OK;
  Shard& S = idx->shards[0];
  CU_TRY(cudaSetDevice(S.dev));
  rank_dedup_kernel<<<static_cast<int>(nq), kDedupThreads, static_cast<size_t>(topN) * 12, S.stream>>>(
      I_dev, D32_dev, D64_dev, in_stride, topN, offset2pid_dev, n_offsets, pid_out_dev, score_out_dev, count_out_dev);
  CU_TRY(cudaGetLastError());
  idx->stats.launches += 1;
  CU_TRY(cudaStreamSynchronize(S.stream));
  return B2F_OK;
}
