/*
 * b2f.h — C ABI of the B200-native exact inner-product top-k engine ("b2f" = B200 flat).
 *
 * This is the drop-in boundary for the dense-retrieval hot path of thunlp/ConvDR:
 * the faiss.IndexFlatIP add / search / reset calls made by
 *   drivers/run_convdr_inference.py::search_one_by_one   (reference :157-242)
 * and the index construction in main()                   (reference :327-370).
 *
 * The reference has no FFI of its own — it binds FAISS through SWIG — so every
 * entry point below cites the FAISS-Python call site in the reference that it
 * replaces.  The Python facade (convdr_b200/faiss_compat.py) binds these with
 * ctypes; INTEGRATION.md shows the stub a ConvDR maintainer would add.
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary;
 *   - every function returns 0 on success, a B2F_ERR_* code otherwise, and never
 *     throws; b2f_last_error() returns a thread-local description;
 *   - "host" pointers are ordinary (pageable or pinned) host memory, "dev"
 *     pointers are CUDA device memory on the index's (first shard's) device;
 *   - vectors are row-major float32 [n, d], d fixed at 768 (reference :353);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with B2F_ERR_NO_DEVICE.
 */
#ifndef B2F_H_
#define B2F_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2F_DIM 768 /* reference drivers/run_convdr_inference.py:353 hard-codes 768 */
#define B2F_MAX_K 2048 /* FAISS-GPU's own limit; reference uses 100 (:316-319) and 1000 */

enum {
  B2F_OK = 0,
  B2F_ERR_INVALID = 1,   /* bad argument (dimension, k, null pointer, ...) */
  B2F_ERR_NO_DEVICE = 2, /* no usable CUDA device / driver */
  B2F_ERR_CUDA = 3,      /* a CUDA runtime / driver call failed */
  B2F_ERR_OOM = 4,       /* device allocation failed */
  B2F_ERR_INTERNAL = 5   /* selection pipeline failed to converge (a bug) */
};

typedef struct b2f_index b2f_index;

/* Scoring engines (b2f_set_option "path"). AUTO picks by batch size. */
enum {
  B2F_PATH_AUTO = 0,
  B2F_PATH_SCAN_F32 = 1,   /* fp32 128-bit loads + warp-shuffle dots (small batches)   */
  B2F_PATH_SCAN_EXACT = 2, /* same scan, fp64 accumulation, total-order keys (robust fallback) */
  B2F_PATH_UMMA_BF16 = 3   /* TMA + tcgen05/TMEM bf16 prefilter, exact rescoring        */
};

/* faiss.get_num_gpus()                                  reference :327 */
int b2f_device_count(void);

/* faiss.IndexFlatIP(768) [+ index_cpu_to_gpu_multiple(vres, vdev, cpu_index, co)
 * with co.shard = True]                                 reference :353, :355-368
 * devices == NULL or n_dev == 0 -> device 0 only.  With n_dev > 1 each add() is
 * split in n_dev contiguous chunks (FAISS IndexShards, successive ids).        */
int b2f_create(int d, const int* devices, int n_dev, b2f_index** out);

/* index.add(passage_embedding)                          reference :180
 * Copies x (the driver deletes its array right after, :203-204); ids are
 * implicit and continue from ntotal.                                          */
int b2f_add(b2f_index* idx, const float* x_host, int64_t n);

/* Same, with explicit int64 labels returned by search instead of positions —
 * folds `passage_embedding2id[I]` (reference :190) into the engine.           */
int b2f_add_with_ids(b2f_index* idx, const float* x_host, const int64_t* ids_host, int64_t n);

/* Zero-copy variant: x_dev is device memory on shard `shard`'s device.         */
int b2f_add_device(b2f_index* idx, int shard, const float* x_dev, int64_t n);

/* Resident load ("search all at once", reference README.md:216; replaces the
 * per-run `pickle.load` + `index.add` of reference :161-180): stream ONE flat
 * shard file (convdr_b200/blocks.py: 64-byte header, float32 rows, int64 passage
 * offsets) into shard `shard`.  n_threads reader threads pread() 24 MB pieces into
 * pinned staging buffers while earlier pieces cross PCIe; the stored offsets become
 * the labels search returns (like b2f_add_with_ids).  Calls for DIFFERENT shards may
 * run concurrently from different host threads.  seconds_out / gbytes_out (may be
 * NULL) report the wall time and the bytes moved.                                 */
int b2f_add_flat_file(b2f_index* idx, int shard, const char* path, int n_threads,
                      double* seconds_out, double* gbytes_out);

/* Writer side of the same format (reference drivers/gen_passage_embeddings.py:146-169
 * + utils/util.py:105-111 dump each rank's arrays as pickles): write the rows and
 * labels of shard `shard` (explicit ids, or the implicit positions) to ONE flat shard
 * file, straight from device memory through pinned staging buffers (the copy of a
 * piece overlaps the write of the previous one); written to `path`.tmp, then renamed. */
int b2f_write_flat_file(b2f_index* idx, int shard, const char* path);

/* Pre-size every shard for `n_per_shard` rows (avoids regrowth copies).        */
int b2f_reserve(b2f_index* idx, int64_t n_per_shard);

/* Append n synthetic rows generated on device: counter-based Philox4x32-10,
 * integer Irwin-Hall components, exact L2 normalisation, times `norm`.
 * Row r of stream (seed, stream) is bit-identical to convdr_b200/synth.py and
 * oracle/synth.c, so CPU checks can regenerate any row.  Rows
 * [first_row, first_row+n) are appended to shard `shard`; their ids are
 * id_base .. id_base+n-1.                                                      */
int b2f_add_synthetic(b2f_index* idx, int shard, int64_t first_row, int64_t n, uint64_t seed,
                      uint64_t stream, float norm, int64_t id_base);

/* D, I = index.search(query_embedding, topN)            reference :182
 * q_host float32 [nq, d]; D float32 [nq, k] sorted descending; I int64 [nq, k];
 * missing results (ntotal < k) are padded with D = -FLT_MAX, I = -1.
 * Scores are the exactly-rounded fp32 value of the fp64 dot product; order is
 * (score desc, insertion position asc).                                        */
int b2f_search(b2f_index* idx, const float* q_host, int64_t nq, int k, float* D_host,
               int64_t* I_host);

/* Filtered search: faiss index.search(x, k, params=faiss.SearchParameters(sel=...)).
 * A selector is built once against one index and reused for many searches.  It is
 * evaluated on the labels search returns (explicit ids, or the implicit positions):
 *   B2F_SEL_RANGE   imin <= id < imax                            (IDSelectorRange)
 *   B2F_SEL_BATCH   id in ids_host[0 .. n_ids), any order, duplicates allowed
 *                                                                (IDSelectorBatch / IDSelectorArray)
 *   B2F_SEL_BITMAP  (bitmap_host[id >> 3] >> (id & 7)) & 1; ids >= 8 n_bytes are not
 *                   selected                                     (IDSelectorBitmap)
 * invert != 0 selects the complement (IDSelectorNot).  Per shard the selector keeps a
 * row bitmap and the lists of the row tiles that hold a selected row: a filtered search
 * streams only those tiles and only selected rows can enter the results, which stay
 * exact; fewer than k selected rows pad with D = -FLT_MAX, I = -1 like faiss.
 * Adding rows or resetting the index makes a selector stale: searching with it then
 * fails with B2F_ERR_INVALID.  Destroy a selector before its index;
 * b2f_selector_destroy first settles the searches still in flight.
 * A NULL selector in the *_sel entry points means no filter.                   */
typedef struct b2f_selector b2f_selector;
enum { B2F_SEL_RANGE = 1, B2F_SEL_BATCH = 2, B2F_SEL_BITMAP = 3 };
int b2f_selector_create(b2f_index* idx, int kind, int invert, int64_t imin, int64_t imax,
                        const int64_t* ids_host, int64_t n_ids, const uint8_t* bitmap_host,
                        int64_t n_bytes, b2f_selector** out);
/* Number of selected rows over all shards. */
int b2f_selector_count(const b2f_selector* sel, int64_t* selected_out);
void b2f_selector_destroy(b2f_selector* sel);
int b2f_search_sel(b2f_index* idx, const b2f_selector* sel, const float* q_host, int64_t nq, int k,
                   float* D_host, int64_t* I_host);

/* Device-resident variant, for any number of shards: q_dev / D_dev / I_dev live on
 * the first shard's device.  The search starts on that shard's index stream
 * (b2f_stream(idx, 0)), so the caller orders q_dev's producer before it; the other
 * shards copy the queries from there, and the merge of their results runs on that
 * stream.  Every stream is synchronised before returning (the candidate-overflow
 * flags are checked on the host, overflowed queries re-run and merged again).  */
int b2f_search_device(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                      int64_t* I_dev);

/* Asynchronous form of b2f_search_device, for any number of shards (q_dev, D_dev,
 * I_dev on the first shard's device): only enqueues and returns; up to 16 searches
 * may be in flight.  Results are ordered on the first shard's index stream
 * (b2f_stream(idx, 0)): later work on that stream may consume them (q_dev must stay
 * valid); the host may read them after b2f_search_finish(), which waits for the
 * streams and re-runs, on the exact engine, any query whose candidate list
 * overflowed (flags are written by the last kernel of a pass straight into mapped
 * host memory) and, with several shards, merges that search again.  Until then such
 * a row carries id -2 in its first slot, the merged row of a multi-shard search
 * too; every other row is final once the stream has passed it.  Every other entry
 * point settles pending searches first.  This is what lets a caller (the NCCL
 * layout in convdr_b200/dist.py, bench.py) queue search -> all-gather -> merge, or
 * several batches, without a host round trip in between.                       */
int b2f_search_device_async(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                            int64_t* I_dev);
int b2f_search_finish(b2f_index* idx);
int b2f_search_device_async_sel(b2f_index* idx, const b2f_selector* sel, const float* q_dev, int64_t nq,
                                int k, float* D_dev, int64_t* I_dev);

/* Merge `n_parts` per-shard results [n_parts, nq, k] (device memory, each part
 * sorted descending, padded with -FLT_MAX / -1) into the global top-k
 * [nq, k] — the device-side replacement of the Python 2-way merge
 * (reference :206-229) and of FAISS IndexShards' CPU merge.  Used after the
 * NCCL all-gather in the one-process-per-GPU layout.                           */
int b2f_merge_device(b2f_index* idx, const float* D_parts_dev, const int64_t* I_parts_dev,
                     int n_parts, int64_t nq, int k, float* D_dev, int64_t* I_dev);

/* Same merge, asynchronous (enqueued on the index stream), over PACKED parts as
 * they arrive from ONE all-gather: part g occupies part_bytes bytes at
 * parts_dev + g*part_bytes and holds D float32 [nq,k] at offset 0 and
 * I int64 [nq,k] at offset i_offset_bytes (both multiples of 8).               */
int b2f_merge_packed_device_async(b2f_index* idx, const void* parts_dev, int n_parts,
                                  int64_t part_bytes, int64_t i_offset_bytes, int64_t nq, int k,
                                  float* D_dev, int64_t* I_dev);

/* EvalDevQuery's ranking clean-up on device (reference :43-69): for each of the nq
 * rows of I_dev (passage offsets, best first; row stride in_stride >= topN) take the
 * first topN entries, translate pid = offset2pid[offset] (a negative offset indexes
 * from the end, like the Python list it replaces), drop every pid that already
 * appeared at a better rank, compact the survivors to the front (pid_out, score_out:
 * [nq, topN]; the tail is filled with pid 0 / score 0 like the reference's
 * `[(0, 0)] * topN`) and report how many survived (count_out [nq]).  Scores come
 * from D32_dev (float32) or D64_dev (float64), whichever is non-NULL.              */
int b2f_rank_dedup_device(b2f_index* idx, const int64_t* I_dev, const float* D32_dev,
                          const double* D64_dev, int64_t nq, int64_t in_stride, int topN,
                          const int64_t* offset2pid_dev, int64_t n_offsets,
                          int64_t* pid_out_dev, double* score_out_dev, int* count_out_dev);

/* Peer-memory exchange for the one-process-per-GPU layout (one single-shard index
 * per rank, all ranks on one NVLink/NVSwitch node): replaces ncclAllGather +
 * merge by two kernels that talk through CUDA-IPC-mapped buffers.
 *   b2f_xchg_create   allocates this rank's exchange buffer for batches up to
 *                     max_nq x max_k and returns its 64-byte cudaIpcMemHandle_t;
 *   b2f_xchg_connect  takes the world x 64 bytes of handles of ALL ranks (rank
 *                     order; exchanged by the caller, e.g. torch.distributed);
 *   b2f_search_xchg_async  local search (ids must be global: add_with_ids /
 *                     add_synthetic) -> push of the packed [nq,k] part into every
 *                     rank's buffer over NVLink -> wait for all ranks' parts ->
 *                     merge into D_dev / I_dev; all enqueued, settle with
 *                     b2f_search_finish.  Collective: every rank must call it with
 *                     the same nq, k.  repush_only != 0 skips the local search
 *                     (used after finish() re-ran overflowed queries; stat
 *                     "merge_saw_overflow" tells every rank when that is needed).
 * Stat "xchg_timeout" is 1 if a rank's part never arrived (~4 s).               */
int b2f_xchg_create(b2f_index* idx, int rank, int world, int64_t max_nq, int max_k, void* handle_out);
int b2f_xchg_connect(b2f_index* idx, const void* handles);
int b2f_search_xchg_async(b2f_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                          int64_t* I_dev, int repush_only);
/* Same collective, filtered: every rank passes a selector built from the same
 * description on its own index.                                                */
int b2f_search_xchg_async_sel(b2f_index* idx, const b2f_selector* sel, const float* q_dev, int64_t nq,
                              int k, float* D_dev, int64_t* I_dev, int repush_only);
/* The same collective as ONE host-buffer call (the end-to-end path of the
 * one-process-per-GPU layout): upload of q_host (straight from the caller's buffer
 * when it is page-locked), local search, push, wait + merge — whose result rows are
 * stored directly into page-locked host memory (the caller's arrays when they are
 * page-locked, else a staging buffer + one memcpy) —, one host wait, and the overflow
 * protocol (local re-run + collective re-push when any rank's list overflowed).     */
int b2f_search_xchg_host(b2f_index* idx, const float* q_host, int64_t nq, int k, float* D_host,
                         int64_t* I_host);
/* The merge of an exchange step is enqueued one search later (the ranks are then
 * coupled with one step of slack instead of a barrier per search; option
 * "xchg_defer", default 1) or by b2f_search_finish.  b2f_xchg_flush enqueues a
 * merge that is still owed WITHOUT waiting, so that a caller can queue its own
 * work (a download of D_dev / I_dev) behind it before the one host wait.        */
int b2f_xchg_flush(b2f_index* idx);

/* faiss IndexFlat.reconstruct_n(i0, ni): copy stored rows [row0, row0+n) of shard
 * `shard` (shard-local positions) back to host memory — inspection / tests.    */
int b2f_reconstruct_n(b2f_index* idx, int shard, int64_t row0, int64_t n, float* out_host);

/* Rows by label: faiss index.reconstruct(key) / reconstruct_batch(keys) / search_and_reconstruct(x, k).
 * A label is what search returns: the explicit id (b2f_add_with_ids, flat files) or the position given by the
 * shard's segments (b2f_add, b2f_add_device; b2f_add_synthetic with its id_base).  Each shard finds a label's
 * row on the GPU through a label index built by its first lookup after an add or reset:
 *   - segment labels: the segments themselves (nothing is built);
 *   - explicit labels stored in ascending order (e.g. one ConvDR block per shard): the label map, in place;
 *   - any other explicit labels: a sorted (label, row) copy, 12 bytes per row (stat "label_index_bytes"),
 *     freed by the next add or reset.
 * The rows are gathered on the GPU, across shards, and returned bit for bit as stored (what b2f_reconstruct_n
 * returns).  A lookup fails with B2F_ERR_INVALID, naming the label, when a label is not in the index, is negative
 * (b2f_reconstruct_batch), or is held by more than one row, within a shard or across shards (duplicate labels
 * stay legal for search; only their lookup is ambiguous).
 *
 * b2f_reconstruct_batch: keys_host [n] in any order, repeats allowed -> out_host float32 [n, d].
 * b2f_search_and_reconstruct_sel: b2f_search_sel (sel may be NULL: no filter), then the rows of the result labels:
 *   R_host float32 [nq, k, d].  D and I are exactly those of b2f_search_sel.  A -1 label (padding: fewer than k
 *   rows, or fewer than k selected rows) gets a row of 0xFF bytes (NaN in every component), as faiss's
 *   Index::search_and_reconstruct does.
 * b2f_search_and_reconstruct_device_sel: the same with q_dev, D_dev, I_dev and R_dev on the first shard's
 *   device; ordered on b2f_stream(idx, 0) like b2f_search_device, synchronised before returning.           */
int b2f_reconstruct_batch(b2f_index* idx, const int64_t* keys_host, int64_t n, float* out_host);
int b2f_search_and_reconstruct_sel(b2f_index* idx, const b2f_selector* sel, const float* q_host, int64_t nq, int k,
                                   float* D_host, int64_t* I_host, float* R_host);
int b2f_search_and_reconstruct_device_sel(b2f_index* idx, const b2f_selector* sel, const float* q_dev, int64_t nq,
                                          int k, float* D_dev, int64_t* I_dev, float* R_dev);

/* index.reset()                                         reference :202 */
int b2f_reset(b2f_index* idx);

/* index.ntotal */
int64_t b2f_ntotal(const b2f_index* idx);

/* Rows on one shard / number of shards. */
int64_t b2f_shard_rows(const b2f_index* idx, int shard);
int b2f_num_shards(const b2f_index* idx);

/* Raw CUDA stream (cudaStream_t) of shard `shard`, for event timing in bench.py. */
void* b2f_stream(b2f_index* idx, int shard);

/* Tuning knobs:
 *   "path" (B2F_PATH_*; AUTO = the tensor engine whenever a shadow exists),
 *   "shadow" (the prefilter copy the tensor engine streams: 0 none, 1 bf16, 2 int8 with one scale per
 *       32-row tile (half the bytes per row, a ~4x wider error margin), 3 AUTO (default): int8 when the
 *       first rows of a shard leave the int8 margin narrow against the spread of the scores, bf16
 *       otherwise; results never depend on it; empty index only), "keep_on_reset" (default 1),
 *   "scan_max_auto" (largest batch AUTO sends to the SIMT scan, default 0 = never),
 *   "center" (default 1: the shadow holds rows minus the mean of the first rows added, so the error
 *       margin follows ||p - mean|| instead of ||p||; empty index only),
 *   "margin_ppm" (scale of the rigorous error margin in parts-per-million, default 1000000),
 *   "worst_case_margin" (1: data-independent 2^-8 bound instead of the per-shard rounding-error
 *       bound; A/B only),
 *   "umma_variant" (tensor engine: 0 auto = QS for passes of up to "qs_max_q" (208) queries, TS above;
 *       2 TS = queries in TMEM, MMA M = 256 query lanes; 3 QS = queries on the MMA N side; 1 = QS with
 *       every query K-block resident in shared memory), "qs_resident_kb" (QS: resident query K-blocks,
 *       default 12; the rest is streamed from L2 through a ring of "qs_q_stages" stages),
 *   "l2_prefetch" (QS: distance in tiles of an optional L2 prefetch warp; default 0 = off, measured slower),
 *   "qs_half_stage" (QS: 8 KB half stages with the 64-byte swizzle when <= 5 full stages fit; default 0, measured slower),
 *   "synth_mean_shift" (b2f_add_synthetic: integer shift M of every component along a fixed sign
 *       vector per seed, 0 = isotropic rows; see convdr_b200/synth.py),
 *   "tighten" (tensor engine: thresholds start at -inf and are tightened inside the one scoring
 *       launch of a pass; minimum pause of the refresher warp in ns, 1..1000000, default 2000),
 *   "tighten_adaptive" (default 1: the pause grows with the elapsed kernel time),
 *   "growth" (phase growth factor of the SIMT scans' phased schedule; also sizes the private list
 *       areas of the tensor engine),
 *   "profile" (1: CUDA events around every scoring / selection launch),
 *   "reset_stats" (any value: zero the counters below).                          */
int b2f_set_option(b2f_index* idx, const char* key, int64_t value);

/* Counters since the last synchronous search started (asynchronous searches
 * accumulate): "launches", "phases", "candidates",
 * "fallback_queries" (queries re-run on the exact engine) and why: "overflow_area" (a private list
 * area was too small), "overflow_survivors" (more rows within the error margin of the k-th score
 * than the survivor buffer holds); "path", "passes", "qs_passes"; with "profile" on also "score_ms",
 * "score_launches", "score_rows" (scoring kernels: device time, launches, rows
 * streamed) and "select_ms" (refresh + final kernels); "shadow_format" (first shard: 0 none,
 * 1 bf16, 2 int8) and "shadow_rho" (AUTO: median 2 eps8 / sigma of the probe, 0 if not measured);
 * "generation" (bumped by every add and reset: a selector built at another generation is stale);
 * "label_index_bytes" (sorted label copies held for b2f_reconstruct_batch and b2f_search_and_reconstruct*, all
 * shards). */
int b2f_get_stat(const b2f_index* idx, const char* key, double* out);

void b2f_destroy(b2f_index* idx);

/* Thread-local description of the last error in this thread. */
const char* b2f_last_error(void);

/* Library build identification ("b2f <version> sm_100a"). */
const char* b2f_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B2F_H_ */
