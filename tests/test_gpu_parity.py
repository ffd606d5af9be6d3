"""GPU parity tests (run on a B200 with `-m gpu`): the CUDA path, called through the C ABI /
faiss facade, against the oracle (FAISS-restated fp32 and fp64 truth) on the same seeded inputs.

Bar (BASELINE.json north_star): ids identical to the reference except at ties within 1e-5 relative
score; scores within 1e-5 relative.  The engine actually reports the correctly rounded fp64 dot, so
against the fp64 truth we additionally require 1e-6.
"""
import os
import tempfile

import numpy as np
import pytest

import convdr_b200.faiss_compat as faiss
from convdr_b200 import FlatIPIndex, driver, synth
from oracle import c_oracle, flat_ip

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# umma_*: the tensor-engine variants — qs (queries streamed on the MMA N side, the default up to 208 queries per
# pass), qsr (same kernel, every query K-block resident in shared memory), ts (queries in TMEM)
# qsh: QS with 8 KB half stages (64B swizzle) wherever <= 5 full stages would fit (161+ queries per pass)
PATHS = ["scan_f32", "scan_exact", "umma_qs", "umma_qsr", "umma_qsh", "umma_ts"]
UMMA_VARIANT = {"umma_qsr": 1, "umma_ts": 2, "umma_qs": 3, "umma_qsh": 3}
RTOL = 1e-5          # the tolerance north_star states
RTOL_TRUTH = 1e-6    # what the exact rescoring actually delivers vs float64


def make_index(path, P=None, devices=None, **opts):
    idx = FlatIPIndex(768, devices=devices)
    if path in UMMA_VARIANT:
        idx.set_option("umma_variant", UMMA_VARIANT[path])
        idx.set_option("qs_half_stage", 1 if path == "umma_qsh" else 0)
        path = "umma_bf16"
    idx.set_option("path", path)
    for k, v in opts.items():
        idx.set_option(k, v)
    if P is not None:
        idx.add(P)
    return idx


def check_against_oracle(D, I, P, Q, k, also_fp32_oracle=True):
    Dt, It = flat_ip.truth_fp64(Q, P, k)
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    r = flat_ip.compare(D, I, Dt, It, score_of, rtol=RTOL)
    assert r["violations"] == 0, r
    valid = It >= 0
    rel = np.abs(D[valid].astype(np.float64) - Dt[valid]) / np.maximum(np.abs(Dt[valid]), 1e-30)
    assert rel.max() <= RTOL_TRUTH, rel.max()
    assert (np.diff(D, axis=1) <= 0).all(), "scores must be sorted descending"
    if also_fp32_oracle:
        Do, Io = flat_ip.knn_inner_product(Q, P, k)
        r2 = flat_ip.compare(D, I, Do, Io, score_of, rtol=RTOL)
        assert r2["violations"] == 0, r2
    return r


@pytest.fixture(scope="module")
def c1_data():
    # BASELINE config 1: 100k x 768, 173 queries
    return c_oracle.synth_block(0, 100000), c_oracle.synth_block(0, 173, stream=1)


@pytest.mark.parametrize("path", PATHS)
def test_config1_100k_173q_top100(path, c1_data):
    P, Q = c1_data
    idx = make_index(path, P)
    assert idx.ntotal == 100000
    D, I = idx.search(Q, 100)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (173, 100)
    r = check_against_oracle(D, I, P, Q, 100)
    assert r["exact_rows"] >= 170
    assert idx.stat("fallback_queries") == 0
    assert int(idx.stat("path")) == {"scan_f32": 1, "scan_exact": 2}.get(path, 3)
    if path in UMMA_VARIANT:
        assert idx.stat("qs_passes") == (0 if path == "umma_ts" else 1)
    assert idx.stat("launches") > 0


@pytest.mark.parametrize("path", PATHS)
def test_results_are_bitwise_path_independent(path, c1_data):
    P, Q = c1_data
    ref = make_index("scan_exact", P[:30000])
    D0, I0 = ref.search(Q[:40], 50)
    idx = make_index(path, P[:30000])
    D, I = idx.search(Q[:40], 50)
    np.testing.assert_array_equal(I, I0)
    np.testing.assert_array_equal(D, D0)


@pytest.mark.parametrize("path", ["scan_f32", "umma_qs", "umma_qsr", "umma_ts"])
def test_top1000_selection_pressure(path, c1_data):
    P, Q = c1_data  # BASELINE config 2's k = 1000 (gen_ranking_data.py negatives), reduced rows
    idx = make_index(path, P)
    D, I = idx.search(Q[:64], 1000)
    check_against_oracle(D, I, P, Q[:64], 1000, also_fp32_oracle=False)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("n", [1, 3, 100, 255, 256, 257, 4095, 18943, 18944, 18945, 40001])
def test_ragged_collection_sizes(path, n, c1_data):
    P, Q = c1_data
    idx = make_index(path, P[:n])
    k = 10
    D, I = idx.search(Q[:21], k)
    if n < k:
        assert (I[:, n:] == -1).all() and (D[:, n:] == -np.float32(3.4028234663852886e38)).all()
    check_against_oracle(D, I, P[:n], Q[:21], k)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("nq", [1, 2, 5, 16, 17, 33, 191, 192, 193, 400])
def test_ragged_query_batches(path, nq):
    P = c_oracle.synth_block(0, 20000, seed=3)
    Q = c_oracle.synth_block(0, nq, seed=3, stream=1)
    idx = make_index(path, P)
    D, I = idx.search(Q, 20)
    check_against_oracle(D, I, P, Q, 20)


@pytest.mark.parametrize("path", PATHS)
def test_empty_index_and_k_larger_than_ntotal(path):
    Q = c_oracle.synth_block(0, 5, stream=1)
    idx = make_index(path)
    D, I = idx.search(Q, 4)
    assert (I == -1).all() and (D == -np.float32(3.4028234663852886e38)).all()
    P = c_oracle.synth_block(0, 7)
    idx.add(P)
    D, I = idx.search(Q, 12)
    assert (I[:, 7:] == -1).all()
    assert sorted(I[0, :7].tolist()) == list(range(7))
    check_against_oracle(D, I, P, Q, 12)


@pytest.mark.parametrize("path", PATHS)
def test_two_adds_equal_one_add_and_reset_readd(path):
    P = c_oracle.synth_block(0, 30000, seed=5)
    Q = c_oracle.synth_block(0, 23, seed=5, stream=1)
    a = make_index(path, P)
    b = make_index(path)
    b.add(P[:11111])
    b.add(P[11111:])
    assert a.ntotal == b.ntotal == 30000
    Da, Ia = a.search(Q, 30)
    Db, Ib = b.search(Q, 30)
    np.testing.assert_array_equal(Ia, Ib)
    np.testing.assert_array_equal(Da, Db)
    b.reset()
    assert b.ntotal == 0
    b.add(P[20000:])
    D, I = b.search(Q, 30)
    check_against_oracle(D, I, P[20000:], Q, 30)


@pytest.mark.parametrize("path", PATHS)
def test_known_answers_identity_and_planted(path):
    P = np.zeros((300, 768), dtype=np.float32)
    P[np.arange(300), np.arange(300)] = 1.0
    Q = np.zeros((2, 768), dtype=np.float32)
    Q[0, 5], Q[0, 7] = 2.0, 1.0
    Q[1, 299], Q[1, 0] = 1.0, 0.5
    D, I = make_index(path, P).search(Q, 3)
    assert I[0, :2].tolist() == [5, 7] and D[0, :2].tolist() == [2.0, 1.0]
    assert I[1, :2].tolist() == [299, 0] and D[1, :2].tolist() == [1.0, 0.5]
    assert D[0, 2] == 0.0 and I[0, 2] == 0   # remaining scores tie at 0 -> lowest index (our total order)
    P = c_oracle.synth_block(0, 50000, seed=1)
    q = c_oracle.synth_block(0, 1, seed=1, stream=1)
    plant = {17: 3.0, 41500: 2.5, 999: 2.0, 4: 1.5}
    for row, s in plant.items():
        P[row] = q[0] * np.float32(s)
    D, I = make_index(path, P).search(q, 4)
    assert I[0].tolist() == [17, 41500, 999, 4]
    np.testing.assert_allclose(D[0], [3.0, 2.5, 2.0, 1.5], rtol=1e-6)


@pytest.mark.parametrize("path", PATHS)
def test_all_equal_scores_use_the_total_order(path):
    """Every row identical: all scores tie.  Candidate lists overflow on the filtering engines and
    the exact engine must finish the query (lowest positions win)."""
    row = c_oracle.synth_block(0, 1, seed=2)
    P = np.tile(row, (60000, 1))
    Q = c_oracle.synth_block(0, 3, seed=2, stream=1)
    idx = make_index(path, P)
    D, I = idx.search(Q, 25)
    assert I.tolist() == [list(range(25))] * 3
    if path != "scan_exact":
        assert idx.stat("fallback_queries") == 3


@pytest.mark.parametrize("path", PATHS)
def test_non_unit_norm_rows_scale_28(path):
    P = c_oracle.synth_block(0, 40000, seed=4, norm=28.0)   # real ANCE scale (SURVEY §8c)
    Q = c_oracle.synth_block(0, 19, seed=4, stream=1, norm=28.0)
    D, I = make_index(path, P).search(Q, 50)
    check_against_oracle(D, I, P, Q, 50)


@pytest.mark.parametrize("path", ["umma_qs", "umma_qsr", "umma_ts", "scan_f32"])
@pytest.mark.parametrize("center", [1, 0])
def test_rows_with_a_common_mean_like_layernorm_outputs(path, center):
    """Embeddings that share a large mean component (cos(p, p') ~ 0.9, norm 28: what LayerNorm-ed ANCE
    vectors look like, reference model/models.py:136-145).  Scores are ~706 +- 3.4, so a Cauchy-Schwarz
    margin on the full norms (2 eps ~ 3.7) would put tens of thousands of rows inside the margin of the
    100th score.  With the rows centred at add time the margin follows ||p - mu|| ~ 9 instead: no list
    overflows and the result is the fp64 truth.  center=0 must stay correct (it may fall back)."""
    P = c_oracle.synth_block(0, 100000, seed=51, norm=28.0, mean_shift=443)
    Q = c_oracle.synth_block(0, 64, seed=51, stream=1, norm=28.0, mean_shift=443)
    idx = make_index(path, None, center=center)
    idx.add(P)
    D, I = idx.search(Q, 100)
    check_against_oracle(D, I, P, Q, 100, also_fp32_oracle=False)
    if center:
        assert idx.stat("fallback_queries") == 0


def test_device_synthetic_rows_with_mean_shift_are_bit_identical_to_host():
    idx = make_index("auto", None, synth_mean_shift=443)
    idx.add_synthetic(3000, first_row=777, seed=5, stream=0, norm=28.0)
    want = synth.block(777, 3000, seed=5, stream=0, norm=28.0, mean_shift=443)
    np.testing.assert_array_equal(idx.reconstruct_n(0, 3000), want)
    Q = c_oracle.synth_block(0, 9, seed=5, stream=1, norm=28.0, mean_shift=443)
    D, I = idx.search(Q, 10)
    Do, Io = flat_ip.truth_fp64(Q, want, 10)
    np.testing.assert_array_equal(I, Io + 777)
    assert idx.stat("fallback_queries") == 0


def test_every_pass_starts_without_the_thresholds_of_earlier_searches():
    """The thresholds live in the shard's workspace, and the scoring launch and finalize_kernel filter on
    them from the first tile on: every pass of both tensor kernels must start from tau = -inf, whatever an
    earlier search or an earlier collection of the same index left behind."""
    P = c_oracle.synth_block(0, 3000, seed=61)
    Qa = c_oracle.synth_block(0, 40, seed=61, stream=1, norm=50.0)     # leaves large thresholds behind
    Qb = c_oracle.synth_block(0, 40, seed=63, stream=1, norm=0.01)     # every score far below them
    for path in ("umma_ts", "umma_qs"):
        small = make_index(path, P)
        big = make_index(path, c_oracle.synth_block(0, 60000, seed=62))
        small.search(Qa, 10)
        big.search(Qa, 10)
        D, I = small.search(Qb, 10)
        check_against_oracle(D, I, P, Qb, 10)
        big.reset()
        big.add(P)
        D, I = big.search(Qb, 10)
        check_against_oracle(D, I, P, Qb, 10)


@pytest.mark.parametrize("path", PATHS)
def test_duplicate_rows_exact_ties_inside_topk(path):
    P = c_oracle.synth_block(0, 30000, seed=6)
    Q = c_oracle.synth_block(0, 8, seed=6, stream=1)
    _, I0 = flat_ip.knn_inner_product(Q, P, 5)
    P[29000:29005] = P[I0[0, :5]]         # exact copies of query 0's top-5, at higher positions
    D, I = make_index(path, P).search(Q, 12)
    Dt, It = flat_ip.truth_fp64(Q, P, 12)
    np.testing.assert_array_equal(I, It)   # (score desc, position asc) is also the truth's order
    assert I[0, 0] < 29000 and I[0, 1] >= 29000 and D[0, 0] == D[0, 1]


def test_add_with_ids_folds_offset_translation():
    P = c_oracle.synth_block(0, 25000, seed=8)
    Q = c_oracle.synth_block(0, 11, seed=8, stream=1)
    ids = (np.arange(25000, dtype=np.int64) * 8 + 3)[::-1].copy()   # strided offsets like block files
    idx = make_index("auto")
    idx.add_with_ids(P, ids)
    D, I = idx.search(Q, 20)
    Do, Io = flat_ip.truth_fp64(Q, P, 20)
    np.testing.assert_array_equal(I, ids[Io])
    np.testing.assert_allclose(D, Do, rtol=RTOL_TRUTH)
    with pytest.raises(RuntimeError):
        idx.add(P[:10])


def test_reconstruct_and_device_synthetic_rows_are_bit_identical_to_host():
    idx = make_index("auto")
    idx.add_synthetic(5000, first_row=123456789012, seed=9, stream=4, norm=3.5)
    got = idx.reconstruct_n(0, 5000)
    want = synth.block(123456789012, 5000, seed=9, stream=4, norm=3.5)
    np.testing.assert_array_equal(got, want)
    Q = c_oracle.synth_block(0, 6, seed=9, stream=1)
    D, I = idx.search(Q, 10)
    Do, Io = flat_ip.truth_fp64(Q, want, 10)
    np.testing.assert_array_equal(I, Io + 123456789012)


@pytest.mark.parametrize("name", ["three_blocks", "one_block", "eight_blocks_k100",
                                  "short_block_wraps_minus_one", "ties_across_blocks"])
def test_driver_search_one_by_one_on_gpu_matches_reference_golden(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", "search_one_by_one.npz"))
    Dg, Ig = z[name + "/D"], z[name + "/I"]
    n, W, nq, topN, dup = (int(v) for v in z[name + "/params"])
    P = synth.block(0, n, seed=7, stream=0)
    if dup:
        P[n - dup:] = P[:dup]
    Q = synth.block(0, nq, seed=7, stream=1)
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(W):
            ids = np.arange(r, n, W, dtype=np.int64)
            flat_ip.write_block(tmp, r, P[ids], ids)
        index = faiss.IndexFlatIP(768)                       # the driver's no --use_gpu path (:369-370)
        D, I = driver.search_one_by_one(tmp, index, Q, topN, verbose=False)
        index2 = faiss.IndexFlatIP(768)
        Dr, Ir = driver.search_resident(tmp, index2, Q, topN)
    assert D.shape == Dg.shape and D.dtype == np.float64 and I.dtype == np.int64
    pad = Dg < -1e38
    np.testing.assert_array_equal(pad, D < -1e38)
    np.testing.assert_array_equal(I[pad], Ig[pad])           # -1 wrapped to the block's last offset, like the reference
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    Dc, Dgc = np.where(pad, -1.0, D), np.where(pad, -1.0, Dg)
    # these collections are tiny (down to 23 rows), so scores near 0 are returned: the golden D
    # (fp32 sgemm) itself carries ~1e-8 absolute rounding, which a purely relative bound cannot absorb
    r = flat_ip.compare(Dc, I, Dgc, Ig, score_of, rtol=RTOL, atol=1e-7)
    assert r["violations"] == 0, r
    if name != "ties_across_blocks":
        assert r["exact_rows"] == nq, r                      # small cases: no near-ties, ids identical
    if name != "short_block_wraps_minus_one":
        r2 = flat_ip.compare(Dr, Ir, Dgc[:, :topN], Ig[:, :topN], score_of, rtol=RTOL, atol=1e-7)
        assert r2["violations"] == 0, r2


def test_multi_gpu_shards_in_one_process_match_single_gpu(gpu_count):
    if gpu_count < 2:
        pytest.skip("needs 2 GPUs (gpurun --gpus 2)")
    P = c_oracle.synth_block(0, 60001, seed=10)
    Q = c_oracle.synth_block(0, 50, seed=10, stream=1)
    one = make_index("auto", P)
    D1, I1 = one.search(Q, 40)
    vres, vdev = faiss.GpuResourcesVector(), faiss.Int32Vector()
    for i in range(gpu_count):
        vdev.push_back(i)
        vres.push_back(faiss.StandardGpuResources())
    co = faiss.GpuMultipleClonerOptions()
    co.shard = True
    multi = faiss.index_cpu_to_gpu_multiple(vres, vdev, faiss.IndexFlatIP(768), co)
    multi.add(P)
    assert multi.num_shards == gpu_count and multi.ntotal == 60001
    Dm, Im = multi.search(Q, 40)
    np.testing.assert_array_equal(Im, I1)
    np.testing.assert_array_equal(Dm, D1)


def test_device_resident_search_and_merge_kernel():
    import torch
    P = c_oracle.synth_block(0, 30000, seed=12)
    Q = c_oracle.synth_block(0, 33, seed=12, stream=1)
    idx = make_index("auto", P)
    Dh, Ih = idx.search(Q, 16)
    qd = torch.from_numpy(Q).cuda()
    Dd, Id = idx.search_device(qd, 16)
    np.testing.assert_array_equal(Id.cpu().numpy(), Ih)
    np.testing.assert_array_equal(Dd.cpu().numpy(), Dh)
    # split the collection in 3 parts, search each, merge on device == search of the whole
    parts = []
    edges = [0, 9000, 21000, 30000]
    for a, b in zip(edges[:-1], edges[1:]):
        sub = make_index("auto")
        sub.add_with_ids(P[a:b], np.arange(a, b, dtype=np.int64))
        parts.append(sub.search_device(qd, 16))
    Dp = torch.stack([p[0] for p in parts]).contiguous()
    Ip = torch.stack([p[1] for p in parts]).contiguous()
    Dm, Im = idx.merge_device(Dp, Ip)
    np.testing.assert_array_equal(Im.cpu().numpy(), Ih)
    np.testing.assert_array_equal(Dm.cpu().numpy(), Dh)


def test_auto_policy_and_invalid_arguments():
    P = c_oracle.synth_block(0, 20000, seed=13)
    idx = make_index("auto", P)
    # AUTO: the tensor engine for every batch size (it streams half the bytes of the fp32 scan and wins from
    # one query on — profiles/r01s2_sweep_8p8M_*.json); per pass, QS (MMA N = batch rounded to 16) up to 208
    # queries, TS (256 query lanes) above
    for nq, passes, qs in ((2, 1, 1), (64, 1, 1), (208, 1, 1), (209, 1, 0), (256, 1, 0), (300, 2, 1)):
        idx.search(c_oracle.synth_block(0, nq, stream=1), 5)
        assert int(idx.stat("path")) == 3
        assert (idx.stat("passes"), idx.stat("qs_passes")) == (passes, qs), nq
    idx.set_option("scan_max_auto", 4)
    idx.search(c_oracle.synth_block(0, 2, stream=1), 5)
    assert int(idx.stat("path")) == 1            # opt-in: tiny batches on the SIMT scan (fp32 128-bit loads)
    with pytest.raises(RuntimeError):
        idx.search(c_oracle.synth_block(0, 2, stream=1), 4096)   # k beyond the supported maximum
    with pytest.raises(AssertionError):
        idx.search(np.zeros((2, 100), dtype=np.float32), 5)
    with pytest.raises(RuntimeError):
        idx.set_option("bootstrap", 1)           # unknown: the dense bootstrap launch was retired
    with pytest.raises(RuntimeError):
        idx.set_option("tighten", 0)             # the phased schedule without in-kernel tightening was retired
    idx.set_option("tighten", 400)               # a refresher pause in ns


def test_asynchronous_device_searches_in_flight_equal_synchronous_ones():
    """b2f_search_device_async: 20 searches queued without a host wait (more than the 16 slots, and a
    batch-size change that regrows the workspace in between) must equal the synchronous results."""
    import torch
    P = c_oracle.synth_block(0, 50000, seed=21)
    idx = make_index("auto", P)
    batches, outs = [], []
    for i in range(20):
        nq = 300 if i == 12 else 40 + i
        q = torch.from_numpy(c_oracle.synth_block(0, nq, seed=100 + i, stream=1)).cuda()
        D = torch.empty((nq, 30), dtype=torch.float32, device="cuda")
        I = torch.empty((nq, 30), dtype=torch.int64, device="cuda")
        idx.search_device_async(q, 30, D, I)
        batches.append(q); outs.append((D, I))
    idx.finish()
    for q, (D, I) in zip(batches, outs):
        Ds, Is = idx.search(q.cpu().numpy(), 30)
        np.testing.assert_array_equal(I.cpu().numpy(), Is)
        np.testing.assert_array_equal(D.cpu().numpy(), Ds)


def test_packed_merge_and_overflow_marker():
    """The packed [D | I] parts of the one-all-gather exchange merge like dense parts, and a part whose
    candidate list overflowed travels with the id -2 marker that the merge kernel reports."""
    import torch
    P = c_oracle.synth_block(0, 60000, seed=22)
    Q = c_oracle.synth_block(0, 13, seed=22, stream=1)
    nq, k = Q.shape[0], 16
    full = make_index("auto", P)
    Dh, Ih = full.search(Q, k)
    qd = torch.from_numpy(Q).cuda()
    i_off = (nq * k * 4 + 15) // 16 * 16
    part = i_off + nq * k * 8
    recv = torch.zeros((3, part), dtype=torch.uint8, device="cuda")
    subs = []
    for g, (a, b) in enumerate([(0, 20000), (20000, 45000), (45000, 60000)]):
        sub = make_index("auto")
        sub.add_with_ids(P[a:b], np.arange(a, b, dtype=np.int64))
        Dl = recv[g, :nq * k * 4].view(torch.float32).view(nq, k)
        Il = recv[g, i_off:].view(torch.int64).view(nq, k)
        sub.search_device_async(qd, k, Dl, Il)
        sub.finish()
        subs.append(sub)
    Dm = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    Im = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    full.merge_packed_device_async(recv, 3, part, i_off, nq, k, Dm, Im)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(Im.cpu().numpy(), Ih)
    np.testing.assert_array_equal(Dm.cpu().numpy(), Dh)
    assert full.stat("merge_saw_overflow") == 0
    recv[1, i_off:].view(torch.int64)[0] = -2            # what finalize_kernel writes for an overflowed row
    full.merge_packed_device_async(recv, 3, part, i_off, nq, k, Dm, Im)
    torch.cuda.synchronize()
    assert full.stat("merge_saw_overflow") == 1
    assert full.stat("merge_saw_overflow") == 0          # read-and-clear


@pytest.mark.parametrize("path", ["umma_ts", "umma_qs", "scan_f32"])
def test_overflowed_rows_carry_the_marker_until_rerun(path):
    """All-equal scores overflow every list: the asynchronous call leaves id -2 in the first slot of
    such rows; finish() re-runs them on the exact engine and the marker is gone."""
    import torch
    row = c_oracle.synth_block(0, 1, seed=2)
    P = np.tile(row, (60000, 1))
    Q = c_oracle.synth_block(0, 3, seed=2, stream=1)
    idx = make_index(path, P)
    qd = torch.from_numpy(Q).cuda()
    D = torch.empty((3, 25), dtype=torch.float32, device="cuda")
    I = torch.empty((3, 25), dtype=torch.int64, device="cuda")
    idx.search_device_async(qd, 25, D, I)
    torch.cuda.synchronize()
    assert I[:, 0].tolist() == [-2, -2, -2]
    idx.finish()
    assert I.cpu().tolist() == [list(range(25))] * 3
    assert idx.stat("fallback_queries") == 3


def test_search_resident_over_flat_shards_matches_block_loop(tmp_path):
    """SURVEY §8 f1/f4: blocks written in the reference's pickle format, converted once to flat shards,
    streamed into the resident index in chunks; one search equals the reference's block loop."""
    from convdr_b200 import blocks
    n_total, W = 30011, 4
    P = c_oracle.synth_block(0, n_total, seed=31)
    Q = c_oracle.synth_block(0, 21, seed=31, stream=1)
    for b in range(W):
        off = blocks.strided_offsets(n_total, b, W)
        blocks.write_block(str(tmp_path), b, P[off], off)
    Do, Io = flat_ip.search_one_by_one(str(tmp_path), flat_ip.IndexFlatIP(768), Q, 40)
    blocks.convert_blocks_to_flat(str(tmp_path))
    idx = make_index("auto")
    Dr, Ir = driver.search_resident(str(tmp_path), idx, Q, 40)
    assert idx.ntotal == n_total
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    r = flat_ip.compare(Dr.astype(np.float32), Ir, Do[:, :40].astype(np.float32), Io[:, :40], score_of, rtol=RTOL)
    assert r["violations"] == 0, r


def test_peer_memory_exchange_equals_nccl_exchange(gpu_count):
    """One process per GPU on EVERY GPU of the box (torchrun, NCCL rendezvous on 127.0.0.1): the peer-memory
    exchange kernels and the ncclAllGather path agree bit for bit with a single index and with the oracle's
    float64 truth, including the overflow re-run (reference: FAISS IndexShards over all GPUs,
    drivers/run_convdr_inference.py:355-368)."""
    import subprocess
    import sys
    if gpu_count < 2:
        pytest.skip("needs 2 GPUs")
    world = min(gpu_count, 8)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "_xchg_worker.py")]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=500)
    assert res.returncode == 0 and f"XCHG_OK {world}" in res.stdout, res.stdout[-6000:] + res.stderr[-3000:]


def test_shard_with_a_block_of_identical_rows_overflows_for_some_queries_only():
    """5000 identical rows (> the survivor capacity of 4096) inside a shard with explicit ids: the few queries
    that rank them high overflow, carry the marker after the asynchronous call, and are settled by
    finish(); all others are untouched.  (The data of the 2-GPU exchange test, one shard of it.)"""
    import torch
    P = c_oracle.synth_block(0, 60000, seed=41)
    P[55000:60000] = P[55000]
    ids = np.arange(30000, 60000, dtype=np.int64)
    idx = make_index("auto")
    idx.add_with_ids(P[30000:], ids)
    ref = make_index("scan_exact")
    ref.add_with_ids(P[30000:], ids)
    Qh = c_oracle.synth_block(0, 173, seed=3, stream=1)
    Qh[5], Qh[100] = P[55000], P[55000] * np.float32(0.5)     # these two rank the identical rows first: overflow
    q = torch.from_numpy(Qh).cuda()
    D = torch.empty((173, 100), dtype=torch.float32, device="cuda")
    I = torch.empty((173, 100), dtype=torch.int64, device="cuda")
    idx.reset_stats()
    idx.search_device_async(q, 100, D, I)
    torch.cuda.synchronize()
    marked = int((I[:, 0] == -2).sum().item())
    assert 2 <= marked < 173
    idx.finish()
    assert idx.stat("fallback_queries") == marked
    Dr, Ir = ref.search(Qh, 100)
    np.testing.assert_array_equal(I.cpu().numpy(), Ir)
    np.testing.assert_array_equal(D.cpu().numpy(), Dr)


# explicit ids: each case keeps the id it has always had, so results stay comparable across versions
@pytest.mark.parametrize("opts", [dict(), dict(tighten_adaptive=0, tighten=400), dict(worst_case_margin=1),
                                  dict(center=0)], ids=["opts0", "opts2", "opts3", "opts5"])
def test_schedule_options_of_the_tensor_engine_give_identical_results(opts, c1_data):
    """Every schedule of the TS engine (adaptive / fixed refresher pacing, data-dependent / worst-case
    margin, centred / uncentred shadow) returns the same bits: the schedule only decides how many
    candidates are looked at, the exact rescoring decides the result."""
    P, Q = c1_data
    base = make_index("umma_qs", P)
    D0, I0 = base.search(Q, 100)
    var = make_index("umma_ts", P, **opts)
    D1, I1 = var.search(Q, 100)
    np.testing.assert_array_equal(I1, I0)
    np.testing.assert_array_equal(D1, D0)
    assert var.stat("fallback_queries") == 0


def test_rank_dedup_kernel_matches_the_restated_evaldevquery():
    """SURVEY §8 f2: offset -> pid translation and the "drop repeated pids" of EvalDevQuery on device."""
    import torch
    rng = np.random.default_rng(5)
    n_off = 5000
    offset2pid = rng.integers(0, 1500, size=n_off).astype(np.int64)           # ~3 offsets per passage: many repeats
    for nq, width, topN, dtype in ((7, 200, 100, np.float64), (3, 1000, 1000, np.float32), (2, 10, 10, np.float64)):
        I = rng.integers(0, n_off, size=(nq, width)).astype(np.int64)
        I[0, 3] = -1                                                          # the reference's wrap (:190)
        D = -np.sort(-rng.random((nq, width)), axis=1).astype(dtype)
        want = flat_ip.eval_rank_dedup(D, I, topN, offset2pid)
        idx = FlatIPIndex(768)
        got = idx.rank_dedup(torch.from_numpy(I).cuda(), torch.from_numpy(D).cuda(), topN,
                             torch.from_numpy(offset2pid).cuda())
        np.testing.assert_array_equal(got[0].cpu().numpy(), want[0])
        np.testing.assert_array_equal(got[1].cpu().numpy(), want[1])
        np.testing.assert_array_equal(got[2].cpu().numpy(), want[2])
        idx.close()


def test_native_flat_file_loader_streams_many_pieces(tmp_path):
    """b2f_add_flat_file: a shard of several 8192-row pieces through the pinned ring equals add_with_ids."""
    from convdr_b200 import blocks
    n = 50001
    P = c_oracle.synth_block(0, n, seed=71)
    ids = np.arange(n, dtype=np.int64) * 3 + 7
    path = blocks.write_flat_shard(str(tmp_path / (blocks.FLAT_NAME % 0)), P, ids)
    a = make_index("auto")
    secs, gb = a.add_flat_file(path, threads=3)
    assert a.ntotal == n and gb == pytest.approx(n * (768 * 4 + 8) / 1e9)
    np.testing.assert_array_equal(a.reconstruct_n(0, n), P)
    b = make_index("auto")
    b.add_with_ids(P, ids)
    Q = c_oracle.synth_block(0, 33, seed=71, stream=1)
    Da, Ia = a.search(Q, 50)
    Db, Ib = b.search(Q, 50)
    np.testing.assert_array_equal(Ia, Ib)
    np.testing.assert_array_equal(Da, Db)
    a.add_flat_file(path)                     # appending a second file keeps the labels of both
    assert a.ntotal == 2 * n
    with pytest.raises(RuntimeError):
        a.add_flat_file(str(tmp_path / "missing.b2f"))


def _synthetic_index(n, **opts):
    idx = make_index("auto", None, **opts)
    idx.reserve(n)
    for a in range(0, n, 1 << 22):
        idx.add_synthetic(min(1 << 22, n - a), first_row=a)
    return idx


def _check_against_full_size_oracle(D, I, Q, sel, k, n):
    """fp64 truth of the selected queries over ALL n rows of the synthetic stream, regenerated on the host block by
    block (oracle/flat_ip_c.c oracle_topk_synth_f64) — detects a missed row, unlike re-scoring the returned ones."""
    Dt, It = c_oracle.topk_synth_f64(Q[sel], k, 0, n)
    score_of = lambda qi, ids: synth.rows(np.asarray(ids).astype(np.uint64)).astype(np.float64) @ Q[sel[qi]].astype(np.float64)
    r = flat_ip.compare(D[sel], I[sel], Dt, It, score_of, rtol=RTOL)
    assert r["violations"] == 0, r
    rel = np.abs(D[sel].astype(np.float64) - Dt) / np.maximum(np.abs(Dt), 1e-30)
    assert rel.max() <= RTOL_TRUTH, rel.max()
    return r


def test_config2_shape_8p8M_rows_173_queries_top1000_against_the_full_size_oracle():
    """BASELINE.json configs[1]: MS MARCO-sized 8,841,823 x 768, the CAsT-19 batch, top-1000 (what
    data/gen_ranking_data.py consumes), single GPU.  At this size the gap near rank 1000 is ~1e-5 of the score:
    where a margin or threshold bug would show first."""
    n, k = 8_841_823, 1000
    idx = _synthetic_index(n)
    Q = c_oracle.synth_block(0, 173, stream=1)
    D, I = idx.search(Q, k)
    assert idx.stat("fallback_queries") == 0 and (np.diff(D, axis=1) <= 0).all()
    _check_against_full_size_oracle(D, I, Q, [0, 21, 43, 86, 129, 150, 165, 172], k, n)
    idx.close()


def test_config3_shape_11p1M_rows_5571_queries_top100_against_the_full_size_oracle():
    """BASELINE.json configs[2]: OR-QuAC-sized 11.1M x 768, all 5,571 test queries in one call (22 passes: 21 of
    256 queries on the TS kernel, the last 195 on QS), top-100; a 16-query subset spread over the passes is
    compared with the full-size oracle."""
    n, k, nq = 11_100_000, 100, 5571
    idx = _synthetic_index(n)
    Q = c_oracle.synth_block(0, nq, stream=1)
    D, I = idx.search(Q, k)
    assert idx.stat("fallback_queries") == 0 and (np.diff(D, axis=1) <= 0).all()
    assert (idx.stat("passes"), idx.stat("qs_passes")) == (22, 1)
    sel = sorted(set(np.linspace(0, nq - 1, 16).astype(int).tolist()))
    _check_against_full_size_oracle(D, I, Q, sel, k, n)
    idx.close()


def test_page_locked_host_buffers_are_used_in_place():
    """b2f_search with page-locked arrays: queries are uploaded straight from the caller's buffer and the last
    kernel stores the result rows straight into the caller's arrays (no staging copies); same bits as the
    pageable path.  Also through a 2-shard... single-shard index with explicit ids and an overflowing query
    (re-run rows are rewritten in place)."""
    import ctypes as C
    import torch
    from convdr_b200 import _lib
    P = c_oracle.synth_block(0, 40000, seed=81)
    P[30000:35000] = P[30000]                     # 5000 identical rows: the planted query overflows and is re-run
    Q = c_oracle.synth_block(0, 37, seed=81, stream=1)
    Q[5] = P[30000]
    idx = make_index("auto", P)
    D0, I0 = idx.search(Q, 50)                    # pageable numpy in / out
    assert idx.stat("fallback_queries") >= 1
    qp = torch.from_numpy(Q).pin_memory()
    Dp = torch.empty((37, 50), dtype=torch.float32).pin_memory()
    Ip = torch.empty((37, 50), dtype=torch.int64).pin_memory()
    Dp.fill_(-1.0); Ip.fill_(-7)
    _lib.check(_lib.load().b2f_search(idx._ensure(), C.c_void_p(qp.data_ptr()), 37, 50, C.c_void_p(Dp.data_ptr()),
                                      C.c_void_p(Ip.data_ptr())))
    np.testing.assert_array_equal(Ip.numpy(), I0)
    np.testing.assert_array_equal(Dp.numpy(), D0)
    check_against_oracle(D0, I0, P, Q, 50, also_fp32_oracle=False)


@pytest.mark.parametrize("n_parts", [2, 5, 8])
def test_merge_kernels_keep_the_tie_order_across_parts(n_parts):
    """Exact ties across parts (the same rows planted in several parts): the merged order must be (score desc,
    part asc, position asc) — the reference's `>=` merge rule (:218) — for the rank-by-counting merge (2-3 parts)
    and for the sort-mode merge (4+ parts)."""
    import torch
    P = c_oracle.synth_block(0, 8000 * n_parts, seed=91)
    Q = c_oracle.synth_block(0, 9, seed=91, stream=1)
    _, I0 = flat_ip.knn_inner_product(Q, P, 4)
    for g in range(1, n_parts):                       # query 0's best rows reappear in every part
        P[8000 * g + 17:8000 * g + 21] = P[I0[0, :4]]
    whole = make_index("auto", P)
    Dw, Iw = whole.search(Q, 30)
    qd = torch.from_numpy(Q).cuda()
    parts = []
    for g in range(n_parts):
        sub = make_index("auto")
        sub.add_with_ids(P[8000 * g:8000 * (g + 1)], np.arange(8000 * g, 8000 * (g + 1), dtype=np.int64))
        parts.append(sub.search_device(qd, 30))
    Dm, Im = whole.merge_device(torch.stack([p[0] for p in parts]).contiguous(),
                                torch.stack([p[1] for p in parts]).contiguous())
    np.testing.assert_array_equal(Im.cpu().numpy(), Iw)
    np.testing.assert_array_equal(Dm.cpu().numpy(), Dw)
    assert (np.diff(Dw[0, :4 * n_parts]) == 0).sum() >= n_parts - 1      # the planted ties are really there


def test_device_side_flat_shard_writer_round_trips(tmp_path):
    """SURVEY §8 f4: b2f_write_flat_file dumps a device-resident shard (several staged pieces) to the flat format;
    numpy's reader and the native loader both get the rows and labels back, explicit or implicit."""
    from convdr_b200 import blocks
    n = 20011
    P = c_oracle.synth_block(0, n, seed=93)
    ids = np.arange(n, dtype=np.int64) * 5 + 2
    a = make_index("auto")
    a.add_with_ids(P, ids)
    paths = blocks.save_index_to_flat(a, str(tmp_path / "labelled"))
    rows, got_ids = blocks.open_flat_shard(paths[0])
    np.testing.assert_array_equal(np.asarray(rows), P)
    np.testing.assert_array_equal(np.asarray(got_ids), ids)
    b = make_index("auto")
    assert blocks.load_flat_into(b, paths) == n
    Q = c_oracle.synth_block(0, 17, seed=93, stream=1)
    Da, Ia = a.search(Q, 40)
    Db, Ib = b.search(Q, 40)
    np.testing.assert_array_equal(Ia, Ib)
    np.testing.assert_array_equal(Da, Db)
    c = make_index("auto", P[:9000])             # implicit ids: the positions
    c.add(P[9000:])
    p2 = str(tmp_path / "implicit.b2f")
    c.write_flat_file(p2)
    _, ids2 = blocks.open_flat_shard(p2)
    np.testing.assert_array_equal(np.asarray(ids2), np.arange(n))
    e = make_index("auto")
    p3 = str(tmp_path / "empty.b2f")
    e.write_flat_file(p3)
    assert blocks.flat_shard_rows(p3) == 0
