"""GPU tests of rows by label: `reconstruct`, `reconstruct_batch`, `search_and_reconstruct` and
`search_and_reconstruct_device` must return, byte for byte, the rows that were added under the labels asked for (or
returned by the search, whose D and I stay those of `search`), on every label form, engine and shard layout.

Layouts: one shard; three shards on device 0 (`devices=[0, 0, 0]`: no peer access to the first device, so those shards
stage their rows and copy them over); with two or more GPUs, every GPU (peer access: rows stored in place)."""
import numpy as np
import pytest

import convdr_b200.faiss_compat as faiss
from convdr_b200 import FlatIPIndex, blocks
from oracle import c_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_FIRST, N_SECOND = 30001, 7            # two adds that do not split evenly over the shards
ENGINES = {"auto_i8": ("auto", 2), "auto_bf16": ("auto", 1), "scan_f32": ("scan_f32", 1), "scan_exact": ("scan_exact", 1)}
LAYOUTS = ["one", "three_on_gpu0", "every_gpu"]
PAD = np.frombuffer(b"\xff" * 4 * 768, dtype=np.float32)


def devices_of(layout, gpu_count):
    if layout == "one":
        return None
    if layout == "three_on_gpu0":
        return [0, 0, 0]
    if gpu_count < 2:
        pytest.skip("needs two GPUs")
    return list(range(gpu_count))


def make_index(devices=None, engine="auto_i8"):
    path, shadow = ENGINES[engine]
    idx = FlatIPIndex(768, devices=devices)
    idx.set_option("path", path)
    idx.set_option("shadow", shadow)
    return idx


@pytest.fixture(scope="module")
def data():
    P = c_oracle.synth_block(0, N_FIRST + N_SECOND, seed=17)
    Q = c_oracle.synth_block(0, 173, seed=17, stream=1)
    return P, Q


def fill(idx, P, labels):
    """Two adds; labels None: implicit positions."""
    for a, b in ((0, N_FIRST), (N_FIRST, P.shape[0])):
        if labels is None:
            idx.add(P[a:b])
        else:
            idx.add_with_ids(P[a:b], labels[a:b])


def labels_of(kind, n):
    if kind == "segments":
        return None
    if kind == "ascending":
        return np.arange(n, dtype=np.int64) * 3 + 1000
    return np.random.default_rng(5).permutation(n).astype(np.int64) * 7 + 11   # shuffled


def rows_by_label(P, labels):
    keys = np.arange(P.shape[0], dtype=np.int64) if labels is None else labels
    return dict(zip(keys.tolist(), range(P.shape[0])))


def check_rows(R, I, P, where):
    """R[i, j] is the source row of I[i, j]; -1 labels give 0xFF rows."""
    R = R.cpu().numpy() if hasattr(R, "cpu") else R
    I = I.cpu().numpy() if hasattr(I, "cpu") else I
    assert R.shape == I.shape + (768,)
    flat_I, flat_R = I.reshape(-1), R.reshape(-1, 768)
    pad = flat_I < 0
    assert flat_R[pad].tobytes() == np.tile(PAD, int(pad.sum())).tobytes()
    src = np.array([where[int(l)] for l in flat_I[~pad]], dtype=np.int64)
    assert flat_R[~pad].tobytes() == P[src].tobytes()


def same(a, b, what=""):
    Da, Ia = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in a)
    Db, Ib = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in b)
    np.testing.assert_array_equal(Ia, Ib, err_msg=what)
    assert Da.tobytes() == Db.tobytes(), what


@pytest.mark.parametrize("kind", ["segments", "ascending", "shuffled"])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_reconstruct_batch_returns_the_source_rows(layout, kind, data, gpu_count):
    P, _ = data
    n = P.shape[0]
    labels = labels_of(kind, n)
    idx = make_index(devices_of(layout, gpu_count))
    fill(idx, P, labels)
    keys = np.arange(n, dtype=np.int64) if labels is None else labels
    order = np.random.default_rng(1).permutation(n)
    assert idx.reconstruct_batch(keys[order]).tobytes() == P[order].tobytes()
    rep = order[[3, 3, 17, 3, n - 1, 0]]          # repeats, any order
    assert idx.reconstruct_batch(keys[rep]).tobytes() == P[rep].tobytes()
    for i in (0, N_FIRST - 1, N_FIRST, n - 1):
        r = idx.reconstruct(int(keys[i]))
        assert r.shape == (768,) and r.dtype == np.float32 and r.tobytes() == P[i].tobytes()
    assert idx.reconstruct_batch(keys[:0]).shape == (0, 768)
    # only a shard whose labels are not in ascending order holds a sorted copy: 12 bytes per row
    assert idx.stat("label_index_bytes") == (12 * n if kind == "shuffled" else 0)
    idx.close()


@pytest.mark.parametrize("files", [1, 2])
def test_flat_file_labels(files, data, tmp_path):
    """A block file holds offsets b, b + W, b + 2W, ...: one file per shard is ascending, two interleave."""
    P, _ = data
    n = P.shape[0] // 2 * 2
    idx = make_index()
    keys = np.empty(n, dtype=np.int64)
    for b in range(files):
        sl = slice(b * n // files, (b + 1) * n // files)
        ids = np.arange(sl.stop - sl.start, dtype=np.int64) * files + b + 10
        keys[sl] = ids
        path = blocks.write_flat_shard(str(tmp_path / f"block{b}.b2f"), P[sl], ids)
        idx.add_flat_file(path)
    order = np.random.default_rng(2).permutation(n)
    assert idx.reconstruct_batch(keys[order]).tobytes() == P[order].tobytes()
    assert idx.stat("label_index_bytes") == (12 * n if files == 2 else 0)


@pytest.mark.parametrize("engine", list(ENGINES))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_search_and_reconstruct_matches_search(layout, engine, data, gpu_count):
    P, Q = data
    n = P.shape[0]
    devices = devices_of(layout, gpu_count)
    q = torch.from_numpy(Q).cuda()
    sels = [None, faiss.IDSelectorRange(1000, 21000), faiss.IDSelectorNot(faiss.IDSelectorRange(9000, 25000))]
    for kind in ("segments", "shuffled"):
        labels = labels_of(kind, n)
        if labels is not None:   # selectors act on labels
            sels[1] = faiss.IDSelectorBatch(labels[::3])
        idx = make_index(devices, engine)
        fill(idx, P, labels)
        where = rows_by_label(P, labels)
        for sel in sels:
            params = None if sel is None else faiss.SearchParameters(sel=sel)
            for nq, k in ((173, 1), (173, 100), (20, 1000)):
                what = f"{layout} {engine} {kind} sel={sel is not None} nq={nq} k={k}"
                ref = idx.search(Q[:nq], k, params=params)
                D, I, R = idx.search_and_reconstruct(Q[:nq], k, params=params)
                same((D, I), ref, what)
                check_rows(R, I, P, where)
                Dd, Id, Rd = idx.search_and_reconstruct_device(q[:nq], k, params=params)
                assert Dd.is_cuda and Id.is_cuda and Rd.is_cuda and Rd.shape == (nq, k, 768)
                same((Dd, Id), ref, what)
                assert Rd.cpu().numpy().tobytes() == R.tobytes(), what
        idx.close()


@pytest.mark.parametrize("layout", LAYOUTS)
def test_padding_rows_are_all_ones(layout, data, gpu_count):
    P, Q = data
    idx = make_index(devices_of(layout, gpu_count))
    idx.add(P[:50])
    D, I, R = idx.search_and_reconstruct(Q[:9], 100)          # k > ntotal
    assert (I[:, 50:] == -1).all() and (I[:, :50] >= 0).all()
    check_rows(R, I, P, rows_by_label(P[:50], None))
    idx.reset()
    fill(idx, P, None)
    sel = faiss.IDSelectorRange(777, 814)                      # 37 selected rows, k = 100
    params = faiss.SearchParameters(sel=sel)
    D, I, R = idx.search_and_reconstruct(Q, 100, params=params)
    assert (I[:, 37:] == -1).all()
    check_rows(R, I, P, rows_by_label(P, None))
    Dd, Id, Rd = idx.search_and_reconstruct_device(torch.from_numpy(Q).cuda(), 100, params=params)
    same((Dd, Id), (D, I))
    assert Rd.cpu().numpy().tobytes() == R.tobytes()
    D0, I0, R0 = idx.search_and_reconstruct(Q[:0], 10)
    assert R0.shape == (0, 10, 768)


@pytest.mark.parametrize("layout", ["one", "three_on_gpu0"])
def test_rows_of_rerun_queries_match_their_final_labels(layout, gpu_count):
    """5000 identical rows (more than the 4096 survivors a list holds): queries that rank them first overflow and are
    re-run on the exact engine; their rows are gathered for the final labels."""
    devices = devices_of(layout, gpu_count)
    G = 1 if devices is None else len(devices)
    n = 10000 * G
    P = c_oracle.synth_block(0, n, seed=41)
    P[n - 5000:] = P[n - 5000]
    ids = np.random.default_rng(3).permutation(n).astype(np.int64) + 30000
    idx = FlatIPIndex(768, devices=devices)
    idx.add_with_ids(P, ids)
    Qh = c_oracle.synth_block(0, 173, seed=3, stream=1)
    Qh[5], Qh[100] = P[n - 5000], P[n - 5000] * np.float32(0.5)
    ref = idx.search(Qh, 100)
    idx.reset_stats()
    D, I, R = idx.search_and_reconstruct(Qh, 100)
    assert idx.stat("fallback_queries") >= 2
    same((D, I), ref)
    check_rows(R, I, P, rows_by_label(P, ids))
    idx.reset_stats()
    Dd, Id, Rd = idx.search_and_reconstruct_device(torch.from_numpy(Qh).cuda(), 100)
    assert idx.stat("fallback_queries") >= 2
    same((Dd, Id), ref)
    assert Rd.cpu().numpy().tobytes() == R.tobytes()


def test_lookup_errors_name_the_label(data):
    P, Q = data
    idx = make_index()
    ids = np.arange(1000, dtype=np.int64) + 500
    idx.add_with_ids(P[:1000], ids)
    with pytest.raises(RuntimeError, match="label 77 is not in the index"):
        idx.reconstruct_batch(np.array([600, 77, 601]))
    with pytest.raises(RuntimeError, match="label -3 is negative"):
        idx.reconstruct(-3)
    # a label held twice in one shard (ascending and shuffled forms): search is fine, its lookup is ambiguous
    for dup in (np.sort(np.r_[ids[:-1], 700]), np.r_[ids[:-1], 700][::-1].copy()):
        idx.reset()
        idx.add_with_ids(P[:1000], dup)
        q = P[np.where(dup == 700)[0][:1]]               # its best match is a row labelled 700
        D, I = idx.search(q, 3)
        assert I[0, 0] == 700
        assert idx.reconstruct(600).tobytes() == P[int(np.where(dup == 600)[0][0])].tobytes()
        with pytest.raises(RuntimeError, match="label 700 is held by more than one row"):
            idx.reconstruct(700)
        with pytest.raises(RuntimeError, match="label 700 is held by more than one row"):
            idx.search_and_reconstruct(q, 3)
    # overlapping segments (two synthetic adds with the same id_base)
    seg = make_index()
    seg.add_synthetic(100, seed=1, id_base=0)
    seg.add_synthetic(100, seed=2, id_base=50)
    assert seg.reconstruct_batch(np.array([10, 149])).tobytes() == np.concatenate(
        [seg.reconstruct_n(10, 1), seg.reconstruct_n(199, 1)]).tobytes()
    with pytest.raises(RuntimeError, match="label 60 is held by more than one row"):
        seg.reconstruct(60)
    with pytest.raises(RuntimeError, match="label 150 is not in the index"):
        seg.reconstruct(150)


@pytest.mark.parametrize("layout", ["three_on_gpu0", "every_gpu"])
def test_label_held_by_two_shards_is_ambiguous(layout, data, gpu_count):
    P, _ = data
    devices = devices_of(layout, gpu_count)
    idx = make_index(devices)
    n = 999
    ids = np.arange(n, dtype=np.int64)
    ids[-1] = 0                                   # the first shard and the last shard both hold label 0
    idx.add_with_ids(P[:n], ids)
    assert idx.search(P[:1], 2)[1][0, 0] == 0
    assert idx.reconstruct(5).tobytes() == P[5].tobytes()
    with pytest.raises(RuntimeError, match="label 0 is held by more than one row"):
        idx.reconstruct_batch(np.array([1, 0, 2]))


@pytest.mark.parametrize("layout", ["one", "three_on_gpu0"])
def test_lookups_follow_add_and_reset(layout, data, gpu_count):
    P, _ = data
    idx = make_index(devices_of(layout, gpu_count))
    shuffled = np.random.default_rng(4).permutation(2000).astype(np.int64)
    idx.add_with_ids(P[:1000], shuffled[:1000])
    assert idx.reconstruct(int(shuffled[3])).tobytes() == P[3].tobytes()
    assert idx.stat("label_index_bytes") == 12 * 1000
    with pytest.raises(RuntimeError, match="not in the index"):
        idx.reconstruct(int(shuffled[1500]))
    idx.add_with_ids(P[1000:2000], shuffled[1000:])
    assert idx.stat("label_index_bytes") == 0                  # freed by the add
    assert idx.reconstruct(int(shuffled[1500])).tobytes() == P[1500].tobytes()
    assert idx.stat("label_index_bytes") == 12 * 2000
    idx.reset()
    assert idx.stat("label_index_bytes") == 0
    idx.add(P[5000:5100])                                       # segment labels 0..99 now
    assert idx.reconstruct_batch(np.arange(100)).tobytes() == P[5000:5100].tobytes()
    assert idx.stat("label_index_bytes") == 0
    with pytest.raises(RuntimeError, match="label 100 is not in the index"):
        idx.reconstruct(100)
