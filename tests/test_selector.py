"""GPU tests of filtered search (faiss SearchParameters(sel=...)): a selected search must return, bit for bit,
what a search over an index holding only the selected rows (with their original labels, in their original order)
returns — on every scoring engine — and agree with the float64 truth over the selected rows."""
import ctypes as C

import numpy as np
import pytest

import convdr_b200.faiss_compat as faiss
from convdr_b200 import FlatIPIndex, _lib
from oracle import c_oracle, flat_ip

pytestmark = pytest.mark.gpu

N = 50000
# (path option, umma_variant, shadow): auto = QS up to 208 queries per pass, TS above (300 queries: one of each)
PATHS = {
    "qs_bf16": ("umma_bf16", 3, 1), "qs_i8": ("umma_bf16", 3, 2),
    "ts_bf16": ("umma_bf16", 2, 1), "ts_i8": ("umma_bf16", 2, 2),
    "auto_bf16": ("umma_bf16", 0, 1), "auto_i8": ("umma_bf16", 0, 2),
    "scan_f32": ("scan_f32", 0, 1), "scan_exact": ("scan_exact", 0, 1),
}


def make_index(path, devices=None, **opts):
    p, variant, shadow = PATHS[path]
    idx = FlatIPIndex(768, devices=devices)
    idx.set_option("path", p)
    idx.set_option("umma_variant", variant)
    idx.set_option("shadow", shadow)
    for k, v in opts.items():
        idx.set_option(k, v)
    return idx


def selectors(n, seed=0):
    rng = np.random.default_rng(seed)
    bm = (rng.random(n) < 0.5)
    return {
        "range_inside": faiss.IDSelectorRange(1000, 9000),
        "batch_1pct": faiss.IDSelectorBatch(rng.choice(n, n // 100, replace=True)),
        "bitmap_50pct": faiss.IDSelectorBitmap(np.packbits(bm, bitorder="little")),
        "not_range": faiss.IDSelectorNot(faiss.IDSelectorRange(3000, 41000)),
        "all_rows": faiss.IDSelectorRange(0, n),
        "fewer_than_k": faiss.IDSelectorRange(777, 814),
        "no_rows": faiss.IDSelectorRange(5, 5),
    }


def subset_index(path, P, labels, mask, devices=None, **opts):
    sub = make_index(path, devices=devices, **opts)
    sub.add_with_ids(P[mask], labels[mask])
    return sub


@pytest.fixture(scope="module")
def data():
    return c_oracle.synth_block(0, N, seed=7), c_oracle.synth_block(0, 300, seed=7, stream=1)


@pytest.mark.parametrize("sel_name", list(selectors(N)))
@pytest.mark.parametrize("path", list(PATHS))
def test_selected_search_is_bit_identical_to_a_subset_index(path, sel_name, data):
    P, Q = data
    sel = selectors(N)[sel_name]
    labels = np.arange(N, dtype=np.int64)
    mask = sel._mask(labels)
    idx = make_index(path)
    idx.add(P)
    sub = subset_index(path, P, labels, mask)
    assert idx.selected_count(sel) == int(mask.sum())
    params = faiss.SearchParameters(sel=sel)
    for nq in (1, 173, 300):
        for k in (1, 100, 1000):
            D, I = idx.search(Q[:nq], k, params=params)
            Ds, Is = sub.search(Q[:nq], k)
            np.testing.assert_array_equal(I, Is, err_msg=f"{path} {sel_name} nq={nq} k={k}")
            assert D.tobytes() == Ds.tobytes(), f"{path} {sel_name} nq={nq} k={k}"
            if sel_name == "all_rows":
                D0, I0 = idx.search(Q[:nq], k)
                assert D.tobytes() == D0.tobytes() and np.array_equal(I, I0)
            if sel_name == "no_rows":
                assert (I == -1).all() and (D == np.float32(-3.4028235e38)).all()
            if sel_name == "fewer_than_k" and k > mask.sum():
                assert (I[:, mask.sum():] == -1).all() and set(I[:, :mask.sum()].ravel()) == set(np.nonzero(mask)[0])
    idx.close()
    sub.close()


@pytest.mark.parametrize("path", ["qs_bf16", "ts_i8", "scan_f32"])
def test_selection_applies_to_explicit_labels(path, data):
    P, Q = data
    labels = (np.arange(N, dtype=np.int64)[::-1] * 3 + 11).copy()    # descending, not positions
    sel = faiss.IDSelectorRange(40000, 100000)
    mask = sel._mask(labels)
    idx = make_index(path)
    idx.add_with_ids(P, labels)
    sub = subset_index(path, P, labels, mask)
    D, I = idx.search(Q[:173], 100, params=faiss.SearchParameters(sel=sel))
    Ds, Is = sub.search(Q[:173], 100)
    assert np.array_equal(I, Is) and D.tobytes() == Ds.tobytes()
    assert np.isin(I, labels[mask]).all()


@pytest.mark.parametrize("path", ["qs_bf16", "ts_bf16", "scan_exact"])
def test_range_spanning_a_shard_boundary(path, data):
    """Two shards (on the same device when there is only one): each filters its own rows by the global labels."""
    P, Q = data
    labels = np.arange(N, dtype=np.int64)
    sel = faiss.IDSelectorRange(N // 2 - 3000, N // 2 + 5000)
    mask = sel._mask(labels)
    idx = make_index(path, devices=[0, 0])
    idx.add(P)
    assert idx.num_shards == 2 and idx.selected_count(sel) == int(mask.sum())
    sub = subset_index(path, P, labels, mask)
    for k in (1, 100, 1000):
        D, I = idx.search(Q[:173], k, params=faiss.SearchParameters(sel=sel))
        Ds, Is = sub.search(Q[:173], k)
        assert np.array_equal(I, Is) and D.tobytes() == Ds.tobytes(), k


@pytest.mark.parametrize("kind", ["isotropic", "common_mean"])
@pytest.mark.parametrize("path", ["qs_bf16", "qs_i8", "ts_bf16", "auto_i8", "scan_f32"])
def test_agrees_with_the_fp64_truth_over_the_selected_rows(path, kind):
    opts = dict(norm=28.0, mean_shift=443) if kind == "common_mean" else {}
    P = c_oracle.synth_block(0, 60000, seed=53, **opts)
    Q = c_oracle.synth_block(0, 64, seed=53, stream=1, **opts)
    rng = np.random.default_rng(1)
    sel = faiss.IDSelectorBitmap(np.packbits(rng.random(60000) < 0.5, bitorder="little"))
    rows = np.nonzero(sel._mask(np.arange(60000)))[0]
    idx = make_index(path)
    idx.add(P)
    D, I = idx.search(Q, 100, params=faiss.SearchParameters(sel=sel))
    Dt, It = flat_ip.truth_fp64(Q, P[rows], 100)
    It = np.where(It >= 0, rows[np.maximum(It, 0)], -1)
    score_of = lambda qi, ids: Q[qi].astype(np.float64) @ P[ids].astype(np.float64).T
    r = flat_ip.compare(D, I, Dt, It, score_of, rtol=1e-5)
    assert r["violations"] == 0, r


@pytest.mark.parametrize("path", [p for p in PATHS if p != "scan_exact"])
def test_overflow_rerun_filters_too(path):
    """All rows equal: every candidate list overflows and the exact engine re-runs the queries; it must return the
    first k SELECTED rows in insertion order."""
    row = c_oracle.synth_block(0, 1, seed=2)
    P = np.tile(row, (60000, 1))
    Q = c_oracle.synth_block(0, 3, seed=2, stream=1)
    sel = faiss.IDSelectorNot(faiss.IDSelectorRange(0, 1000))
    idx = make_index(path)
    idx.add(P)
    D, I = idx.search(Q, 25, params=faiss.SearchParameters(sel=sel))
    assert I.tolist() == [list(range(1000, 1025))] * 3
    assert idx.stat("fallback_queries") > 0


def test_async_searches_with_different_selectors_settle_with_one_finish(data):
    torch = pytest.importorskip("torch")
    P, Q = data
    idx = make_index("auto_bf16")
    idx.add(P)
    sels = list(selectors(N).values())
    q = torch.from_numpy(Q[:173]).cuda()
    outs = []
    for s in sels:
        D = torch.empty((173, 100), dtype=torch.float32, device="cuda")
        I = torch.empty((173, 100), dtype=torch.int64, device="cuda")
        idx.search_device_async(q, 100, D, I, params=faiss.SearchParameters(sel=s))
        outs.append((D, I))
    idx.finish()
    for s, (D, I) in zip(sels, outs):
        Dr, Ir = idx.search(Q[:173], 100, params=faiss.SearchParameters(sel=s))
        assert np.array_equal(I.cpu().numpy(), Ir) and D.cpu().numpy().tobytes() == Dr.tobytes()
    Dd, Id = idx.search_device(q, 100, params=faiss.SearchParameters(sel=sels[1]))
    Dr, Ir = idx.search(Q[:173], 100, params=faiss.SearchParameters(sel=sels[1]))
    assert np.array_equal(Id.cpu().numpy(), Ir)


def test_two_gpus_in_one_process_equal_one_gpu(gpu_count, data):
    if gpu_count < 2:
        pytest.skip("needs two GPUs")
    P, Q = data
    for sel in selectors(N).values():
        one = make_index("auto_bf16")
        one.add(P)
        two = make_index("auto_bf16", devices=[0, 1])
        two.add(P)
        params = faiss.SearchParameters(sel=sel)
        D1, I1 = one.search(Q[:173], 100, params=params)
        D2, I2 = two.search(Q[:173], 100, params=params)
        assert np.array_equal(I1, I2) and D1.tobytes() == D2.tobytes()


def test_stale_selector_fails_and_the_facade_rebuilds(data):
    P, Q = data
    lib = _lib.load()
    idx = make_index("qs_bf16")
    idx.add(P[:30000])
    h = idx._ensure()
    sel = C.c_void_p()
    _lib.check(lib.b2f_selector_create(h, 1, 0, 100, 20000, None, 0, None, 0, C.byref(sel)))
    cnt = C.c_int64()
    _lib.check(lib.b2f_selector_count(sel, C.byref(cnt)))
    assert cnt.value == 19900
    D = np.empty((5, 10), dtype=np.float32)
    I = np.empty((5, 10), dtype=np.int64)
    q = np.ascontiguousarray(Q[:5])
    _lib.check(lib.b2f_search_sel(h, sel, q.ctypes.data, 5, 10, D.ctypes.data, I.ctypes.data))
    idx.add(P[30000:])
    assert lib.b2f_search_sel(h, sel, q.ctypes.data, 5, 10, D.ctypes.data, I.ctypes.data) == 1
    assert "stale" in _lib.last_error()
    lib.b2f_selector_destroy(sel)
    # the facade keys its compiled selectors by the index generation: the same object is rebuilt after an add
    s = faiss.IDSelectorRange(29000, 31000)
    assert idx.selected_count(s) == 2000
    idx.reset()
    assert idx.selected_count(s) == 0
    idx.add(P[:30500])
    assert idx.selected_count(s) == 1500


@pytest.mark.parametrize("path,tile_rows", [("qs_bf16", 256), ("ts_bf16", 64)])
def test_profile_counts_only_the_listed_tiles(path, tile_rows):
    n = 400000
    idx = make_index(path, profile=1)
    idx.add_synthetic(n, seed=9)
    Q = c_oracle.synth_block(0, 173, seed=9, stream=1)
    lo, hi = 123457, 123457 + n // 10
    idx.search(Q, 100, params=faiss.SearchParameters(sel=faiss.IDSelectorRange(lo, hi)))
    tiles = (hi - 1) // tile_rows - lo // tile_rows + 1
    assert idx.stat("score_rows") == tiles * tile_rows
    assert abs(idx.stat("score_rows") / n - 0.1) < 0.01
