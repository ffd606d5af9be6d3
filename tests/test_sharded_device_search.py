"""GPU tests of CUDA-tensor queries on an index sharded over several devices of one process: `search_device`,
`search_device_into` and queued `search_device_async` + `finish()` must return, bit for bit, what the host
`search` of the same index and a single-shard index return.

Every behaviour runs on one GPU with three shards on device 0 (`devices=[0, 0, 0]`): those shards have no peer
access to the first device, so they take the path that copies the queries out and the parts back.  With two or
more GPUs the same tests also run over every GPU (peer access: parts are stored straight into the first device's
memory), plus the check that queries on another device are refused."""
import ctypes as C

import numpy as np
import pytest

import convdr_b200.faiss_compat as faiss
from convdr_b200 import FlatIPIndex, _lib
from oracle import c_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_FIRST, N_SECOND = 30001, 7            # two adds that do not split evenly over the shards
# path option and shadow format: the tensor engine with the int8 and the bf16 shadow, the fp32 scan, the exact scan
ENGINES = {"auto_i8": ("auto", 2), "auto_bf16": ("auto", 1), "scan_f32": ("scan_f32", 1), "scan_exact": ("scan_exact", 1)}
LAYOUTS = ["three_on_gpu0", "every_gpu"]


def devices_of(layout, gpu_count):
    if layout == "three_on_gpu0":
        return [0, 0, 0]
    if gpu_count < 2:
        pytest.skip("needs two GPUs")
    return list(range(gpu_count))


def make_index(engine, devices=None):
    path, shadow = ENGINES[engine]
    idx = FlatIPIndex(768, devices=devices)
    idx.set_option("path", path)
    idx.set_option("shadow", shadow)
    return idx


def fill(idx, P, ids):
    if ids is None:
        idx.add(P[:N_FIRST])
        idx.add(P[N_FIRST:])
    else:
        idx.add_with_ids(P[:N_FIRST], ids[:N_FIRST])
        idx.add_with_ids(P[N_FIRST:], ids[N_FIRST:])


def same(a, b, what=""):
    """Bit-identical (D, I) pairs; either side may be CUDA tensors."""
    Da, Ia = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in a)
    Db, Ib = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in b)
    np.testing.assert_array_equal(Ia, Ib, err_msg=what)
    assert Da.tobytes() == Db.tobytes(), what


@pytest.fixture(scope="module")
def data():
    P = c_oracle.synth_block(0, N_FIRST + N_SECOND, seed=17)
    Q = c_oracle.synth_block(0, 300, seed=17, stream=1)
    return P, Q


@pytest.mark.parametrize("ids", ["implicit", "explicit"])
@pytest.mark.parametrize("engine", list(ENGINES))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_device_search_is_bit_identical_to_host_search_and_to_one_shard(layout, engine, ids, data, gpu_count):
    P, Q = data
    labels = None if ids == "implicit" else (np.arange(P.shape[0], dtype=np.int64)[::-1] * 5 + 3).copy()
    idx = make_index(engine, devices_of(layout, gpu_count))
    fill(idx, P, labels)
    one = make_index(engine)
    fill(one, P, labels)
    assert idx.ntotal == one.ntotal == N_FIRST + N_SECOND and idx.num_shards > 1
    q = torch.from_numpy(Q).cuda()
    for nq in (1, 173, 209, 300):
        for k in (1, 100, 1000, 2048):
            what = f"{layout} {engine} {ids} nq={nq} k={k}"
            dev = idx.search_device(q[:nq], k)
            same(dev, idx.search(Q[:nq], k), what)
            same(dev, one.search(Q[:nq], k), what)
            D = torch.empty((nq, k), dtype=torch.float32, device="cuda")
            I = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            idx.search_device_into(q[:nq], k, D, I)
            same((D, I), dev, what)
    assert idx.stat("fallback_queries") == 0
    with pytest.raises(RuntimeError):
        idx.search_device(q[:5], 2049)
    D0, I0 = idx.search_device(q[:0], 10)
    assert D0.shape == (0, 10) and I0.shape == (0, 10) and D0.is_cuda and I0.is_cuda
    idx.close()
    one.close()


@pytest.mark.parametrize("layout", LAYOUTS)
def test_index_with_fewer_rows_than_shards(layout, data, gpu_count):
    P, Q = data
    devices = devices_of(layout, gpu_count)
    n = len(devices) - 1
    idx = make_index("auto_bf16", devices)
    idx.add(P[:n])
    assert min(idx.shard_rows(g) for g in range(idx.num_shards)) == 0
    one = make_index("auto_bf16")
    one.add(P[:n])
    q = torch.from_numpy(Q[:173]).cuda()
    for k in (1, 5, 100):
        dev = idx.search_device(q, k)
        same(dev, one.search(Q[:173], k), f"k={k}")
        assert (dev[1][:, n:] == -1).all()
        D = torch.empty((173, k), dtype=torch.float32, device="cuda")
        I = torch.empty((173, k), dtype=torch.int64, device="cuda")
        idx.search_device_async(q, k, D, I)
        idx.finish()
        same((D, I), dev, f"async k={k}")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_queued_searches_settle_with_one_finish(layout, data, gpu_count):
    """20 queued searches with mixed batch sizes, k and selectors: a host search after the fourth settles the queue,
    the tenth batch (300 queries, more than the workspaces were sized for) settles and regrows them, and the last ten
    are in flight together."""
    P, Q = data
    idx = make_index("auto_i8", devices_of(layout, gpu_count))
    fill(idx, P, None)
    q = torch.from_numpy(Q).cuda()
    sels = [None, faiss.IDSelectorRange(1000, 21000), faiss.IDSelectorNot(faiss.IDSelectorRange(9000, 25000)),
            faiss.IDSelectorBatch(np.arange(5, N_FIRST, 97))]
    plan = [(209, 1000)] + [((1, 173, 40, 209)[i % 4], (100, 10, 1000, 1)[(i // 2) % 4]) for i in range(1, 20)]
    plan[9] = (300, 100)
    plan = [(nq, k, sels[i % len(sels)]) for i, (nq, k) in enumerate(plan)]
    outs = []
    for i, (nq, k, sel) in enumerate(plan):
        D = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        I = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        params = None if sel is None else faiss.SearchParameters(sel=sel)
        idx.search_device_async(q[:nq], k, D, I, params=params)
        outs.append((D, I))
        if i == 3:
            mid = idx.search(Q[:50], 100)
    idx.finish()
    same(mid, idx.search_device(q[:50], 100), "host search in the middle")
    for (nq, k, sel), got in zip(plan, outs):
        params = None if sel is None else faiss.SearchParameters(sel=sel)
        same(got, idx.search_device(q[:nq], k, params=params), f"nq={nq} k={k}")
        same(got, idx.search(Q[:nq], k, params=params), f"nq={nq} k={k}")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_overflowed_rows_carry_the_marker_until_finish(layout, gpu_count):
    """5000 identical rows (more than the 4096 survivors a list holds) in the last shard: the queries that rank
    them first overflow there.  After the queued search and a device synchronise their merged rows carry id -2 in
    slot 0 and every other row is already final; finish() re-runs them on that shard and merges again."""
    devices = devices_of(layout, gpu_count)
    G = len(devices)
    n = 10000 * G
    P = c_oracle.synth_block(0, n, seed=41)
    P[n - 5000:] = P[n - 5000]
    ids = np.arange(30000, 30000 + n, dtype=np.int64)
    idx = FlatIPIndex(768, devices=devices)
    idx.add_with_ids(P, ids)
    assert idx.shard_rows(G - 1) == 10000
    ref = FlatIPIndex(768)
    ref.set_option("path", "scan_exact")
    ref.add_with_ids(P, ids)
    Qh = c_oracle.synth_block(0, 173, seed=3, stream=1)
    Qh[5], Qh[100] = P[n - 5000], P[n - 5000] * np.float32(0.5)
    Dr, Ir = ref.search(Qh, 100)
    q = torch.from_numpy(Qh).cuda()
    D = torch.empty((173, 100), dtype=torch.float32, device="cuda")
    I = torch.empty((173, 100), dtype=torch.int64, device="cuda")
    idx.reset_stats()
    idx.search_device_async(q, 100, D, I)
    torch.cuda.synchronize()
    marked = (I[:, 0] == -2).cpu().numpy()
    assert marked[5] and marked[100] and 2 <= marked.sum() < 173
    np.testing.assert_array_equal(I.cpu().numpy()[~marked], Ir[~marked])
    np.testing.assert_array_equal(D.cpu().numpy()[~marked], Dr[~marked])
    idx.finish()
    same((D, I), (Dr, Ir))
    assert idx.stat("fallback_queries") == marked.sum()
    launches = idx.stat("launches")
    Ds, Is = idx.search_device(q, 100)      # the synchronous form: re-run and merged again before it returns
    same((Ds, Is), (Dr, Ir))
    assert idx.stat("fallback_queries") == marked.sum() and idx.stat("launches") == launches
    same(idx.search(Qh, 100), (Dr, Ir))


@pytest.mark.parametrize("layout", LAYOUTS)
def test_filtered_device_search_equals_filtered_host_search(layout, data, gpu_count):
    P, Q = data
    n = P.shape[0]
    rng = np.random.default_rng(0)
    sels = {
        "range": faiss.IDSelectorRange(8000, 23000),
        "batch": faiss.IDSelectorBatch(rng.choice(n, n // 100, replace=True)),
        "bitmap": faiss.IDSelectorBitmap(np.packbits(rng.random(n) < 0.5, bitorder="little")),
        "not": faiss.IDSelectorNot(faiss.IDSelectorRange(3000, 26000)),
        "fewer_than_k": faiss.IDSelectorRange(777, 814),
        "no_rows": faiss.IDSelectorRange(5, 5),
    }
    idx = make_index("auto_i8", devices_of(layout, gpu_count))
    fill(idx, P, None)
    q = torch.from_numpy(Q[:173]).cuda()
    for name, sel in sels.items():
        params = faiss.SearchParameters(sel=sel)
        for k in (1, 100, 1000):
            dev = idx.search_device(q, k, params=params)
            same(dev, idx.search(Q[:173], k, params=params), f"{name} k={k}")
            if name == "no_rows":
                assert (dev[1] == -1).all()
    # a selector built before an add is stale: the queued search refuses it
    lib = _lib.load()
    h = idx._ensure()
    sel = C.c_void_p()
    _lib.check(lib.b2f_selector_create(h, 1, 0, 100, 20000, None, 0, None, 0, C.byref(sel)))
    D = torch.empty((173, 10), dtype=torch.float32, device="cuda")
    I = torch.empty((173, 10), dtype=torch.int64, device="cuda")
    _lib.check(lib.b2f_search_device_async_sel(h, sel, q.data_ptr(), 173, 10, D.data_ptr(), I.data_ptr()))
    idx.finish()
    idx.add(P[:10])
    assert lib.b2f_search_device_async_sel(h, sel, q.data_ptr(), 173, 10, D.data_ptr(), I.data_ptr()) == 1
    assert "stale" in _lib.last_error()
    lib.b2f_selector_destroy(sel)


@pytest.mark.parametrize("devices", [None, [0, 0, 0]])
def test_search_waits_for_the_queries_of_the_current_stream(devices, data):
    """The queries are produced on a side stream behind a long sleep; with that stream current, the index stream
    must not read them before they are written."""
    P, Q = data
    idx = make_index("auto_bf16", devices)
    fill(idx, P, None)
    ref = idx.search(Q[:173] * np.float32(2), 100)
    base = torch.from_numpy(Q[:173]).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        q = base * 2
        same(idx.search_device(q, 100), ref, "search_device")
        torch.cuda._sleep(200_000_000)
        q2 = base * 2
        D = torch.empty((173, 100), dtype=torch.float32, device="cuda")
        I = torch.empty((173, 100), dtype=torch.int64, device="cuda")
        idx.search_device_async(q2, 100, D, I)
        idx.finish()
        same((D, I), ref, "search_device_async")


def test_queries_on_another_device_than_the_first_shard_are_refused(data, gpu_count):
    if gpu_count < 2:
        pytest.skip("needs two GPUs")
    P, Q = data
    idx = make_index("auto_bf16", list(range(gpu_count)))
    fill(idx, P, None)
    q1 = torch.from_numpy(Q[:8]).to("cuda:1")
    with pytest.raises(AssertionError):
        idx.search_device(q1, 10)
    D = torch.empty((8, 10), dtype=torch.float32, device="cuda:0")
    I = torch.empty((8, 10), dtype=torch.int64, device="cuda:0")
    with pytest.raises(AssertionError):
        idx.search_device_async(q1, 10, D, I)
    q0 = torch.from_numpy(Q[:8]).cuda()
    with pytest.raises(AssertionError):
        idx.search_device_into(q0, 10, D, I.to("cuda:1"))
