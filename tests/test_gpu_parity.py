"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C-ABI
against the committed reference goldens and the CPU oracle.  Bit-exact for the
integer-valued matrices; normalised matrices within 1e-5 relative (in practice
they are bit-identical too, the epilogue uses the reference's fp64 formula)."""
import os
import pickle
import sys

import numpy as np
import pytest

import gio
from oracle.gk_oracle import SPOracle, WLOracle, gen, wl_partitions

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def eng():
    from grakel_b200 import _lib
    return _lib.get_engine()


def _k():
    import grakel_b200
    return grakel_b200


def _same(a, b, exact=True):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape
    if exact:
        assert np.array_equal(a, b, equal_nan=True), f"max abs diff {np.nanmax(np.abs(a - b))}"
    else:
        np.testing.assert_allclose(a, b, rtol=1e-5, atol=0, equal_nan=True)


# --------------------------------------------------------------- Gram kernels
@pytest.mark.parametrize("n,d,hi", [(64, 64, 5), (300, 200, 20), (520, 130, 256), (1000, 1500, 7), (129, 65, 3)])
def test_tcgen05_gram_matches_integer_matmul(eng, n, d, hi):
    rs = np.random.RandomState(n + d)
    C = (rs.rand(n, d) < 0.2) * rs.randint(1, hi + 1, size=(n, d))
    exact = (C.astype(np.int64) @ C.astype(np.int64).T).astype(np.float64)
    tc, simt = eng.selftest_gram(C)
    _same(simt, exact)
    _same(tc, exact)


# --------------------------------------------------------------- WL
def _run_case(X, Y, out):
    k = _k()
    for key, rec in out.items():
        parts = key.split("_")
        if "error" in rec:
            continue
        if parts[0] == "wl":
            est = k.WeisfeilerLehman(n_iter=int(parts[1][1:]), normalize=parts[2] == "n")
        else:
            est = k.ShortestPath(with_labels=parts[1] == "l", algorithm_type="_".join(parts[2:-1]),
                                 normalize=parts[-1] == "n")
        with np.errstate(all="ignore"):
            _same(est.fit_transform(X), rec["fit_transform"])
            if "transform" in rec:
                _same(est.transform(Y), rec["transform"])


def test_spellings_all_kernels():
    g = gio.load(os.path.join(G, "spellings.json.gz"))
    for name, case in g["cases"].items():
        _run_case(gio.dec_dataset(case["X"]), None, case["out"])


@pytest.mark.parametrize("tag", ["unit", "intw"])
def test_fit_then_transform_with_unseen_labels(tag):
    d = gio.load(os.path.join(G, "fit_transform.json.gz"))[tag]
    _run_case(gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"]), d["out"])


def test_real_weights_both_path_sum_orders():
    """Real-valued weights: path lengths are compared by exact float equality (shortest_path.py:472, 511) and the
    reference's two algorithms associate the sums differently (SURVEY 7), so the device reproduces each bit for bit:
    the fp64 k-ordered Floyd-Warshall (adjacency input / forced FW) and Dijkstra's left-to-right sums (edge
    dictionaries / forced dijkstra: the least fixed point of d[v] = min fl(d[u] + w), sp_dijkstra_order_apsp)."""
    d = gio.load(os.path.join(G, "fit_transform.json.gz"))["realw"]
    X, Y = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    _run_case(X, Y, d["out"])


def test_dijkstra_order_goldens_from_the_reference():
    """tests/golden/make_golden_dijkstra.py: edge dictionaries with weights from {0.1, 0.2, 0.3, 0.7, 1.1} -- path
    lengths coincide only when the sums associate as in the reference -- through ShortestPath (auto -> dijkstra),
    its Floyd-Warshall twin (different matrix), WL over ShortestPath and ShortestPathAttr(algorithm_type="dijkstra")."""
    sys.path.insert(0, G)
    from make_golden_dijkstra import gen_real
    k = _k()
    ref = np.load(os.path.join(G, "dijkstra_real.npz"))
    X = gen_real(40, 12, 21)
    fit, new = X[:30], X[30:]
    for tag, wl in (("lab", True), ("nolab", False)):
        e = k.ShortestPath(with_labels=wl)
        _same(e.fit_transform(fit), ref[f"dj_{tag}_K"])
        _same(e.transform(new), ref[f"dj_{tag}_Kt"])
        _same(k.ShortestPath(with_labels=wl, algorithm_type="floyd_warshall").fit_transform(fit), ref[f"fw_{tag}_K"])
    _same(k.ShortestPath(normalize=True).fit_transform(fit), ref["dj_norm_K"])
    w = k.WeisfeilerLehman(n_iter=2, base_graph_kernel=k.ShortestPath)
    _same(w.fit_transform(fit), ref["wlsp_K"])
    _same(w.transform(new), ref["wlsp_Kt"])
    A = gen_real(7, 8, 5, attr=3)
    np.testing.assert_allclose(k.ShortestPathAttr(algorithm_type="dijkstra").fit_transform(A), ref["attr_dj_K"], rtol=1e-5)


def test_mutag_goldens():
    k = _k()
    X = gio.dec_dataset(gio.load(os.path.join(G, "mutag_graphs.json.gz")))
    ref = np.load(os.path.join(G, "mutag_out.npz"))
    for h in (3, 5):
        K = k.WeisfeilerLehman(n_iter=h).fit_transform(X)
        assert K.dtype == np.float64 and K.flags.c_contiguous
        _same(K, ref[f"wl_h{h}"])
    _same(k.ShortestPath().fit_transform(X), ref["sp"])
    tr, te = ref["split_train"].tolist(), ref["split_test"].tolist()
    wl = k.WeisfeilerLehman(n_iter=3, normalize=True)
    _same(wl.fit_transform([X[i] for i in tr]), ref["wl_h3_norm_train"])
    wl2 = pickle.loads(pickle.dumps(wl))  # fitted state is host-resident
    _same(wl2.transform([X[i] for i in te]), ref["wl_h3_norm_test"])
    sp = k.ShortestPath(normalize=True)
    _same(sp.fit_transform([X[i] for i in tr]), ref["sp_norm_train"])
    _same(sp.transform([X[i] for i in te]), ref["sp_norm_test"])
    # GraphKernel front door == direct class (graph_kernels.py:405)
    gk = k.GraphKernel(kernel=[{"name": "WL", "n_iter": 3}, "subtree_wl"], normalize=True)
    _same(gk.fit_transform([X[i] for i in tr]), ref["wl_h3_norm_train"])
    # PSD like grakel/tests/test_kernels.py:516-520
    assert np.linalg.eigvalsh(k.WeisfeilerLehman(n_iter=5).fit_transform(X)).min() > -1e-5


def test_config1_gram_labels_and_dims(eng):
    k = _k()
    ref = np.load(os.path.join(G, "config1_out.npz"))
    X = gen(188, 18, 0)
    wl = k.WeisfeilerLehman(n_iter=3)
    K = wl.fit_transform(X)
    _same(K, ref["K"])
    assert list(wl.stats_.level_dims[:4]) == ref["D"].tolist()
    _same(wl.diagonal(), np.diagonal(ref["K"]))
    _same(k.WeisfeilerLehman(n_iter=3, normalize=True).fit_transform(X), ref["Knorm"])
    # label partition parity per level against the oracle (SURVEY 8c)
    o = WLOracle(n_iter=3)
    _, levels = o.fit_transform(X, return_levels=True)
    parts = wl_partitions(levels)
    V = wl.X.block.n_vertices
    for lv in range(4):
        dev = eng.wl_labels(lv, V).astype(np.int64)
        ren = {}
        canon = np.fromiter((ren.setdefault(int(x), len(ren)) for x in dev), dtype=np.int64, count=V)
        assert np.array_equal(canon, parts[lv]), f"level {lv} partition differs"
        if lv:  # device ids are already first-occurrence ranks
            assert np.array_equal(dev, canon)
    # exact CUDA-core Gram == tensor-core Gram
    Ks, _, _ = eng.gram(188, simt=True)
    _same(Ks, ref["K"])
    Kf, _, _ = eng.gram(188, dtype=np.float32, full_tiles=True)
    _same(Kf.astype(np.float64), ref["K"])


@pytest.mark.parametrize("T", ["1", "2", "8", "64", "4096"])
def test_head_tail_split_is_exact_for_every_threshold(T, monkeypatch, eng):
    """K must not depend on where the column-frequency threshold falls: all-dense (T=1),
    mixed, and all-tail (T=4096: every shared column goes through atomic pair updates)."""
    monkeypatch.setenv("GRAKEL_B200_FORCE_T", T)
    k = _k()
    ref = np.load(os.path.join(G, "config1_out.npz"))
    X = gen(188, 18, 0)
    wl = k.WeisfeilerLehman(n_iter=3)
    _same(wl.fit_transform(X), ref["K"])
    if T == "4096":
        assert int(wl.stats_.n_dense_columns) == 0 and int(wl.stats_.n_tail_columns) > 0
    _same(k.WeisfeilerLehman(n_iter=3, normalize=True).fit_transform(X), ref["Knorm"])
    Kf, _, _ = eng.gram(188, dtype=np.float32)
    _same(Kf.astype(np.float64), ref["K"])
    d = gio.load(os.path.join(G, "fit_transform.json.gz"))["unit"]
    Xd, Yd = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    for key in ("wl_h4_u", "wl_h4_n"):
        est = k.WeisfeilerLehman(n_iter=4, normalize=key.endswith("n"))
        _same(est.fit_transform(Xd), d["out"][key]["fit_transform"])
        _same(est.transform(Yd), d["out"][key]["transform"])
    with np.errstate(all="ignore"):
        for key in ("sp_l_auto_u", "sp_l_auto_n"):
            est = k.ShortestPath(normalize=key.endswith("n"))
            _same(est.fit_transform(Xd), d["out"][key]["fit_transform"])
            _same(est.transform(Yd), d["out"][key]["transform"])


@pytest.mark.parametrize("n", [1000, 1003, 260])
def test_fp32_output_paths_equal_fp64(eng, n):
    """fp32 K (TMA-store epilogue when rows are 16-byte aligned, vector-store epilogue otherwise)
    must hold the same integers as the fp64 K, in square, row-block and rectangular mode."""
    from grakel_b200.packing import pack, label_ids
    X = gen(n, 14, 11)
    b = pack(X, "wl", len_ok=lambda m: m >= 2)
    ids, _ = label_ids(b.labels, None)
    eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids)
    eng.wl_features(3)
    K64, d64, _ = eng.gram(n)
    for kw in ({}, {"dense_all": True}, {"full_tiles": True}):
        K32, _, _ = eng.gram(n, dtype=np.float32, **kw)
        assert np.array_equal(K32.astype(np.float64), K64), kw
    rb, re_ = n // 3, n // 3 + 300 if n > 600 else n // 3 + 50
    Kr, _, _ = eng.gram(n, dtype=np.float32, row_range=(rb, re_))
    assert np.array_equal(Kr.astype(np.float64), K64[rb:re_])
    nf = n - 128
    Kt64, _, yd = eng.gram(n, n_fit=nf)
    Kt32, _, _ = eng.gram(n, n_fit=nf, dtype=np.float32)
    assert np.array_equal(Kt32.astype(np.float64), Kt64) and Kt64.shape == (128, nf)
    assert np.array_equal(yd, d64[nf:])


@pytest.mark.parametrize("n", [1000, 260, 3000])
def test_cta_pair_gemm_equals_one_cta_gemm(eng, n, monkeypatch):
    """gram_tc2_kernel (tcgen05 cta_group::2, 256 x 256 tiles per two-CTA cluster; GRAKEL_B200_CTA2=0 turns it off) must
    write the same fp32 integers as the one-CTA kernel and as the fp64 matrix: square (mirrored SYRK tiles),
    every column dense, full tiles, a row block, and the rectangular transform shape."""
    from grakel_b200.packing import pack, label_ids
    X = gen(n, 14, 17)
    b = pack(X, "wl", len_ok=lambda m: m >= 2)
    ids, _ = label_ids(b.labels, None)
    eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids)
    eng.wl_features(3)
    K64, _, _ = eng.gram(n)
    nf = n - 136
    Kt64, _, _ = eng.gram(n, n_fit=nf)
    rb, re_ = n // 3, n // 3 + (700 if n > 2000 else 100)
    st = _k()._lib.GkStats()
    for cta2 in ("1", "0"):  # the default (CTA pairs) and the one-CTA kernel
        monkeypatch.setenv("GRAKEL_B200_CTA2", cta2)
        for kw in ({}, {"dense_all": True}, {"full_tiles": True}):
            K32, _, _ = eng.gram(n, dtype=np.float32, stats=st, **kw)
            assert np.array_equal(K32.astype(np.float64), K64), (cta2, kw)
        assert int(st.gram_path) == 1
        Kr, _, _ = eng.gram(n, dtype=np.float32, row_range=(rb, re_))
        assert np.array_equal(Kr.astype(np.float64), K64[rb:re_])
        Kt32, _, _ = eng.gram(n, n_fit=nf, dtype=np.float32)
        assert np.array_equal(Kt32.astype(np.float64), Kt64)


def test_wide_counts_take_the_exact_integer_path():
    """A feature count above 256 is not exact in bf16: the engine must switch to the exact
    u64 CUDA-core Gram on its own (gram_path 2) and still match the oracle bit for bit."""
    k = _k()
    rs = np.random.RandomState(5)
    X = []
    for n in (400, 350, 30, 500):
        A = (rs.rand(n, n) < 0.01).astype(float)
        A = ((A + A.T) > 0).astype(float)
        np.fill_diagonal(A, 0)
        X.append([A, {i: int(i % 10 == 0) for i in range(n)}])  # 90 % of the vertices share a label -> counts up to 450
    wl = k.WeisfeilerLehman(n_iter=2)
    K = wl.fit_transform(X)
    assert int(wl.stats_.max_count) > 256 and int(wl.stats_.gram_path) == 2
    _same(K, WLOracle(n_iter=2).fit_transform(X))
    sp = k.ShortestPath()
    Ks = sp.fit_transform(X[2:3] + X[:1])
    assert int(sp.stats_.gram_path) == 2
    _same(Ks, SPOracle().fit_transform(X[2:3] + X[:1]))


def test_vertex_histogram_is_level0():
    k = _k()
    X = gen(60, 12, 5)
    K = k.VertexHistogram().fit_transform(X)
    Ko = WLOracle(n_iter=1)
    Ko.fit_transform(X)
    _same(K, Ko.levels[0].gram())


def test_high_degree_and_empty_edge_graphs():
    """degree > 32 goes through the warp-per-vertex signature kernel; graphs without
    edges and isolated vertices still count (SURVEY 7: they add to K)."""
    k = _k()
    rs = np.random.RandomState(3)
    X = []
    for n in (70, 150, 40):
        A = np.zeros((n, n))
        A[0, 1:] = A[1:, 0] = 1  # star: hub degree n-1
        extra = rs.rand(n, n) < 0.05
        A = ((A + extra + extra.T) > 0).astype(float)
        np.fill_diagonal(A, 0)
        X.append([A, {i: int(rs.randint(3)) for i in range(n)}])
    X.append([np.zeros((5, 5)), {i: i % 2 for i in range(5)}])
    X.append([{(0, 0): 1.0}, {0: 1}])  # single vertex with a self loop
    for h in (1, 4):
        _same(k.WeisfeilerLehman(n_iter=h).fit_transform(X), WLOracle(n_iter=h).fit_transform(X))
    with np.errstate(all="ignore"):
        _same(k.ShortestPath().fit_transform(X[:4]), SPOracle().fit_transform(X[:4]))


@pytest.mark.parametrize("fused", ["0", "1", "1-multitile", "v1"])
def test_wl_fused_and_multikernel_paths_agree(fused, monkeypatch, eng):
    """The persistent cooperative WL kernel (wl_fused.cuh) and the per-level kernels (wl.cuh)
    must produce the same labels (first-occurrence ids), level sizes and Gram matrix -- on a
    sparse set (thread-per-vertex signatures), on a set with hubs of degree > 32 (warp path)
    and on a block smaller than the grid (empty CTA ranges)."""
    if fused == "1-multitile":  # several tiles per CTA: shared memory is re-staged per tile and level (large inputs)
        monkeypatch.setenv("GRAKEL_B200_WL_TILES_PER_CTA", "3")
        fused = "1"
    if fused == "v1":  # the first-generation fused kernel (dense ranks, two barriers per level)
        monkeypatch.setenv("GRAKEL_B200_WL_V1", "1")
        fused = "1"
    monkeypatch.setenv("GRAKEL_B200_WL_FUSED", fused)
    k = _k()
    rs = np.random.RandomState(11)
    dense = []
    for n in (70, 33, 150, 12):
        A = (rs.rand(n, n) < 0.3).astype(float)
        A = ((A + A.T) > 0).astype(float)
        np.fill_diagonal(A, 0)
        dense.append([A, {i: int(rs.randint(3)) for i in range(n)}])
    for X, h in ((gen(300, 18, 7), 4), (dense, 3), (gen(3, 6, 2), 2)):
        wl = k.WeisfeilerLehman(n_iter=h)
        K = wl.fit_transform(X)
        o = WLOracle(n_iter=h)
        Ko, levels = o.fit_transform(X, return_levels=True)
        _same(K, Ko)
        parts = wl_partitions(levels)
        V = wl.X.block.n_vertices
        for lv in range(1, h + 1):
            dev = eng.wl_labels(lv, V).astype(np.int64)
            assert np.array_equal(dev, parts[lv]), f"level {lv} labels differ (fused={fused})"
        assert list(wl.stats_.level_dims[1:h + 1]) == [int(parts[lv].max()) + 1 for lv in range(1, h + 1)]
        # fit then transform goes through the same kernel with n_fit < n_graphs
        _same(k.WeisfeilerLehman(n_iter=h).fit(X[:-1]).transform(X[-1:]), WLOracle(n_iter=h).fit_transform(X)[-1:, :-1])


def test_fp32_transport_with_host_widening_is_exact(monkeypatch):
    """Default delivery: K crosses PCIe as fp32 -- the upper triangle only for the square case -- and is widened,
    mirrored (and normalised in fp64) by the library's host threads (host_deliver.h); it must be bit-identical to
    the plain fp64 transport of a device-side fp64 result (GRAKEL_B200_WIDEN=0), also for sizes that are not a
    multiple of the band, the strip or the 8 x 8 transpose block, for transform (rectangular) and normalised results."""
    k = _k()
    for n, nbar in ((257, 10), (1031, 8), (2500, 6)):
        X = gen(n, nbar, 9)
        monkeypatch.setenv("GRAKEL_B200_WIDEN", "0")
        K0 = k.WeisfeilerLehman(n_iter=2).fit_transform(X)
        Kn0 = k.WeisfeilerLehman(n_iter=2, normalize=True).fit_transform(X)
        monkeypatch.delenv("GRAKEL_B200_WIDEN", raising=False)
        K1 = k.WeisfeilerLehman(n_iter=2).fit_transform(X)
        assert K1.dtype == np.float64 and K1.flags.c_contiguous
        _same(K1, K0)
        _same(k.WeisfeilerLehman(n_iter=2, normalize=True).fit_transform(X), Kn0)
        Kt = k.WeisfeilerLehman(n_iter=2).fit(X[:-5]).transform(X[-5:])
        _same(Kt, K0[-5:, :-5])
        monkeypatch.setenv("GRAKEL_B200_NO_TRI", "1")  # all rows as fp32 instead of the triangle
        _same(k.WeisfeilerLehman(n_iter=2).fit_transform(X), K0)
        monkeypatch.delenv("GRAKEL_B200_NO_TRI", raising=False)


def test_asynchronous_pass_equals_the_synchronous_route(monkeypatch):
    """gk_wl_gram: the one-synchronisation pass (head/tail threshold chosen on the device, buffers sized by the
    capacities earlier passes left) must give the matrix, self similarities and statistics of gk_wl_features +
    gk_gram bit for bit -- for the float64 host delivery, the library-owned device result and the dense-all mode --
    and must fall back by itself when a capacity does not fit (a larger block packed on the same handle)."""
    from grakel_b200 import _lib
    from grakel_b200.packing import pack, label_ids
    eng = _lib.Engine(0)

    def load(X):
        b = pack(X, "wl")
        ids, _ = label_ids(b.labels, None, sort_new=False)
        eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids)
        return b.n_graphs

    def sync_route(n, h, **kw):
        s = eng.wl_features(h)
        K, xd, _ = eng.gram(n, stats=s, **kw)
        return K, xd, s

    for n_graphs, nbar, h in ((700, 14, 3), (1800, 9, 4)):  # the second block is larger: capacities of the first do not fit
        n = load(gen(n_graphs, nbar, 31))
        K0, xd0, s0 = sync_route(n, h)
        assert s0.gemm_launches > 0
        for rep in range(3):
            K1, xd1, s1 = eng.wl_gram(h, want_diag=True)
            _same(K1, K0)
            assert np.array_equal(xd1, xd0)
            assert [s1.level_dims[i] for i in range(h + 1)] == [s0.level_dims[i] for i in range(h + 1)]
            assert (s1.threshold, s1.n_dense_columns, s1.n_tail_columns, s1.tail_updates) == \
                   (s0.threshold, s0.n_dense_columns, s0.n_tail_columns, s0.tail_updates)
        assert s1.gemm_launches == 0, "the asynchronous pass was expected to run (gemm_launches marks the synchronous gk_gram)"
        # library-owned fp32 device result
        _, _, s2 = eng.wl_gram(h, out=False, dtype=np.float32)
        assert s2.gemm_launches == 0
        full = np.empty((n, n), dtype=np.float32)
        eng.fetch(full)
        _same(full, K0)
        # every shared column dense
        Kd, _, s3 = eng.wl_gram(h, dense_all=True)
        _same(Kd, K0)
        assert s3.n_tail_columns == 0
        # the tail inside the GEMM epilogue: one entry per block applied there, the rest through the overflow list; and
        # the separate tail kernel
        for name, val in (("GRAKEL_B200_TB_CAP", "1"), ("GRAKEL_B200_TB_CAP", "0"), ("GRAKEL_B200_TAIL_FUSED", "0")):
            monkeypatch.setenv(name, val)
            K5, _, s5 = eng.wl_gram(h)
            assert s5.gemm_launches == 0
            _same(K5, K0)
            monkeypatch.delenv(name)
        # the switch
        monkeypatch.setenv("GRAKEL_B200_NO_ASYNC", "1")
        K4, _, s4 = eng.wl_gram(h)
        assert s4.gemm_launches > 0
        _same(K4, K0)
        monkeypatch.delenv("GRAKEL_B200_NO_ASYNC")
    # the oracle, through the one-call host form (pack + gk_wl_gram), twice: synchronous first, asynchronous second
    X = gen(300, 12, 5)
    b = pack(X, "wl")
    ids, _ = label_ids(b.labels, None, sort_new=False)
    Ko = WLOracle(n_iter=3).fit_transform(X)
    e2 = _lib.Engine(0)
    for rep in range(3):
        out = np.empty((b.n_graphs, b.n_graphs), dtype=np.float64)
        e2.wl_fit_transform_raw(b.graph_ptr, b.row_ptr, b.col_idx, ids, 3, out)
        _same(out, Ko)


# --------------------------------------------------------------- SP
def test_apsp_known_answers(eng):
    """grakel/tests/test_graph.py:40,62-65 and doc/documentation/introduction.rst:313-343."""
    k = _k()
    from grakel_b200.packing import pack, label_ids
    inf = float("inf")
    exp = np.array([[0.0, 1.0, inf, 3.0], [1.0, 0.0, inf, 2.0], [2.0, 3.0, 0.0, 1.0], [1.0, 2.0, inf, 0.0]])
    A = np.array([[1, 1, 0, 3], [1, 0, 0, 2], [2, 3, 0, 1], [1, 0, 0, 0]])
    lab = {0: "banana", 1: "cherry", 2: "banana", 3: "cherry"}
    D = {"a": {"a": 1, "b": 1, "d": 3}, "b": {"a": 1, "d": 2}, "c": {"a": 2, "b": 3, "d": 1}, "d": {"a": 1}}
    for g, L in ((A, lab), (D, {"a": "banana", "b": "cherry", "c": "banana", "d": "cherry"})):
        b = pack([[g, L]], "sp", want_weights=True)
        ids, _ = label_ids(b.labels, None, sort_new=False)
        eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids, b.weights)
        eng.sp_features(with_labels=True, keep_dist=True)
        assert np.array_equal(eng.sp_distances(0, 4), exp)
    H2O = [[[0, 1, 1], [1, 0, 0], [1, 0, 0]], {0: "O", 1: "H", 2: "H"}]
    H3O = [[[0, 1, 1, 1], [1, 0, 0, 0], [1, 0, 0, 0], [1, 0, 0, 0]], {0: "O", 1: "H", 2: "H", 3: "H"}]
    sp = k.ShortestPath()
    assert sp.fit_transform([H2O]).tolist() == [[12.0]]
    assert sp.transform([H3O]).tolist() == [[24.0]]
    sp = k.ShortestPath(normalize=True)
    assert sp.fit_transform([H2O]).tolist() == [[1.0]]
    assert abs(sp.transform([H3O])[0, 0] - 0.94280904) < 1e-8


def test_config3_small_and_large_graph_path():
    k = _k()
    ref = np.load(os.path.join(G, "config3_small_out.npz"))
    sp = k.ShortestPath()
    _same(sp.fit_transform(gen(40, 60, 0, as_adj=True)), ref["K"])
    assert int(sp.stats_.n_columns) == int(ref["D"])
    # graphs whose distance matrix does not fit shared memory use the global-memory path
    X = gen(3, 420, 9, as_adj=True) + gen(5, 30, 9, as_adj=True)
    _same(k.ShortestPath().fit_transform(X), SPOracle().fit_transform(X))
    _same(k.ShortestPath(with_labels=False).fit_transform(X), SPOracle(with_labels=False).fit_transform(X))


# --------------------------------------------------------------- SP-attr
@pytest.mark.parametrize("mode", ["tf32x3", "fp64"])
def test_shortest_path_attr_matches_reference_loop(mode, monkeypatch):
    """Golden from the real reference's 4-deep loop (shortest_path.py:151-162) on tiny graphs, then the oracle's
    feature-map form on a config-5 shaped subset and SURVEY 8c's real-reference K[0,:5] of config 5.

    Default path: tcgen05 kind::tf32 GEMM on a hi/lo split of the fp64 features (3 passes, fp32 accumulation folded
    into fp64 every few hundred MMAs, rows scaled by powers of two so the range is fp64's); error within 1e-5 of
    sum_k |phi_ik| |phi_jk|, i.e. 1e-5 relative here, where the attributes are non-negative (observed ~2e-6; signed
    attributes: normwise only, tests/test_spattr_edges.py).  GRAKEL_B200_SPATTR_F64=1: the fp64 CUDA-core Gram, 1e-9
    elementwise.  Self similarities (the diagonal and what normalisation divides by) are exact fp64 in both."""
    from oracle.gk_oracle import SPAttrOracle
    tol = 1e-9 if mode == "fp64" else 1e-5
    if mode == "fp64":
        monkeypatch.setenv("GRAKEL_B200_SPATTR_F64", "1")
    else:
        monkeypatch.delenv("GRAKEL_B200_SPATTR_F64", raising=False)
    k = _k()
    d = gio.load(os.path.join(G, "spattr.json.gz"))
    X, Y = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    est = k.ShortestPathAttr()
    K = est.fit_transform(X)
    np.testing.assert_allclose(K, np.asarray(d["K"]), rtol=tol)
    assert np.array_equal(K, K.T)
    np.testing.assert_allclose(np.diagonal(K), np.diagonal(np.asarray(d["K"])), rtol=1e-12)
    np.testing.assert_allclose(est.transform(Y), np.asarray(d["Kt"]), rtol=tol)
    est = k.ShortestPathAttr(normalize=True)
    np.testing.assert_allclose(est.fit_transform(X), np.asarray(d["Kn"]), rtol=tol)
    np.testing.assert_allclose(est.transform(Y), np.asarray(d["Ktn"]), rtol=tol)
    Xc = gen(24, 40, 0, attr=16, as_adj=True)  # first graphs of BASELINE config 5
    Ko = SPAttrOracle().fit_transform(Xc)
    Kd = k.GraphKernel(kernel={"name": "shortest_path", "as_attributes": True}).fit_transform(Xc)
    np.testing.assert_allclose(Kd, Ko, rtol=tol)
    np.testing.assert_allclose(Kd[0, :5], [837683.171027, 2683836.635183, 1663520.495733, 1549141.171651, 2537314.325017],
                               rtol=max(tol, 1e-9))  # SURVEY.md 8c: real-reference K[0,:5] of config 5
    if mode == "tf32x3":  # the observed error, not just the bound: a regression to plain tf32 (1e-3) or bf16 would show
        err = float(np.max(np.abs(Kd - Ko) / np.abs(Ko)))
        assert err < 3e-6, err
        # a few hundred graphs: several row tiles, k-chunk folding, mirrored tiles, against the fp64 device Gram
        Xm = gen(300, 30, 3, attr=16, as_adj=True)
        K32 = k.ShortestPathAttr().fit_transform(Xm)
        monkeypatch.setenv("GRAKEL_B200_SPATTR_F64", "1")
        K64 = k.ShortestPathAttr().fit_transform(Xm)
        assert np.array_equal(K32, K32.T)
        np.testing.assert_allclose(K32, K64, rtol=3e-6)
    # a metric that is np.dot in disguise takes the generic pairwise route (device APSP + host contraction): same matrix
    Kp = k.ShortestPathAttr(metric=lambda a, b: float(np.dot(a, b))).fit_transform(Xc[:3])
    np.testing.assert_allclose(Kp, Ko[:3, :3], rtol=1e-9)


def test_spattr_user_metric_against_reference_goldens():
    """ShortestPathAttr(metric=<callable>): shortest-path matrices from the device (gk_spattr_features ->
    gk_sp_distances; unit weights and real-valued weights in Dijkstra order), the reference's per-pair contraction on
    the host through the generic driver (kernel.py:236-296, shortest_path.py:130-164).  Goldens: the real reference
    (tests/golden/make_golden_spattr_metric.py).  Tolerance 1e-9: only the summation order differs."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk_spattr_metric", os.path.join(G, "make_golden_spattr_metric.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    k = _k()
    ref = np.load(os.path.join(G, "spattr_metric.npz"))
    X = mk.gen_attr(9, 7, 11)
    fit, new = X[:6], X[6:]
    e = k.ShortestPathAttr(metric=mk.rbf)
    K = e.fit_transform(fit)
    np.testing.assert_allclose(K, ref["unit_K"], rtol=1e-9)
    np.testing.assert_allclose(e.transform(new), ref["unit_Kt"], rtol=1e-9)
    e = k.ShortestPathAttr(metric=mk.rbf, normalize=True)
    np.testing.assert_allclose(e.fit_transform(fit), ref["unit_Kn"], rtol=1e-9)
    np.testing.assert_allclose(e.transform(new), ref["unit_Ktn"], rtol=1e-9)
    W = mk.gen_attr(6, 6, 12, real_weights=True)
    e = k.ShortestPathAttr(metric=mk.rbf)
    np.testing.assert_allclose(e.fit_transform(W[:4]), ref["real_K"], rtol=1e-9)
    np.testing.assert_allclose(e.transform(W[4:]), ref["real_Kt"], rtol=1e-9)
    # through GraphKernel, as the reference spells it
    gk_ = k.GraphKernel(kernel={"name": "shortest_path", "as_attributes": True, "metric": mk.rbf})
    np.testing.assert_allclose(gk_.fit_transform(fit), ref["unit_K"], rtol=1e-9)


# --------------------------------------------------------------- BASELINE sizes
def test_config2_full_size_properties():
    """N = 10 000, h = 5 (BASELINE config 2): checksums + sampled rows from the real
    reference run (tests/golden/make_golden.py --big) and size-independent properties."""
    k = _k()
    rows = np.load(os.path.join(G, "config2_rows.npz"))
    big = gio.load(os.path.join(G, "big_summaries.json.gz"))["config2"]
    X = gen(10000, 40, 0)
    wl = k.WeisfeilerLehman(n_iter=5)
    K = wl.fit_transform(X)
    assert K.shape == (10000, 10000)
    assert list(wl.stats_.level_dims[:6]) == big["D"]
    assert float(K.sum()) == big["sum"] == 22925628586.0
    assert float(np.trace(K)) == big["trace"] and float(K.max()) == big["max"]
    assert np.array_equal(K[rows["rows"]], rows["K_rows"].astype(np.float64))
    assert np.array_equal(np.diagonal(K), rows["diag"].astype(np.float64))
    assert np.array_equal(K, K.T)  # symmetry (mirrored tiles)
    assert int(wl.stats_.gram_path) == 1  # tensor-core path for the head columns
    # all shared columns on the tensor cores gives the same matrix
    from grakel_b200 import _lib
    Kd, _, _ = _lib.get_engine().gram(10000, dtype=np.float32, dense_all=True)
    assert np.array_equal(Kd, K.astype(np.float32))


def test_config3_full_size_properties():
    k = _k()
    rows = np.load(os.path.join(G, "config3_rows.npz"))
    big = gio.load(os.path.join(G, "big_summaries.json.gz"))["config3"]
    sp = k.ShortestPath()
    K = sp.fit_transform(gen(5000, 60, 0, as_adj=True))
    assert int(sp.stats_.n_columns) == big["D"] == 476
    assert float(K.sum()) == big["sum"] and float(np.trace(K)) == big["trace"] and float(K.max()) == big["max"]
    assert np.array_equal(K[rows["rows"]], rows["K_rows"].astype(np.float64))
    assert np.array_equal(K, K.T)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["er60", "er25_deep"])
def test_exported_level_dictionaries_equal_the_references(name):
    """`WeisfeilerLehman._inv_labels[i]` for every level (weisfeiler_lehman.py:208-257): device relabel ->
    gk_wl_labels -> the reference's credential strings and numbering, against the real reference's dictionaries
    (tests/golden/make_golden_invlabels.py).  Asking for a level does not disturb the fitted state."""
    import gzip
    import json
    with gzip.open(os.path.join(G, "inv_labels.json.gz"), "rt") as f:
        case = json.load(f)[name]
    c = case["params"]
    X = gen(c["N"], c["nbar"], c["seed"], nl=c["nl"])
    k = _k()
    wl = k.WeisfeilerLehman(n_iter=c["n_iter"])
    K = wl.fit_transform(X)
    for i, pairs in case["levels"].items():
        want = {(key if int(i) else int(key)): v for key, v in pairs}
        assert wl._inv_labels[int(i)] == want, f"level {i}"
    assert len(wl.wl_labels_) == c["n_iter"] + 1
    Kt = wl.transform(X[:5])
    _same(Kt, K[:5])
    w2 = pickle.loads(pickle.dumps(wl))
    assert sorted(w2._inv_labels) == list(range(c["n_iter"] + 1))
