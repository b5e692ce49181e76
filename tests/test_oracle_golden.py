"""Pin the CPU oracle (oracle/gk_oracle.py) to vectors produced by the real
reference (tests/golden/make_golden.py).  CPU-only; runs everywhere."""
import os

import numpy as np
import pytest

import gio
from oracle.gk_oracle import SPAttrOracle, SPOracle, WLOracle, OGraph, gen

G = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return gio.load(os.path.join(G, name))


def _eq(a, b, exact=True):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape
    if exact:
        assert np.array_equal(a, b, equal_nan=True)
    else:
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, equal_nan=True)


def _check_out(X, Y, out):
    for key, rec in out.items():
        parts = key.split("_")
        if parts[0] == "wl":
            h, norm = int(parts[1][1:]), parts[2] == "n"
            o = WLOracle(n_iter=h, normalize=norm)
            _eq(o.fit_transform(X), rec["fit_transform"])
            if "D" in rec:
                assert [lv.X.shape[1] for lv in o.levels] == rec["D"]
            if "transform" in rec:
                _eq(o.transform(Y), rec["transform"])
        else:
            wlab, alg, norm = parts[1] == "l", "_".join(parts[2:-1]), parts[-1] == "n"
            if "error" in rec:
                continue
            o = SPOracle(with_labels=wlab, algorithm_type=alg, normalize=norm)
            with np.errstate(all="ignore"):
                _eq(o.fit_transform(X), rec["fit_transform"])
                if "transform" in rec:
                    _eq(o.transform(Y), rec["transform"])


def test_spellings():
    g = _load("spellings.json.gz")
    for name, case in g["cases"].items():
        _check_out(gio.dec_dataset(case["X"]), None, case["out"])


@pytest.mark.parametrize("tag", ["unit", "intw", "realw"])
def test_fit_transform_unseen_labels(tag):
    d = _load("fit_transform.json.gz")[tag]
    X, Y = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    out = d["out"]
    if tag == "realw":
        # real weights: the reference's own Dijkstra and Floyd-Warshall paths give
        # different float keys (SURVEY 7 "hard parts"); the oracle's Dijkstra is a
        # heap, not the reference's priority_dict, so only the FW/auto(adjacency) path
        # is pinned bit-exactly.
        out = {k: v for k, v in out.items() if "dijkstra" not in k}
    _check_out(X, Y, out)


def test_mutag():
    X = gio.dec_dataset(_load("mutag_graphs.json.gz"))
    ref = np.load(os.path.join(G, "mutag_out.npz"))
    for h in (3, 5):
        _eq(WLOracle(n_iter=h).fit_transform(X), ref[f"wl_h{h}"])
    _eq(SPOracle().fit_transform(X), ref["sp"])
    tr, te = ref["split_train"].tolist(), ref["split_test"].tolist()
    o = WLOracle(n_iter=3, normalize=True)
    _eq(o.fit_transform([X[i] for i in tr]), ref["wl_h3_norm_train"])
    _eq(o.transform([X[i] for i in te]), ref["wl_h3_norm_test"])
    o = SPOracle(normalize=True)
    _eq(o.fit_transform([X[i] for i in tr]), ref["sp_norm_train"])
    _eq(o.transform([X[i] for i in te]), ref["sp_norm_test"])


def test_config1():
    ref = np.load(os.path.join(G, "config1_out.npz"))
    o = WLOracle(n_iter=3)
    K = o.fit_transform(gen(188, 18, 0))
    _eq(K, ref["K"])
    assert [lv.X.shape[1] for lv in o.levels] == ref["D"].tolist()
    assert K.sum() == 1607302 and np.trace(K) == 22060  # SURVEY.md 8c
    _eq(WLOracle(n_iter=3, normalize=True).fit_transform(gen(188, 18, 0)), ref["Knorm"])


def test_config3_small():
    ref = np.load(os.path.join(G, "config3_small_out.npz"))
    o = SPOracle()
    _eq(o.fit_transform(gen(40, 60, 0, as_adj=True)), ref["K"])
    assert len(o.enum) == int(ref["D"])


def test_spattr():
    d = _load("spattr.json.gz")
    X, Y = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    o = SPAttrOracle()
    np.testing.assert_allclose(o.fit_transform(X), np.asarray(d["K"]), rtol=1e-12)
    np.testing.assert_allclose(o.transform(Y), np.asarray(d["Kt"]), rtol=1e-12)
    o = SPAttrOracle(normalize=True)
    np.testing.assert_allclose(o.fit_transform(X), np.asarray(d["Kn"]), rtol=1e-12)
    np.testing.assert_allclose(o.transform(Y), np.asarray(d["Ktn"]), rtol=1e-12)


def test_spattr_dense_reference():
    """tests/spattr_ref.py, the fp64 feature-matrix restatement the device ShortestPathAttr tests compare with
    (K = Phi Phi^T), against the real reference: fit_transform / transform, raw and normalised, and the path sums in
    Dijkstra's order on real-valued weights (its Floyd-Warshall twin gives a different matrix there)."""
    import sys
    from spattr_ref import spattr_ref
    sys.path.insert(0, G)
    from make_golden_dijkstra import gen_real
    d = _load("spattr.json.gz")
    X, Y = gio.dec_dataset(d["X"]), gio.dec_dataset(d["Y"])
    for key, Yk, norm in (("K", None, False), ("Kt", Y, False), ("Kn", None, True), ("Ktn", Y, True)):
        K, K_abs, drow, dcol = spattr_ref(X, Yk, normalize=norm)
        np.testing.assert_allclose(K, np.asarray(d[key]), rtol=1e-12)
        assert np.all(np.abs(K) <= K_abs * (1 + 1e-12))
    K, K_abs, drow, dcol = spattr_ref(X)
    assert np.array_equal(K, K.T) and np.array_equal(np.diagonal(K), drow) and np.array_equal(drow, dcol)
    np.testing.assert_allclose(K_abs, K, rtol=1e-12)  # non-negative attributes: the error scale is K itself
    A = gen_real(7, 8, 5, attr=3)
    ref = np.load(os.path.join(G, "dijkstra_real.npz"))["attr_dj_K"]
    np.testing.assert_allclose(spattr_ref(A, algorithm_type="dijkstra")[0], ref, rtol=1e-12)
    assert not np.allclose(spattr_ref(A, algorithm_type="floyd_warshall")[0], ref, rtol=1e-6)


def test_apsp_known_answer():
    """The reference's own APSP known-answer (grakel/tests/test_graph.py:40,62-65
    adjacency input with a self loop; :80-83,119-122 the same graph as a nested
    edge dictionary): directed, weighted, one unreachable vertex."""
    inf = float("inf")
    exp = np.array([[0.0, 1.0, inf, 3.0], [1.0, 0.0, inf, 2.0], [2.0, 3.0, 0.0, 1.0], [1.0, 2.0, inf, 0.0]])
    A = np.array([[1, 1, 0, 3], [1, 0, 0, 2], [2, 3, 0, 1], [1, 0, 0, 0]])
    lab = {0: "banana", 1: "cherry", 2: "banana", 3: "cherry"}
    g = OGraph(A, lab)
    assert np.array_equal(g.shortest_paths("auto"), exp)
    assert np.array_equal(g.dijkstra_all(), exp)
    D = {"a": {"a": 1, "b": 1, "d": 3}, "b": {"a": 1, "d": 2}, "c": {"a": 2, "b": 3, "d": 1}, "d": {"a": 1}}
    g = OGraph(D, {"a": "banana", "b": "cherry", "c": "banana", "d": "cherry"})
    assert np.array_equal(g.shortest_paths("auto"), exp)
    assert np.array_equal(g.floyd_warshall(), exp)
    assert g.index_labels() == lab


def test_doc_known_answers():
    """doc/documentation/introduction.rst:313-343: SP(H2O)=12, SP(H2O,H3O)=24,
    normalised 1.0 / 0.94280904."""
    H2O = [[[0, 1, 1], [1, 0, 0], [1, 0, 0]], {0: "O", 1: "H", 2: "H"}]
    H3O = [[[0, 1, 1, 1], [1, 0, 0, 0], [1, 0, 0, 0], [1, 0, 0, 0]], {0: "O", 1: "H", 2: "H", 3: "H"}]
    o = SPOracle()
    assert o.fit_transform([H2O]).tolist() == [[12.0]]
    assert o.transform([H3O]).tolist() == [[24.0]]
    o = SPOracle(normalize=True)
    assert o.fit_transform([H2O]).tolist() == [[1.0]]
    assert abs(o.transform([H3O])[0, 0] - 0.94280904) < 1e-8
