"""SURVEY 8(f) rank 4: TU-format files -> packed CSR through the C-ABI reader (gk_tu_*), and the packed-block
fast path of the estimators.

CPU (-m "not gpu"): the native reader against (a) the oracle's restatement of read_data, (b) digests of the REAL
reference's read_data on its own bundled datasets (tests/golden/tu_digest.json; the MUTAG and Cuneiform files are
stored in tests/golden/tu_datasets.tar.xz), (c) the reference's MUTAG kernel matrices through the numpy model of the
device pipeline.
GPU (-m gpu): estimators fed with blocks read from files against the same goldens."""
import json
import os
import tarfile

import numpy as np
import pytest

import blockref
import gio
import tu_io
from grakel_b200 import (ShortestPath, ShortestPathAttr, VertexHistogram, WeisfeilerLehman,
                         WeisfeilerLehmanOptimalAssignment)
from grakel_b200.datasets import read_tu
from grakel_b200.packing import Block, label_ids, pack
from oracle.gk_oracle import WLOAOracle, gen, read_data_oracle, tu_digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def _mutag():
    return gio.dec_dataset(gio.load(os.path.join(G, "mutag_graphs.json.gz")))


def _elements_of(bunch, mode):
    """Back from a packed block to read_data-style elements (global 1-based node ids)."""
    b, node = bunch.data, bunch.node_ids
    out = []
    for g in range(b.n_graphs):
        v0, v1 = int(b.graph_ptr[g]), int(b.graph_ptr[g + 1])
        edges = set()
        for v in range(v0, v1):
            for k in range(int(b.row_ptr[v]), int(b.row_ptr[v + 1])):
                edges.add((int(node[v]), int(node[b.col_idx[k]])))
        if b.attrs is not None:
            lab = {int(node[v]): [float(x) for x in b.attrs[v]] for v in range(v0, v1)}
        elif b.labels is not None:
            lab = {int(node[v]): int(b.labels[v]) for v in range(v0, v1)}
        else:
            lab = {int(node[v]): 0 for v in range(v0, v1)}
        out.append([edges, lab, {}])
    return out


@pytest.fixture(scope="module")
def mutag_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("tu")
    X = _mutag()
    tu_io.write_tu(str(d), "MUTAG", X, classes=[1 if i % 3 else -1 for i in range(len(X))])
    return str(d)


@pytest.fixture(scope="module")
def bundled_dir(tmp_path_factory):
    """The reference's bundled MUTAG and Cuneiform datasets (tests/data of ysig/GraKeL, without Cuneiform's edge
    attributes, which read_data does not read), extracted from tests/golden/tu_datasets.tar.xz."""
    d = tmp_path_factory.mktemp("bundled")
    with tarfile.open(os.path.join(G, "tu_datasets.tar.xz")) as t:
        t.extractall(d, filter="data")
    return str(d)


# ------------------------------------------------------------------ reader vs read_data
@pytest.mark.parametrize("kernel,mode", [("WL", "wl"), ("SP", "sp")])
def test_reader_matches_the_read_data_restatement(mutag_dir, kernel, mode):
    ref, classes = read_data_oracle(mutag_dir, "MUTAG")
    got = read_tu(mutag_dir, "MUTAG", kernel=kernel)
    assert tu_digest(_elements_of(got, mode), mode) == tu_digest(ref, mode)
    assert np.array_equal(got.target, classes)
    assert got.data.mode == mode and got.data.n_graphs == 188


@pytest.mark.parametrize("name", ["MUTAG", "Cuneiform"])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("attr", [False, True])
def test_reader_matches_the_real_reference_on_its_bundled_datasets(bundled_dir, name, sym, attr):
    gold = json.load(open(os.path.join(G, "tu_digest.json")))[f"{name}_sym{int(sym)}_attr{int(attr)}"]
    if "error" in gold:  # Cuneiform's two-column node_labels.txt: int() raises ValueError in read_data
        with pytest.raises(ValueError):
            read_tu(bundled_dir, name, kernel="WL", is_symmetric=sym, prefer_attr_nodes=attr)
        return
    for kernel, mode in (("WL", "wl"), ("SP", "sp")):
        got = read_tu(bundled_dir, name, kernel=kernel, is_symmetric=sym, prefer_attr_nodes=attr)
        assert got.data.n_graphs == gold["graphs"]
        assert tu_digest(_elements_of(got, mode), mode) == gold[mode]
        assert int(got.target.sum()) == gold["classes_sum"]
        assert len(got.edge_labels) == gold["edge_label_entries"] and int(got.edge_labels.sum()) == gold["edge_label_sum"]
    # and the oracle's restatement of read_data agrees with the real one
    ref, _ = read_data_oracle(bundled_dir, name, is_symmetric=sym, prefer_attr_nodes=attr)
    assert tu_digest(ref, "wl") == gold["wl"] and tu_digest(ref, "sp") == gold["sp"]


def test_reader_edge_semantics(tmp_path):
    d = str(tmp_path)
    # two graphs; a duplicated edge line, a one-directional edge, an isolated node (5), a self loop
    X = [[[(1, 2), (2, 1), (1, 2), (2, 3)], {1: 7, 2: 8, 3: 7}], [[(4, 4), (4, 6)], {4: 1, 5: 2, 6: 3}]]
    EL = [{(1, 2): 5, (2, 1): 6, (2, 3): 9}, {(4, 4): 1, (4, 6): 2}]
    EL[0][(1, 2)] = 4  # the last line of a repeated pair wins (base.py:262-266)
    tu_io.write_tu(d, "T", X, classes=[0, 1], edge_labels=EL)
    b = read_tu(d, "T", kernel="WL")
    assert b.data.graph_ptr.tolist() == [0, 3, 6] and b.data.row_ptr.tolist() == [0, 1, 3, 3, 5, 5, 5]
    assert b.data.col_idx.tolist() == [1, 0, 2, 3, 5] and b.edge_labels.tolist() == [4, 6, 9, 1, 2]
    assert b.data.labels.tolist() == [7, 8, 7, 1, 2, 3]
    s = read_tu(d, "T", kernel="SP")  # node 5 occurs in no edge: not a vertex for ShortestPath / WL-OA
    assert s.data.graph_ptr.tolist() == [0, 3, 5] and s.node_ids.tolist() == [1, 2, 3, 4, 6]
    y = read_tu(d, "T", kernel="WL", is_symmetric=True)  # reverse edges added
    assert y.data.row_ptr.tolist() == [0, 1, 3, 4, 6, 6, 7] and y.data.col_idx.tolist() == [1, 0, 2, 1, 3, 5, 3]
    ref, _ = read_data_oracle(d, "T", is_symmetric=True)
    assert tu_digest(_elements_of(y, "wl"), "wl") == tu_digest(ref, "wl")
    assert sorted(ref[0][2].items()) == [((1, 2), 4), ((2, 1), 4), ((2, 3), 9), ((3, 2), 9)]
    assert y.edge_labels.tolist() == [4, 4, 9, 9, 1, 2, 2]
    # no label file + produce_labels_nodes: out-degree without self loops; nodes of degree 0 stay unlabelled
    tu_io.write_tu(str(tmp_path / "n"), "T", X, node_labels=False)
    dg = read_tu(str(tmp_path / "n"), "T", kernel="SP", with_classes=False, produce_labels_nodes=True, is_symmetric=True)
    assert dg.data.labels.tolist() == [1, 2, 1, 1, 1] and dg.node_ids.tolist() == [1, 2, 3, 4, 6]
    ref, _ = read_data_oracle(str(tmp_path / "n"), "T", is_symmetric=True, produce_labels_nodes=True)
    assert tu_digest(_elements_of(dg, "sp"), "sp") == tu_digest(ref, "sp")


def test_reader_errors(tmp_path):
    d = str(tmp_path)
    with pytest.raises(ValueError, match="graph_indicator"):
        read_tu(d, "missing")
    X = [[[(1, 2)], {1: 0, 2: 0}], [[(3, 3)], {3: 1}]]
    tu_io.write_tu(d, "T", X)
    with pytest.raises(ValueError, match="classes"):
        read_tu(d, "T")  # with_classes but no graph_labels file
    with pytest.raises(ValueError):
        read_tu(d, "T", kernel="RW")
    open(os.path.join(d, "T_A.txt"), "a").write("1, 3\n")  # joins two graphs: KeyError in the reference
    with pytest.raises(ValueError, match="different graphs"):
        read_tu(d, "T", with_classes=False)
    open(os.path.join(d, "T_A.txt"), "w").write("1, x\n")
    with pytest.raises(ValueError, match="not an integer"):
        read_tu(d, "T", with_classes=False)
    open(os.path.join(d, "T_A.txt"), "w").write("1, 9\n")
    with pytest.raises(ValueError, match="out of range"):
        read_tu(d, "T", with_classes=False)
    b = read_tu(str(tmp_path), "T", with_classes=False) if False else None
    assert b is None
    with pytest.raises(ValueError, match="another kernel"):  # a WL block handed to ShortestPath
        tu_io.write_tu(d, "U", X)
        ShortestPath().fit(read_tu(d, "U", kernel="WL", with_classes=False).data)


def test_vectorised_label_ids_match_the_generic_path():
    rs = np.random.RandomState(0)
    lab = rs.randint(-3, 9, size=200).astype(np.int32)
    for sort_new in (True, False):
        a, da = label_ids(lab, None, sort_new=sort_new)
        b, db = label_ids(lab.tolist(), None, sort_new=sort_new)
        assert np.array_equal(a, b) and da == db
        known = {int(k): i for i, k in enumerate([4, 0, -3])}
        a, da = label_ids(lab, known, sort_new=sort_new)
        b, db = label_ids(lab.tolist(), known, sort_new=sort_new)
        assert np.array_equal(a, b) and da == db


# ------------------------------------------------------------------ packed blocks through the device model
def test_mutag_blocks_reproduce_the_reference_matrices_on_the_device_model(mutag_dir):
    ref = np.load(os.path.join(G, "mutag_out.npz"))
    b = read_tu(mutag_dir, "MUTAG", kernel="WL", with_classes=False).data
    est = WeisfeilerLehman(n_iter=3)
    est._method_calling = 1
    est.initialize()
    f = est.parse_input(b)  # the packed fast path: no per-graph Python
    assert f.block is b
    K, _, _ = blockref.wl_gram_block(f.block, f.ids, 3)
    assert np.array_equal(K, ref["wl_h3"])
    s = read_tu(mutag_dir, "MUTAG", kernel="SP", with_classes=False).data
    sp = ShortestPath()
    sp._method_calling = 1
    sp.initialize()
    f = sp.parse_input(s)
    K, _, _ = blockref.sp_gram_block(f.block, f.ids)
    assert np.array_equal(K, ref["sp"])
    # same block as the Python packer builds from the element list (vertex order = node id order)
    p = pack(_mutag(), "wl")
    assert np.array_equal(p.graph_ptr, b.graph_ptr) and np.array_equal(p.row_ptr, b.row_ptr)
    assert np.array_equal(p.col_idx, b.col_idx) and list(p.labels) == b.labels.tolist()


# ------------------------------------------------------------------ the CUDA path
@pytest.mark.gpu
def test_gpu_estimators_accept_blocks_read_from_files(mutag_dir, tmp_path):
    ref = np.load(os.path.join(G, "mutag_out.npz"))
    wl = read_tu(mutag_dir, "MUTAG", kernel="WL", with_classes=False).data
    sp = read_tu(mutag_dir, "MUTAG", kernel="SP", with_classes=False).data
    for h in (3, 5):
        assert np.array_equal(WeisfeilerLehman(n_iter=h).fit_transform(wl), ref[f"wl_h{h}"])
    assert np.array_equal(ShortestPath().fit_transform(sp), ref["sp"])
    X = _mutag()
    assert np.array_equal(VertexHistogram().fit_transform(wl), VertexHistogram().fit_transform(X))
    assert np.array_equal(WeisfeilerLehmanOptimalAssignment(n_iter=4).fit_transform(sp)[:60, :60],
                          np.load(os.path.join(G, "wloa.npz"))["oa_mutag_h4"])
    # fit on one file set, transform another (train / test split written as two datasets)
    tr, te = X[:150], X[150:]
    tu_io.write_tu(str(tmp_path), "TR", tr)
    shift = min(te[0][1]) - 1
    te0 = [[[(a - shift, b - shift) for a, b in g], {v - shift: l for v, l in lab.items()}] for g, lab in te]
    tu_io.write_tu(str(tmp_path), "TE", te0)
    for est, kern in ((WeisfeilerLehman(n_iter=3, normalize=True), "WL"), (ShortestPath(normalize=True), "SP"),
                      (WeisfeilerLehmanOptimalAssignment(n_iter=3), "WL-OA")):
        a = read_tu(str(tmp_path), "TR", kernel=kern, with_classes=False).data
        b = read_tu(str(tmp_path), "TE", kernel=kern, with_classes=False).data
        e2 = type(est)(**est.get_params())
        Kf, Kt = est.fit_transform(a), est.transform(b)
        assert np.array_equal(Kf, e2.fit_transform(tr)) and np.array_equal(Kt, e2.transform(te))


@pytest.mark.gpu
def test_gpu_attribute_blocks(tmp_path):
    X = gen(12, 10, 4, attr=3)
    Xr = tu_io.renumber(X)
    tu_io.write_tu(str(tmp_path), "A", [[g, {v: 0 for v in l}] for g, l in Xr], attributes={v: a for _, l in Xr for v, a in l.items()})
    b = read_tu(str(tmp_path), "A", kernel="SP", with_classes=False, prefer_attr_nodes=True).data
    keep = [i for i, (g, _l) in enumerate(X) if len(g)]  # graphs with at least one edge
    K = ShortestPathAttr().fit_transform(b)
    Kl = ShortestPathAttr().fit_transform([X[i] for i in keep])
    np.testing.assert_allclose(K[np.ix_(keep, keep)], Kl, rtol=1e-9)
