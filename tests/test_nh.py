"""NeighborhoodHash (neighborhood_hash.py).  Goldens come from the REAL reference (tests/golden/make_golden_nh.py ->
tests/golden/nh.npz).

CPU (-m "not gpu"): the oracle restatement and the numpy model of the device pipeline (tests/nh_ref.py) against the
goldens bit for bit; the estimator's host logic (label set, hash dictionary, RandomState consumption, level-0 labels,
None seeding), its errors, dispatch and pickling.  GPU (-m gpu): the CUDA path through the C-ABI."""
import os
import pickle
import tempfile
import warnings

import numpy as np
import pytest

import nh_ref
from grakel_b200 import GraphKernel, NeighborhoodHash
from grakel_b200.packing import Block
from nh_ref import NHOracle, nh_pipeline_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
REF = np.load(os.path.join(G, "nh.npz"))

import importlib.util  # noqa: E402

_spec = importlib.util.spec_from_file_location("make_golden_nh", os.path.join(G, "make_golden_nh.py"))
mg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mg)
SETS = mg.nh_sets()
CASES = [(s, t, R, b) for s in SETS for (t, R, b) in mg.CASES]
IDS = ["%s-%s-R%d-b%d" % c for c in CASES]


def _tag(s, t, R, b):
    return f"{s}_{t}_R{R}_b{b}"


def _eq(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(a, b), f"max abs diff {np.max(np.abs(a - b)) if a.size else 0}"


def _est(t, R, b):
    return NeighborhoodHash(R=R, nh_type=t, bits=b, random_state=R * 100 + b)


def _golden_dict(tag):
    return dict(zip(REF[tag + "_hk"].tolist(), REF[tag + "_hv"].tolist()))


# ------------------------------------------------------------------ oracle vs the real reference
@pytest.mark.parametrize("s,t,R,b", CASES, ids=IDS)
def test_oracle_matches_reference(s, t, R, b):
    fit, new = SETS[s]
    tag = _tag(s, t, R, b)
    o = NHOracle(R=R, nh_type=t, bits=b, random_state=R * 100 + b)
    _eq(o.fit_transform(fit), REF[tag + "_K"])
    assert list(o.hash_dict.items()) == list(_golden_dict(tag).items())  # same keys, values AND iteration order
    _eq(o.transform(new), REF[tag + "_Kt"])


def test_oracle_matches_reference_on_mutag():
    X = mg.mutag()
    for t in ("simple", "count_sensitive"):
        _eq(NHOracle(R=3, nh_type=t, random_state=5).fit_transform(X), REF[f"mutag_{t}"])


def test_the_goldens_exercise_the_corner_cases():
    # more labels than 2^bits (5 labels, bits = 2): the chunked draws of :165-181
    assert len(REF["small_simple_R1_b2_hk"]) > 4
    # count-sensitive labels above the mask: ROT(l ^ occ, occ) with occ % bits == 0 is not masked
    fit, _ = SETS["hubs"]
    o = NHOracle(R=3, nh_type="count_sensitive", bits=2, random_state=302).fit(fit)
    assert max(l for _, lv in o.X for lab in lv for l in lab.values() if l is not None) > 3
    # unseen transform labels: None reaches the histogram's exclusion
    _, new = SETS["small"]
    o = NHOracle(R=3, random_state=308).fit(SETS["small"][0])
    ys = [o._levels(g, L) for g, L in o._graphs(new)]
    assert any(l is None for lv in ys for lab in lv for l in lab.values())


# ------------------------------------------------------------------ estimator host logic (no device)
def _fit_host(est, X):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return est.fit(X)


@pytest.mark.parametrize("s,t,R,b", CASES, ids=IDS)
def test_host_hash_dictionary_and_random_state(s, t, R, b):
    fit, _ = SETS[s]
    tag = _tag(s, t, R, b)
    e = _fit_host(_est(t, R, b), fit)
    assert list(e._labels_hash_dict.items()) == list(_golden_dict(tag).items())
    assert e.random_state_.randint(1 << 30) == int(REF[tag + "_rs"][0])  # transform draws nothing
    _fit_host(e, fit)  # a second fit continues the same RandomState
    assert list(e._labels_hash_dict.values()) == REF[tag + "_hv2"].tolist()


@pytest.mark.parametrize("s,t,R,b", CASES, ids=IDS)
def test_pipeline_model_matches_reference(s, t, R, b):
    """labels0 of the estimator -> the numpy model of the device pipeline -> the reference's matrices."""
    fit, new = SETS[s]
    tag = _tag(s, t, R, b)
    e = _fit_host(_est(t, R, b), fit)
    K, _ = nh_pipeline_model(e.X.block, e.X.ids, R, b, t == "count_sensitive")
    _eq(K, REF[tag + "_K"])
    yb, _ = e._pack(new)
    y0 = e._labels0(yb, e._labels_hash_dict)
    if s == "small":
        assert np.any(y0 == -1)  # unseen labels are seeded as None
    assert np.all(e.X.ids >= 0)
    Kt, _ = nh_pipeline_model(Block.concat(e.X.block, yb), np.concatenate([e.X.ids, y0]), R, b, t == "count_sensitive",
                              n_fit=e.X.block.n_graphs)
    _eq(Kt, REF[tag + "_Kt"])


def test_labels0_follow_the_hash_dictionary():
    fit, _ = SETS["adj"]
    e = _fit_host(NeighborhoodHash(R=2, random_state=1), fit)
    lab = [fit[g][1][v] for g in range(len(fit)) for v in range(len(fit[g][1]))]  # adjacency: vertices = range(n)
    assert e.X.ids.tolist() == [e._labels_hash_dict[l] for l in lab]


def _tu_block(d):
    from grakel_b200.datasets import read_tu
    mg.write_mutag_tu(os.path.join(d, "MUTAG"))
    return read_tu(d, "MUTAG", kernel="NH").data


def test_tu_block_label_set_and_model():
    """A packed TU block: the label set comes from the packed labels in graph order; equal to read_data + the real
    NH."""
    with tempfile.TemporaryDirectory() as d:
        blk = _tu_block(d)
    for t in ("simple", "count_sensitive"):
        e = NeighborhoodHash(R=3, nh_type=t, random_state=6).fit(blk)
        K, _ = nh_pipeline_model(e.X.block, e.X.ids, 3, 8, t == "count_sensitive")
        _eq(K, REF[f"tu_{t}"])


def test_string_labels_against_the_oracle():
    """String labels: the set order depends on PYTHONHASHSEED, so the check is in-process against the oracle."""
    fit, new = SETS["small"]
    names = "abcdefghij"
    fs = [[g, {v: names[l] for v, l in L.items()}] for g, L in fit]
    ns = [[g, {v: names[l] for v, l in L.items()}] for g, L in new]
    for t in ("simple", "count_sensitive"):
        e = _fit_host(NeighborhoodHash(R=3, nh_type=t, bits=4, random_state=9), fs)
        o = NHOracle(R=3, nh_type=t, bits=4, random_state=9).fit(fs)
        assert list(e._labels_hash_dict.items()) == list(o.hash_dict.items())
        K, _ = nh_pipeline_model(e.X.block, e.X.ids, 3, 4, t == "count_sensitive")
        _eq(K, o.fit_transform(fs))
        yb, _ = e._pack(ns)
        Kt, _ = nh_pipeline_model(Block.concat(e.X.block, yb), np.concatenate([e.X.ids, e._labels0(yb, e._labels_hash_dict)]),
                                  3, 4, t == "count_sensitive", n_fit=e.X.block.n_graphs)
        _eq(Kt, o.transform(ns))


def test_error_behaviour():
    fit, _ = SETS["small"]
    for kw, msg in ((dict(R=0), "R must be"), (dict(R=2.0), "R must be"), (dict(nh_type="x"), "unrecognised"),
                    (dict(bits=0), "illegal number of bits"), (dict(bits=3.0), "illegal number of bits")):
        with pytest.raises(TypeError, match=msg):
            NeighborhoodHash(**kw).fit(fit)
    with pytest.raises(ValueError, match="Maximum allowed size exceeded"):  # numpy's choice(2**64, ...)
        NeighborhoodHash(bits=64).fit(fit)
    e = NeighborhoodHash()
    with pytest.raises(ValueError, match="`fit` input cannot be None"):
        e.fit(None)
    with pytest.raises(TypeError, match="input must be an iterable"):
        e.fit(5)
    with pytest.raises(TypeError, match="each element of X"):
        e.fit([5])
    with pytest.raises(TypeError, match="each element of X"):
        e.fit([[1, 2, 3, 4]])
    with pytest.warns(UserWarning, match="Ignoring empty element"), pytest.raises(ValueError, match="parsed input is empty"):
        e.fit([[]])
    with pytest.raises(ValueError, match="Graph does not have any labels"):
        e.fit([[{(0, 1): 1}, {}]])
    with pytest.warns(UserWarning, match="Labels must be provided"), pytest.raises(UnboundLocalError):
        e.fit([[fit[0][0]]] + fit)  # a one-member element first: the reference's unbound `vertices`
    with pytest.warns(UserWarning, match="Labels must be provided"), pytest.raises(AttributeError):
        e.fit(fit + [[fit[0][0]]])  # ... later: the previous graph's variables, then list.neighbors
    with pytest.raises(ZeroDivisionError):
        NeighborhoodHash().fit_transform(fit + [[{}, {0: 1}]])  # a graph without vertices: 0 / 0.0
    e = _fit_host(NeighborhoodHash(random_state=0), fit + [[{}, {0: 1}]])  # fit alone does not divide
    assert e.X.block.n_graphs == len(fit) + 1
    with pytest.raises(ValueError, match="`transform` input cannot be None"):
        e.transform(None)
    with pytest.warns(UserWarning, match="Ignoring empty element"):
        K = e.transform([[]])  # the reference returns an empty matrix here
    assert K.shape == (0, len(fit) + 1) and e.diagonal() == (1.0, 1.0)
    with pytest.raises(ZeroDivisionError):
        e.transform([[{}, {0: 1}]])
    with pytest.warns(UserWarning), pytest.raises(UnboundLocalError):
        e.transform([[fit[0][0]]])


def test_diagonal_and_normalize_are_the_references():
    e = NeighborhoodHash(normalize=True, verbose=True)
    assert e.verbose is False and e.get_params()["normalize"] is True
    assert e.diagonal() == 1.0


def test_dispatch_and_pickling():
    for name in ("NH", "neighborhood_hash"):
        gk = GraphKernel(kernel={"name": name, "R": 2, "nh_type": "count_sensitive", "bits": 5, "random_state": 3})
        gk.initialize()
        k = gk.kernel_
        assert isinstance(k, NeighborhoodHash)
        assert (k.R, k.nh_type, k.bits, k.random_state) == (2, "count_sensitive", 5, 3)
    with pytest.raises(NotImplementedError):
        GraphKernel(kernel="random_walk").initialize()
    fit, _ = SETS["small"]
    e = _fit_host(NeighborhoodHash(R=2, random_state=4), fit)
    f = pickle.loads(pickle.dumps(e))
    assert f._labels_hash_dict == e._labels_hash_dict and np.array_equal(f.X.ids, e.X.ids)
    assert f.random_state_.randint(1 << 30) == e.random_state_.randint(1 << 30)


# ------------------------------------------------------------------ the CUDA path
def _run_golden(s, t, R, b):
    fit, new = SETS[s]
    tag = _tag(s, t, R, b)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        e = _est(t, R, b)
        _eq(e.fit_transform(fit), REF[tag + "_K"])
        assert e.diagonal() == float(REF[tag + "_d"])
        _eq(e.transform(new), REF[tag + "_Kt"])
        assert e.diagonal() == tuple(REF[tag + "_dt"].tolist())
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("s,t,R,b", CASES, ids=IDS)
def test_gpu_nh_matches_reference(s, t, R, b):
    _run_golden(s, t, R, b)


@pytest.mark.gpu
def test_gpu_nh_mutag_tu_and_dispatch():
    X = mg.mutag()
    for t in ("simple", "count_sensitive"):
        _eq(NeighborhoodHash(R=3, nh_type=t, random_state=5).fit_transform(X), REF[f"mutag_{t}"])
        _eq(GraphKernel(kernel={"name": "NH", "R": 3, "nh_type": t, "random_state": 5}).fit_transform(X),
            REF[f"mutag_{t}"])
        with tempfile.TemporaryDirectory() as d:
            blk = _tu_block(d)
        _eq(NeighborhoodHash(R=3, nh_type=t, random_state=6).fit_transform(blk), REF[f"tu_{t}"])


@pytest.mark.gpu
def test_gpu_nh_nystroem_shapes():
    fit, new = SETS["small"]
    gk = GraphKernel(kernel={"name": "NH", "R": 2, "random_state": 0}, Nystroem=10, random_state=0)
    Z = gk.fit_transform(fit)
    assert Z.shape == (len(fit), 10) and np.all(np.isfinite(Z))
    assert gk.transform(new).shape == (len(new), 10)


@pytest.mark.gpu
@pytest.mark.parametrize("cs", [False, True])
def test_gpu_nh_labels_equal_the_oracle(cs):
    """gk_nh_labels per level, per vertex (adjacency input: packed vertex v of a graph is its vertex v), None included."""
    from grakel_b200 import _lib
    fit, new = SETS["hubs"] if cs else SETS["adj"]
    b = 2 if cs else 8
    t = "count_sensitive" if cs else "simple"
    e = NeighborhoodHash(R=3, nh_type=t, bits=b, random_state=1).fit(fit)
    yb, _ = e._pack(new)
    blk = Block.concat(e.X.block, yb)
    lab0 = np.concatenate([e.X.ids, e._labels0(yb, e._labels_hash_dict)])
    o = NHOracle(R=3, nh_type=t, bits=b, hash_dict=e._labels_hash_dict)
    want = [lv for g, L in o._graphs(list(fit) + list(new)) for lv in [o._levels(g, L)]]
    _, model = nh_pipeline_model(blk, lab0, 3, b, cs)
    with _lib.engine() as eng:
        eng.pack(blk.graph_ptr, blk.row_ptr, blk.col_idx)
        eng.nh_features(3, b, cs, lab0)
        for r in range(3):
            got = eng.nh_labels(r, blk.n_vertices)
            exp = np.array([nh_ref.NONE64 if lv[r][v] is None else np.uint64(lv[r][v])
                            for lv in want for v in sorted(lv[r])], dtype=np.uint64)
            assert np.array_equal(got, exp)
            assert np.array_equal(got, model[r])


@pytest.mark.gpu
@pytest.mark.parametrize("path", [None, "1", "4096", "simt"])
def test_gpu_nh_against_the_oracle_on_every_gram_path(path, monkeypatch):
    """300 graphs, R = 3, fit + transform with unseen labels: the default head/tail split, every column on the tensor
    cores (T = 1), every column through the pair-update tail (T = 4096), and the CUDA-core Gram."""
    from grakel_b200 import _lib
    from oracle.gk_oracle import gen
    if path in ("1", "4096"):
        monkeypatch.setenv("GRAKEL_B200_FORCE_T", path)
    X = gen(300, 16, 21, nl=3)
    fit, new = X[:220], X[220:]
    for _g, l in new[::3]:
        l[0] = 99
    for t in ("simple", "count_sensitive"):
        e = NeighborhoodHash(R=3, nh_type=t, random_state=2)
        K = e.fit_transform(fit)
        o = NHOracle(R=3, nh_type=t, hash_dict=e._labels_hash_dict)
        _eq(K, o.fit_transform(fit))
        Kt = e.transform(new)
        _eq(Kt, o.transform(new))
        if path == "simt":
            yb, _ = e._pack(new)
            blk = Block.concat(e.X.block, yb)
            with _lib.engine() as eng:
                eng.pack(blk.graph_ptr, blk.row_ptr, blk.col_idx)
                eng.nh_features(3, 8, t == "count_sensitive",
                                np.concatenate([e.X.ids, e._labels0(yb, e._labels_hash_dict)]))
                st = _lib.GkStats()
                _eq(eng.nh_gram(blk.n_graphs, n_fit=len(fit), simt=True, stats=st), Kt)
                assert st.gram_path == 2


@pytest.mark.gpu
@pytest.mark.parametrize("t", ["simple", "count_sensitive"])
def test_gpu_nh_full_size_properties(t):
    """BASELINE config 2's graphs (10 000, R = 3): K is exactly symmetric with a unit diagonal, 0 <= K <= 1, and a
    48-graph sub-matrix equals the oracle on that subset with the estimator's hash dictionary (the dictionary depends
    on the whole label set)."""
    from oracle.gk_oracle import gen
    X = gen(10000, 40, 0)
    e = NeighborhoodHash(R=3, nh_type=t, random_state=0)
    K = e.fit_transform(X)
    assert K.shape == (10000, 10000) and K.dtype == np.float64
    assert np.array_equal(K, K.T)
    assert np.all(np.diagonal(K) == 1.0)
    assert np.all((K >= 0) & (K <= 1))
    pick = np.random.RandomState(3).choice(len(X), 48, replace=False)
    sub = [X[i] for i in pick]
    _eq(K[np.ix_(pick, pick)], NHOracle(R=3, nh_type=t, hash_dict=e._labels_hash_dict).fit_transform(sub))
    assert e.stats_.n_levels == 3 and e.stats_.n_entries == 3 * e.X.block.n_vertices
