"""ShortestPathAttr (metric=np.dot) on the device against a dense fp64 reference (tests/spattr_ref.py: K = Phi Phi^T,
pinned to the real reference in test_oracle_golden.py), where the tensor-core Gram can go wrong: signed attributes,
attributes far from unit size, feature maps wider than one shared-memory chunk, the largest attribute dimension, tile
and k-block edges of N and D, graphs without edges, and the inputs the feature kernel must refuse.

Every case asserts, for fit_transform and for transform:
  entries      |K_dev - K_ref| <= tol * K_abs,  K_abs = |Phi| |Phi|^T  (tol 1e-5 on the tensor cores; 1e-12 on the
               fp64 CUDA-core Gram, GRAKEL_B200_SPATTR_F64=1).  For non-negative attributes K_abs = K_ref.
  diagonal     the self similarities to 1e-12 relative,
  symmetry     K exactly symmetric,
  normalised   |Kn_dev - Kn_ref| <= tol * K_abs / sqrt(d_i d_j)  (NaN exactly where the reference has NaN)."""
import warnings

import numpy as np
import pytest

from oracle.gk_oracle import gen
from spattr_ref import spattr_phi, spattr_ref

pytestmark = pytest.mark.gpu

ROUTES = ["tf32x3", "fp64"]
TOL = {"tf32x3": 1e-5, "fp64": 1e-12}


@pytest.fixture(params=ROUTES)
def route(request, monkeypatch):
    if request.param == "fp64":
        monkeypatch.setenv("GRAKEL_B200_SPATTR_F64", "1")
    else:
        monkeypatch.delenv("GRAKEL_B200_SPATTR_F64", raising=False)
    monkeypatch.delenv("GRAKEL_B200_SPATTR_CHUNK", raising=False)
    return request.param


def _k():
    import grakel_b200
    return grakel_b200


# ------------------------------------------------------------------ inputs (seeded)
def _attrs(X, kind, seed):
    """Replace the attributes of gen(..., attr=da): 'rand' keeps U[0, 1), 'centred' is U[-0.5, 0.5), 'randn' N(0, 1)."""
    rs = np.random.RandomState(seed)
    out = []
    for A, L in X:
        if kind == "centred":
            L = {i: v - 0.5 for i, v in L.items()}
        elif kind == "randn":
            L = {i: rs.randn(len(v)) for i, v in L.items()}
        out.append([A, L])
    return out


def _graphs(N, nbar, seed, da, kind="centred"):
    return _attrs(gen(N, nbar, seed, attr=da, as_adj=True), kind, seed + 1)


def _scaled(X, s):
    return [[A, {i: np.ldexp(v, s) for i, v in L.items()}] for A, L in X]


def _real_graphs(N, nbar, seed, da, as_adj):
    """ER graphs (average degree 4) with random real edge weights, so that nearly every vertex pair of every graph has
    its own path length: a few hundred distinct lengths for a dozen graphs.  Adjacency matrices or edge dictionaries;
    N(0, 1) attributes."""
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(N):
        n = int(rs.randint(nbar // 2, nbar + nbar // 2 + 1))
        iu = np.triu_indices(n, 1)
        m = rs.rand(len(iu[0])) < 4.0 / (n - 1)
        a, b = iu[0][m], iu[1][m]
        if len(a) == 0:
            a, b = np.array([0]), np.array([1])
        w = 0.05 + rs.rand(len(a))
        L = {i: rs.randn(da) for i in range(n)}
        if as_adj:
            A = np.zeros((n, n))
            A[a, b] = w
            A[b, a] = w
            out.append([A, L])
        else:
            g = {}
            for x, y, wt in zip(a.tolist(), b.tolist(), w.tolist()):
                g[(x, y)] = wt
                g[(y, x)] = wt
            out.append([g, L])
    return out


def _paths(N, L, seed, da=1):
    """Path graphs of 2 .. L + 1 vertices, the first one of L + 1: exactly the path lengths 1 .. L, i.e. D = L * da^2."""
    rs = np.random.RandomState(seed)
    out = []
    for g in range(N):
        n = L + 1 if g == 0 else int(rs.randint(2, L + 2))
        A = np.zeros((n, n))
        i = np.arange(n - 1)
        A[i, i + 1] = A[i + 1, i] = 1.0
        out.append([A, {v: rs.randn(da) for v in range(n)}])
    return out


# ------------------------------------------------------------------ the contract
def _entries(Kd, ref, tol, what):
    K, K_abs = ref[0], ref[1]
    Kd = np.asarray(Kd)
    assert Kd.dtype == np.float64 and Kd.shape == K.shape, (what, Kd.shape, K.shape)
    nan = np.isnan(K)
    assert np.array_equal(np.isnan(Kd), nan), f"{what}: NaN pattern differs ({int(np.isnan(Kd).sum())} vs {int(nan.sum())})"
    err = np.abs(Kd[~nan] - K[~nan])
    bound = tol * K_abs[~nan]
    ok = err <= bound
    if not ok.all():
        i = int(np.argmax(np.where(ok, 0, 1)))
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.size} entries outside {tol:g} * K_abs; first: "
                             f"device {Kd[~nan][i]!r} reference {K[~nan][i]!r} K_abs {K_abs[~nan][i]!r}")


def _run(X, Y=None, normalize=False, algorithm_type="auto"):
    """Device K of fit_transform(X) (Y None) or of transform(Y) after fit(X), and the self similarities (rows, cols)."""
    est = _k().ShortestPathAttr(normalize=normalize, algorithm_type=algorithm_type)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # graphs without features: "normalizing it yields NaNs"
        K = est.fit_transform(X)
        if Y is None:
            d = est.diagonal()
            return K, d, d
        Kt = est.transform(Y)
        dx, dy = est.diagonal()
        return Kt, dy, dx


def _check(X, Y=None, route="tf32x3", algorithm_type="auto", norm=True):
    """The whole contract for fit_transform(X) (Y None) or transform(Y); returns (K_dev, K_ref, K_abs)."""
    tol = TOL[route]
    ref = spattr_ref(X, Y, algorithm_type)
    Kd, drow, dcol = _run(X, Y, algorithm_type=algorithm_type)
    what = "fit_transform" if Y is None else "transform"
    _entries(Kd, ref, tol, what)
    np.testing.assert_allclose(drow, ref[2], rtol=1e-12, atol=0)
    np.testing.assert_allclose(dcol, ref[3], rtol=1e-12, atol=0)
    if Y is None:
        assert np.array_equal(Kd, Kd.T), "K is not exactly symmetric"
        np.testing.assert_allclose(np.diagonal(Kd), ref[2], rtol=1e-12, atol=0)
    if norm:
        Kn = _run(X, Y, normalize=True, algorithm_type=algorithm_type)[0]
        _entries(Kn, spattr_ref(X, Y, algorithm_type, normalize=True), tol, what + " normalised")
    return Kd, ref[0], ref[1]


def _check_fit_and_transform(X, Y, route, algorithm_type="auto"):
    _check(X, None, route, algorithm_type)
    _check(X, Y, route, algorithm_type)


# ------------------------------------------------------------------ signed attributes
@pytest.mark.parametrize("kind", ["centred", "randn"])
@pytest.mark.parametrize("da", [1, 3, 16])
def test_signed_attributes(route, kind, da):
    """Zero-mean attributes: entries cancel, so the tensor-core error is bounded by K_abs, not by |K|.  ~300 graphs:
    several 128-row tiles, mirrored tiles and k-chunk folds."""
    X = _graphs(310, 20 if da == 16 else 30, 40 + da, da, kind)
    _check_fit_and_transform(X[:270], X[270:], route)


def test_signed_attributes_observed_error(monkeypatch):
    """The observed error, not just the bound: a fall back to plain tf32 (~1e-3) or bf16 would show."""
    monkeypatch.delenv("GRAKEL_B200_SPATTR_F64", raising=False)
    monkeypatch.delenv("GRAKEL_B200_SPATTR_CHUNK", raising=False)
    X = _graphs(300, 20, 56, 16, "centred")
    Kd, K, K_abs = _check(X, None, norm=False)
    seen = K_abs > 0
    err = float(np.max(np.abs(Kd - K)[seen] / K_abs[seen]))
    assert err < 3e-6, err


# ------------------------------------------------------------------ scale
SCALES = [-128, -64, -40, -24, -8, 8, 24, 40, 64, 128]


@pytest.fixture(scope="module")
def scale_base():
    """Unscaled device results, computed once per (attributes, route)."""
    return {}


@pytest.mark.parametrize("s", SCALES)
@pytest.mark.parametrize("kind", ["rand", "centred"])
def test_attribute_scale(route, kind, s, scale_base):
    """Attributes times 2^s scale Phi by 2^(2s) and K by 2^(4s): from |s| ~ 26 (on config-5-like graphs) upwards that is
    outside fp32's range, which the tensor-core route must not inherit.  The device result scales bit for bit (every
    row is split at its own power of two), and its normalised matrix does not change for |s| <= 64; above that d_i d_j
    overflows fp64 in the reference's own K / sqrt(d_i d_j), and the contract against the reference applies."""
    X0 = _graphs(48, 16, 77, 3, kind)
    fit, new = X0[:36], X0[36:]
    key = (kind, route)
    if key not in scale_base:
        scale_base[key] = {(Y is None, norm): _run(fit, Y, normalize=norm)[0] for Y in (None, new) for norm in (False, True)}
    base = scale_base[key]
    Xs = _scaled(X0, s)
    fs, ns = Xs[:36], Xs[36:]
    for Y, Yb in ((None, None), (ns, new)):
        Kd = _check(fs, Y, route)[0]
        assert np.array_equal(Kd, np.ldexp(base[(Y is None, False)], 4 * s)), "K(2^s a) != 2^(4s) K(a)"
        if abs(s) <= 64:
            Kn = _run(fs, Y, normalize=True)[0]
            assert np.array_equal(Kn, base[(Y is None, True)], equal_nan=True), "normalised K depends on the scale"


# ------------------------------------------------------------------ wide feature maps
@pytest.mark.parametrize("as_adj,algorithm_type", [(True, "floyd_warshall"), (False, "dijkstra")])
def test_many_path_lengths(route, as_adj, algorithm_type):
    """Real-valued weights and da = 8: several hundred distinct path lengths, more than one shared-memory chunk of
    spattr_accumulate (about 390 blocks of 8 x 8 fit), in both path-sum orders."""
    X = _real_graphs(16, 10, 5, 8, as_adj)
    n_max = max(len(L) for _, L in X)
    chunk = (200 * 1024 - (n_max * 8 * 8 + n_max * n_max * 2 + 64)) // (64 * 8)  # blocks per chunk (gk_spattr_features)
    assert spattr_phi(X[:12], None, algorithm_type).shape[1] // 64 > chunk
    _check_fit_and_transform(X[:12], X[12:], route, algorithm_type)


@pytest.mark.parametrize("weights", ["unit", "real"])
def test_attribute_dimension_32(route, weights):
    """da = 32, the largest attribute dimension: 1024 features per path length, 24 lengths per shared-memory chunk."""
    if weights == "unit":
        X = _graphs(40, 12, 8, 32, "randn")
        _check_fit_and_transform(X[:30], X[30:], route)
    else:
        X = _real_graphs(8, 8, 9, 32, as_adj=False)
        _check_fit_and_transform(X[:6], X[6:], route, "dijkstra")


@pytest.mark.parametrize("chunk", ["1", "3"])
def test_k_chunk_setting(monkeypatch, chunk):
    """GRAKEL_B200_SPATTR_CHUNK: k-blocks per fp32 accumulator before the fold into fp64."""
    monkeypatch.delenv("GRAKEL_B200_SPATTR_F64", raising=False)
    monkeypatch.setenv("GRAKEL_B200_SPATTR_CHUNK", chunk)
    X = _real_graphs(16, 10, 5, 8, True)
    _check_fit_and_transform(X[:12], X[12:], "tf32x3", "floyd_warshall")


# ------------------------------------------------------------------ shapes
@pytest.mark.parametrize("N", [1, 2, 127, 128, 129, 255, 256, 257])
def test_square_sizes(route, N):
    _check(_graphs(N, 8, 100 + N, 2), None, route)


@pytest.mark.parametrize("n_fit,n_y", [(1, 1), (255, 1), (257, 129)])
def test_transform_sizes(route, n_fit, n_y):
    X = _graphs(n_fit + n_y, 8, 200 + n_fit, 2)
    _check(X[:n_fit], X[n_fit:], route)


@pytest.mark.parametrize("da,L", [(1, 1), (3, 1), (1, 31), (1, 32), (1, 33)])
def test_feature_widths(route, da, L):
    """D = L * da^2 columns: one block, and widths just below, at and above one 32-column k-block (D = 33: Dp / 32 = 2
    k-blocks, not a multiple of the 8-block chunk)."""
    X = _paths(40, L, 300 + L + da, da)
    assert spattr_phi(X).shape[1] == L * da * da
    _check_fit_and_transform(X[:30], X[30:], route)


def test_graph_without_edges(route):
    """A graph without edges has no path lengths: a zero row of Phi, K row 0, normalised row NaN (0 / 0, as the
    reference gives it under np.errstate)."""
    X = _graphs(24, 8, 400, 3)
    rs = np.random.RandomState(401)
    empty = [np.zeros((3, 3)), {i: rs.randn(3) for i in range(3)}]
    X = X[:5] + [empty] + X[5:] + [empty]
    fit, new = X[:20], X[20:]
    _check(fit, None, route)
    _check(fit, new, route)
    K = _run(fit)[0]
    assert not K[5].any() and not K[:, 5].any()
    Kn = _run(fit, normalize=True)[0]
    assert np.isnan(Kn[5]).all() and np.isnan(Kn[:, 5]).all()
    assert np.isnan(_run(fit, new, normalize=True)[0][-1]).all()


# ------------------------------------------------------------------ limits
def test_attribute_dimension_above_32_raises():
    with pytest.raises(NotImplementedError, match="attribute dimension above 32"):
        _k().ShortestPathAttr().fit_transform(_graphs(4, 8, 500, 33))


def test_graph_above_shared_memory_budget_raises():
    """spattr_accumulate keeps a graph's block ids (2 bytes per vertex pair) and attributes in shared memory: a graph of
    330 vertices (218 KB) does not fit."""
    X = _graphs(3, 8, 501, 1) + _paths(1, 329, 502)
    assert X[-1][0].shape == (330, 330)
    with pytest.raises(NotImplementedError, match="graph too large"):
        _k().ShortestPathAttr().fit_transform(X)
