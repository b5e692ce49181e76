"""Estimator classes of the hot path, mirroring the reference's operator API.

Same class names, constructor signatures, method names and error behaviour as
grakel.kernels.{Kernel, WeisfeilerLehman, VertexHistogram, ShortestPath,
ShortestPathAttr} (kernel.py:23-456, weisfeiler_lehman.py:23-555,
vertex_histogram.py:23-219, shortest_path.py:16-515), but every kernel matrix is
produced by the CUDA engine behind `grakel_b200._lib` -- there is no CPU path.

Fitted state is host-resident numpy / Python objects (a packed CSR `Block` and
the level-0 label dictionary), so fitted estimators pickle like the reference's
(grakel/tests/test_common.py:53-58); device buffers are re-created on demand.
"""
from __future__ import annotations

import copy
import warnings
from collections.abc import Iterable

import numpy as np
from sklearn.base import BaseEstimator, TransformerMixin
from sklearn.exceptions import NotFittedError
from sklearn.utils import check_random_state
from sklearn.utils.validation import check_is_fitted

from . import _lib
from .packing import Block, Graph, label_ids, pack


class Fitted:
    """What `fit` keeps: the packed graphs, their level-0 label ids, the label dictionary."""

    def __init__(self, block, ids, dictionary):
        self.block = block
        self.ids = ids
        self.dictionary = dictionary

    def __len__(self):
        return self.block.n_graphs


class Kernel(BaseEstimator, TransformerMixin):
    """Estimator contract of grakel.kernels.Kernel (kernel.py:23-456).

    Subclasses provide `parse_input` (host packing) and `_device_features`
    (which feature kernel to run); fit / transform / fit_transform / diagonal /
    set_params behave as in the reference."""

    X = None
    _graph_format = "dictionary"
    _method_calling = 0
    _nan_to_num = False

    def __init__(self, n_jobs=None, normalize=False, verbose=False):
        self.verbose = verbose
        self.n_jobs = n_jobs
        self.normalize = normalize
        self._initialized = dict(n_jobs=False)

    # ---- reference protocol --------------------------------------------------
    def fit(self, X, y=None):
        self._is_transformed = False
        self._method_calling = 1
        self.initialize()
        if X is None:
            raise ValueError("`fit` input cannot be None")
        self.X = self.parse_input(X)
        return self

    def transform(self, X):
        self._method_calling = 3
        check_is_fitted(self, ["X"])
        if X is None:
            raise ValueError("`transform` input cannot be None")
        Y = self.parse_input(X)
        K, xdiag, ydiag = self._run(Block.concat(self.X.block, Y.block), np.concatenate([self.X.ids, Y.ids]),
                                    n_fit=self.X.block.n_graphs)
        self._X_diag = xdiag  # kernel.py:160-164 computes it on demand; the joint run returns it anyway
        self._Y_diag = ydiag
        self._is_transformed = True
        if self.normalize:
            self._warn_unnormalizable(self._X_diag, ydiag)
        return K

    def fit_transform(self, X, y=None):
        self._method_calling = 2
        self.fit(X)
        K, xdiag, _ = self._run(self.X.block, self.X.ids, n_fit=self.X.block.n_graphs)
        self._X_diag = xdiag
        if self.normalize:
            self._warn_unnormalizable(xdiag)
        return K

    def diagonal(self):
        check_is_fitted(self, ["X"])
        try:
            check_is_fitted(self, ["_X_diag"])
        except NotFittedError:
            _, self._X_diag, _ = self._run(self.X.block, self.X.ids, n_fit=self.X.block.n_graphs, want_matrix=False)
        if getattr(self, "_is_transformed", False):
            return self._X_diag, self._Y_diag
        return self._X_diag

    def _warn_unnormalizable(self, *diagonals):
        """kernel.py:206-234: say why a normalised matrix contains NaNs."""
        name = type(self).__name__
        for d in diagonals:
            d = np.asarray(d, dtype=float)
            if np.any(d == 0):
                warnings.warn(name + " has zero self similarities, so normalizing it yields NaNs: those graphs "
                              "have no features this kernel can see. Either drop them or pass normalize=False.",
                              RuntimeWarning)
                break

    def initialize(self):
        """kernel.py:386-399.  `n_jobs` is validated and then ignored: the whole Gram
        matrix is one device job (ShortestPath already ignores it, shortest_path.py:239-242)."""
        if not self._initialized["n_jobs"]:
            if type(self.n_jobs) is not int and self.n_jobs is not None:
                raise ValueError("n_jobs parameter must be an int indicating the number of jobs as in joblib or None")
            self._parallel = None
            self._initialized["n_jobs"] = True

    def parse_input(self, X):
        raise NotImplementedError

    def pairwise_operation(self, x, y):
        raise NotImplementedError("Pairwise operation is not implemented!")

    # ---- generic pairwise driver (kernel.py:236-296, 298-336) ---------------------
    # For kernels whose value needs a per-pair Python callback (ShortestPathAttr with a user metric): `self.X` is then
    # a plain list of per-graph items produced on the device and the matrix is filled pair by pair on the host, in the
    # reference's order and with its symmetrisation.  The Gram kernels never take this route.
    def _calculate_kernel_matrix(self, Y=None):
        if Y is None:
            n = len(self.X)
            K = np.zeros(shape=(n, n))
            cache = []
            for i, x in enumerate(self.X):
                K[i, i] = self.pairwise_operation(x, x)
                for j, y in enumerate(cache):
                    K[j, i] = self.pairwise_operation(y, x)
                cache.append(x)
            return np.triu(K) + np.triu(K, 1).T
        K = np.zeros(shape=(len(Y), len(self.X)))
        for j, y in enumerate(Y):
            for i, x in enumerate(self.X):
                K[j, i] = self.pairwise_operation(y, x)
        return K

    def _pairwise_fit_transform(self, X):
        self._method_calling = 2
        self.fit(X)
        km = self._calculate_kernel_matrix()
        self._X_diag = np.diagonal(km).copy()
        if self.normalize:  # kernel.py:196-203
            self._warn_unnormalizable(self._X_diag)
            with np.errstate(invalid="ignore", divide="ignore"):
                km = km / np.sqrt(np.outer(self._X_diag, self._X_diag))
        return km

    def _pairwise_transform(self, X):
        self._method_calling = 3
        check_is_fitted(self, ["X"])
        if X is None:
            raise ValueError("`transform` input cannot be None")
        Y = self.parse_input(X)
        km = self._calculate_kernel_matrix(Y)
        self._Y = Y
        self._is_transformed = True
        if self.normalize:  # kernel.py:155-164
            X_diag, Y_diag = self._pairwise_diagonal()
            self._warn_unnormalizable(X_diag, Y_diag)
            with np.errstate(invalid="ignore", divide="ignore"):
                km /= np.sqrt(np.outer(Y_diag, X_diag))
        return km

    def _pairwise_diagonal(self):
        check_is_fitted(self, ["X"])
        try:
            check_is_fitted(self, ["_X_diag"])
        except NotFittedError:
            self._X_diag = np.array([self.pairwise_operation(x, x) for x in self.X], dtype=float)
        if getattr(self, "_is_transformed", False) and hasattr(self, "_Y"):
            self._Y_diag = np.array([self.pairwise_operation(y, y) for y in self._Y], dtype=float)
            return self._X_diag, self._Y_diag
        return self._X_diag

    def set_params(self, **params):
        """kernel.py:417-433: a changed parameter is re-validated at the next fit."""
        if len(self._initialized):
            params = copy.deepcopy(params)
            for key in params:
                key, delim, sub_key = key.partition("__")
                if delim:
                    if sub_key in self._initialized:
                        self._initialized[sub_key] = False
                elif key in self._initialized:
                    self._initialized[key] = False
        super().set_params(**params)
        return self

    # ---- device side ---------------------------------------------------------
    def _device_features(self, engine):
        raise NotImplementedError

    def _run(self, block, ids, n_fit, want_matrix=True):
        """pack -> feature kernels -> Gram, all on the device.  Returns (K, xdiag, ydiag)."""
        with _lib.engine(getattr(self, "device_", None)) as eng:
            eng.pack(block.graph_ptr, block.row_ptr, block.col_idx, ids, block.weights, block.attrs)
            self.stats_ = self._device_features(eng)
            K, xd, yd = eng.gram(block.n_graphs, n_fit=n_fit, normalize=bool(self.normalize) and want_matrix,
                                 nan_to_num=self._nan_to_num, out=None if want_matrix else False,
                                 stats=self.stats_)
        if self.verbose:
            print(type(self).__name__, self.stats_.as_dict())
        return K, xd, yd


# ------------------------------------------------------------------------------
class VertexHistogram(Kernel):
    """Vertex histogram kernel (vertex_histogram.py:23-219): K = Phi Phi^T with
    Phi[g, l] = number of vertices of g carrying label l."""

    def __init__(self, n_jobs=None, normalize=False, verbose=False, sparse="auto"):
        super().__init__(n_jobs=n_jobs, normalize=normalize, verbose=verbose)
        self.sparse = sparse
        self._initialized.update({"sparse": True})

    def parse_input(self, X):
        from .packing import iter_elements
        if self._method_calling in (1, 2):
            known = None
        else:
            known = self.X.dictionary
        if isinstance(X, Block):  # packed input (datasets.read_tu): only the label multisets matter
            X.require("wl")
            block = Block(X.graph_ptr, np.zeros(X.n_vertices + 1, dtype=np.int64), np.zeros(0, dtype=np.int64), None,
                          X.labels)
            labels = X.labels
        else:
            sizes, labels = [0], []
            for _, _g, L in iter_elements(X, lambda n: n in (2, 3)):
                vals = list(L.values())
                labels.extend(vals)
                sizes.append(sizes[-1] + len(vals))
            if len(sizes) == 1:
                raise ValueError("parsed input is empty")
            block = Block(np.asarray(sizes), np.zeros(sizes[-1] + 1, dtype=np.int64), np.zeros(0, dtype=np.int64),
                          None, labels)
        if known is None:
            ids, new = label_ids(labels, None, sort_new=False)
            dictionary = new
            self.sparse_ = True
        else:
            ids, new = label_ids(labels, known, sort_new=False)
            dictionary = known
        return Fitted(block, ids, dictionary)

    def _device_features(self, eng):
        return eng.wl_features(0)


# ------------------------------------------------------------------------------
def _path_sum_order(block, algorithm_type):
    """Which of the reference's two shortest-path algorithms defines the path sums of a block with real-valued
    weights: "auto" runs Floyd-Warshall on adjacency input and Dijkstra on edge dictionaries (shortest_path.py:244-252,
    graph.py:652-656), and the two round differently (SURVEY 7).  Returns True for Dijkstra's order.  Integer-valued
    weights give the same distances either way."""
    if block.weights is None or not np.any(block.weights != np.rint(block.weights)):
        return False
    if algorithm_type == "floyd_warshall":
        return False
    if algorithm_type == "dijkstra":
        return True
    if block.all_adjacency:
        return False
    if getattr(block, "any_adjacency", False):
        raise NotImplementedError("real-valued edge weights with adjacency and dictionary inputs mixed in one call: the "
                                  "reference would use a different algorithm per graph; pass algorithm_type explicitly")
    return True


def _edge_label_values(X):
    """Edge-label values per element, with the element checks of EdgeHistogram.parse_input
    (edge_histogram.py:76-103): elements must have exactly three members (graph, node labels,
    edge labels) or be `Graph` objects; only the VALUES of the edge-label dictionary are used."""
    if not isinstance(X, Iterable):
        raise TypeError("input must be an iterable\n")
    out = []
    for idx, x in enumerate(iter(X)):
        if isinstance(x, Graph):
            if not x.edge_labels:
                raise ValueError("Graph does not have any labels for edges.")
            L = x.edge_labels
        else:
            is_iter = isinstance(x, Iterable)
            if is_iter:
                x = list(x)
            if not (is_iter and len(x) in (0, 3)):
                raise TypeError("each element of X must be either a graph object or a list with at least a graph like "
                                "object and node labels dict \n")
            if len(x) == 0:
                warnings.warn("Ignoring empty element on index: " + str(idx))
                continue
            L = x[2]
        out.append(list(L.values()))
    if not out:
        raise ValueError("parsed input is empty")
    return out


class EdgeHistogram(Kernel):
    """Edge histogram kernel (edge_histogram.py:23-212): K = Phi Phi^T with
    Phi[g, l] = number of edge-label entries of g equal to l.  On the device this is the
    vertex-histogram path over a block whose "vertices" are the edge-label entries."""

    _levels = 0

    def __init__(self, n_jobs=None, normalize=False, verbose=False, sparse="auto"):
        super().__init__(n_jobs=n_jobs, normalize=normalize, verbose=verbose)
        self.sparse = sparse
        self._initialized.update({"sparse": True})

    def initialize(self):
        if not self._initialized["n_jobs"]:  # edge_histogram.py:48-52
            if self.n_jobs is not None:
                warnings.warn("no implemented parallelization for EdgeHistogram")
            self._initialized["n_jobs"] = True

    def parse_input(self, X):
        values = _edge_label_values(X)
        sizes = np.concatenate([[0], np.cumsum([len(v) for v in values])])
        labels = [l for v in values for l in v]
        block = Block(sizes, np.zeros(int(sizes[-1]) + 1, dtype=np.int64), np.zeros(0, dtype=np.int64), None, labels)
        if self._method_calling in (1, 2):
            ids, dictionary = label_ids(labels, None, sort_new=False)
            self._labels = dictionary
            self.sparse_ = True
            return Fitted(block, ids, dictionary)
        ids, _ = label_ids(labels, self.X.dictionary, sort_new=False)
        return Fitted(block, ids, self.X.dictionary)

    def _device_features(self, eng):
        return eng.wl_features(self._levels)


# ------------------------------------------------------------------------------
class _LevelDictionaries(dict):
    """`_inv_labels` of a fitted WL estimator (weisfeiler_lehman.py:208-257): level 0 is built on the host by `fit`;
    the dictionaries of the levels >= 1 -- credential string -> compressed label, in the reference's own numbering --
    are exported from the device relabelling the first time one of them is asked for."""

    def __init__(self, level0, owner):
        super().__init__({0: level0})
        self._owner = owner

    def __missing__(self, level):
        owner = self._owner
        if owner is None or type(level) is not int or not 0 < level < owner._n_iter:
            raise KeyError(level)
        self.update(owner._export_level_dictionaries())
        return dict.__getitem__(self, level)

    def __reduce__(self):  # pickles as what has been materialised plus the owner
        return (_restore_level_dictionaries, (dict(self), self._owner))


def _restore_level_dictionaries(content, owner):
    d = _LevelDictionaries(content.get(0), owner)
    d.update(content)
    return d


def wl_reference_dictionaries(row_ptr, col_idx, level0_ids, n_level0, classes):
    """The reference's per-level label dictionaries from the device partition.

    `classes[i]` (i >= 1) holds one class id per vertex (any numbering; `gk_wl_labels`).  The reference names a
    class by the string  str(own label) + "," + str(sorted neighbour labels)  over the labels of level i-1, sorts the
    distinct strings and numbers them on from where the previous level stopped (weisfeiler_lehman.py:223-246).
    One string per CLASS is built here (from the class's first vertex), not one per vertex.
    Returns ({level: {credential: label}}, [reference label of every vertex, per level])."""
    prev = np.asarray(level0_ids, dtype=np.int64)
    count = int(n_level0)
    out, labels = {}, [prev]
    for i in range(1, len(classes)):
        uniq, first, inv = np.unique(np.asarray(classes[i]), return_index=True, return_inverse=True)
        creds = []
        for v in first.tolist():
            nb = prev[col_idx[row_ptr[v]:row_ptr[v + 1]]]
            creds.append(str(int(prev[v])) + "," + str(sorted(nb.tolist())))
        if len(set(creds)) != len(creds):
            raise RuntimeError("two classes of level %d share a signature: the device partition is not the "
                               "reference's" % i)
        order = sorted(range(len(creds)), key=creds.__getitem__)
        new_id = np.empty(len(uniq), dtype=np.int64)
        new_id[order] = count + np.arange(len(uniq), dtype=np.int64)
        out[i] = {creds[k]: count + r for r, k in enumerate(order)}
        prev = new_id[inv.reshape(-1)]
        labels.append(prev)
        count += len(uniq)
    return out, labels


# ------------------------------------------------------------------------------
class WeisfeilerLehman(Kernel):
    """Weisfeiler-Lehman subtree kernel (weisfeiler_lehman.py:23-555).

    K = sum over levels 0..n_iter of the vertex-histogram kernel on the level's
    compressed labels.  Only the subtree base kernel (`VertexHistogram`, the
    reference default) runs on the device."""

    _graph_format = "dictionary"
    _nan_to_num = True

    def __init__(self, n_jobs=None, verbose=False, normalize=False, n_iter=5, base_graph_kernel=VertexHistogram):
        super().__init__(n_jobs=n_jobs, verbose=verbose, normalize=normalize)
        self.n_iter = n_iter
        self.base_graph_kernel = base_graph_kernel
        self._initialized.update({"n_iter": False, "base_graph_kernel": False})
        self._base_graph_kernel = None

    def initialize(self):
        super().initialize()
        if not self._initialized["base_graph_kernel"]:  # weisfeiler_lehman.py:77-109
            base = self.base_graph_kernel
            if base is None:
                base, params = VertexHistogram, dict()
            elif type(base) is type and issubclass(base, Kernel):
                params = dict()
            else:
                try:
                    base, params = base
                except Exception:
                    raise TypeError("Base kernel was not formulated in the correct way. Check documentation.")
                if not (type(base) is type and issubclass(base, Kernel)):
                    raise TypeError("The first argument must be a valid grakel.kernel.kernel Object")
                if type(params) is not dict:
                    raise ValueError("If the second argument of base kernel exists, it must be a dictionary between "
                                     "parameters names and values")
                params.pop("normalize", None)
            if base not in (VertexHistogram, EdgeHistogram, ShortestPath):
                raise NotImplementedError("grakel_b200 runs WeisfeilerLehman over VertexHistogram (the subtree kernel), "
                                          "EdgeHistogram or ShortestPath; other base kernels are outside the device "
                                          "hot path")
            if base is ShortestPath:
                if not params.get("with_labels", True):
                    raise NotImplementedError("WeisfeilerLehman over ShortestPath(with_labels=False) ignores the WL "
                                              "labels; use (n_iter + 1) * ShortestPath(with_labels=False)")
                if params.get("algorithm_type", "auto") not in ("auto", "floyd_warshall", "dijkstra"):
                    raise ValueError('Unsupported "algorithm_type"')
            params["normalize"] = False
            params["verbose"] = self.verbose
            params["n_jobs"] = None
            self._base_graph_kernel = base
            self._params = params
            self._initialized["base_graph_kernel"] = True
        if not self._initialized["n_iter"]:  # :111-115
            if type(self.n_iter) is not int or self.n_iter <= 0:
                raise TypeError("'n_iter' must be a positive integer")
            self._n_iter = self.n_iter + 1
            self._initialized["n_iter"] = True

    def _pack_for_base(self, X, len_ok):
        """One block per base kernel: the subtree kernel needs the adjacency structure only, the
        shortest-path base also the edge weights; the edge-histogram base never looks at the graph --
        its block has one "vertex" per edge-label entry and no edges, so that every WL round reproduces
        the same partition and K = (n_iter + 1) * K_EH, exactly what the reference computes by fitting
        one EdgeHistogram per level on unchanged edge labels (weisfeiler_lehman.py:157-169, 260-270)."""
        base = self._base_graph_kernel
        if isinstance(X, Block):  # packed input (datasets.read_tu)
            if base is EdgeHistogram:
                raise NotImplementedError("packed blocks carry no edge-label entries; pass the list of graphs")
            return X.require("wl")
        if base is EdgeHistogram:
            if not isinstance(X, Iterable):
                raise TypeError("input must be an iterable\n")
            X = list(X)
            pack(X, "wl", len_ok=len_ok)  # the reference builds the Graph + node labels first: same errors
            values = _edge_label_values(X)
            sizes = np.concatenate([[0], np.cumsum([len(v) for v in values])])
            return Block(sizes, np.zeros(int(sizes[-1]) + 1, dtype=np.int64), np.zeros(0, dtype=np.int64), None,
                         [l for v in values for l in v])
        if base is ShortestPath:
            # the base kernel receives the edge DICTIONARY of every graph (weisfeiler_lehman.py:188, 218):
            # Dijkstra semantics whatever the input spelling; labels are the WL vertex set
            return pack(X, "wl", len_ok=len_ok, want_weights=True)
        return pack(X, "wl", len_ok=len_ok)

    def parse_input(self, X):
        if self._method_calling in (1, 2):
            if hasattr(self, "_X_diag"):
                delattr(self, "_X_diag")
            if not isinstance(X, (Iterable, Block)):
                raise TypeError("input must be an iterable\n")
            block = self._pack_for_base(X, lambda n: n >= 2)  # weisfeiler_lehman.py:152
            self._nx = block.n_graphs
            ids, dictionary = label_ids(block.labels, None, sort_new=True)  # :199-206
            self._inv_labels = _LevelDictionaries(dictionary, self)
            return Fitted(block, ids, dictionary)
        if self._method_calling != 3:
            raise ValueError("method call must be called either from fit or fit-transform")
        block = self._pack_for_base(X, lambda n: n in (2, 3))  # :367
        ids, _ = label_ids(block.labels, self._inv_labels[0], sort_new=True)  # :417-418
        return Fitted(block, ids, self._inv_labels[0])

    def fit_transform(self, X, y=None):
        self._method_calling = 2
        self._is_transformed = False
        self.initialize()
        if X is None:
            raise ValueError("transform input cannot be None")
        self.X = self.parse_input(X)
        K, xdiag, _ = self._run(self.X.block, self.X.ids, n_fit=self._nx)
        self._X_diag = xdiag
        return K

    def fit(self, X, y=None):
        self._is_transformed = False
        self._method_calling = 1
        self.initialize()
        if X is None:
            raise ValueError("`fit` input cannot be None")
        self.X = self.parse_input(X)
        return self

    def transform(self, X):
        self._method_calling = 3
        check_is_fitted(self, ["X", "_nx", "_inv_labels"])
        if X is None:
            raise ValueError("transform input cannot be None")
        if not isinstance(X, (Iterable, Block)):
            raise ValueError("input must be an iterable\n")
        Y = self.parse_input(X)
        K, xdiag, ydiag = self._run(Block.concat(self.X.block, Y.block), np.concatenate([self.X.ids, Y.ids]),
                                    n_fit=self._nx)
        self._X_diag = xdiag
        self._Y_diag = ydiag
        self._is_transformed = True
        return K

    def _device_features(self, eng):
        if self._base_graph_kernel is ShortestPath:
            return eng.wl_sp_features(self._n_iter - 1, dijkstra_order=True)  # the base kernel gets edge dictionaries
        return eng.wl_features(self._n_iter - 1)

    def _run(self, block, ids, n_fit, want_matrix=True):
        """The plain subtree fit_transform (square, un-normalised) is ONE C call, gk_wl_gram: relabel, column statistics,
        head/tail decision on the device, GEMM, tail and delivery with a single host synchronisation."""
        if (want_matrix and not self.normalize and n_fit == block.n_graphs and self._base_graph_kernel is VertexHistogram
                and type(self) is WeisfeilerLehman):
            with _lib.engine(getattr(self, "device_", None)) as eng:
                eng.pack(block.graph_ptr, block.row_ptr, block.col_idx, ids, block.weights, block.attrs)
                K, xd, self.stats_ = eng.wl_gram(self._n_iter - 1, want_diag=True)
            if self.verbose:
                print(type(self).__name__, self.stats_.as_dict())
            return K, xd, None
        return super()._run(block, ids, n_fit, want_matrix)

    def _export_level_dictionaries(self):
        """`_inv_labels[i]` for i >= 1 (weisfeiler_lehman.py:257): the fitted graphs are relabelled on the device, the
        per-level classes come back through `gk_wl_labels`, and the host names every class the way the reference
        does.  Also keeps `wl_labels_`: the reference's compressed label of every packed vertex, per level."""
        check_is_fitted(self, ["X", "_nx"])
        block, ids = self.X.block, self.X.ids
        with _lib.engine(getattr(self, "device_", None)) as eng:
            eng.pack(block.graph_ptr, block.row_ptr, block.col_idx, ids, None, None)
            eng.wl_features(self._n_iter - 1)
            classes = [ids] + [eng.wl_labels(lv, block.n_vertices) for lv in range(1, self._n_iter)]
        out, self.wl_labels_ = wl_reference_dictionaries(np.asarray(block.row_ptr), np.asarray(block.col_idx), ids,
                                                         len(self.X.dictionary), classes)
        return out


# ------------------------------------------------------------------------------
class WeisfeilerLehmanOptimalAssignment(Kernel):
    """Weisfeiler-Lehman optimal-assignment kernel (weisfeiler_lehman_optimal_assignment.py:19-481):
    K[i, j] = sum over the WL label hierarchy of min(#vertices of i, #vertices of j) carrying the label.

    The reference fills K with an O(N^2) Python loop of histogram intersections (:257-266); here the WL
    feature block is expanded to unary form on the device (`gk_wl_oa_features`) and the same Gram as the
    subtree kernel returns the intersections exactly.  `sparse` only selects the reference's storage
    of Hs and does not change K; it is accepted and ignored."""

    _graph_format = "dictionary"
    _nan_to_num = True

    def __init__(self, n_jobs=None, verbose=False, normalize=False, n_iter=5, sparse=False):
        super().__init__(n_jobs=n_jobs, verbose=verbose, normalize=normalize)
        self.n_iter = n_iter
        self.sparse = sparse
        self._initialized.update({"n_iter": False, "sparse": True})

    def initialize(self):
        super().initialize()
        if not self._initialized["n_iter"]:  # :68-72
            if type(self.n_iter) is not int or self.n_iter <= 0:
                raise TypeError("'n_iter' must be a positive integer")
            self._n_iter = self.n_iter + 1
            self._initialized["n_iter"] = True
        if not self._initialized["sparse"]:
            self._initialized["sparse"] = False

    def parse_input(self, X):
        msg = ("each element of X must be either a graph object or a list with at least a graph like object and "
               "node labels dict \n")
        if self._method_calling in (1, 2):
            if hasattr(self, "_X_diag"):
                delattr(self, "_X_diag")
            if isinstance(X, Block):  # packed input (datasets.read_tu)
                block = X.require("sp", "wloa")
            elif not isinstance(X, Iterable):
                raise TypeError("input must be an iterable\n")
            else:
                block = pack(X, "wloa", len_ok=lambda n: n >= 2, type_error_msg=msg)  # :113
            self._nx = block.n_graphs
            ids, dictionary = label_ids(block.labels, None, sort_new=True)  # :157-161
            self._inv_labels = {0: dictionary}
            self._hierarchy = {"root": {"parent": None, "w": 0, "omega": 0}}  # fitted marker; the tree lives on the device
            return Fitted(block, ids, dictionary)
        if self._method_calling != 3:
            raise ValueError("method call must be called either from fit or fit-transform")
        if isinstance(X, Block):
            block = X.require("sp", "wloa")
        else:
            try:
                block = pack(X, "wloa", len_ok=lambda n: n in (2, 3), type_error_msg=msg)  # :323
            except TypeError as e:  # transform raises ValueError for malformed elements (:344-346)
                raise ValueError("each element of X must have at least one and at most 3 elements\n") from e
        ids, _ = label_ids(block.labels, self._inv_labels[0], sort_new=True)  # :356-359
        return Fitted(block, ids, self._inv_labels[0])

    def fit_transform(self, X, y=None):
        self._method_calling = 2
        self._is_transformed = False
        self.initialize()
        if X is None:
            raise ValueError("transform input cannot be None")
        self.X = self.parse_input(X)
        K, xdiag, _ = self._run(self.X.block, self.X.ids, n_fit=self._nx)
        self._X_diag = xdiag
        return K

    def transform(self, X):
        self._method_calling = 3
        check_is_fitted(self, ["X", "_nx", "_hierarchy", "_inv_labels"])
        if X is None:
            raise ValueError("transform input cannot be None")
        if not isinstance(X, (Iterable, Block)):
            raise ValueError("input must be an iterable\n")
        Y = self.parse_input(X)
        K, xdiag, ydiag = self._run(Block.concat(self.X.block, Y.block), np.concatenate([self.X.ids, Y.ids]),
                                    n_fit=self._nx)
        self._X_diag = xdiag
        self._Y_diag = ydiag
        self._is_transformed = True
        return K

    def _device_features(self, eng):
        return eng.wl_oa_features(self._n_iter - 1)


# ------------------------------------------------------------------------------
class ShortestPath(Kernel):
    """Shortest-path kernel (shortest_path.py:167-515): features are
    (l(u), l(v), d(u,v)) triples (or d(u,v) alone with with_labels=False) over ordered
    vertex pairs at finite distance; K = Phi Phi^T."""

    def __init__(self, n_jobs=None, normalize=False, verbose=False, with_labels=True, algorithm_type="auto"):
        super().__init__(n_jobs=n_jobs, normalize=normalize, verbose=verbose)
        self.with_labels = with_labels
        self.algorithm_type = algorithm_type
        self._initialized.update({"with_labels": False, "algorithm_type": False})

    def initialize(self):
        if not self._initialized["n_jobs"]:  # shortest_path.py:239-242
            if self.n_jobs is not None:
                warnings.warn("no implemented parallelization for ShortestPath")
            self._initialized["n_jobs"] = True
        if not self._initialized["algorithm_type"]:  # :244-252
            if self.algorithm_type == "auto":
                self._graph_format = "auto"
            elif self.algorithm_type == "floyd_warshall":
                self._graph_format = "adjacency"
            elif self.algorithm_type == "dijkstra":
                self._graph_format = "dictionary"
            else:
                raise ValueError('Unsupported "algorithm_type"')
        self._lt = "vertex" if self.with_labels else "none"

    def parse_input(self, X):
        wl = bool(self.with_labels)
        # Floyd-Warshall treats a 0 entry as "no edge" (graph.py:1786); Dijkstra walks every
        # listed edge.  "auto" picks FW for adjacency input and Dijkstra for dictionaries, so
        # zero-weight dictionary edges only disappear when FW is forced.
        if isinstance(X, Block):  # packed input (datasets.read_tu): unit weights, dictionary semantics
            block = X.require("sp", labels=wl)
        else:
            block = pack(X, "sp", need_labels=wl, len_ok=lambda n: n in (2, 3) or (n == 1 and not wl),
                         want_weights=True, fw_zero_is_absent=self.algorithm_type == "floyd_warshall",
                         type_error_msg="each element of X must have at least one and at most 3 elements\n")
        # real-valued weights: feature keys compare path lengths by exact float equality (shortest_path.py:472, 511)
        # and the reference's Dijkstra and Floyd-Warshall round differently; the device reproduces whichever the
        # reference would run (k-ordered fp64 Floyd-Warshall, or the Dijkstra-order fixed point of sp_dijkstra_order_apsp)
        dj = _path_sum_order(block, self.algorithm_type)
        if self._method_calling in (1, 2):
            self._dijkstra_order = dj
        elif dj != getattr(self, "_dijkstra_order", dj) and block.weights is not None:
            self._dijkstra_order = self._dijkstra_order or dj
        if self._method_calling in (1, 2):
            self._nx = block.n_graphs
            if wl:
                ids, dictionary = label_ids(block.labels, None, sort_new=False)
            else:
                ids, dictionary = None, {}
            self._enum = dictionary  # fitted marker (the reference keeps the feature enumeration here)
            return Fitted(block, ids, dictionary)
        self._ny = block.n_graphs
        if wl:
            ids, _ = label_ids(block.labels, self.X.dictionary, sort_new=False)
        else:
            ids = None
        return Fitted(block, ids, self.X.dictionary)

    def fit_transform(self, X, y=None):
        self._method_calling = 2
        self.fit(X)  # resets _method_calling to 1 like shortest_path.py:392-393
        K, xdiag, _ = self._run(self.X.block, self.X.ids, n_fit=self._nx)
        self._X_diag = xdiag
        return K

    def transform(self, X):
        self._method_calling = 3
        check_is_fitted(self, ["X", "_nx", "_enum"])
        if X is None:
            raise ValueError("transform input cannot be None")
        Y = self.parse_input(X)
        ids = None if self.X.ids is None else np.concatenate([self.X.ids, Y.ids])
        K, xdiag, ydiag = self._run(Block.concat(self.X.block, Y.block), ids, n_fit=self._nx)
        self._X_diag = xdiag
        self._Y_diag = ydiag
        self._is_transformed = True
        return K

    def diagonal(self):
        out = super().diagonal()
        if isinstance(out, tuple):  # shortest_path.py:359-366: X diagonal as a column
            return np.reshape(out[0], (-1, 1)), out[1]
        return np.reshape(out, (-1, 1))

    def _device_features(self, eng):
        return eng.sp_features(with_labels=bool(self.with_labels), dijkstra_order=bool(getattr(self, "_dijkstra_order", False)))


class ShortestPathAttr(Kernel):
    """Shortest-path kernel on node attributes (shortest_path.py:16-164)."""

    def __init__(self, n_jobs=None, normalize=False, verbose=False, algorithm_type="auto", metric=np.dot):
        super().__init__(n_jobs=n_jobs, normalize=normalize, verbose=verbose)
        self.algorithm_type = algorithm_type
        self.metric = metric
        self._initialized.update({"algorithm_type": False, "metric": False})

    def initialize(self):
        super().initialize()
        if not self._initialized["algorithm_type"]:
            if self.algorithm_type not in ("auto", "floyd_warshall", "dijkstra"):
                raise ValueError("Unsupported value " + str(self.algorithm_type) + ' for "algorithm_type"')
            self._initialized["algorithm_type"] = True
        if not self._initialized["metric"]:
            if not callable(self.metric):
                raise TypeError('"metric" must be callable')
            self._initialized["metric"] = True

    def _bilinear(self):
        """The explicit feature map (and with it the tensor-core Gram) is valid for the default metric only."""
        return self.metric is np.dot

    def parse_input(self, X):
        if not self._bilinear():
            return self._parse_pairs(X)
        if isinstance(X, Block):  # packed input (datasets.read_tu(prefer_attr_nodes=True))
            if X.require("sp", labels=False).attrs is None:
                raise ValueError("Graph does not have any labels for vertices.")
            return Fitted(X, None, {})
        block = pack(X, "sp", need_labels=True, len_ok=lambda n: n in (2, 3), want_weights=True,
                     fw_zero_is_absent=self.algorithm_type == "floyd_warshall", attributes=True,
                     type_error_msg="each element of X must be either a graph or an iterable with at least 2 and at "
                                    "most 3 elements\n")
        self._dijkstra_order = _path_sum_order(block, self.algorithm_type) or getattr(self, "_dijkstra_order", False)
        return Fitted(block, None, {})

    # ---- a user metric: shortest-path matrices on the device, the reference's per-pair contraction on the host
    def _parse_pairs(self, X):
        """shortest_path.py:77-129 for a callable metric: one (S, phi) tuple per graph.  S comes from the device APSP
        kernels (gk_spattr_features -> gk_sp_distances; the path-sum order the reference would use), phi are the
        attribute rows.  The metric is a Python callback per attribute pair by definition, so the contraction of
        shortest_path.py:130-164 runs on the host (`pairwise_operation`), through the generic driver of the base
        class (kernel.py:236-296)."""
        if isinstance(X, Block):
            block = X.require("sp", labels=False)
            if block.attrs is None:
                raise ValueError("Graph does not have any labels for vertices.")
        else:
            block = pack(X, "sp", need_labels=True, len_ok=lambda n: n in (2, 3), want_weights=True,
                         fw_zero_is_absent=self.algorithm_type == "floyd_warshall", attributes=True,
                         type_error_msg="each element of X must be either a graph or an iterable with at least 2 and at "
                                        "most 3 elements\n")
        dj = _path_sum_order(block, self.algorithm_type)
        items = []
        with _lib.engine(getattr(self, "device_", None)) as eng:
            eng.pack(block.graph_ptr, block.row_ptr, block.col_idx, None, block.weights, block.attrs)
            self.stats_ = eng.spattr_features(dijkstra_order=bool(dj))
            gp = block.graph_ptr
            for g in range(block.n_graphs):
                n = int(gp[g + 1] - gp[g])
                S = eng.sp_distances(g, n) if n else np.zeros((0, 0))
                items.append((S, np.array(block.attrs[gp[g]:gp[g + 1]], dtype=float)))
        return items

    def pairwise_operation(self, x, y):
        """shortest_path.py:130-164, vectorised over the path lengths: sum over ordered vertex pairs (i, j) of x and
        (k, m) of y with equal finite shortest-path length of metric(phi_x[i], phi_y[k]) * metric(phi_x[j], phi_y[m])."""
        Sx, phi_x = x
        Sy, phi_y = y
        nx, ny = Sx.shape[0], Sy.shape[0]
        if nx < 2 or ny < 2:
            return 0
        M = np.empty((nx, ny), dtype=float)
        for i in range(nx):
            for k in range(ny):
                M[i, k] = self.metric(phi_x[i], phi_y[k])
        offx, offy = ~np.eye(nx, dtype=bool), ~np.eye(ny, dtype=bool)
        fx, fy = offx & np.isfinite(Sx), offy & np.isfinite(Sy)
        kernel = 0.0
        for d in np.intersect1d(np.unique(Sx[fx]), np.unique(Sy[fy])):
            Ax = (fx & (Sx == d)).astype(float)
            Ay = fy & (Sy == d)
            kernel += float(np.sum((M.T @ Ax @ M)[Ay]))
        return kernel

    def diagonal(self):
        if not self._bilinear():
            return self._pairwise_diagonal()
        return super().diagonal()

    def fit_transform(self, X, y=None):
        self.initialize()
        if not self._bilinear():
            return self._pairwise_fit_transform(X)
        self._method_calling = 2
        self.fit(X)
        K, xdiag, _ = self._run(self.X.block, None, n_fit=self.X.block.n_graphs)
        self._X_diag = xdiag
        if self.normalize:
            self._warn_unnormalizable(xdiag)
        return K

    def transform(self, X):
        if not self._bilinear():
            return self._pairwise_transform(X)
        self._method_calling = 3
        check_is_fitted(self, ["X"])
        if X is None:
            raise ValueError("`transform` input cannot be None")
        Y = self.parse_input(X)
        K, xdiag, ydiag = self._run(Block.concat(self.X.block, Y.block), None, n_fit=self.X.block.n_graphs)
        self._X_diag = xdiag
        self._Y_diag = ydiag
        self._is_transformed = True
        if self.normalize:
            self._warn_unnormalizable(xdiag, ydiag)
        return K

    def _device_features(self, eng):
        return eng.spattr_features(dijkstra_order=bool(getattr(self, "_dijkstra_order", False)))


# ------------------------------------------------------------------------------
_NH_ELEMENT_MSG = ("each element of X must be either a graph object or a list with at least a graph like object and "
                   "node labels dict \n")


def _nh_elements(X):
    """The reference's element loop (neighborhood_hash.py:127-159, 272-313) without the graph work: yields the node-label
    dict of every element that becomes a graph, warns on empty elements, raises as the reference does.

    A one-member element warns and then reaches the graph tuple with the previous element's variables: the reference
    fails there with UnboundLocalError for the first graph and AttributeError (a list has no `neighbors`) afterwards."""
    i = 0
    for idx, x in enumerate(X):
        if isinstance(x, Graph):
            x = x.as_element()
        is_iter = isinstance(x, Iterable)
        if is_iter:
            x = list(x)
        if not (is_iter and len(x) in (0, 1, 2, 3)):
            raise TypeError(_NH_ELEMENT_MSG)
        if len(x) == 0:
            warnings.warn("Ignoring empty element on index: " + str(idx))
            continue
        if len(x) == 1:
            warnings.warn("Ignoring empty element on index: " + str(i) + "\nLabels must be provided.")
            if i == 0:
                raise UnboundLocalError("cannot access local variable 'vertices' where it is not associated with a value")
            raise AttributeError("'list' object has no attribute 'neighbors'")
        i += 1
        yield x[1]


class NeighborhoodHash(Kernel):
    """Neighborhood hashing kernel (neighborhood_hash.py:14-570, Hido & Kashima): every vertex label is hashed R times
    from its own label and its out-neighbours' labels (a bit rotation and XORs, :367-504), and
    K[i, j] = mean over the R levels of c_r / (n_i + n_j - c_r), c_r the multiset intersection of the two graphs' level-r
    labels, n the vertex counts (:531-570).

    The host builds the reference's label set and hash dictionary (:157, 164-189) with the same sequence of set
    operations and RandomState draws, so `_labels_hash_dict` and `random_state_` end up as the reference leaves them;
    the relabel levels, the per-level intersections (a unary-expanded histogram through the integer Gram) and the fp64
    combine run on the device (`gk_nh_features` / `gk_nh_gram`).  `normalize` and `n_jobs` are accepted and have no
    effect, as in the reference: the matrix is already normalised and `diagonal()` returns 1.0 (:343-365)."""

    _graph_format = "dictionary"

    def __init__(self, n_jobs=None, normalize=False, verbose=False, random_state=None, R=3, nh_type="simple", bits=8):
        super().__init__(n_jobs=n_jobs, normalize=normalize, verbose=False)  # :50-52: verbose is dropped
        self.random_state = random_state
        self.R = R
        self.nh_type = nh_type
        self.bits = bits
        self._initialized.update({"random_state": False, "R": False, "nh_type": False, "bits": False})

    def initialize(self):
        """:61-89"""
        super().initialize()
        if not self._initialized["random_state"]:
            self.random_state_ = check_random_state(self.random_state)
            self._initialized["random_state"] = True
        if not self._initialized["R"]:
            if type(self.R) is not int or self.R <= 0:
                raise TypeError("R must be an intger bigger than zero")
            self._initialized["R"] = True
        if not self._initialized["nh_type"]:
            if self.nh_type not in ("simple", "count_sensitive"):
                raise TypeError("unrecognised neighborhood hashing type")
            self._nh_cs = self.nh_type == "count_sensitive"
            self._initialized["nh_type"] = True
        if not self._initialized["bits"]:
            if type(self.bits) is not int or self.bits <= 0:
                raise TypeError("illegal number of bits for hashing")
            self._max_number = 1 << self.bits
            self._mask = self._max_number - 1
            self._initialized["bits"] = True

    # ---- host logic
    def _pack(self, X):
        """(block, per-graph label-value iterables in graph order) of a fit or transform input."""
        if isinstance(X, Block):  # packed input (datasets.read_tu): the label set comes from the packed labels
            block = X.require("sp", "wloa")
            gp = block.graph_ptr
            lab = block.labels.tolist() if isinstance(block.labels, np.ndarray) else list(block.labels)
            return block, (lab[gp[g]:gp[g + 1]] for g in range(block.n_graphs))
        if not isinstance(X, Iterable):
            raise TypeError("input must be an iterable\n")
        if type(X) is not list:
            X = list(X)
        label_dicts = list(_nh_elements(X))  # element checks, warnings and errors in the reference's order
        if not label_dicts:
            return None, ()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # the empty-element warnings were given above
            block = pack(X, "wloa", len_ok=lambda n: n in (2, 3), type_error_msg=_NH_ELEMENT_MSG)
        return block, (L.values() for L in label_dicts)

    def _hash_labels(self, label_values):
        """:157, 164-189: the label set, built with `|=` in graph order, zipped with draws from random_state_."""
        labels_hash_set = set()
        for vals in label_values:
            labels_hash_set |= set(vals)
        rs, M = self.random_state_, self._max_number
        if len(labels_hash_set) > M:
            warnings.warn("Number of labels is smaller than" "the biggest possible.. " "Collisions will appear on the "
                          "new labels.")
            nl, nrl = list(), len(labels_hash_set)
            while nrl > M:
                nl += rs.choice(M, M, replace=False).tolist()
                nrl -= M
            if nrl > 0:
                nl += rs.choice(M, nrl, replace=False).tolist()
        else:
            nl = rs.choice(M, len(labels_hash_set), replace=False).tolist()
        return dict(zip(labels_hash_set, nl))

    @staticmethod
    def _labels0(block, hash_dict):
        """Hashed level-0 label of every packed vertex, -1 for a label outside the dictionary (None, :299)."""
        labels = block.labels
        if isinstance(labels, np.ndarray):
            uniq, inv = np.unique(labels, return_inverse=True)
            hv = np.fromiter((hash_dict.get(u, -1) for u in uniq.tolist()), dtype=np.int64, count=len(uniq))
            return hv[inv.ravel()]
        return np.fromiter((hash_dict.get(l, -1) for l in labels), dtype=np.int64, count=len(labels))

    # ---- reference protocol
    def fit(self, X, y=None):
        """:91-206"""
        self._method_calling = 1
        self._is_transformed = False
        self.initialize()
        if X is None:
            raise ValueError("`fit` input cannot be None")
        block, label_values = self._pack(X)
        if block is None:
            raise ValueError("parsed input is empty")
        self._labels_hash_dict = self._hash_labels(label_values)
        self.X = Fitted(block, self._labels0(block, self._labels_hash_dict), self._labels_hash_dict)
        return self

    def fit_transform(self, X, y=None):
        """:208-237"""
        self._method_calling = 2
        self.fit(X)
        if np.any(np.diff(self.X.block.graph_ptr) == 0):
            raise ZeroDivisionError("float division by zero")  # a graph without vertices against itself: 0 / 0.0
        return self._run(self.X.block, self.X.ids, n_fit=self.X.block.n_graphs)

    def transform(self, X):
        """:239-322"""
        self._method_calling = 3
        check_is_fitted(self, ["X"])
        if X is None:
            raise ValueError("`transform` input cannot be None")
        block, _ = self._pack(X)
        self._is_transformed = True
        n_fit = self.X.block.n_graphs
        if block is None:  # the reference builds an empty matrix when every element was empty
            return np.zeros((0, n_fit))
        if np.any(np.diff(block.graph_ptr) == 0) and np.any(np.diff(self.X.block.graph_ptr) == 0):
            raise ZeroDivisionError("float division by zero")
        ids = np.concatenate([self.X.ids, self._labels0(block, self._labels_hash_dict)])
        return self._run(Block.concat(self.X.block, block), ids, n_fit=n_fit)

    def diagonal(self):
        """:343-365: the matrix is normalised by construction."""
        if getattr(self, "_is_transformed", False):
            return 1.0, 1.0
        return 1.0

    def _run(self, block, labels0, n_fit):
        """pack -> R relabel levels -> per-level intersections and the fp64 combine, all on the device."""
        with _lib.engine(getattr(self, "device_", None)) as eng:
            eng.pack(block.graph_ptr, block.row_ptr, block.col_idx)
            self.stats_ = eng.nh_features(self.R, self.bits, self._nh_cs, labels0)
            self.stats_gram_ = _lib.GkStats()
            K = eng.nh_gram(block.n_graphs, n_fit=n_fit, stats=self.stats_gram_)
        return K
