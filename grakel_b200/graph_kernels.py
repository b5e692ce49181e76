"""`GraphKernel`: the name -> kernel dispatcher of the reference (grakel/graph_kernels.py:77-571), restricted to
the kernels of the device hot path:

    "weisfeiler_lehman" / "WL"  (framework; base "vertex_histogram"/"subtree_wl"/"VH"/"ST-WL", "shortest_path", ...)
    "vertex_histogram" / "subtree_wl" / "VH" / "ST-WL"
    "shortest_path" / "SP"      (+ with_labels, algorithm_type, as_attributes)
    "edge_histogram" / "EH"
    "core_framework" / "CORE"   (framework; base "shortest_path" or "weisfeiler_lehman" ...)
    "weisfeiler_lehman_optimal_assignment" / "WL-OA"
    "neighborhood_hash" / "NH"  (R, nh_type, bits, random_state: the reference's dispatcher does not pass its own
                                 random_state to this kernel, graph_kernels.py:524-525, so a seed goes in the dict)

Any other reference kernel name raises NotImplementedError (not ValueError, which the reference reserves for
unknown names).  The public surface (constructor parameters, `fit` / `transform` / `fit_transform`, the fitted
attributes `kernel_`, `nystroem_`, `components_`, `component_indices_`, `nystroem_normalization_`, the error
messages) is the reference's; the implementation is a name registry plus a small low-rank-map helper.

Nystroem (graph_kernels.py:311-335, 367, 403): `Nystroem=n` picks n basis graphs at random, and every later matrix
is K(X, basis) @ W^T with W = K(basis, basis)^(-1/2).  The large object of that computation is the m x n cross
matrix -- n is ~100, so it is megabytes, not the N x N matrix -- and it comes from the device like any other
`transform`; the n x n inverse square root is host linear algebra.
"""
import copy
import warnings

import numpy as np
from sklearn.base import BaseEstimator, TransformerMixin
from sklearn.utils import check_random_state
from sklearn.utils.validation import check_is_fitted

from .core_framework import CoreFramework
from .kernels import (EdgeHistogram, NeighborhoodHash, ShortestPath, ShortestPathAttr, VertexHistogram,
                      WeisfeilerLehman, WeisfeilerLehmanOptimalAssignment)

default_n_components = 100

# reference names outside the hot path (graph_kernels.py:38-64)
_OUTSIDE = frozenset((
    "random_walk", "RW", "graphlet_sampling", "GR", "subgraph_matching", "SM", "multiscale_laplacian", "ML",
    "lovasz_theta", "LOVT", "svm_theta", "SVMT", "neighborhood_subgraph_pairwise_distance",
    "NSPD", "odd_sth", "ODD", "propagation", "PR", "pyramid_match", "PM", "graph_hopper", "GH", "hadamard_code", "HC"))


def _shortest_path(params):
    return (ShortestPathAttr if params.pop("as_attributes", False) else ShortestPath), params


# name -> (is a framework that takes the rest of the list as its base kernel, builder(params) -> (class, params))
_REGISTRY = {}
for _names, _framework, _build in (
        (("vertex_histogram", "subtree_wl", "VH", "ST-WL"), False, lambda p: (VertexHistogram, p)),
        (("edge_histogram", "EH"), False, lambda p: (EdgeHistogram, p)),
        (("weisfeiler_lehman_optimal_assignment", "WL-OA"), False, lambda p: (WeisfeilerLehmanOptimalAssignment, p)),
        (("shortest_path", "SP"), False, _shortest_path),
        (("neighborhood_hash", "NH"), False, lambda p: (NeighborhoodHash, p)),
        (("weisfeiler_lehman", "WL"), True, lambda p: (WeisfeilerLehman, p)),
        (("core_framework", "CORE"), True, lambda p: (CoreFramework, p))):
    for _n in _names:
        _REGISTRY[_n] = (_framework, _build)


class _LowRankMap:
    """K(., basis) -> K(., basis) @ W^T with W = K(basis, basis)^(-1/2): the Nystroem feature map.

    K_bb is symmetric; with its eigen-pairs (l_i, u_i) the matrix the reference builds from an SVD
    (`U / sqrt(max(S, 1e-12)) @ V`, graph_kernels.py:326-329) is  sum_i sign(l_i) / sqrt(max(|l_i|, 1e-12)) u_i u_i^T
    -- singular values are |l_i|, and the right singular vector of a negative eigenvalue is -u_i."""

    def __init__(self, k_bb):
        k_bb = np.asarray(k_bb, dtype=np.float64)
        lam, vec = np.linalg.eigh((k_bb + k_bb.T) * 0.5)
        scale = np.where(lam < 0, -1.0, 1.0) / np.sqrt(np.maximum(np.abs(lam), 1e-12))
        self.matrix = (vec * scale) @ vec.T

    def apply(self, k_xb):
        return np.asarray(k_xb).dot(self.matrix.T)


class GraphKernel(BaseEstimator, TransformerMixin):
    def __init__(self, kernel="shortest_path", normalize=False, verbose=False, n_jobs=None, random_state=None,
                 Nystroem=False):
        self.kernel = kernel
        self.normalize = normalize
        self.verbose = verbose
        self.n_jobs = n_jobs
        self.random_state = random_state
        self.Nystroem = Nystroem
        self._initialized = dict.fromkeys(("kernel", "Nystroem", "random_state", "normalize", "verbose", "n_jobs"), False)

    # ---- estimator protocol
    def fit(self, X, y=None):
        self.initialize()
        if not self.nystroem_:
            self.kernel_.fit(X)
            return self
        X = list(X)
        wanted = self.nystroem_
        if wanted > len(X):
            warnings.warn("n_components > n_samples. This is not possible.\nn_components was set to n_samples, "
                          "which results in inefficient evaluation of the full kernel.")
        n_basis = min(len(X), wanted)
        order = self.random_state_.permutation(len(X))
        self.components_ = [X[i] for i in order[:n_basis]]
        self.component_indices_ = order
        self._map = _LowRankMap(self.kernel_.fit_transform(self.components_))
        self.nystroem_normalization_ = self._map.matrix
        self.nystroem_ = n_basis
        return self

    def transform(self, X):
        check_is_fitted(self, "kernel_")
        K = self.kernel_.transform(X)
        if getattr(self, "nystroem_", False):
            check_is_fitted(self, "components_")
            return K.dot(self.nystroem_normalization_.T)
        return K

    def fit_transform(self, X, y=None):
        self.initialize()
        if not self.nystroem_:
            return self.kernel_.fit_transform(X)
        X = list(X)
        return self.fit(X).transform(X)

    # ---- parameters
    def initialize(self):
        todo = [p for p, done in self._initialized.items() if not done]
        if "Nystroem" in todo:
            self.nystroem_ = self._n_components(self.Nystroem)
            self._initialized["Nystroem"] = True
        if any(p != "Nystroem" for p in todo):
            if "random_state" in todo:
                self.random_state_ = check_random_state(self.random_state)
            spec = self.kernel
            if type(spec) in (dict, str):
                spec = [spec]
            elif type(spec) is not list:
                raise ValueError('A "kernel" must be defined at the __init__ function of the graph kernel generic '
                                 "wrapper. Valid kernel types are dict, str, and list of dict or str.")
            cls, params = self.make_kernel_(copy.deepcopy(spec),
                                            {"verbose": self.verbose, "normalize": self.normalize, "n_jobs": self.n_jobs})
            self.kernel_ = cls(**params)
            for p in self._initialized:
                self._initialized[p] = True

    @staticmethod
    def _n_components(value):
        if type(value) not in (int, bool):
            raise ValueError("Nystroem parameter must be an int, indicating the number of components or a boolean")
        if value is False:
            return False
        if value is True or value in (0, -1):
            return default_n_components
        if value <= 0:
            raise ValueError("number of nystroem components must be positive")
        return value

    def make_kernel_(self, kernel_list, hidden_args):
        """(class, constructor parameters) of the first entry of `kernel_list`; a framework entry takes the rest of
        the list as its base kernel (graph_kernels.py:452-554)."""
        head = kernel_list.pop(0)
        if type(head) is str:
            name, params = head, {}
        elif type(head) is dict:
            if "name" not in head:
                raise ValueError('each dictionary concerning a kernel must have a "name" parameter designating '
                                 "the kernel")
            params = head
            name = params.pop("name")
        else:
            raise ValueError("each element of the list of kernels must be a dictionary or a string")
        for key, val in hidden_args.items():
            if key in params:
                warnings.warn("Overriding global kernel attribute " + str(key) + " with " + str(val) +
                              ". Please set this attribute as an argument of GraphKernel.")
            params[key] = val
        entry = _REGISTRY.get(name)
        if entry is None:
            if name in _OUTSIDE:
                raise NotImplementedError("kernel '" + str(name) + "' is outside the device hot path of grakel_b200 "
                                          "(WL-subtree, vertex histogram, edge histogram, shortest path, WL-OA, "
                                          "neighborhood hash)")
            raise ValueError("Unsupported kernel: " + str(name))
        framework, build = entry
        if framework:
            if kernel_list:
                params["base_graph_kernel"] = self.make_kernel_(kernel_list, {})
        elif kernel_list:
            warnings.warn("Kernel List not empty while reaching a base-kernel - the rest kernel names will be "
                          "ignored")
        return build(params)

    def set_params(self, **params):
        for key in params:
            head, _, sub = key.partition("__")
            flag = sub if sub else head
            if flag in self._initialized:
                self._initialized[flag] = False
        super().set_params(**copy.deepcopy(params))
        return self
