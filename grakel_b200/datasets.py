"""TU-format datasets straight into packed CSR blocks (SURVEY 8(f) rank 4).

`read_tu` replaces, for the kernels of the hot path, the pair
``grakel.datasets.read_data`` (datasets/base.py:135-290: five text files parsed line by line into
per-graph Python sets and dictionaries) + the per-graph ``Graph`` parsing every ``fit`` repeats
(graph.py:147-230, 982-1053).  The files are parsed by the C-ABI reader (`gk_tu_*`, host code in
csrc/tu_reader.h) into the arrays `gk_pack_csr` takes; the result is a `Block` that every estimator of
this package accepts in place of the list of graphs (`fit`, `transform`, `fit_transform`).

The vertex set of a block depends on the kernel, exactly as in the reference:
  * "WL" / "VH"      every labelled node                     (weisfeiler_lehman.py:234 walks the label keys)
  * "SP" / "WL-OA"   the nodes that occur in an edge         (graph.py:1613-1631; edge-dictionary keys)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from .packing import Block

_MODES = {"WL": 0, "VH": 0, "weisfeiler_lehman": 0, "vertex_histogram": 0, "subtree_wl": 0, "ST-WL": 0,
          "SP": 1, "shortest_path": 1, "WL-OA": 1, "weisfeiler_lehman_optimal_assignment": 1,
          "NH": 1, "neighborhood_hash": 1}
GK_TU_SYMMETRIC, GK_TU_ATTR_NODES, GK_TU_DEGREE_LABELS = 1, 2, 4


class Bunch(dict):
    """`sklearn.utils.Bunch`-like result of read_tu: .data (Block), .target (classes), .edge_labels, .node_ids."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


def read_tu(path, name, kernel="WL", with_classes=True, is_symmetric=False, prefer_attr_nodes=False,
            produce_labels_nodes=False):
    """Read `<path>/<name>/<name>_*.txt` (read_data's layout) or `<path>/<name>_*.txt` into one packed block
    for `kernel`.

    Parameters follow `read_data` (base.py:135-143): `is_symmetric` adds the reverse of every edge line,
    `prefer_attr_nodes` loads node attributes instead of node labels (for ShortestPathAttr),
    `produce_labels_nodes` labels nodes by their degree when the dataset has no node labels."""
    if kernel not in _MODES:
        raise ValueError("read_tu packs for WL / VH / SP / WL-OA / NH; got " + repr(kernel))
    mode = _MODES[kernel]
    lib = _lib.load_library()

    def check(rc):
        if rc != 0:
            raise ValueError(lib.gk_last_error().decode())

    flags = (GK_TU_SYMMETRIC if is_symmetric else 0) | (GK_TU_ATTR_NODES if prefer_attr_nodes else 0) | \
            (GK_TU_DEGREE_LABELS if produce_labels_nodes else 0)
    t = C.c_void_p()
    path = str(path)
    if os.path.isdir(os.path.join(path, str(name))):  # read_data's layout: ./<name>/<name>_A.txt (base.py:181-191)
        path = os.path.join(path, str(name))
    check(lib.gk_tu_open(path.encode(), str(name).encode(), flags, C.byref(t)))
    try:
        info = (C.c_int64 * 8)()
        check(lib.gk_tu_info(t, info))
        n_graphs, has_nl, has_el, has_cls, attr_dim = int(info[0]), bool(info[3]), bool(info[4]), bool(info[5]), int(info[6])
        V, E = C.c_int64(), C.c_int64()
        check(lib.gk_tu_pack(t, mode, C.byref(V), C.byref(E)))
        V, E = V.value, E.value
        gp = np.empty(n_graphs + 1, dtype=np.int32)
        rp = np.empty(V + 1, dtype=np.int32)
        ci = np.empty(E, dtype=np.int32)
        use_attr = prefer_attr_nodes and attr_dim > 0
        labelled = (has_nl or produce_labels_nodes) and not use_attr
        lab = np.empty(V, dtype=np.int32) if labelled else None
        el = np.empty(E, dtype=np.int32) if has_el else None
        at = np.empty((V, attr_dim), dtype=np.float64) if use_attr else None
        cls = np.empty(n_graphs, dtype=np.int32) if (with_classes and has_cls) else None
        node = np.empty(V, dtype=np.int32)
        p = _lib._ptr
        check(lib.gk_tu_fill(t, p(gp), p(rp), p(ci), p(lab), p(el), p(at), p(cls), p(node)))
    finally:
        lib.gk_tu_close(t)
    block = Block(gp, rp, ci, None, lab, at, all_adjacency=False)
    block.mode = "wl" if mode == 0 else "sp"
    out = Bunch(data=block, edge_labels=el, node_ids=node)
    if with_classes:
        if cls is None:
            raise ValueError("the dataset has no graph classes (<name>_graph_labels.txt)")
        out["target"] = cls.astype(int)
    return out
