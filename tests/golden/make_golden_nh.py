"""Golden fixtures for NeighborhoodHash, produced by the REAL reference (neighborhood_hash.py).  Inputs are
regenerated from seeds (`nh_sets` below), only the reference's outputs are stored (tests/golden/nh.npz).  Integer
labels only: the iteration order of a set of strings depends on PYTHONHASHSEED.

    GRAKEL_REF=baseline/_ref python tests/golden/make_golden_nh.py
"""
import os
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..", "..")
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, ".."))  # tests/: tu_io


def nh_sets():
    """name -> (fit elements, transform elements or None).

    small_*: seeded sparse graphs with five labels (more than 2^2), the transform set carries labels 7, 8 that the fit
    set lacks (None spreads from them); adj: the same as adjacency matrices; hubs: stars whose centre has 4 - 9
    neighbours of two labels, so that bits = 2 count-sensitive labels outgrow the mask (occ % bits == 0, occ >= 4)."""
    from oracle.gk_oracle import gen
    X = gen(40, 12, 31, nl=5)
    rs = np.random.RandomState(7)
    for _g, l in X[30:][::2]:
        for v in list(l)[::5]:
            l[v] = 7 + int(rs.randint(2))
    out = {"small": (X[:30], X[30:])}
    A = gen(24, 10, 32, nl=4, as_adj=True)
    out["adj"] = (A[:18], A[18:])
    hubs = []
    for i in range(16):
        k = 4 + i % 6
        n = k + 1 + int(rs.randint(3))
        M = np.zeros((n, n))
        M[0, 1:k + 1] = M[1:k + 1, 0] = 1
        for a in range(k + 1, n):  # a tail hanging off the last leaf
            M[a, a - 1] = M[a - 1, a] = 1
        hubs.append([M, {v: int(rs.randint(2)) if v else 2 for v in range(n)}])
    out["hubs"] = (hubs[:12], hubs[12:])
    return out


CASES = [(t, R, b) for t in ("simple", "count_sensitive") for R in (1, 3) for b in (2, 8)]


def mutag():
    import gio
    return gio.dec_dataset(gio.load(os.path.join(HERE, "mutag_graphs.json.gz")))[:60]


def write_mutag_tu(path):
    import tu_io
    X = mutag()
    tu_io.write_tu(path, "MUTAG", X, classes=[1 if i % 3 else -1 for i in range(len(X))],
                   edge_labels=[{e: 0 for e in el[0]} for el in X])  # read_data wants MUTAG's edge-label file


if __name__ == "__main__":
    sys.path.insert(0, os.environ.get("GRAKEL_REF", os.path.join(ROOT, "baseline", "_ref")))
    from grakel import NeighborhoodHash as RefNH  # the reference
    from grakel.datasets.base import read_data
    warnings.simplefilter("ignore")
    out = {}
    for name, (fit, new) in nh_sets().items():
        for t, R, b in CASES:
            tag = f"{name}_{t}_R{R}_b{b}"
            k = RefNH(R=R, nh_type=t, bits=b, random_state=R * 100 + b)
            out[tag + "_K"] = k.fit_transform(fit)
            out[tag + "_hk"] = np.array(list(k._labels_hash_dict.keys()), dtype=np.int64)
            out[tag + "_hv"] = np.array(list(k._labels_hash_dict.values()), dtype=np.int64)
            out[tag + "_d"] = np.array(k.diagonal(), dtype=float)
            out[tag + "_Kt"] = k.transform(new)
            out[tag + "_dt"] = np.array(k.diagonal(), dtype=float)
            out[tag + "_rs"] = np.array([k.random_state_.randint(1 << 30)])  # RandomState consumption
            k.fit(fit)  # a second fit draws again from the same random_state_
            out[tag + "_hv2"] = np.array(list(k._labels_hash_dict.values()), dtype=np.int64)
    for t in ("simple", "count_sensitive"):
        out[f"mutag_{t}"] = RefNH(R=3, nh_type=t, random_state=5).fit_transform(mutag())
        with tempfile.TemporaryDirectory() as d:  # read_data reads ./<name>/<name>_*.txt
            write_mutag_tu(os.path.join(d, "MUTAG"))
            cwd = os.getcwd()
            os.chdir(d)
            try:
                data = read_data("MUTAG", with_classes=True).data
            finally:
                os.chdir(cwd)
            out[f"tu_{t}"] = RefNH(R=3, nh_type=t, random_state=6).fit_transform(data)
    np.savez_compressed(os.path.join(HERE, "nh.npz"), **out)
    for k, v in out.items():
        if k.endswith("_K") or k.startswith(("mutag", "tu")):
            print(k, v.shape, float(np.nansum(v)))
