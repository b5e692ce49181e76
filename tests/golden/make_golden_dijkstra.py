"""Golden fixtures for real-valued edge weights with the reference's DIJKSTRA path sums, produced by the REAL
reference (baseline/_ref, or GRAKEL_REF): ShortestPath on edge-dictionary inputs (algorithm_type "auto" -> dijkstra,
graph.py:652-656, 1712-1764), with and without labels, fit_transform + transform, the Floyd-Warshall matrices of the
same graphs for contrast (the two differ: SURVEY 7), WeisfeilerLehman over ShortestPath, and ShortestPathAttr with
algorithm_type="dijkstra".  Inputs are regenerated from the seed; only the reference's matrices are stored.

    python tests/golden/make_golden_dijkstra.py
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..", "..")


def gen_real(n_graphs, nbar, seed, attr=0):
    """ER graphs (avg degree 4) as {(u, v): w} with symmetric weights from a few non-dyadic reals -- path lengths
    coincide across graphs only when the sums associate the same way (0.1 + 0.2 != 0.3 in binary) --; labels or
    attribute vectors."""
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n_graphs):
        n = int(rs.randint(nbar // 2, nbar + nbar // 2 + 1))
        iu = np.triu_indices(n, 1)
        m = rs.rand(len(iu[0])) < 4.0 / (n - 1)
        g = {}
        for a, b in zip(iu[0][m].tolist(), iu[1][m].tolist()):
            w = float(rs.choice([0.1, 0.2, 0.3, 0.7, 1.1]))
            g[(a, b)] = w
            g[(b, a)] = w
        if not g:
            g[(0, 1)] = g[(1, 0)] = 1.25
        L = {i: (rs.rand(attr) if attr else int(rs.randint(4))) for i in range(n)}
        out.append([g, L])
    return out


if __name__ == "__main__":
    # the reference is imported only to write the fixtures: the tests import gen_real from here without it
    sys.path.insert(0, os.environ.get("GRAKEL_REF", os.path.join(ROOT, "baseline", "_ref")))
    from grakel import ShortestPath, ShortestPathAttr, WeisfeilerLehman  # (the reference)
    warnings.simplefilter("ignore")
    out = {}
    X = gen_real(40, 12, 21)
    fit, new = X[:30], X[30:]
    for tag, wl in (("lab", True), ("nolab", False)):
        e = ShortestPath(with_labels=wl)
        out[f"dj_{tag}_K"] = e.fit_transform(fit)
        out[f"dj_{tag}_Kt"] = e.transform(new)
        out[f"fw_{tag}_K"] = ShortestPath(with_labels=wl, algorithm_type="floyd_warshall").fit_transform(fit)
    assert not np.array_equal(out["dj_nolab_K"], out["fw_nolab_K"]), "the two algorithms were expected to differ"
    out["dj_norm_K"] = ShortestPath(normalize=True).fit_transform(fit)
    w = WeisfeilerLehman(n_iter=2, base_graph_kernel=ShortestPath)
    out["wlsp_K"] = w.fit_transform(fit)
    out["wlsp_Kt"] = w.transform(new)
    A = gen_real(7, 8, 5, attr=3)
    out["attr_dj_K"] = ShortestPathAttr(algorithm_type="dijkstra").fit_transform(A)
    np.savez_compressed(os.path.join(HERE, "dijkstra_real.npz"), **out)
    for k, v in out.items():
        print(k, v.shape, float(np.nansum(v)))
