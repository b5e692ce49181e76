"""NeighborhoodHash on the CPU, twice (no device, no reference needed):

* `NHOracle` restates neighborhood_hash.py:91-570 over the oracle's graph parser (`OGraph`: the reference's vertex set
  and out-neighbour order), with an injectable hash dictionary: a sub-matrix of a large fit equals the oracle on that
  subset run with the estimator's fitted `_labels_hash_dict`.
* `nh_pipeline_model` follows the device pipeline on a packed block (grakel_b200/csrc/nh.cuh): u64 labels with the
  all-ones None, the per-slot count-sensitive rule over CSR rows, dense per-level columns, the unary expansion and its
  integer Gram, the fp64 combine.
"""
from collections import Counter
from collections.abc import Iterable

import numpy as np
from sklearn.utils import check_random_state

from oracle.gk_oracle import OGraph

NONE64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def nh_rot(n, d, bits):
    """ROT of :367-390"""
    mask = (1 << bits) - 1
    m = d % bits
    return ((n << m) & mask) | ((n & mask) >> (bits - m)) if m > 0 else n


def nh_hash(lu, nbr_labels, bits, count_sensitive):
    """One vertex of NH_ (:392-447); None in, None out."""
    if lu is None or any(l is None for l in nbr_labels):
        return None
    out = nh_rot(lu, 1, bits)
    if not count_sensitive:
        for l in nbr_labels:
            out ^= l
        return out
    mask = (1 << bits) - 1
    srt = sorted(nbr_labels, key=lambda l: l & mask)  # the LSD radix sort of :468-491 is this stable sort
    i = 0
    while i < len(srt):
        j = i
        while j < len(srt) and srt[j] == srt[i]:
            j += 1
        occ = j - i
        out ^= nh_rot(srt[i] ^ occ, occ, bits)
        i = j
    return out


def hash_dictionary(label_dicts, bits, random_state):
    """:157, 164-189 -> (dictionary, the RandomState after the draws)"""
    rs = check_random_state(random_state)
    s = set()
    for L in label_dicts:
        s |= set(L.values())
    M = 1 << bits
    nl, nrl = [], len(s)
    while nrl > M:
        nl += rs.choice(M, M, replace=False).tolist()
        nrl -= M
    if nrl > 0:
        nl += rs.choice(M, nrl, replace=False).tolist()
    return dict(zip(s, nl)), rs


class NHOracle:
    def __init__(self, R=3, nh_type="simple", bits=8, random_state=None, hash_dict=None):
        self.R, self.bits, self.cs = R, bits, nh_type == "count_sensitive"
        self.random_state = random_state
        self.hash_dict = hash_dict

    @staticmethod
    def _graphs(X):
        if not isinstance(X, Iterable):
            raise TypeError("input must be an iterable\n")
        out = []
        for x in X:
            x = list(x)
            if len(x) == 0:
                continue
            out.append((OGraph(x[0], x[1]), x[1]))
        if not out:
            raise ValueError("parsed input is empty")
        return out

    def _levels(self, g, L):
        """[R] dicts vertex -> label (None = unseen)"""
        lab = {v: self.hash_dict.get(l) for v, l in L.items()}
        verts = g.verts
        levels = []
        for _ in range(self.R):
            lab = {u: nh_hash(lab[u], [lab[n] for n in g.ed[u]], self.bits, self.cs) for u in verts}
            levels.append(lab)
        return levels

    def fit(self, X):
        gs = self._graphs(X)
        if self.hash_dict is None:
            self.hash_dict, self.random_state_ = hash_dictionary([L for _, L in gs], self.bits, self.random_state)
        self.X = [(len(g.verts), self._levels(g, L)) for g, L in gs]
        return self

    def _pair(self, x, y):
        (nx, lx), (ny, ly) = x, y
        a = []
        for r in range(self.R):
            cx = Counter(l for l in lx[r].values() if l is not None)
            cy = Counter(l for l in ly[r].values() if l is not None)
            c = sum(min(n, cy[l]) for l, n in cx.items() if l in cy)
            a.append(c / float(nx + ny - c))
        return sum(a) / (1.0 * self.R)  # the built-in sum, as :340 (compensated for floats since CPython 3.12)

    def fit_transform(self, X):
        self.fit(X)
        n = len(self.X)
        K = np.zeros((n, n))
        for i in range(n):
            for j in range(i, n):
                K[i, j] = K[j, i] = self._pair(self.X[i], self.X[j])
        return K

    def transform(self, Y):
        ys = [(len(g.verts), self._levels(g, L)) for g, L in self._graphs(Y)]
        return np.array([[self._pair(y, x) for x in self.X] for y in ys]).reshape(len(ys), len(self.X))


# ---------------------------------------------------------------------------------------------------------- device model
def nh_relabel_model(row_ptr, col_idx, lab, bits, count_sensitive):
    """One level of nh_relabel over the packed CSR: the per-slot rule of nh_cs_term, u64 labels, all ones = None."""
    mask = (1 << bits) - 1
    V = len(row_ptr) - 1
    out = np.empty(V, dtype=np.uint64)
    lab_py = [int(x) for x in lab]
    NONE = int(NONE64)
    for v in range(V):
        b, e = int(row_ptr[v]), int(row_ptr[v + 1])
        nb = [lab_py[int(c)] for c in col_idx[b:e]]
        if lab_py[v] == NONE or NONE in nb:
            out[v] = NONE64
            continue
        x = 0
        for i, l in enumerate(nb):
            if not count_sensitive:
                x ^= l
                continue
            k = l & mask
            prev = next((nb[j] for j in range(i - 1, -1, -1) if nb[j] & mask == k), None)
            if prev == l:
                continue
            occ = 1
            for j in range(i + 1, len(nb)):
                if nb[j] & mask == k:
                    if nb[j] != l:
                        break
                    occ += 1
            x ^= nh_rot(l ^ occ, occ, bits)
        out[v] = np.uint64(nh_rot(lab_py[v], 1, bits) ^ x)
    return out


def nh_pipeline_model(block, labels0, R, bits, count_sensitive, n_fit=None):
    """(K, [R] u64 label arrays) of the device pipeline on a packed block; labels0 int64, -1 = None."""
    gp = np.asarray(block.graph_ptr, dtype=np.int64)
    N = len(gp) - 1
    n_fit = N if n_fit is None else n_fit
    vgraph = np.repeat(np.arange(N), np.diff(gp))
    nv = np.diff(gp).astype(np.int64)
    lab = np.asarray(labels0, dtype=np.int64).astype(np.uint64)
    levels = []
    K = None
    rows = np.arange(N) if n_fit == N else np.arange(n_fit, N)
    for r in range(R):
        lab = nh_relabel_model(block.row_ptr, block.col_idx, lab, bits, count_sensitive)
        levels.append(lab)
        ok = lab != NONE64
        # dense columns of the labels present, count block, thermometer expansion, integer Gram
        _, col = np.unique(lab[ok], return_inverse=True)
        D = int(col.max()) + 1 if len(col) else 0
        cnt = np.zeros((N, max(D, 1)), dtype=np.int64)
        np.add.at(cnt, (vgraph[ok], col), 1)
        colmax = cnt.max(axis=0)
        base = np.concatenate([[0], np.cumsum(colmax)])
        U = np.zeros((N, int(base[-1]) or 1), dtype=np.int64)
        for g, c in zip(*np.nonzero(cnt)):
            U[g, base[c]:base[c] + cnt[g, c]] = 1
        C = (U[rows] @ U[:n_fit].T).astype(np.float64)
        a = C / (nv[rows][:, None] + nv[:n_fit][None, :] - C)
        if r == 0:
            K, comp = a, np.zeros_like(a)
        else:  # nh_combine: Neumaier's compensated sum, as CPython's sum() of floats
            t = K + a
            comp = comp + np.where(np.abs(K) >= np.abs(a), (K - t) + a, (a - t) + K)
            K = t
    K = np.where((comp != 0) & np.isfinite(comp), K + comp, K)
    return K / float(R), levels
