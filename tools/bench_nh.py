"""NeighborhoodHash on BASELINE config 2's graphs (gen(10000, 40, 0), R = 3, bits = 8), both hash types.

Reports, per type:
  * device-resident ms of one gk_nh_features + gk_nh_gram pass (K stays on the device), CUDA events after warm-up, with
    the stage times the library returns: relabel, level histograms + unary expansion, the R level Grams, the fp64
    combine.  Working set: the R fp32 level Grams (3 x 400 MB) and the fp64 K (800 MB) are far above the 126 MB L2.
  * end-to-end ms of NeighborhoodHash().fit_transform(list) (host packing and hashing, device, fp64 copy to the host);
  * the bound of every stage, from shapes: HBM bytes over 7.7 TB/s, or dense tensor FLOPs over 2 250 TFLOP/s (BF16);
  * the reference's pairs/s on a prefix of the graphs (when the reference is installed under baseline/_ref).
One JSON line on stdout and in --out.

    python tools/bench_nh.py --out profiles/r04_nh_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM = 7.7e12      # B/s, HGX B200 data sheet, one GPU
TC_BF16 = 2.25e15  # dense FLOP/s, same source


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown (%s)" % e}


def device_pass(X, t, warmup, steps):
    from grakel_b200 import NeighborhoodHash, _lib
    est = NeighborhoodHash(R=3, nh_type=t, bits=8, random_state=0).fit(X)
    blk, lab0 = est.X.block, est.X.ids
    N = blk.n_graphs
    rows = []
    with _lib.engine() as eng:
        eng.pack(blk.graph_ptr, blk.row_ptr, blk.col_idx)
        for i in range(warmup + steps):
            sf, sg = _lib.GkStats(), _lib.GkStats()
            eng.event_record(0)
            sf = eng.nh_features(3, 8, t == "count_sensitive", lab0)
            eng.nh_gram(N, out=False, stats=sg)
            eng.event_record(1)
            eng.sync()
            if i >= warmup:
                rows.append((eng.event_elapsed(0, 1), sf.ms_features, sf.ms_panel, sg.ms_gemm, sg.ms_tail))
        dense_cols = sg.n_dense_columns
    a = np.array(rows)
    med = np.median(a, axis=0)
    V = blk.n_vertices
    R = 3
    # bounds from shapes
    b_relabel = R * (V * 8 * 2 + len(blk.col_idx) * (4 + 8) + (V + 1) * 4) / HBM  # labels in/out, neighbour gathers
    b_gram_store = R * N * N * 4 / HBM  # each level Gram written once in fp32
    b_gram_mma = R * N * N * max(int(dense_cols), 0) / TC_BF16  # symmetric: N^2 Dc MACs = 2 N^2 Dc / 2 flops per level
    b_combine = (R * N * N * 4 + N * N * 8) / HBM  # R fp32 level Grams read, fp64 K written once
    return {
        "type": t, "steps": steps,
        "ms_pass_median": float(med[0]), "ms_pass_min": float(a[:, 0].min()), "ms_pass_max": float(a[:, 0].max()),
        "ms_relabel": float(med[1]), "ms_hist_expand": float(med[2]), "ms_level_grams": float(med[3]),
        "ms_combine": float(med[4]),
        "bound_ms": {"relabel_hbm": b_relabel * 1e3, "level_grams_store_hbm": b_gram_store * 1e3,
                     "level_grams_head_mma_last_level": b_gram_mma * 1e3, "combine_hbm": b_combine * 1e3},
        "n_vertices": V, "n_graphs": N, "head_columns_last_level": int(dense_cols),
    }


def e2e(X, t, reps):
    from grakel_b200 import NeighborhoodHash
    NeighborhoodHash(R=3, nh_type=t, random_state=0).fit_transform(X)  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        NeighborhoodHash(R=3, nh_type=t, random_state=0).fit_transform(X)
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def reference_rate(X, t, n):
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "grakel")):
        return None
    sys.path.insert(0, ref)
    from grakel import NeighborhoodHash as RefNH
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        RefNH(R=3, nh_type=t, random_state=0).fit_transform(X[:n])
        dt = time.perf_counter() - t0
    return {"graphs": n, "seconds": dt, "pairs_per_s": n * (n + 1) / 2 / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--ref-graphs", type=int, default=300)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from oracle.gk_oracle import gen
    X = gen(10000, 40, 0)
    res = {"workload": "NeighborhoodHash R=3 bits=8 on gen(10000, 40, 0)", **card(), "per_type": []}
    for t in ("simple", "count_sensitive"):
        d = device_pass(X, t, a.warmup, a.steps)
        d["ms_fit_transform_e2e"] = e2e(X, t, a.e2e_reps)
        r = reference_rate(X, t, a.ref_graphs)
        d["reference"] = r if r is not None else "not measured (reference not installed)"
        if r is not None:
            d["device_pairs_per_s"] = 10000 * 10001 / 2 / (d["ms_pass_median"] / 1e3)
        res["per_type"].append(d)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
