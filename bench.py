#!/usr/bin/env python
"""bench.py -- graph-pairs/sec of the N x N WL-subtree Gram matrix (BASELINE.json).

Workload (N=1, and every rank at N>1): BASELINE config 2 -- 10 000 synthetic
Erdos-Renyi labelled graphs (avg 40 nodes, 7 labels, seed 0), WL-subtree h=5.
A "step" is one pass of the hot path over that batch: WL relabel of all graphs
(one persistent kernel), feature block, dense bf16 head panel, tcgen05 Gram GEMM,
exact sparse tail, diagonal / output.

  value      pairs/s with the packed CSR already resident in HBM and K left in HBM
             (CUDA events on the engine's stream, max over ranks)
  e2e        pairs/s through the C-ABI one-call entry point gk_wl_fit_transform with
             PINNED HOST buffers: CSR H2D and the float64 K on the host inside the timed region
             (K crosses PCIe as the fp32 upper triangle and is widened + mirrored by host threads)
  e2e_api    SURVEY 8(d)'s T_e2e: WeisfeilerLehman(n_iter=5).fit_transform(python list of graphs) ->
             fresh float64 ndarray, time.perf_counter around the call (packing, H2D, device, delivery)
  roofline   the tcgen05 Gram GEMM (CTA-pair kernel): algorithmic flops N(N+1)*D_c (upper-triangular
             tiles, SURVEY 8d) / CUDA-event duration vs the measured bf16 BURST peak (a 0.2 ms launch
             inside a step that is mostly not tensor work)
  cpu_baseline / --impl reference
             the UNMODIFIED reference (ysig/GraKeL installed in baseline/_ref by baseline/build_ref.sh):
             grakel.WeisfeilerLehman(n_iter=5).fit_transform on a bounded prefix of the same graphs on
             the box's host cores, with n_jobs=None (library default) and n_jobs=cpu_count (its best
             setting); the oracle port stands in only if baseline/_ref is missing ("kind": "port")

N > 1 (torchrun): weak scaling -- the graph count grows as 10 000 * sqrt(N) so every rank owns
the same number of K entries; every rank relabels the (replicated, tiny) CSR block and
computes a contiguous row block of K -- no data-path collective;
value = (graphs^2) / max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_GRAPHS, NBAR, H, SEED = 10000, 40, 5, 0
CPU_SAMPLE = 3000  # largest prefix the bounded CPU sample may use


# the Gram GEMM gk_gram launches for fp32 output (grakel_b200/csrc/api.cu): CTA pairs unless switched off
GEMM_KERNEL = ("gram_tc_kernel<float,false> (tcgen05 cta_group::1 bf16 SYRK, 128x256 tiles)"
               if os.environ.get("GRAKEL_B200_CTA2", "1") == "0" else
               "gram_tc2_kernel (tcgen05 cta_group::2 bf16 SYRK, 256x256 tile per two-CTA cluster)")


def pack_workload(n_graphs):
    """Seeded generator of SURVEY 8d, packed straight to CSR (vectorised; the Python
    list-of-dicts form is only built for the CPU arm)."""
    rs = np.random.RandomState(SEED)
    gp, rp, ci, lab = [0], [np.zeros(1, dtype=np.int64)], [], []
    e_tot = 0
    for _ in range(n_graphs):
        n = int(rs.randint(NBAR // 2, NBAR + NBAR // 2 + 1))
        p = 4.0 / (n - 1)
        iu = np.triu_indices(n, 1)
        m = rs.rand(len(iu[0])) < p
        a, b = iu[0][m], iu[1][m]
        L = rs.randint(7, size=n)  # same stream as n independent rs.randint(7) draws
        src = np.concatenate([a, b])
        dst = np.concatenate([b, a])
        order = np.lexsort((dst, src))
        src, dst = src[order], dst[order]
        cnt = np.bincount(src, minlength=n)
        rp.append(e_tot + np.cumsum(cnt))
        ci.append(dst + gp[-1])
        lab.append(L)
        e_tot += len(src)
        gp.append(gp[-1] + n)
    return (np.asarray(gp, dtype=np.int32), np.concatenate(rp).astype(np.int32),
            np.concatenate(ci).astype(np.int32), np.concatenate(lab).astype(np.int32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 8 and r[4 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1683.9), d.get("hbm_gbs", 6582.5), \
            "measured (MEASURED_PEAKS.json, BURST bf16: the GEMM is a 0.2 ms launch inside a mostly non-tensor step)"
    return 1683.9, 6582.5, "fallback (B200_PROFILING.md)"


def kernel_source_sha1():
    """sha1 over the sources of the Gram GEMM kernels: profiles/traffic.json is only valid for the kernel it was captured from."""
    import hashlib
    h = hashlib.sha1()
    for f in ("gram_tc.cuh", "gram_tc2.cuh"):
        h.update(open(os.path.join(ROOT, "grakel_b200", "csrc", f), "rb").read())
    return h.hexdigest()


def measured_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture (profiles/traffic.json),
    or None -- also None when the GEMM sources changed since the capture (the file carries their sha1)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if d.get("gemm_source_sha1") != kernel_source_sha1():
            return None
        for k, v in d.items():
            if isinstance(v, dict) and key in k:
                return v["dram_read_bytes"] + v["dram_write_bytes"]
    except Exception:
        pass
    return None


def gen_list(n_graphs, nbar=NBAR, seed=SEED, attr=0, as_adj=False):
    """The seeded generator of SURVEY 8(d) in its Python-list form (what the reference API takes):
    [{(u, v): 1, (v, u): 1, ...}, {vertex: label}] per graph; `as_adj`: dense float adjacency instead of the edge
    dictionary (SP configs), `attr`: d-dimensional U[0,1) attribute vectors instead of labels (config 5)."""
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n_graphs):
        n = int(rs.randint(nbar // 2, nbar + nbar // 2 + 1))
        p = 4.0 / (n - 1)
        iu = np.triu_indices(n, 1)
        m = rs.rand(len(iu[0])) < p
        a, b = iu[0][m], iu[1][m]
        L = {i: rs.rand(attr) for i in range(n)} if attr else {i: int(rs.randint(7)) for i in range(n)}
        if as_adj:
            A = np.zeros((n, n))
            A[a, b] = 1.0
            g = A + A.T
        else:
            g = {}
            for x, y in zip(a.tolist(), b.tolist()):
                g[(x, y)] = 1
                g[(y, x)] = 1
        out.append([g, L])
    return out


def dump_rows(n_rows, n_cols):
    """Sorted, seeded sample of row indices for --dump-outputs: the same rows on every run with the same arguments,
    few enough that their fp32 and fp64 copies stay under 48 MB together."""
    k = int(min(n_rows, 256, max(1, 48e6 // (12 * n_cols))))
    return np.sort(np.random.RandomState(20240).choice(n_rows, size=k, replace=False))


def bind_to_gpu_node(torch, local):
    """Run this process on the CPUs of the NUMA node the GPU hangs off (what `numactl --cpunodebind` would do): host
    buffers the bench allocates (pinned CSR / K) then live next to the GPU's PCIe root.  Returns the node or None."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def host_info():
    info = {"logical_cores": os.cpu_count()}
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["cpu_model"] = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_info
        info["threadpools"] = [{k: t.get(k) for k in ("user_api", "internal_api", "num_threads")} for t in threadpool_info()]
    except Exception:
        pass
    return info


def reference_estimator():
    """(factory(n_jobs) -> estimator, kind): the real GraKeL from baseline/_ref, else the oracle port."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "grakel")):
        sys.path.insert(0, ref)
        try:
            from grakel.kernels import WeisfeilerLehman as RefWL
            return (lambda nj: RefWL(n_iter=H, n_jobs=nj)), "reference"
        except Exception as e:  # pragma: no cover
            print("baseline/_ref import failed (%r): falling back to the oracle port" % (e,), file=sys.stderr)
            sys.path.remove(ref)
    from oracle.gk_oracle import WLOracle
    return (lambda nj: WLOracle(n_iter=H, n_jobs=nj)), "port"


def cpu_arm(steps=1, warmup=0, budget_s=12.0, n_max=CPU_SAMPLE):
    """The reference's CPU fit_transform on a prefix of the workload.  A timed probe (600 graphs, both n_jobs
    settings) picks the faster setting and the prefix length (cost ~ n^2) so that warmup + steps runs take about
    `budget_s` seconds, capped at `n_max` graphs.  Returns a dict with pairs/s of the chosen setting, of
    n_jobs=None on the same prefix, seconds/step, the prefix length and the kind of implementation."""
    make, kind = reference_estimator()
    X = gen_list(n_max)
    ncpu = os.cpu_count() or 1
    probe = min(600, n_max)
    tp = {}
    for nj in (None, ncpu):
        make(nj).fit_transform(X[:200])  # warm-up (imports, thread pool)
        t = time.perf_counter()
        make(nj).fit_transform(X[:probe])
        tp[nj] = time.perf_counter() - t
    best = min(tp, key=tp.get)
    n_sample = int(min(n_max, max(probe, probe * np.sqrt(budget_s / max(steps + warmup, 1) / tp[best]))))
    n_sample -= n_sample % 100
    Xs = X[:n_sample]
    for _ in range(warmup):
        make(best).fit_transform(Xs)
    ts = []
    for _ in range(steps):
        t = time.perf_counter()
        K = make(best).fit_transform(Xs)
        ts.append(time.perf_counter() - t)
        assert K.shape == (n_sample, n_sample)
        del K
    t_best = float(np.mean(ts))
    t = time.perf_counter()
    make(ncpu if best is None else None).fit_transform(Xs)  # the other setting, once, on the same prefix
    t_other = time.perf_counter() - t
    t_default, t_all = (t_best, t_other) if best is None else (t_other, t_best)
    return {"value": n_sample * n_sample / t_best, "seconds_per_step": t_best, "n_sample": n_sample, "kind": kind,
            "n_jobs": "None" if best is None else ncpu,
            "pairs_per_s_n_jobs_None": n_sample * n_sample / t_default,
            "pairs_per_s_n_jobs_all": n_sample * n_sample / t_all,
            "threads_useful": 1 if best is None else min(ncpu, H + 1)}


def cpu_baseline_obj(r, n_total):
    return {"value": r["value"], "unit": "pairs/s", "cores": r["threads_useful"], "kind": r["kind"],
            "sample": f"first {r['n_sample']} of the {n_total} graphs ({r['n_sample'] ** 2} ordered pairs per step), "
                      f"{r['seconds_per_step']:.2f} s per fit_transform with n_jobs={r['n_jobs']} (joblib threads over the "
                      f"{H + 1} WL levels, weisfeiler_lehman.py:279-285)",
            "n_jobs_None_pairs_per_s": r["pairs_per_s_n_jobs_None"], "n_jobs_all_pairs_per_s": r["pairs_per_s_n_jobs_all"],
            "host": host_info()}


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_arm(steps=args.steps, warmup=args.warmup, budget_s=110.0, n_max=4000)
    val, t, n = r["value"], r["seconds_per_step"], r["n_sample"]
    line = {
        "impl": "reference", "metric": "graph-pairs/sec, N x N WL-subtree (h=5) Gram", "value": val,
        "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"config2: {N_GRAPHS} ER graphs (avg {NBAR} nodes, 7 labels, seed {SEED}), WL-subtree h={H}",
                   "parallelism": f"host CPU, grakel.WeisfeilerLehman(n_iter={H}, n_jobs={r['n_jobs']}).fit_transform"},
        "cpu_baseline": cpu_baseline_obj(r, N_GRAPHS),
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def other_paths(eng, local, X2, with_cpu, steps):
    """BASELINE configs 3 (ShortestPath, 5 000 graphs, avg 60 nodes) and 5 (ShortestPathAttr, 2 000 graphs, d = 16) and
    WL-OA on the graphs of config 2: one GPU, CSR resident in HBM -> K resident in HBM, CUDA events on the engine's
    stream, `steps` timed steps each; each with its dominant kernel against the stated roof (SURVEY 8d) and the real
    reference on a bounded sample beside it."""
    from grakel_b200.packing import label_ids, pack
    peak_tf, peak_hbm, _ = peaks()
    out = {}

    def timed(fn, warmup=3):
        for _ in range(warmup):
            st = fn()
        eng.event_record(4)
        for _ in range(steps):
            st = fn()
        eng.event_record(5)
        return eng.event_elapsed(4, 5) / steps, st

    def ref_time(make, X):
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
            est = make()
            t0 = time.perf_counter()
            est.fit_transform(X)
            return time.perf_counter() - t0, "reference"
        except Exception as e:  # pragma: no cover
            return None, "unavailable: %r" % (e,)

    sm_clock = 1.965e9
    # ---- config 3
    X = gen_list(5000, 60, 0, as_adj=True)
    b = pack(X, "sp", want_weights=True)
    ids, _ = label_ids(b.labels, None, sort_new=False)
    eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids, b.weights)
    n = b.n_graphs
    sizes = np.diff(b.graph_ptr).astype(np.float64)

    def step3():
        st = eng.sp_features(with_labels=True)
        eng.gram(n, out=False, dtype=np.float32, stats=st, want_diag=False)
        return st
    ms, st = timed(step3)
    relax = float((sizes ** 3).sum())
    D3 = int(st.n_columns)
    c3 = {"workload": "config3: 5000 ER graphs (avg 60 nodes, 7 labels, seed 0), ShortestPath(with_labels=True), adjacency input",
          "ms_per_step": ms, "pairs_per_s": n * n / (ms * 1e-3),
          "stages_ms": {"apsp+histogram (sp_bfs_hist)": st.ms_features, "columns+panel": st.ms_panel, "gram_gemm": st.ms_gemm, "tail": st.ms_tail},
          "features_D": D3, "head_columns": int(st.n_dense_columns),
          "roofline": {"kernel": "sp_bfs_hist<W> (all-sources bitmask BFS + labelled path histogram, one CTA per graph)", "bound": "alu",
                       "achieved": relax / (st.ms_features * 1e-3), "peak": 148 * 128 * sm_clock, "unit": "Floyd-Warshall-equivalent min-plus/s",
                       "frac": relax / (st.ms_features * 1e-3) / (148 * 128 * sm_clock),
                       "note": "algorithmic work = sum n^3 relaxations of the reference's Floyd-Warshall (graph.py:1767-1794); the bitmask BFS does "
                               "n (n + m) / 64 word operations instead, hence a 'fraction' that may exceed what the ALUs could relax one by one",
                       "hbm_GBps_compulsory": (4.0 * (int(b.graph_ptr[-1]) + int(b.row_ptr[-1])) + 4.0 * int(b.graph_ptr[-1])) / (st.ms_features * 1e-3) / 1e9},
          "roofline_gram": {"kernel": GEMM_KERNEL, "bound": "tensor", "achieved": float(n) * (n + 1) * int(st.n_dense_columns) / (st.ms_gemm * 1e-3) / 1e12 if st.ms_gemm > 0 else 0.0,
                            "peak": peak_tf, "unit": "TFLOP/s",
                            "frac": float(n) * (n + 1) * int(st.n_dense_columns) / (st.ms_gemm * 1e-3) / 1e12 / peak_tf if st.ms_gemm > 0 else 0.0,
                            "note": "K-store-bound at this size: 100 MB of fp32 K for %d head columns" % int(st.n_dense_columns)}}
    if with_cpu:
        m = 300
        def mk():
            from grakel.kernels import ShortestPath as RefSP
            return RefSP()
        t, kind = ref_time(mk, X[:m])
        c3["cpu_baseline"] = {"value": m * m / t if t else None, "unit": "pairs/s", "cores": 1, "kind": kind,
                              "sample": "first %d of the 5000 graphs, grakel.ShortestPath().fit_transform (ignores n_jobs), %s s" % (m, "%.1f" % t if t else "-")}
    out["config3_sp"] = c3
    del X
    # ---- config 5
    X = gen_list(2000, 40, 0, attr=16, as_adj=True)
    b = pack(X, "sp", need_labels=True, attributes=True, want_weights=True)
    eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, None, b.weights, b.attrs)
    n = b.n_graphs

    def step5():
        st = eng.spattr_features()
        eng.gram(n, out=False, dtype=np.float64, stats=st, want_diag=False)
        return st
    ms, st = timed(step5, warmup=2)
    D5 = int(st.n_columns)
    tf32_peak = peak_tf / 2.0
    fl = 2.0 * n * n * D5
    c5 = {"workload": "config5: 2000 ER graphs (avg 40 nodes, fp attributes d=16, seed 0), ShortestPathAttr(metric=np.dot)",
          "ms_per_step": ms, "pairs_per_s": n * n / (ms * 1e-3), "feature_dim": D5, "distance_blocks": int(st.level_dims[0]),
          "stages_ms": {"apsp + feature map (fp64)": st.ms_features, "gram (3xTF32 tcgen05, fp64 result)": st.ms_gemm},
          "roofline": {"kernel": "gram_tc_kernel<double,false,tf32> (tcgen05 kind::tf32, hi/lo split: 3 passes over the k range)", "bound": "tensor",
                       "achieved": fl / (st.ms_gemm * 1e-3) / 1e12 if st.ms_gemm > 0 else 0.0, "peak": tf32_peak, "unit": "TFLOP/s",
                       "frac": fl / (st.ms_gemm * 1e-3) / 1e12 / tf32_peak if st.ms_gemm > 0 else 0.0, "passes": 3,
                       "note": "algorithmic 2 N^2 D flops (SURVEY 8d: split passes are not counted); peak = half the measured bf16 burst peak "
                               "(tf32 runs at half the bf16 rate); the launch includes the split, the fp64 fold of the k-chunks and the mirror pass"}}
    if with_cpu:
        m = 5
        def mk5():
            from grakel.kernels import ShortestPathAttr as RefSPA
            return RefSPA()
        t, kind = ref_time(mk5, X[:m])
        c5["cpu_baseline"] = {"value": m * m / t if t else None, "unit": "pairs/s", "cores": 1, "kind": kind,
                              "sample": "first %d of the 2000 graphs (%d unordered pairs), grakel.ShortestPathAttr().fit_transform, %s s" % (m, m * (m + 1) // 2, "%.1f" % t if t else "-")}
    out["config5_spattr"] = c5
    del X
    # ---- WL-OA on the graphs of config 2
    b = pack(X2, "wloa", len_ok=lambda k: k >= 2)
    ids, _ = label_ids(b.labels, None, sort_new=True)
    eng.pack(b.graph_ptr, b.row_ptr, b.col_idx, ids)
    n = b.n_graphs

    def step_oa():
        st = eng.wl_oa_features(H)
        eng.gram(n, out=False, dtype=np.float32, stats=st, want_diag=False)
        return st
    ms, st = timed(step_oa)
    oa = {"workload": "WL-OA (n_iter=5) on the graphs of config 2", "ms_per_step": ms, "pairs_per_s": n * n / (ms * 1e-3),
          "stages_ms": {"wl + unary expansion": st.ms_features, "columns+panel": st.ms_panel, "gram_gemm": st.ms_gemm, "tail": st.ms_tail},
          "unary_columns": int(st.n_columns), "unary_entries": int(st.n_entries), "head_columns": int(st.n_dense_columns),
          "roofline": {"kernel": GEMM_KERNEL, "bound": "tensor", "achieved": float(n) * (n + 1) * int(st.n_dense_columns) / (st.ms_gemm * 1e-3) / 1e12 if st.ms_gemm > 0 else 0.0,
                       "peak": peak_tf, "unit": "TFLOP/s",
                       "frac": float(n) * (n + 1) * int(st.n_dense_columns) / (st.ms_gemm * 1e-3) / 1e12 / peak_tf if st.ms_gemm > 0 else 0.0}}
    if with_cpu:
        m = 150
        def mko():
            from grakel.kernels import WeisfeilerLehmanOptimalAssignment as RefOA
            return RefOA(n_iter=H)
        t, kind = ref_time(mko, X2[:m])
        oa["cpu_baseline"] = {"value": m * m / t if t else None, "unit": "pairs/s", "cores": 1, "kind": kind,
                              "sample": "first %d graphs, grakel.WeisfeilerLehmanOptimalAssignment(n_iter=5).fit_transform, %s s" % (m, "%.1f" % t if t else "-")}
    out["config2_wloa"] = oa
    return out


def run_config4(eng, n4, rank, world, local, dist, torch, _lib, steps):
    """BASELINE config 4: WL-subtree (h=5) Gram of n4 graphs, row-tiled over the ranks (GK_DIST tiles, mirrored halves
    over NVLink) and assembled on EVERY rank by the in-place all-gather of gk_gram(GK_DIST_GATHER).  Returns rank 0's
    report; parity = prefix of the assembled matrix against a single-GPU run, checksum equal on all ranks."""
    gp, rp, ci, lab = pack_workload(n4)
    eng.pack(gp, rp, ci, lab)
    rb, re_ = eng.comm_rows(n4)
    ts, t_feat, t_gemm, t_tail = [], [], [], []
    for it in range(2 + steps):
        dist.barrier()
        torch.cuda.synchronize()
        eng.event_record(2)
        s = eng.wl_features(H)
        eng.gram(n4, out=False, dtype=np.float32, row_range=(rb, re_), stats=s, want_diag=False, gather=True)
        eng.event_record(3)
        ms = eng.event_elapsed(2, 3)
        if it >= 2:
            ts.append(ms); t_feat.append(s.ms_features); t_gemm.append(s.ms_panel + s.ms_gemm); t_tail.append(s.ms_tail)
    tt = torch.tensor([float(np.mean(ts))], device="cuda")
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ptr, rows, cols, ld, _ = eng.result_device()

    class _View:  # zero-copy torch view of the library-owned fp32 result
        __cuda_array_interface__ = {"data": (ptr, False), "shape": (rows, ld), "typestr": "<f4", "version": 3}
    Kd = torch.as_tensor(_View(), device="cuda")[:, :cols]
    cs = 0.0
    for r0 in range(0, rows, 4096):  # fp64 checksum in row chunks
        cs += float(Kd[r0:r0 + 4096].double().sum().item())
    Kfull = Kd[: min(2048, n4), : min(2048, n4)].cpu().numpy()
    cst = torch.tensor([cs], device="cuda", dtype=torch.float64)
    lo, hi = cst.clone(), cst.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    ok_prefix = None
    if rank == 0:
        p1 = min(2048, n4)
        e1 = _lib.Engine(local)
        e1.pack(*pack_workload(p1))
        s1 = e1.wl_features(H)
        K1, _, _ = e1.gram(p1, dtype=np.float32, stats=s1, want_diag=False)
        ok_prefix = bool(np.array_equal(Kfull[:p1, :p1], K1))
        del e1
    ms = float(tt.item())
    from grakel_b200.dist import TILE, rows_per_rank
    per = rows_per_rank(n4, world, TILE)
    gather_bytes_in = (world - 1) * per * ld * 4
    t_other = float(np.mean(t_feat)) + float(np.mean(t_gemm))
    t_gather = float(np.mean(t_tail))  # barrier + tail + all-gather (tev[7] -> end of the device work)
    return {"workload": f"config4: {n4} ER graphs (avg {NBAR} nodes, 7 labels, seed {SEED}), WL-subtree h={H}, K on every rank",
            "n_gpus": world, "ms_per_step": ms, "pairs_per_s": n4 * n4 / (ms * 1e-3),
            "ms_relabel_replicated": float(np.mean(t_feat)), "ms_columns_panel_gemm": float(np.mean(t_gemm)),
            "ms_barrier_tail_allgather": t_gather,
            "allgather_bytes_in_per_rank": int(gather_bytes_in),
            "allgather_GBps_in_per_rank": gather_bytes_in / (t_gather * 1e-3) / 1e9 if t_gather > 0 else None,
            "nvlink5_peak_GBps_per_direction": 900.0,
            "result_bytes_per_rank": int(world * per * ld * 4),
            "checksum": cs, "checksum_equal_on_all_ranks": bool(lo.item() == hi.item()),
            "prefix_equals_single_gpu": ok_prefix,
            "note": "the all-gather moves (G-1)/G of a 4 N^2-byte matrix INTO every GPU: at NVLink-5 rates that is longer than the "
                    "whole compute, so the step is bandwidth-bound by construction; compute is what hides behind it, not the reverse"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--graphs", type=int, default=N_GRAPHS)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-paths", action="store_true", help="skip configs 3 / 5 / WL-OA")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy: a seeded sample of rows of K from "
                         "the device-resident pass (K_rows, fp32) and from the C-ABI end-to-end call (K_e2e_rows, fp64), "
                         "their global row numbers (K_row_ids) and the whole diagonal (K_diag); rank 0's rows at N > 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    # rank 0 prints exactly one JSON line on stdout.  Libraries write there too (NCCL prints its version banner
    # at NCCL_DEBUG=VERSION and above, straight to file descriptor 1), so descriptor 1 is pointed at stderr for the
    # whole run and the JSON line goes to a private duplicate of the original stdout.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0)
    numa_node = bind_to_gpu_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from grakel_b200 import _lib
    eng = _lib.Engine(local)

    # weak scaling: ordered pairs per GPU stay fixed (N = 10 000 * sqrt(world) graphs), every rank
    # produces the same number of K entries; N = 1 is exactly BASELINE config 2
    n = int(round(args.graphs * np.sqrt(world)))
    gp, rp, ci, lab = pack_workload(n)
    V, E = int(gp[-1]), int(rp[-1])
    if world > 1:
        # C-ABI communicator (gk_comm_init): NCCL id broadcast over torch.distributed, everything else in the library
        from grakel_b200.dist import comm_init
        comm_init(eng)
        rb, re_ = eng.comm_rows(n)
    else:
        rb, re_ = 0, n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------ device-resident steps
    eng.pack(gp, rp, ci, lab)
    st = _lib.GkStats()

    def step():
        if world == 1:
            # one C call for the whole pass (gk_wl_gram): features, column statistics, head/tail decision on the
            # device, panel, GEMM, tail -- a single host synchronisation at the end
            return eng.wl_gram(H, out=False, dtype=np.float32)[2]
        s = eng.wl_features(H)
        eng.gram(n, out=False, dtype=np.float32, row_range=(rb, re_), stats=s, want_diag=False, dist=True)
        return s

    gemm_ms, feat_ms, panel_ms, tail_ms, launches = [], [], [], [], 0
    # the clock sampler (an nvidia-smi process) starts BEFORE the warm-up: its start-up talks to the driver for tens of
    # milliseconds and would otherwise sit on top of a timed region that is itself only ~15 ms long
    with ClockSampler(local) as clk:
        n_warm = max(args.warmup, 200)  # untimed; the same count on every rank (the multi-GPU step is collective)
        for _ in range(n_warm):
            st = step()
        barrier()
        eng.event_record(0)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            st = step()
            gemm_ms.append(st.ms_gemm)
            feat_ms.append(st.ms_features)
            panel_ms.append(st.ms_panel)
            tail_ms.append(st.ms_tail)
            launches += int(st.kernel_launches + st.gemm_launches)
        eng.event_record(1)
        dev_ms = eng.event_elapsed(0, 1)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
    dump, rows = None, None
    if args.dump_outputs and rank == 0:
        # K of the last timed step is still in the library-owned device buffer; later calls overwrite it
        Kf = np.empty((re_ - rb, n), dtype=np.float32)
        eng.fetch(Kf)
        rows = dump_rows(re_ - rb, n)
        dump = {"K_rows": Kf[rows], "K_row_ids": (rb + rows).astype(np.float64),
                "K_diag": Kf[np.arange(re_ - rb), rb + np.arange(re_ - rb)]}
        del Kf
    t_ms = torch.tensor([dev_ms], device="cuda")
    stages_per_rank = None
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        mine = {"rank": rank, "ms_per_step": dev_ms / args.steps, "wl_features": float(np.mean(feat_ms)), "columns+panel(+barrier)": float(np.mean(panel_ms)),
                "gram_gemm": float(np.mean(gemm_ms)), "barrier+tail": float(np.mean(tail_ms)), "tiles": int(st.gemm_tiles)}
        stages_per_rank = [None] * world
        dist.all_gather_object(stages_per_rank, mine)
    ms_step = float(t_ms.item()) / args.steps
    value = n * n / (ms_step * 1e-3)

    # ------------------------------------------------ end to end through the C-ABI
    e2e = None
    if not args.no_e2e:
        kr = re_ - rb if world > 1 else n
        Kh = torch.empty((kr, n), dtype=torch.float64).pin_memory().numpy()
        gp_p, rp_p, ci_p, lab_p = [torch.from_numpy(a).pin_memory().numpy() for a in (gp, rp, ci, lab)]

        def e2e_step():
            if world == 1:
                return eng.wl_fit_transform_raw(gp_p, rp_p, ci_p, lab_p, H, Kh)
            eng.pack(gp_p, rp_p, ci_p, lab_p)
            s = eng.wl_features(H)
            eng.gram(n, out=Kh, dtype=np.float64, row_range=(rb, re_), stats=s, want_diag=False, dist=True)
            return s

        for _ in range(int(os.environ.get("GRAKEL_B200_E2E_WARMUP", "4"))):
            e2e_step()
        barrier()
        import gc
        if os.environ.get("GRAKEL_B200_BENCH_GC", "1") == "0":
            gc.collect(); gc.disable()
        t0 = time.perf_counter()
        per_step = []
        for _ in range(args.steps):
            t1 = time.perf_counter()
            es = e2e_step()
            per_step.append((time.perf_counter() - t1) * 1e3)
        barrier()
        e2e_t = torch.tensor([(time.perf_counter() - t0) / args.steps], device="cuda")
        if dump is not None:
            dump["K_e2e_rows"] = Kh[rows]  # before the breakdown below writes Kh again
        if world > 1:
            dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        e2e = {"value": n * n / float(e2e_t.item()), "unit": "pairs/s",
               "h2d_bytes_per_step": int(gp.nbytes + rp.nbytes + ci.nbytes + lab.nbytes),
               "d2h_bytes_per_step": int(kr * n * 8), "ms_per_step": float(e2e_t.item()) * 1e3,
               "ms_per_step_min_median_max": [float(np.min(per_step)), float(np.median(per_step)), float(np.max(per_step))],
               "ms_each_step": [round(float(x), 2) for x in per_step],
               "api": "gk_wl_fit_transform (C-ABI), pinned host CSR in, pinned float64 K out (fp32 upper triangle over "
                      "PCIe, widened + mirrored by host threads)",
               "pcie_d2h_bytes_per_step": int(n * (n + 1) // 2 * 4) if world == 1 else int(kr * n * 4),
               "last_step_ms": {"h2d+pack": es.ms_h2d, "features": es.ms_features, "columns+panel": es.ms_panel,
                                "gemm": es.ms_gemm, "tail": es.ms_tail, "d2h": es.ms_d2h}}
        # host-side breakdown of one e2e step (wall clock, separate C calls)
        tb = {}
        t0 = time.perf_counter(); eng.pack(gp_p, rp_p, ci_p, lab_p); tb["pack_csr(host scans + H2D)"] = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter(); s_ = eng.wl_features(H); tb["wl_features"] = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter(); eng.gram(n, out=Kh, dtype=np.float64, row_range=(rb, re_) if world > 1 else None, stats=s_, want_diag=False, dist=world > 1)
        tb["gram + D2H"] = (time.perf_counter() - t0) * 1e3
        e2e["host_wall_ms"] = tb
        if rank == 0 and world == 1 and n == N_GRAPHS:
            assert float(Kh.sum()) == 22925628586.0, "K checksum differs from the reference golden"

    # ------------------------------------------------ multi-GPU: parity of the tiled result, BASELINE config 4
    dist_check, config4 = None, None
    if world > 1:
        # every rank's row block against rows of a single-GPU run of a prefix (an entry depends on its two graphs only)
        eng.gram(n, out=False, dtype=np.float32, row_range=(rb, re_), stats=st, want_diag=False, dist=True)
        p1 = min(1536, n)
        ok = True
        if rb < p1:
            blk = np.empty((min(re_, p1) - rb, n), dtype=np.float32)
            full = np.empty((re_ - rb, n), dtype=np.float32)
            eng.fetch(full)
            blk[:] = full[: blk.shape[0]]
            e1 = _lib.Engine(local)
            e1.pack(*pack_workload(p1))
            s1 = e1.wl_features(H)
            K1, _, _ = e1.gram(p1, dtype=np.float32, stats=s1, want_diag=False)
            ok = bool(np.array_equal(blk[:, :p1], K1[rb:rb + blk.shape[0]]))
            del e1
        okt = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        dist_check = {"row_blocks_equal_single_gpu_prefix": bool(okt.item() == 1), "prefix": p1}
        n4 = int(os.environ.get("GRAKEL_B200_CONFIG4_GRAPHS", "50000" if world == 8 else "0"))
        if n4 > 0:
            config4 = run_config4(eng, n4, rank, world, local, dist, torch, _lib, args.steps)

    # ------------------------------------------------ end to end through the Python API (SURVEY 8d T_e2e)
    e2e_api, paths = None, None
    if not args.no_e2e and world == 1 and rank == 0:
        from grakel_b200 import WeisfeilerLehman
        _lib.set_default_device(local)
        t0 = time.perf_counter()
        X = gen_list(n)
        t_gen = time.perf_counter() - t0
        ts = []
        for i in range(2 + args.steps):
            t0 = time.perf_counter()
            est = WeisfeilerLehman(n_iter=H)
            Ka = est.fit_transform(X)
            ts.append(time.perf_counter() - t0)
            if i == 0:
                assert Ka.dtype == np.float64 and Ka.shape == (n, n) and Ka.flags.c_contiguous
                if n == N_GRAPHS:
                    assert float(Ka.sum()) == 22925628586.0, "K checksum (Python API) differs from the reference golden"
            del Ka
        # host-side split of one more call
        from grakel_b200 import packing
        t0 = time.perf_counter(); blk = packing.pack(X, "wl", len_ok=lambda k: k >= 2); t_pack = time.perf_counter() - t0
        t0 = time.perf_counter(); packing.label_ids(blk.labels, None, True); t_ids = time.perf_counter() - t0
        t_api = float(np.mean(ts[2:]))
        e2e_api = {"value": n * n / t_api, "unit": "pairs/s", "ms_per_step": t_api * 1e3,
                   "api": f"grakel_b200.WeisfeilerLehman(n_iter={H}).fit_transform(list of [edge dict, label dict]) -> fresh float64 ndarray",
                   "first_call_ms": ts[0] * 1e3, "min_ms": float(np.min(ts[2:])) * 1e3,
                   "host_ms": {"pack(list -> CSR)": t_pack * 1e3, "label_ids": t_ids * 1e3},
                   "result_buffer": "pooled huge-page host mapping (gk_host_alloc); first_call_ms includes faulting it in",
                   "list_build_ms_not_timed": t_gen * 1e3}
        if not args.no_paths:
            try:
                paths = other_paths(eng, local, X, not args.no_cpu, args.steps)
            except Exception as e:  # the headline line must survive a failure of the secondary measurements
                paths = {"error": repr(e)}
        del X

    def leave():
        """Multi-rank exit: every rank has finished its device work (barrier), rank 0 has printed; the process then ends
        without tearing down two NCCL communicators, IPC mappings and the CUDA context in interpreter-finalisation order
        (one exit-time SIGSEGV in ~5 runs of the 2-GPU job otherwise; gk_comm_destroy / Engine.close remain the API)."""
        barrier()
        real_stdout.flush()
        sys.stderr.flush()
        os._exit(0)

    if rank != 0:
        if world > 1:
            leave()
        return

    # the tensor-bound configuration of the same GEMM kernel (every shared column dense), for the
    # "GEMM % of tensor-core peak" half of the BASELINE metric
    dense = None
    if world == 1:
        ds = _lib.GkStats()
        dms = []
        for i in range(3 + 5):
            eng.gram(n, out=False, dtype=np.float32, stats=ds, want_diag=False, dense_all=True)
            if i >= 3:
                dms.append(ds.ms_gemm)
        dflops = float(n) * (n + 1) * int(ds.n_dense_columns)
        dense = {"dense_columns": int(ds.n_dense_columns), "ms_per_launch": float(np.mean(dms)),
                 "flops_per_launch": dflops, "achieved_tflops": dflops / (np.mean(dms) * 1e-3) / 1e12}
    peak_tf, peak_hbm, peak_src = peaks()
    Dc = int(st.n_dense_columns)
    g_ms = float(np.mean(gemm_ms))
    # multi-GPU: the SYRK tiles are shared between the ranks (each computed once); rank 0's share = its tile count
    flops = (2.0 * 256 * 256 * Dc * int(st.gemm_tiles)) if world > 1 else (float(n) * (n + 1) * Dc)
    achieved = flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    line = {
        "metric": "graph-pairs/sec, N x N WL-subtree (h=5) Gram", "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "warmup_run": n_warm, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 x bf16 -> f32 (exact integers)",
        "data": "synthetic",
        "config": {"workload": f"config2: {n} ER graphs (avg {NBAR} nodes, 7 labels, seed {SEED}), WL-subtree h={H}",
                   "vertices": V, "directed_edges": E, "feature_columns": int(st.n_columns), "nnz": int(st.n_entries),
                   "dense_columns_Dc": Dc,
                   "parallelism": (f"rows of K tiled over {world} GPUs (gk_comm_init / GK_DIST): SYRK tiles shared, mirrored halves "
                                   f"stored into the owner's row block over NVLink by the GEMM epilogue; CSR + relabel replicated")
                   if world > 1 else "1 GPU",
                   "host_numa_node": numa_node,
                   "l2": "per-step working set (panel %.0f MB + K %.0f MB) exceeds the 126 MB L2" %
                         (n * ((Dc + 63) // 64 * 64) * 2 / 1e6, (re_ - rb if world > 1 else n) * n * 4 / 1e6)},
        "clocks": clk.summary(),
        "e2e": e2e,
        "e2e_api": e2e_api,
        "other_paths": paths,
        "stages_ms_per_rank": stages_per_rank,
        "dist_check": dist_check,
        "config4": config4,
        "gpu_launches": launches,
        "roofline": {"kernel": GEMM_KERNEL, "bound": "tensor",
                     "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                     "traffic": measured_traffic("hybrid") if (world == 1 and n == N_GRAPHS) else None,
                     "traffic_unit": "bytes/launch (ncu dram read+write, profiles/traffic.json)",
                     "peak_source": peak_src, "flops_per_launch": flops, "ms_per_launch": g_ms,
                     "share_of_step": g_ms / ms_step},
        "roofline_store": {"kernel": "gram_tc_kernel epilogue (K written once, fp32)", "bound": "hbm",
                           "achieved": (re_ - rb if world > 1 else n) * n * 4 / (g_ms * 1e-3) / 1e9 if g_ms > 0 else 0.0,
                           "peak": peak_hbm, "unit": "GB/s",
                           "frac": ((re_ - rb if world > 1 else n) * n * 4 / (g_ms * 1e-3) / 1e9 / peak_hbm) if g_ms > 0 else 0.0},
        # the other large kernel of a step, against the HBM roof with SURVEY 8(d)'s algorithmic bytes: K1 relabel
        # (12V + 4E + 4) + K2 compaction 16V per iteration, K3 histogram 4V + 8 nnz_i per level.  It is bound by
        # dependent L2 operations and two grid barriers per level, not by bytes (DESIGN.md 4.1) -- the fraction says so.
        "roofline_relabel": (lambda b, ms: {"kernel": "wl_fused2_kernel (all WL levels, one persistent cooperative launch, one grid barrier per level)", "bound": "hbm",
                                            "algorithmic_bytes": b, "ms_per_launch": ms, "achieved": b / (ms * 1e-3) / 1e9,
                                            "peak": peak_hbm, "unit": "GB/s", "frac": b / (ms * 1e-3) / 1e9 / peak_hbm,
                                            "share_of_step": ms / ms_step})(
            float(H * (12 * V + 4 * E + 4 + 16 * V) + (H + 1) * 4 * V + 8 * int(st.n_entries)), float(np.mean(feat_ms))),
        "stages_ms": {"wl_features": float(np.mean(feat_ms)), "columns+panel": float(np.mean(panel_ms)),
                      "gram_gemm": g_ms, "tail_pairs": float(np.mean(tail_ms)), "wall_ms_per_step": wall_ms / args.steps},
        "head_tail": {"threshold_T": int(st.threshold), "head_columns": Dc, "tail_columns": int(st.n_tail_columns),
                      "tail_pair_updates": int(st.tail_updates)},
        "dense_gemm_mode": dense,
    }
    if not args.no_cpu and world == 1:
        os.sched_setaffinity(0, all_cpus)  # the CPU leg may use every core of the box
        line["cpu_baseline"] = cpu_baseline_obj(cpu_arm(steps=1, budget_s=12.0), n)
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a))
        print("bench: wrote %s to %s" % (", ".join(sorted(dump)), args.dump_outputs), file=sys.stderr)
    print(json.dumps(line), file=real_stdout, flush=True)
    if world > 1:
        leave()


if __name__ == "__main__":
    main()
