/* grakel_b200 -- C-ABI of the B200-native graph-kernel Gram engine.
 *
 * This header is the drop-in boundary for the hot path of ysig/GraKeL
 * (reference v0.1.11):  N x N Gram matrices of the Weisfeiler-Lehman subtree
 * kernel and the Shortest-Path kernels.  The reference has no FFI on this path
 * (it is pure Python + numpy/scipy); its only native precedent is the Cython
 * `cdef extern` block grakel/kernels/_c_functions/header.pxd:1-4 over
 * include/functions.hpp:4-5 (raw pointers + sizes, results by out-pointer).
 * The entry points below follow that convention: extern "C", plain pointers and
 * sizes, caller-owned host buffers, library-owned device memory behind an
 * opaque handle, int status return (0 = ok, <0 = error; text via gk_last_error).
 *
 * What each entry point replaces in the reference:
 *
 *   gk_pack_csr          Graph.__init__/build_graph/_import_*  (graph.py:147-230,
 *                        912-1053) + get_edge_dictionary/get_labels
 *                        (graph.py:1182-1204, 689-772) -- after the Python layer
 *                        has normalised the input into one CSR block.
 *   gk_wl_features       WeisfeilerLehman.parse_input relabel loop
 *                        (weisfeiler_lehman.py:199-258) + VertexHistogram.parse_input
 *                        (vertex_histogram.py:57-154) for every level.
 *   gk_sp_features       Graph.build_shortest_path_matrix / floyd_warshall / dijkstra
 *                        (graph.py:588-687, 1712-1794) + ShortestPath.parse_input
 *                        pair histogram (shortest_path.py:468-490).
 *   gk_wl_sp_features    the WL level loop with ShortestPath as base kernel
 *                        (weisfeiler_lehman.py:260-270, "WL-SP" of doc/benchmarks).
 *   gk_wl_oa_features    WeisfeilerLehmanOptimalAssignment.parse_input + the O(N^2) Python loop of
 *                        histogram intersections (weisfeiler_lehman_optimal_assignment.py:78-229,
 *                        257-266, 433-437).
 *   gk_nh_features, gk_nh_gram, gk_nh_labels
 *                        NeighborhoodHash.fit / transform / pairwise_operation
 *                        (neighborhood_hash.py:91-341, 392-570), see below.
 *   gk_spattr_features   ShortestPathAttr.parse_input + the bilinear pair kernel
 *                        (shortest_path.py:77-164) as an explicit feature map.
 *   gk_gram              VertexHistogram._calculate_kernel_matrix
 *                        (vertex_histogram.py:156-184), np.sum over levels
 *                        (weisfeiler_lehman.py:270), np.dot(phi, phi.T)
 *                        (shortest_path.py:404 / :312), the diagonals
 *                        (vertex_histogram.py:186-219, shortest_path.py:320-368) and
 *                        the normalisation (weisfeiler_lehman.py:324-327, 494-498;
 *                        shortest_path.py:314-316, 407-408).
 *   gk_wl_fit_transform, gk_sp_fit_transform
 *                        one-call forms of the above with HOST buffers in and out:
 *                        WeisfeilerLehman.fit_transform (weisfeiler_lehman.py:292-328),
 *                        ShortestPath.fit_transform (shortest_path.py:370-410).
 *
 * Fit + transform.  The reference keeps per-level dictionaries at fit time and
 * re-applies them to new graphs (weisfeiler_lehman.py:330-500).  Here the same
 * result is obtained by packing the fitted graphs X followed by the new graphs Y
 * into one block and relabelling them jointly: a Y feature is "seen" iff its
 * column also occurs in an X graph, unseen columns contribute nothing to
 * K[y, x] and are counted in Y's self-similarity, exactly as
 * vertex_histogram.py:179 / :211-217 and shortest_path.py:312 / :365 do.
 * `n_fit` below is the number of leading graphs that form X.
 */
#ifndef GRAKEL_B200_H
#define GRAKEL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gk_handle gk_handle;

/* output element type of K */
#define GK_F32 0
#define GK_F64 1

/* gk_gram flags */
#define GK_NORMALIZE 1   /* K_ij / sqrt(d_i d_j) in fp64 (weisfeiler_lehman.py:326) */
#define GK_NAN_TO_NUM 2  /* WL only: np.nan_to_num on the normalised matrix          */
#define GK_GRAM_SIMT 4   /* use the exact int64 CUDA-core Gram (verification / wide counts) */
#define GK_OUT_DEVICE 8  /* K_out is a DEVICE pointer (e.g. a torch tensor)          */
#define GK_FULL_TILES 16 /* square case: compute every tile, no mirroring            */
#define GK_DENSE_ALL 32  /* contract every shared column on the tensor cores (no sparse tail) */

/* gk_sp_features flags */
#define GK_SP_WITH_LABELS 1
#define GK_SP_KEEP_DIST 2    /* keep fp64 APSP matrices for gk_sp_distances (tests) */
#define GK_SP_DIJKSTRA_ORDER 4 /* real-valued weights: path sums associate as in dijkstra (graph.py:1712-1764), not as in
                                floyd_warshall (:1767-1794); integer-valued distances are the same either way */

/* error codes */
#define GK_OK 0
#define GK_ERR_CUDA -1
#define GK_ERR_ARG -2
#define GK_ERR_STATE -3
#define GK_ERR_RANGE -4   /* a count or Gram value leaves the exactly representable range */
#define GK_ERR_UNSUPPORTED -5

/* Per-call statistics (all optional; pass NULL).  Times are CUDA-event
 * milliseconds on the handle's stream. */
typedef struct gk_stats {
  int64_t n_graphs, n_vertices, n_edges;
  int64_t n_levels;          /* WL: h+1 */
  int64_t level_dims[64];    /* WL: distinct labels per level (= D_i of the reference) */
  int64_t n_columns;         /* total feature columns D */
  int64_t n_entries;         /* nnz of the feature block */
  int64_t n_dense_columns;   /* D_c: "head" columns contracted by the tensor-core GEMM */
  int64_t n_tail_columns;    /* low-frequency columns contracted by exact atomic pair updates */
  int64_t tail_updates;      /* number of those pair updates */
  int64_t threshold;         /* T: columns in more than T graphs are head columns */
  int64_t max_count;         /* largest single feature count */
  int64_t max_diag;          /* largest self-similarity */
  int64_t hash_retries;      /* WL: relabel passes repeated after a detected hash collision */
  int64_t gram_path;         /* 1 = tcgen05 bf16 tensor-core GEMM, 2 = exact int64 CUDA-core Gram, 3 = no contracted columns */
  int64_t gemm_tiles;        /* output tiles computed */
  int64_t gemm_launches;     /* kernels launched by the last gk_gram */
  int64_t kernel_launches;   /* kernels launched by the last features call */
  float ms_h2d, ms_features, ms_panel, ms_gemm, ms_tail, ms_d2h, ms_total;
} gk_stats;

int gk_version(void);
const char* gk_last_error(void);

int gk_create(int device_ordinal, gk_handle** out);
int gk_destroy(gk_handle* h);
int gk_sync(gk_handle* h);

/* Upload one packed CSR block (host pointers).
 *   graph_ptr[n_graphs+1]  vertex offsets, graph g owns vertices [graph_ptr[g], graph_ptr[g+1])
 *   row_ptr[V+1]           out-edge offsets per vertex (V = graph_ptr[n_graphs])
 *   col_idx[E]             GLOBAL vertex id of each out-neighbour (same graph)
 *   labels[V]              dense non-negative id of the vertex label (level 0), or NULL
 *   weights[E]             edge weights (fp64) or NULL for unit weights
 *   attrs[V*attr_dim]      fp64 node attributes or NULL                                  */
int gk_pack_csr(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr, const int32_t* row_ptr,
                const int32_t* col_idx, const int32_t* labels, const double* weights,
                const double* attrs, int32_t attr_dim);

/* Build the sparse feature block of the packed graphs on the device. */
int gk_wl_features(gk_handle* h, int32_t n_iter, gk_stats* stats);
int gk_sp_features(gk_handle* h, int32_t flags, gk_stats* stats);
int gk_spattr_features(gk_handle* h, int32_t flags /* GK_SP_DIJKSTRA_ORDER or 0 */, gk_stats* stats);
/* WeisfeilerLehman(base_graph_kernel=ShortestPath), weisfeiler_lehman.py:260-270 over
 * shortest_path.py:370-410: n_iter WL rounds, then the labelled shortest-path histogram of every
 * level in one feature block (level-unique label ids => disjoint columns), so that one gk_gram
 * returns the sum of the per-level matrices. */
int gk_wl_sp_features(gk_handle* h, int32_t n_iter, int32_t flags, gk_stats* stats);

/* WeisfeilerLehmanOptimalAssignment (weisfeiler_lehman_optimal_assignment.py:78-279): the WL feature
 * block of all levels in unary ("thermometer") form -- column c with count k becomes k columns holding 1
 * -- so that gk_gram's dot products are the histogram intersections sum_c min(Hs[i,c], Hs[j,c]) of
 * :257-266 / :433-437, the self similarities the row sums of :459-461, exactly (integers). */
int gk_wl_oa_features(gk_handle* h, int32_t n_iter, gk_stats* stats);

/* NeighborhoodHash (neighborhood_hash.py:91-206, 239-322, 324-341, 392-570).
 *
 * gk_nh_features replaces the R applications of NH_ (neighborhood_hash.py:191-201, 307-310: the simple hash of
 * :392-418 or, with GK_NH_COUNT_SENSITIVE, the count-sensitive hash of :420-504) and prepares every level for the
 * merge of nh_compare_labels (:531-570) as a unary-expanded histogram (the intersection c_r is a dot product).
 *   labels0[V]  level-0 hashed label of every packed vertex (_labels_hash_dict[label], :189-194), -1 = None
 *               (a transform label unseen at fit time, :299-300)
 *   bits        1 .. 63 (the reference's `bits`, :83-88)
 * stats: n_levels = R, level_dims[r] = distinct non-None labels of level r, n_columns / n_entries = columns / entries
 * of the R expanded blocks, ms_features = the relabel, ms_panel = the level histograms and expansions.
 *
 * gk_nh_gram replaces pairwise_operation over all pairs (:324-341, kernel.py:257-284):
 * K[i, j] = sum(a_0 .. a_{R-1}) / R with a_r = c_r / (double)(n_i + n_j - c_r), n = the graph's packed vertex count
 * (None vertices included), the sum compensated as CPython's built-in sum() adds floats (Neumaier, CPython >= 3.12).  fp64 only.  n_fit == n_graphs: the square, symmetric fit_transform matrix;
 * n_fit < n_graphs: [(n_graphs - n_fit) x n_fit], rows = Y graphs.  flags: GK_OUT_DEVICE (K_out is a device pointer,
 * row pitch ld), GK_GRAM_SIMT / GK_DENSE_ALL select the path of the per-level integer Grams.  K_out == NULL keeps
 * K on the device (gk_result_device / gk_fetch).  stats: ms_gemm = the R level Grams, ms_tail = the fp64 combine,
 * ms_d2h = the copy to the host; gram_path / threshold / n_dense_columns are those of the last level.
 *
 * gk_nh_labels: the u64 labels of level `level` (0 .. R-1) per packed vertex, UINT64_MAX = None (tests). */
#define GK_NH_COUNT_SENSITIVE 1
int gk_nh_features(gk_handle* h, int32_t R, int32_t bits, int32_t flags, const int64_t* labels0, gk_stats* stats);
int gk_nh_gram(gk_handle* h, int64_t n_fit, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld,
               gk_stats* stats);
int gk_nh_labels(gk_handle* h, int32_t level, uint64_t* out);

/* Gram matrix of the current feature block.
 *   n_fit == n_graphs : K is [n_graphs x n_graphs]                      (fit_transform)
 *   n_fit <  n_graphs : K is [(n_graphs-n_fit) x n_fit], rows = Y graphs (transform)
 *   row_begin,row_end : only rows [row_begin,row_end) of K are computed and written
 *                       (multi-GPU row tiling); K_out points at row `row_begin`.
 *   K_out may be NULL (result stays on the device; see gk_fetch).
 *   xdiag[n_fit], ydiag[n_graphs-n_fit] : self-similarities (fp64, host) or NULL.      */
int gk_gram(gk_handle* h, int64_t n_fit, int32_t flags, int64_t row_begin, int64_t row_end,
            void* K_out, int32_t out_dtype, int64_t ld, double* xdiag, double* ydiag,
            gk_stats* stats);

/* Row map: packed graph g contributes to row row_of_graph[g] of K (n_rows rows in total; gk_gram's
 * n_fit / row ranges / diagonals then count rows).  Used by CoreFramework (core_framework.py:177-223):
 * the k-core subgraphs of every graph are packed as separate graphs with level-tagged labels (their
 * feature columns are therefore disjoint) and mapped back to their graph's row, so one Gram equals the
 * reference's scatter-add of one base-kernel matrix per core level.  Cleared by gk_pack_csr;
 * n_rows <= 0 restores the identity. */
int gk_set_row_map(gk_handle* h, int64_t n_rows, const int32_t* row_of_graph);

/* ---- multi-GPU: one process per GPU, one handle per process (SURVEY 8b/8e: the N x N output tiled over GPUs,
 * a final all-gather over NVLink only when the whole matrix must live on every device).
 * Every rank packs the same block and runs the same feature call (the relabel prologue is replicated: the whole
 * graph set is a few tens of MB); gk_gram with GK_DIST then computes the rank's row block [gk_comm_rows) of K.
 * The SYRK tiles are shared between the ranks -- each off-diagonal 256 x 256 tile is computed once, by one of
 * the two ranks that own its rows / columns -- and the GEMM epilogue stores the mirrored half straight into the
 * owning rank's row block through peer-mapped memory (CUDA IPC over NVLink), so the exchange overlaps the MMA
 * tile by tile and no rank recomputes what another one has.  NCCL carries the bootstrap, the handle exchange,
 * the two barriers of a call and, with GK_DIST_GATHER, the in-place all-gather of the finished row blocks
 * (BASELINE config 4: the full fp32 K on every rank, library-owned: gk_result_device / gk_fetch).
 * gk_comm_unique_id: rank 0 creates the 128-byte NCCL id, the application hands it to every rank (any channel).
 * All of these are collective: every rank calls them in the same order with the same sizes. */
#define GK_DIST 64          /* gk_gram flag: row block of this rank, tiles shared with the peers */
#define GK_DIST_GATHER 128  /* gk_gram flag: GK_DIST + all-gather, the full K stays on every device */
int gk_comm_unique_id(void* out128);
int gk_comm_init(gk_handle* h, int32_t nranks, int32_t rank, const void* unique_id128);
int gk_comm_destroy(gk_handle* h);  /* collective; gk_destroy calls it */
/* the row block of this rank: ceil(n_rows / nranks) rounded up to 256 rows per rank (identity without a communicator) */
int gk_comm_rows(gk_handle* h, int64_t n_rows, int64_t* row_begin, int64_t* row_end);
/* library-owned device result of the last gk_gram (valid until the next call on the handle) */
int gk_result_device(gk_handle* h, void** ptr, int64_t* rows, int64_t* cols, int64_t* ld, int32_t* dtype);
/* host-only (tests): the {row, column} tile list gk_gram(GK_DIST) gives rank `rank` of `nranks` */
int gk_selftest_dist_tiles(int64_t n_rows, int32_t nranks, int32_t rank, int32_t* tiles_xy, int64_t cap, int64_t* n_tiles);

/* Copy rows of the device-resident K of the last gk_gram to the host. */
int gk_fetch(gk_handle* h, void* K_out, int32_t out_dtype, int64_t ld);

/* WL inspection (parity tests): compressed label of every vertex at `level`
 * (dense ids, first-occurrence order) */
int gk_wl_labels(gk_handle* h, int32_t level, int32_t* out);

/* APSP matrix of graph g (n x n fp64, inf = unreachable): after gk_sp_features(GK_SP_KEEP_DIST), or after
 * gk_spattr_features -- the (S, phi) tuples of shortest_path.py:77-129 that ShortestPathAttr with a user `metric`
 * contracts pair by pair on the host (grakel/kernels/shortest_path.py:130-164, kernel.py:236-296) */
int gk_sp_distances(gk_handle* h, int64_t g, double* out);

/* WL features + square Gram of the packed block in ONE call: gk_wl_features followed by gk_gram(n_fit = N)
 * (weisfeiler_lehman.py:199-328 for fit_transform).  When the request is the plain square case with an fp32 device
 * result (flags 0 / GK_OUT_DEVICE / GK_DENSE_ALL; K_out NULL = library-owned, a device pointer, or a float64 host
 * matrix) the whole pass is enqueued without a host synchronisation in the middle: the head/tail threshold is chosen
 * on the device and the host sizes buffers by the capacities earlier passes left; anything that does not fit (first
 * call, hash collision, counts beyond the exact range) repeats through the two synchronous calls. */
int gk_wl_gram(gk_handle* h, int32_t n_iter, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld,
               double* xdiag, gk_stats* stats);

/* One-call forms with host buffers (the e2e path that bench.py times). */
int gk_wl_fit_transform(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr,
                        const int32_t* row_ptr, const int32_t* col_idx, const int32_t* labels,
                        int32_t n_iter, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld,
                        double* diag, gk_stats* stats);
int gk_sp_fit_transform(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr,
                        const int32_t* row_ptr, const int32_t* col_idx, const int32_t* labels,
                        const double* weights, int32_t sp_flags, int32_t flags, void* K_out,
                        int32_t out_dtype, int64_t ld, double* diag, gk_stats* stats);

/* ---- TU-format dataset files -> packed CSR block (host side; no device work).
 * Replaces grakel/datasets/base.py:135-290 (read_data: <name>_graph_indicator.txt, _A.txt, _node_labels.txt,
 * _node_attributes.txt, _edge_labels.txt, _graph_labels.txt parsed into per-graph Python sets and dicts) and
 * the per-graph Graph parsing that follows it (graph.py:147-230, 982-1053): the arrays gk_tu_fill writes are
 * exactly what gk_pack_csr takes.  Edge semantics as in read_data: an edge line belongs to the graph of its
 * source, GK_TU_SYMMETRIC adds the reverse edge (base.py:216-218), duplicates collapse, the last edge-label
 * line of a pair wins (:262-266). */
typedef struct gk_tu gk_tu;
#define GK_TU_SYMMETRIC 1      /* read_data(is_symmetric=True) */
#define GK_TU_ATTR_NODES 2     /* read_data(prefer_attr_nodes=True): node attributes instead of node labels */
#define GK_TU_DEGREE_LABELS 4  /* read_data(produce_labels_nodes=True) when there is no node-label file */
/* vertex set of the packed block */
#define GK_TU_LABELLED_NODES 0 /* every labelled node: what WeisfeilerLehman / VertexHistogram walk */
#define GK_TU_EDGE_NODES 1     /* nodes that occur in an edge: ShortestPath(+Attr) and WL-OA (edge-dictionary keys) */
int gk_tu_open(const char* dir, const char* name, int32_t flags, gk_tu** out);
/* info[0..7] = graphs, nodes, edge lines, has node labels, has edge labels, has classes, attribute dim, 0 */
int gk_tu_info(const gk_tu* t, int64_t* info);
/* choose the vertex set, build the CSR; returns the sizes of the arrays gk_tu_fill writes */
int gk_tu_pack(gk_tu* t, int32_t mode, int64_t* n_vertices, int64_t* n_edges);
/* graph_ptr[graphs+1], row_ptr[V+1], col_idx[E] (GLOBAL vertex ids, rows sorted), node_labels[V] (raw integer
 * labels), edge_labels[E], attrs[V*dim], classes[graphs], node_of_vertex[V] (1-based file node id); any may be NULL */
int gk_tu_fill(const gk_tu* t, int32_t* graph_ptr, int32_t* row_ptr, int32_t* col_idx, int32_t* node_labels,
               int32_t* edge_labels, double* attrs, int32_t* classes, int32_t* node_of_vertex);
int gk_tu_close(gk_tu* t);

/* CUDA-event timing on the handle's stream (bench.py). */
int gk_event_record(gk_handle* h, int32_t slot);            /* slot in [0,16) */
int gk_event_elapsed(gk_handle* h, int32_t a, int32_t b, float* ms);

/* cudaProfilerStart / cudaProfilerStop (on != 0 / on == 0): lets a profiler capture one
 * steady-state pass (tools/profile_step.py under `ncu --profile-from-start off`). */
int gk_profiler_range(int32_t on);

/* Self-test of the tensor-core Gram on a dense count matrix (tests only):
 * counts[n*d] (uint16), out_tc / out_simt [n*n] fp64. */
int gk_selftest_gram(gk_handle* h, int64_t n, int64_t d, const uint16_t* counts, double* out_tc,
                     double* out_simt);

/* ---- float64 result buffers on the host (the reference returns a fresh float64 ndarray, kernel.py:167-204).
 * gk_host_alloc maps `bytes` of anonymous memory with transparent huge pages requested; gk_host_free returns
 * the block to a small per-process pool (GRAKEL_B200_HOST_POOL_MB, default 2048; 0 = unmap at once), so a loop
 * of fit_transform calls re-uses already-faulted pages.  The Python layer wraps the block in an ndarray whose
 * finaliser calls gk_host_free.  Any host pointer is accepted as K_out of gk_gram; these are just the fast ones. */
int gk_host_alloc(int64_t bytes, void** out);
int gk_host_free(void* p, int64_t bytes);

/* Host-only self test of the result delivery (tests only; no device needed): src[rows*cols] fp32 on the host
 * -> dst[rows*cols] fp64 through the same band / widen / mirror code gk_gram uses after its D2H copies.
 * mode 0: symmetric square, upper triangle only; 1: all rows; 2: all rows, normalised by diag (+ nan_to_num). */
int gk_selftest_deliver(int32_t mode, int64_t rows, int64_t cols, const float* src, const double* diag,
                        int32_t nan_to_num, double* dst);

#ifdef __cplusplus
}
#endif
#endif
