// Shared declarations of the grakel_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>

#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/grakel_b200.h"

namespace gk {

// ---------------------------------------------------------------- errors
extern thread_local std::string g_last_error;

inline int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

#define GK_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      return gk::fail(GK_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) +   \
                                       " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
    }                                                                                      \
  } while (0)

#define GK_TRY(expr)          \
  do {                        \
    int _r = (expr);          \
    if (_r != GK_OK) return _r; \
  } while (0)

// ---------------------------------------------------------------- buffers
// Grow-only device buffer: the engine is called repeatedly on same-sized
// workloads (bench loop, fit then transform), so capacity is kept between calls.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return GK_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + (bytes >> 3) + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      return fail(GK_ERR_CUDA, std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e));
    }
    cap = want;
    return GK_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinBuf {  // pinned host staging (D2H of small scalars, H2D of CSR)
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return GK_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMallocHost(&p, bytes + 256);
    if (e != cudaSuccess) return fail(GK_ERR_CUDA, std::string("cudaMallocHost: ") + cudaGetErrorString(e));
    cap = bytes + 256;
    return GK_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr unsigned long long EMPTY64 = ~0ULL;
constexpr int MAX_LEVELS = 64;

// Device-side scalars the pipeline reads back once per phase.
struct DevScalars {
  long long level_dims[MAX_LEVELS];      // distinct labels per WL level
  long long level_base[MAX_LEVELS + 1];  // first column id of each level
  unsigned int collision;                // WL: a hash collision was detected (-> retry with new seed)
  unsigned int ft_overflow;              // feature table probe overflow (cannot happen at load <= 0.5)
  unsigned long long n_entries;          // nnz of the feature block
  unsigned long long max_count;          // largest count
  unsigned long long max_diag;           // largest self similarity
  long long n_dense;                     // D_c
  unsigned long long sp_coo;             // wl_fused2: self-similarity units of frozen vertices (= sum of diag_frozen)
  unsigned int sp_dict_size;             // SP: number of distinct (lu,lv,d) keys
  unsigned int sp_nonint;                // SP: a non-integer / out-of-range distance was met
};

static_assert(sizeof(DevScalars) % 8 == 0, "cleared as 64-bit words");

}  // namespace gk

// The opaque handle of the C-ABI.
struct gk_handle {
  int dev = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // side stream: independent kernels of one phase run concurrently
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_stage[4] = {};  // D2H staging ring of host_deliver.h
  cudaEvent_t ev[16] = {};
  cudaEvent_t tev[8] = {};  // internal stage timers

  // ---- packed graphs
  int64_t N = 0, V = 0, E = 0;
  int32_t n_labels0 = 0;
  bool has_weights = false, unit_weights = true;
  int32_t attr_dim = 0;
  int32_t max_degree = 0, max_graph_size = 0;
  gk::DevBuf graph_ptr, row_ptr, col_idx, labels0, weights, attrs, vgraph;
  bool has_labels = false;  // the current block was packed with vertex labels (labels0 may hold an older block's)
  gk::DevBuf sp_lists;      // graph lists of the shortest-path launches (kept apart from large_list: gk_wl_features reads that)
  gk::DevBuf large_list;  // vertices with degree > group width
  int64_t n_large = 0;
  int group_width = 32;

  // ---- WL scratch
  int n_levels = 0;
  gk::DevBuf labels_all;  // [(h+1) * V] int32
  gk::DevBuf sig_nbr;     // [E] sorted neighbour labels of the current level
  gk::DevBuf slot_of;     // [V] hash slot, then representative vertex
  gk::DevBuf ht_keys, ht_rep;
  size_t ht_cap = 0;
  gk::DevBuf flags, block_sums;
  gk::DevBuf wlf_buf;  // fused WL kernel: [cta_vbeg (G+1) | cta_count (G) | barrier]
  gk::DevBuf wl_payload;  // fused WL kernel v2: [2][ht_cap] 32-byte slot payloads (the installing vertex's signature)
  gk::DevBuf wl_single;  // fused WL kernels: one byte per vertex (singleton class / frozen)
  gk::DevBuf diag_frozen;  // fused WL kernel v2: frozen vertices' share of the self similarities (u64 per graph)
  bool wl_sparse_ids = false;  // labels of levels >= 1 are representative vertex ids (wl_fused2), not dense ranks
  gk::DevBuf scalars;  // gk::DevScalars
  gk::PinBuf h_scalars;

  // ---- feature block (hash table of (graph, column) -> count)
  gk::DevBuf ft_keys, ft_cnt;
  size_t ft_cap = 0;
  int64_t n_columns = 0;
  bool features_ready = false;
  int64_t feat_serial = 0;   // bumped whenever the feature block changes state
  int64_t pro_serial = -1;   // feat_serial for which gk_wl_features already ran the Gram prologue (square case):
                             // self similarities finished, column histogram on the host -- gk_gram then needs no
                             // host synchronisation before its launches
  int feature_kind = 0;  // 1 = WL, 2 = SP, 3 = SP-attr (dense fp32 features), 4 = NeighborhoodHash levels

  gk::DevBuf oa_keys, oa_cnt, oa_colcnt;  // WL-OA: unary-expanded block, swapped with ft_keys / ft_cnt / colcnt
  // NeighborhoodHash (nh.cuh): u64 labels [R + 1][V] (slot 0 = hashed level-0 input), the R unary-expanded level
  // blocks [R][V] keys / counts, [R][V + 1] graphs per column, [R][N] self similarities; sort / scan scratch; the fp32
  // level Gram
  gk::DevBuf nh_labels, nh_keys, nh_cnt, nh_colcnt, nh_diag, nh_tmp, nh_kf;
  int nh_R = 0;
  // ---- columns / panel / diag
  gk::DevBuf colcnt, colmin, colmax, colslot, col_flags3, col_block_sums, colstats;
  int64_t col_cap = 0;  // allocated length of the per-column arrays
  gk::DevBuf part_max, part_new;  // per-CTA partials of the feature kernels
  int64_t n_part = 0;
  gk::DevBuf tail_desc, tail_ent, tail_cur;
  gk::PinBuf h_colstats;
  gk::DevBuf tb_cnt, tb_ent, tb_ovf;  // tail fused into the GEMM epilogue: per-block update lists + overflow (features.cuh tail_bucket)
  gk::DevBuf gram_dyn;   // gk::GramDyn: device-side decisions of the asynchronous pass (gk_wl_gram)
  gk::PinBuf h_dyn;
  gk::DevBuf diag_u64, diag_f64;
  gk::DevBuf row_map, diag_rows;  // gk_set_row_map: packed graph -> row of K (0 rows = identity)
  int64_t n_rows = 0;
  gk::DevBuf panel;
  int64_t Dc = 0, Dc_pad = 0;

  // ---- SP scratch
  gk::DevBuf sp_dist;      // global-memory distance matrices for graphs too large for smem
  gk::DevBuf sp_dict_keys; // (lu,lv,d) -> column dictionary
  gk::DevBuf sp_dict_ids;
  gk::DevBuf sp_dkeys;     // real-valued weights: dictionary of distance bit patterns
  size_t sp_dict_cap = 0;
  gk::DevBuf sp_graph_off; // per-graph offset into sp_dist (for gk_sp_distances)
  int sp_flags = 0;
  int sp_dist_esz = 0;     // gk_spattr_features: element size of the matrices it left in sp_dist (2 = u16, 8 = fp64)

  // ---- SP-attr dense fp32 feature matrix
  gk::DevBuf fattr;
  int64_t fattr_dim = 0;

  // ---- GEMM
  gk::DevBuf tiles;  // int2 list
  gk::PinBuf h_tiles;
  gk::PinBuf h_bands;  // band table of the u16 result transport (its own buffer: h_tiles may still feed an async copy)
  gk::DevBuf K;      // device-resident result of the last gk_gram
  int64_t K_rows = 0, K_cols = 0, K_ld = 0;  // K_ld: row pitch in elements (>= K_cols)
  int K_dtype = GK_F32;
  gk::DevBuf K_stage;  // fp64 staging when K is kept as f32 but fetched as f64

  gk::PinBuf h_stage;  // pinned staging ring of the result delivery
  gk::PinBuf h_diag;   // self similarities on the host (normalisation during the widening)
  int64_t launches = 0;
  void* comm = nullptr;  // gk::Comm (comm.h) after gk_comm_init
};
