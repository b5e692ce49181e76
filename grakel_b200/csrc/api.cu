// C-ABI of the grakel_b200 engine (see include/grakel_b200.h for the contract and
// the reference file:line each entry point replaces).  sm_100a only.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <atomic>
#include <thread>

#include <immintrin.h>
#include <pthread.h>
#include <sched.h>

#include <cuda_profiler_api.h>

#include "common.cuh"
#include "features.cuh"
#include "gram_tc.cuh"
#include "gram_tc2.cuh"
#include "sp.cuh"
#include "spattr.cuh"
#include "wl.cuh"
#include "wl_fused.cuh"
#include "wl_fused2.cuh"
#include "wl_oa.cuh"
#include "nh.cuh"
#include "tu_reader.h"
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "comm.h"

namespace gk {
thread_local std::string g_last_error;

static inline size_t next_pow2(size_t x) {
  size_t p = 1;
  while (p < x) p <<= 1;
  return p;
}
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static int make_panel_map(CUtensorMap* m, void* base, long long cols, long long rows, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return GK_OK;
}

// fp32 (tf32 operand) panel: 32 elements = one 128-byte swizzle row per k-block
static int make_panel_map_f32(CUtensorMap* m, void* base, long long cols, long long rows, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  cuuint32_t box[2] = {(cuuint32_t)BK_TF32, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled(f32 panel) failed: " + std::to_string((int)r));
  return GK_OK;
}

// fp32 K as a 2-D tensor for TMA stores of 32x32 blocks (128-byte swizzle)
static int make_out_map(CUtensorMap* m, void* base, long long cols, long long rows, long long ld) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GK_ERR_CUDA, "cuTensorMapEncodeTiled(out) failed: " + std::to_string((int)r));
  return GK_OK;
}

static int read_scalars(gk_handle* h, DevScalars** out) {
  GK_TRY(h->h_scalars.ensure(sizeof(DevScalars)));
  GK_CUDA(cudaMemcpyAsync(h->h_scalars.p, h->scalars.p, sizeof(DevScalars), cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  *out = h->h_scalars.as<DevScalars>();
  return GK_OK;
}

static float ev_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  return ms;
}

}  // namespace gk

using namespace gk;

// extra host-side state that does not belong in the POD-ish handle header
struct HandleExtra {
  std::vector<int> graph_ptr;
  std::vector<int> graph_eptr;  // first edge of each graph (row_ptr[graph_ptr[g]])
  std::vector<long long> sp_goff;
  // fused WL kernel: the tile partition of the packed block (device copy in wlf_buf) is kept between calls
  bool wl_tiles_valid = false;
  bool wl_tiles_fused = false;
  int wl_n_tiles = 0;
  long long wl_tiles_key = -1;  // GRAKEL_B200_WL_TILES_PER_CTA the partition was built with
  // Gram prologue run by gk_wl_features (pro_serial): what gk_gram would otherwise read back after a synchronisation
  ColStats pro_hist;
  long long pro_max_count = 0, pro_max_diag = 0, pro_n_entries = 0;
  // GEMM tile list on the device (h->tiles): rebuilt and uploaded only when its key changes
  long long tiles_key[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
  long long tiles_n = 0;
  long long head_dc_pad = 0;  // panel width of the last pass whose threshold came from the cost model (not GK_DENSE_ALL / FORCE_T)
  // gk_nh_features: per level, the expanded block's columns and entries (what gk_nh_gram hands to gk_gram)
  std::vector<long long> nh_cols, nh_entries;
};
static std::vector<std::pair<gk_handle*, HandleExtra*>> g_extra;
static HandleExtra* extra_of(gk_handle* h) {
  for (auto& p : g_extra)
    if (p.first == h) return p.second;
  HandleExtra* e = new HandleExtra();
  g_extra.emplace_back(h, e);
  return e;
}
static void drop_extra(gk_handle* h) {
  for (size_t i = 0; i < g_extra.size(); ++i)
    if (g_extra[i].first == h) {
      delete g_extra[i].second;
      g_extra.erase(g_extra.begin() + i);
      return;
    }
}

#define LAUNCH_CHECK(h)                                 \
  do {                                                  \
    (h)->launches++;                                    \
    GK_CUDA(cudaGetLastError());                        \
  } while (0)

extern "C" {

int gk_version(void) { return 100; }
const char* gk_last_error(void) { return g_last_error.c_str(); }

int gk_create(int device_ordinal, gk_handle** out) {
  if (!out) return fail(GK_ERR_ARG, "gk_create: out is NULL");
  int n = 0;
  GK_CUDA(cudaGetDeviceCount(&n));
  if (device_ordinal < 0 || device_ordinal >= n) return fail(GK_ERR_ARG, "gk_create: bad device ordinal");
  GK_CUDA(cudaSetDevice(device_ordinal));
  cudaDeviceProp prop;
  GK_CUDA(cudaGetDeviceProperties(&prop, device_ordinal));
  if (prop.major != 10) {
    return fail(GK_ERR_UNSUPPORTED, std::string("grakel_b200 needs an sm_100a (B200) device, found sm_") +
                                        std::to_string(prop.major) + std::to_string(prop.minor));
  }
  gk_handle* h = new gk_handle();
  h->dev = device_ordinal;
  h->sm_count = prop.multiProcessorCount;
  GK_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  GK_CUDA(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
  GK_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  GK_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  for (auto& e : h->ev_stage) GK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto& e : h->ev) GK_CUDA(cudaEventCreate(&e));
  for (auto& e : h->tev) GK_CUDA(cudaEventCreate(&e));
  GK_TRY(h->scalars.ensure(sizeof(DevScalars)));
  GK_TRY(h->h_scalars.ensure(sizeof(DevScalars)));
  GK_CUDA(cudaFuncSetAttribute(gram_tc_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
  GK_CUDA(cudaFuncSetAttribute(gram_tc_kernel<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
  GK_CUDA(cudaFuncSetAttribute(gram_tc_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
  GK_CUDA(cudaFuncSetAttribute(gram_tc_kernel<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
  GK_CUDA(cudaFuncSetAttribute(gram_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM));
  GK_CUDA(cudaFuncSetAttribute(gram_tc_kernel<double, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
  GK_CUDA(cudaFuncSetAttribute(wl_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WLF_SMEM));
  GK_CUDA(cudaFuncSetAttribute(wl_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, WLF_SMEM));
  GK_CUDA(cudaFuncSetAttribute(wl_fused2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WLF2_SMEM));
  GK_CUDA(cudaFuncSetAttribute(wl_fused2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, WLF2_SMEM));
  *out = h;
  return GK_OK;
}

// --------------------------------------------------------------------------- multi-GPU (comm.h)
int gk_comm_unique_id(void* out128) {
  if (!out128) return fail(GK_ERR_ARG, "gk_comm_unique_id: null argument");
  NcclApi* api = nccl_api();
  if (!api->lib || !api->error.empty()) return fail(GK_ERR_UNSUPPORTED, "gk_comm_unique_id: " + api->error);
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  GK_NCCL(api, api->GetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return GK_OK;
}

int gk_comm_destroy(gk_handle* h) {
  if (!h || !h->comm) return GK_OK;
  Comm* c = reinterpret_cast<Comm*>(h->comm);
  cudaSetDevice(h->dev);
  cudaStreamSynchronize(h->stream);
  for (int r = 0; r < c->nranks; ++r)
    if (r != c->rank && c->peer_base[r]) { cudaIpcCloseMemHandle(c->peer_base[r]); c->peer_base[r] = nullptr; }
  // collective: nobody frees an exported block (gk_destroy does, right after this) before every peer has unmapped it
  if (c->comm && c->nranks > 1 && nccl_api()->AllReduce) {
    nccl_api()->AllReduce(c->d_token, c->d_token, 1, ncclInt32, ncclSum, c->comm, h->stream);
    cudaStreamSynchronize(h->stream);
  }
  if (c->d_token) cudaFree(c->d_token);
  if (c->d_handles) cudaFree(c->d_handles);
  NcclApi* api = nccl_api();
  if (c->comm && api->CommDestroy) api->CommDestroy(c->comm);
  delete c;
  h->comm = nullptr;
  return GK_OK;
}

int gk_comm_init(gk_handle* h, int32_t nranks, int32_t rank, const void* unique_id128) {
  if (!h || !unique_id128) return fail(GK_ERR_ARG, "gk_comm_init: null argument");
  if (nranks < 1 || nranks > DIST_MAX_RANKS || rank < 0 || rank >= nranks) return fail(GK_ERR_ARG, "gk_comm_init: 1..8 ranks");
  if (h->comm) return fail(GK_ERR_STATE, "gk_comm_init: the handle already has a communicator");
  NcclApi* api = nccl_api();
  if (!api->lib || !api->error.empty()) return fail(GK_ERR_UNSUPPORTED, "gk_comm_init: " + api->error);
  GK_CUDA(cudaSetDevice(h->dev));
  Comm* c = new Comm();
  c->nranks = nranks; c->rank = rank;
  ncclUniqueId id;
  memcpy(&id, unique_id128, sizeof(id));
  ncclResult_t r = api->CommInitRank(&c->comm, nranks, id, rank);
  if (r != ncclSuccess) { delete c; return fail(GK_ERR_CUDA, std::string("ncclCommInitRank: ") + api->GetErrorString(r)); }
  if (cudaMalloc(&c->d_token, 256) != cudaSuccess || cudaMalloc(&c->d_handles, (size_t)(nranks + 1) * 64) != cudaSuccess) {
    delete c;
    return fail(GK_ERR_CUDA, "gk_comm_init: cudaMalloc failed");
  }
  cudaMemset(c->d_token, 0, 256);
  h->comm = c;
  return GK_OK;
}

int gk_comm_rows(gk_handle* h, int64_t n_rows, int64_t* row_begin, int64_t* row_end) {
  if (!h || !row_begin || !row_end || n_rows < 0) return fail(GK_ERR_ARG, "gk_comm_rows: bad arguments");
  Comm* c = reinterpret_cast<Comm*>(h->comm);
  const int nranks = c ? c->nranks : 1, rank = c ? c->rank : 0;
  const long long per = dist_rows_per_rank(n_rows, nranks);
  *row_begin = std::min<long long>(n_rows, rank * per);
  *row_end = std::min<long long>(n_rows, (rank + 1) * per);
  return GK_OK;
}

// Host-only: the tile list of one rank (tests of the partition; no device, no communicator needed)
int gk_selftest_dist_tiles(int64_t n_rows, int32_t nranks, int32_t rank, int32_t* tiles_xy, int64_t cap, int64_t* n_tiles) {
  if (!n_tiles || nranks < 1 || nranks > DIST_MAX_RANKS || rank < 0 || rank >= nranks) return fail(GK_ERR_ARG, "gk_selftest_dist_tiles: bad arguments");
  std::vector<int2> t;
  dist_tiles(n_rows, nranks, rank, t);
  *n_tiles = (int64_t)t.size();
  if (tiles_xy)
    for (size_t i = 0; i < t.size() && (int64_t)i < cap; ++i) { tiles_xy[2 * i] = t[i].x; tiles_xy[2 * i + 1] = t[i].y; }
  return GK_OK;
}

int gk_destroy(gk_handle* h) {
  if (!h) return GK_OK;
  cudaSetDevice(h->dev);
  cudaStreamSynchronize(h->stream);
  gk::DevBuf* bufs[] = {&h->graph_ptr, &h->row_ptr, &h->col_idx, &h->labels0, &h->weights, &h->attrs, &h->vgraph,
                        &h->large_list, &h->labels_all, &h->sig_nbr, &h->slot_of, &h->ht_keys, &h->ht_rep,
                        &h->flags, &h->block_sums, &h->scalars, &h->ft_keys, &h->ft_cnt, &h->colcnt,
                        &h->colmin, &h->colmax, &h->colslot, &h->col_flags3, &h->col_block_sums, &h->colstats, &h->tail_desc,
                        &h->tail_ent, &h->tail_cur, &h->part_max, &h->part_new, &h->diag_u64, &h->diag_f64, &h->panel,
                        &h->sp_dist, &h->sp_dict_keys, &h->sp_dict_ids, &h->sp_dkeys, &h->sp_graph_off, &h->fattr, &h->fattr_exp, &h->tiles,
                        &h->K, &h->K_stage, &h->wlf_buf, &h->row_map, &h->diag_rows, &h->oa_keys, &h->oa_cnt, &h->oa_colcnt, &h->wl_single,
                        &h->diag_frozen, &h->sp_lists, &h->wl_payload, &h->gram_dyn, &h->tb_cnt, &h->tb_ent, &h->tb_ovf,
                        &h->nh_labels, &h->nh_keys, &h->nh_cnt, &h->nh_colcnt, &h->nh_diag, &h->nh_tmp, &h->nh_kf};
  for (auto* b : bufs) b->release();
  h->h_scalars.release();
  h->h_colstats.release();
  h->h_dyn.release();
  h->h_tiles.release();
  h->h_stage.release();
  h->h_diag.release();
  h->h_bands.release();
  for (auto& e : h->ev) cudaEventDestroy(e);
  for (auto& e : h->tev) cudaEventDestroy(e);
  cudaStreamDestroy(h->stream);
  cudaStreamDestroy(h->stream2);
  cudaEventDestroy(h->ev_fork);
  cudaEventDestroy(h->ev_join);
  for (auto& e : h->ev_stage) cudaEventDestroy(e);
  gk_comm_destroy(h);
  drop_extra(h);
  delete h;
  return GK_OK;
}

int gk_sync(gk_handle* h) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

int gk_event_record(gk_handle* h, int32_t slot) {
  if (!h || slot < 0 || slot >= 16) return fail(GK_ERR_ARG, "gk_event_record: bad slot");
  GK_CUDA(cudaEventRecord(h->ev[slot], h->stream));
  return GK_OK;
}
int gk_event_elapsed(gk_handle* h, int32_t a, int32_t b, float* ms) {
  if (!h || !ms || a < 0 || a >= 16 || b < 0 || b >= 16) return fail(GK_ERR_ARG, "gk_event_elapsed: bad args");
  GK_CUDA(cudaEventSynchronize(h->ev[b]));
  GK_CUDA(cudaEventElapsedTime(ms, h->ev[a], h->ev[b]));
  return GK_OK;
}

// ncu/nsys capture range (tools/profile_step.py runs under `--profile-from-start off`)
int gk_profiler_range(int32_t on) {
  GK_CUDA(on ? cudaProfilerStart() : cudaProfilerStop());
  return GK_OK;
}

// ---------------------------------------------------------------------------
int gk_pack_csr(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr, const int32_t* row_ptr,
                const int32_t* col_idx, const int32_t* labels, const double* weights, const double* attrs,
                int32_t attr_dim) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (n_graphs <= 0 || !graph_ptr || !row_ptr) return fail(GK_ERR_ARG, "gk_pack_csr: empty input");
  if (n_graphs >= (1LL << 31) - 1) return fail(GK_ERR_ARG, "gk_pack_csr: too many graphs");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t N = n_graphs;
  const int64_t V = graph_ptr[N];
  if (graph_ptr[0] != 0 || V < 0) return fail(GK_ERR_ARG, "gk_pack_csr: bad graph_ptr");
  if (V >= (1LL << 26)) return fail(GK_ERR_ARG, "gk_pack_csr: more than 2^26 vertices in one block");
  const int64_t E = V ? row_ptr[V] : 0;
  if (E < 0 || (E > 0 && !col_idx)) return fail(GK_ERR_ARG, "gk_pack_csr: bad row_ptr / col_idx");
  // graph sizes (N small); every per-vertex / per-edge scan runs on the device below
  int max_n = 0;
  for (int64_t g = 0; g < N; ++g) {
    const int n = graph_ptr[g + 1] - graph_ptr[g];
    if (n < 0 || graph_ptr[g + 1] > V) return fail(GK_ERR_ARG, "gk_pack_csr: graph_ptr not monotone");
    max_n = std::max(max_n, n);
  }
  h->N = N; h->V = V; h->E = E;
  h->has_weights = weights != nullptr;
  h->has_labels = labels != nullptr;
  h->attr_dim = attrs ? attr_dim : 0;
  h->max_graph_size = max_n;
  h->features_ready = false; h->feat_serial++;
  h->feature_kind = 0;
  h->n_rows = 0;  // a new block starts without a row map
  HandleExtra* ex = extra_of(h);
  ex->wl_tiles_valid = false;
  ex->graph_ptr.assign(graph_ptr, graph_ptr + N + 1);
  ex->graph_eptr.resize(N + 1);
  for (int64_t g = 0; g <= N; ++g) ex->graph_eptr[g] = V ? row_ptr[graph_ptr[g]] : 0;

  GK_CUDA(cudaEventRecord(h->tev[0], h->stream));
  GK_TRY(h->graph_ptr.ensure((N + 1) * 4));
  GK_TRY(h->row_ptr.ensure((V + 1) * 4));
  GK_TRY(h->col_idx.ensure(std::max<int64_t>(E, 1) * 4));
  GK_TRY(h->vgraph.ensure(std::max<int64_t>(V, 1) * 4));
  GK_TRY(h->large_list.ensure(std::max<int64_t>(V, 1) * 4 + 64));
  GK_CUDA(cudaMemcpyAsync(h->graph_ptr.p, graph_ptr, (N + 1) * 4, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaMemcpyAsync(h->row_ptr.p, row_ptr, (V + 1) * 4, cudaMemcpyHostToDevice, h->stream));
  if (E) GK_CUDA(cudaMemcpyAsync(h->col_idx.p, col_idx, E * 4, cudaMemcpyHostToDevice, h->stream));
  if (labels) {
    GK_TRY(h->labels0.ensure(std::max<int64_t>(V, 1) * 4));
    GK_CUDA(cudaMemcpyAsync(h->labels0.p, labels, V * 4, cudaMemcpyHostToDevice, h->stream));
  }
  if (weights && E) {
    GK_TRY(h->weights.ensure(E * 8));
    GK_CUDA(cudaMemcpyAsync(h->weights.p, weights, E * 8, cudaMemcpyHostToDevice, h->stream));
  }
  if (attrs && attr_dim > 0) {
    GK_TRY(h->attrs.ensure((size_t)V * attr_dim * 8));
    GK_CUDA(cudaMemcpyAsync(h->attrs.p, attrs, (size_t)V * attr_dim * 8, cudaMemcpyHostToDevice, h->stream));
  }
  // device-side statistics + validation (degree histogram, bounds, labels, weights)
  int* d_scan = reinterpret_cast<int*>(h->scalars.as<DevScalars>()) ;  // reuse the scalar block as 16 ints
  GK_CUDA(cudaMemsetAsync(d_scan, 0, 64, h->stream));
  int hscan[16] = {0};
  if (V) {
    fill_vgraph<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, (int)N, h->graph_ptr.as<int>(), h->vgraph.as<int>());
    LAUNCH_CHECK(h);
    pack_scan<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, (int)E, h->graph_ptr.as<int>(), h->vgraph.as<int>(),
                                                   h->row_ptr.as<int>(), h->col_idx.as<int>(),
                                                   labels ? h->labels0.as<int>() : nullptr, d_scan);
    LAUNCH_CHECK(h);
    if (weights && E) {
      pack_scan_weights<<<h->sm_count * 4, 256, 0, h->stream>>>(E, h->weights.as<double>(), d_scan);
      LAUNCH_CHECK(h);
    }
    GK_CUDA(cudaMemcpyAsync(h->h_scalars.p, d_scan, 64, cudaMemcpyDeviceToHost, h->stream));
    GK_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(hscan, h->h_scalars.p, 64);
  }
  if (hscan[6] & 1) return fail(GK_ERR_ARG, "gk_pack_csr: row_ptr not monotone");
  if (hscan[6] & 2) return fail(GK_ERR_ARG, "gk_pack_csr: edge leaves its graph");
  if (hscan[6] & 4) return fail(GK_ERR_ARG, "gk_pack_csr: negative label id");
  if (hscan[8] & 2) return fail(GK_ERR_UNSUPPORTED, "gk_pack_csr: negative or NaN edge weight");
  h->n_labels0 = labels ? hscan[7] + 1 : 0;
  h->unit_weights = !(hscan[8] & 1);
  h->max_degree = hscan[5];
  // WL signature kernel choice: one thread per vertex for degree <= 8 (cost ~1 lane), else
  // 16 or 32 lanes per vertex; vertices above the width take the warp-per-vertex kernel.
  {
    const long long above8 = (long long)hscan[2] + hscan[3] + hscan[4], above16 = (long long)hscan[3] + hscan[4],
                    above32 = hscan[4];
    const long long c8 = (long long)V * 1 + above8 * 32, c16 = (long long)V * 16 + above16 * 32,
                    c32 = (long long)V * 32 + above32 * 32;
    h->group_width = 8;
    h->n_large = above8;
    long long best = c8;
    if (c16 < best) { best = c16; h->group_width = 16; h->n_large = above16; }
    if (c32 < best) { best = c32; h->group_width = 32; h->n_large = above32; }
  }
  if (h->n_large) {
    GK_CUDA(cudaMemsetAsync(d_scan, 0, 4, h->stream));
    pack_large_list<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, h->row_ptr.as<int>(), h->group_width,
                                                         h->large_list.as<int>(), d_scan);
    LAUNCH_CHECK(h);
  }
  GK_CUDA(cudaEventRecord(h->tev[1], h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));  // caller buffers may be reused once we return
  return GK_OK;
}

// ---------------------------------------------------------------------------
}  // extern "C"

template <int G>
static void launch_sig_small(gk_handle* h, const int* lab_in, unsigned long long seed) {
  const long long threads = (long long)h->V * G;
  wl_sig_small<G><<<cdiv(threads, 256), 256, 0, h->stream>>>(
      (int)h->V, h->row_ptr.as<int>(), h->col_idx.as<int>(), lab_in, h->sig_nbr.as<int>(), seed,
      h->ht_keys.as<unsigned long long>(), h->ht_rep.as<int>(), (unsigned)(h->ht_cap - 1), h->slot_of.as<int>());
}

// (re)allocate and clear the statistics the feature kernels maintain at insert time
static int reset_feature_stats(gk_handle* h, int64_t col_cap, int64_t n_part, FeatStats* st, bool clear = true) {
  col_cap = std::max<int64_t>(col_cap, 1);
  n_part = std::max<int64_t>(n_part, 1);
  GK_TRY(h->part_max.ensure(n_part * 4));
  GK_TRY(h->part_new.ensure(n_part * 4));
  h->n_part = n_part;
  if (clear) {
    GK_CUDA(cudaMemsetAsync(h->part_max.p, 0, n_part * 4, h->stream));
    GK_CUDA(cudaMemsetAsync(h->part_new.p, 0, n_part * 4, h->stream));
  }
  st->part_max = h->part_max.as<unsigned>();
  st->part_new = h->part_new.as<unsigned>();
  GK_TRY(h->colcnt.ensure(col_cap * 4));
  GK_TRY(h->diag_u64.ensure(h->N * 8));
  h->col_cap = col_cap;
  if (clear) {
    GK_CUDA(cudaMemsetAsync(h->colcnt.p, 0, col_cap * 4, h->stream));
    GK_CUDA(cudaMemsetAsync(h->diag_u64.p, 0, h->N * 8, h->stream));
  }
  st->colcnt = h->colcnt.as<unsigned>();
  st->diag = h->diag_u64.as<unsigned long long>();
  st->sc = h->scalars.as<DevScalars>();
  return GK_OK;
}

static int init_scalars(gk_handle* h, int n_labels0) {
  DevScalars* hs = h->h_scalars.as<DevScalars>();
  memset(hs, 0, sizeof(DevScalars));
  hs->level_dims[0] = n_labels0;
  hs->level_base[0] = 0;
  hs->level_base[1] = n_labels0;
  GK_CUDA(cudaMemcpyAsync(h->scalars.p, hs, sizeof(DevScalars), cudaMemcpyHostToDevice, h->stream));
  // the pinned struct is reused for read-back; make sure the upload has consumed it
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

// What gk_wl_features decides and allocates before its first launch (shared with the asynchronous pass, gk_wl_gram)
struct WlPlan {
  int L = 0, G = 0, nb = 0, n_tiles = 0;
  bool fused = false;
  size_t ft_level_cap = 0;
};

static int wl_setup(gk_handle* h, int n_iter, WlPlan* pl) {
  const int64_t V = h->V, E = h->E;
  const int L = n_iter + 1;
  GK_TRY(h->labels_all.ensure((size_t)L * V * 4));
  GK_TRY(h->sig_nbr.ensure(std::max<int64_t>(E, 1) * 4 * 2));  // wl_fused2 double-buffers the rows by level parity
  GK_TRY(h->slot_of.ensure(V * 4));
  GK_TRY(h->flags.ensure(V * 4));
  const int nb = cdiv(V, 256);
  GK_TRY(h->block_sums.ensure((size_t)nb * 4));
  // >= 2 V slots (load <= 0.5 at the one level where almost every vertex is a class of its own; frozen vertices stop
  // inserting after it): three rotating tables stay L2-resident up to ~1.3 M vertices.  Measured against 4 V:
  // 0.229 vs 0.239 ms at config 2, 0.618 vs 0.655 ms at 28 284 graphs (profiles/r02n_table_factor.txt).
  size_t table_factor = 2;
  if (const char* e = getenv("GRAKEL_B200_WL_TABLE_FACTOR")) table_factor = (size_t)std::max(2, atoi(e));
  h->ht_cap = std::max<size_t>(next_pow2((size_t)V * table_factor), 1024);
  GK_TRY(h->ht_keys.ensure(h->ht_cap * 8 * 3));  // three tables: the fused kernel rotates them over the levels
  GK_TRY(h->ht_rep.ensure(h->ht_cap * 4 * 2));
  const size_t ft_level_cap = std::max<size_t>(next_pow2((size_t)V * 2), 1024);  // one L2-sized sub-table per level
  // Fused persistent kernel (wl_fused.cuh) whenever the graphs can be cut into shared-memory tiles of
  // whole graphs; otherwise (a graph above the tile capacity) the multi-kernel path below.
  bool fused = true;
  if (const char* e = getenv("GRAKEL_B200_WL_FUSED")) fused = atoi(e) != 0;
  const int G = std::min(h->sm_count, 1024);
  int n_tiles = 0;
  long long tiles_env = 0;
  if (const char* e = getenv("GRAKEL_B200_WL_TILES_PER_CTA")) tiles_env = atoi(e);
  if (fused && extra_of(h)->wl_tiles_valid && extra_of(h)->wl_tiles_key == tiles_env) {
    // same packed block as the last call: the partition is still in wlf_buf (the kernels only touch its barrier word)
    fused = extra_of(h)->wl_tiles_fused;
    n_tiles = extra_of(h)->wl_n_tiles;
  } else if (fused) {
    HandleExtra* ex = extra_of(h);
    std::vector<int> tv, ct(G + 1, 0);
    bool ok = false;
    int64_t per0 = std::max<int64_t>(1, std::max((V + (int64_t)G * WLF_TILE_V - 1) / ((int64_t)G * WLF_TILE_V),
                                                  (E + (int64_t)G * WLF_TILE_E - 1) / ((int64_t)G * WLF_TILE_E)));
    if (const char* e = getenv("GRAKEL_B200_WL_TILES_PER_CTA")) per0 = std::max<int64_t>(per0, atoi(e));  // tests: multi-tile CTAs on small inputs
    for (int per = (int)per0;
         per <= 4096 && !ok; per *= 2) {
      // G * per tiles of whole graphs, balanced by vertex count
      const int T = G * per;
      tv.assign(T + 1, 0);
      size_t g = 0;
      for (int t = 1; t < T; ++t) {
        const long long want = (long long)V * t / T;
        while (g < (size_t)h->N && ex->graph_ptr[g] < want) ++g;
        tv[t] = (int)g;
      }
      tv[T] = (int)h->N;
      ok = true;
      for (int t = 0; t < T && ok; ++t) {
        const int nv = ex->graph_ptr[tv[t + 1]] - ex->graph_ptr[tv[t]];
        const int ne = ex->graph_eptr[tv[t + 1]] - ex->graph_eptr[tv[t]];
        if (nv > WLF_TILE_V || ne > WLF_TILE_E) ok = false;
      }
      if (ok) {
        n_tiles = T;
        for (int t = 0; t <= T; ++t) tv[t] = ex->graph_ptr[tv[t]];  // graph index -> first vertex
        for (int c = 0; c <= G; ++c) ct[c] = c * per;
        long long max_cta = 0;
        for (int c = 0; c < G; ++c) max_cta = std::max<long long>(max_cta, tv[ct[c + 1]] - tv[ct[c]]);
        if (max_cta >= (1 << WLF_RANK_BITS)) ok = false;
      }
      if (h->max_graph_size > WLF_TILE_V) break;
    }
    fused = ok;
    if (fused) {
      // layout of wlf_buf (ints): [tile_vbeg (T+1) | cta_tile (G+1) | cta_count (G) | barrier]
      const size_t n_int = (size_t)(n_tiles + 1) + (G + 1) + G + 1;
      GK_TRY(h->wlf_buf.ensure(n_int * 4));
      GK_TRY(h->h_tiles.ensure(((size_t)n_tiles + G + 2) * 4));
      int* hp = h->h_tiles.as<int>();
      memcpy(hp, tv.data(), (size_t)(n_tiles + 1) * 4);
      memcpy(hp + n_tiles + 1, ct.data(), (size_t)(G + 1) * 4);
      GK_CUDA(cudaMemcpyAsync(h->wlf_buf.p, hp, ((size_t)n_tiles + G + 2) * 4, cudaMemcpyHostToDevice, h->stream));
    }
    ex->wl_tiles_valid = true; ex->wl_tiles_fused = fused; ex->wl_n_tiles = n_tiles; ex->wl_tiles_key = tiles_env;
  }
  // feature block: the multi-kernel path fills one open-addressing sub-table per level, the fused
  // kernel appends at most V entries per level to the same arrays used as a COO list
  h->ft_cap = fused ? std::max<size_t>((size_t)V * L, 1) : ft_level_cap * (size_t)L;
  if (h->ft_cap > (1ULL << 31)) return fail(GK_ERR_ARG, "gk_wl_features: feature table too large");
  GK_TRY(h->ft_keys.ensure(h->ft_cap * 8));
  GK_TRY(h->ft_cnt.ensure(h->ft_cap * 4));
  pl->L = L; pl->G = G; pl->nb = nb; pl->n_tiles = n_tiles; pl->fused = fused; pl->ft_level_cap = ft_level_cap;
  return GK_OK;
}

// prepare + wl_fused2 on the handle's stream; no synchronisation
static int wl_launch_v2(gk_handle* h, const WlPlan& pl, unsigned long long seed, const FeatStats& fst, bool prof) {
  const int64_t V = h->V, E = h->E;
  const int L = pl.L, G = pl.G, n_tiles = pl.n_tiles;
  DevScalars* sc = h->scalars.as<DevScalars>();
  int* labels_all = h->labels_all.as<int>();
  {
      // wl_fused2.cuh: labels = representative vertex ids (one grid barrier per level), frozen singleton classes
      int* wb = h->wlf_buf.as<int>();
      int* d_cta_tile = wb + n_tiles + 1;
      unsigned* d_barrier = reinterpret_cast<unsigned*>(d_cta_tile + G + 1 + G);
      GK_TRY(h->wl_single.ensure((size_t)V + 16));
      GK_TRY(h->diag_frozen.ensure((size_t)h->N * 8));
      {  // one launch clears everything the kernel expects cleared (no host upload, no synchronisation)
        Wlf2Prepare q;
        q.sc = sc; q.n_labels0 = h->n_labels0;
        q.part_max = h->part_max.as<unsigned>(); q.part_new = h->part_new.as<unsigned>(); q.n_part = h->n_part;
        q.colcnt = h->colcnt.as<unsigned>(); q.col_cap = h->col_cap;
        q.diag = h->diag_u64.as<unsigned long long>(); q.diag_frozen = h->diag_frozen.as<unsigned long long>(); q.n_graphs = h->N;
        q.barrier = d_barrier;
        q.frozen = h->wl_single.as<unsigned char>(); q.V = V;
        q.table1 = L > 1 ? h->ht_keys.as<unsigned long long>() + h->ht_cap : nullptr; q.ht_cap = (long long)h->ht_cap;
        wlf2_prepare_kernel<<<h->sm_count * 2, 1024, 0, h->stream>>>(q);
        LAUNCH_CHECK(h);
      }
      WlFused2Params fp;
      memset(&fp, 0, sizeof(fp));
      fp.V = (int)V; fp.L = L; fp.n_labels0 = h->n_labels0;
      fp.graph_ptr = h->graph_ptr.as<int>();
      fp.row_ptr = h->row_ptr.as<int>(); fp.col_idx = h->col_idx.as<int>(); fp.vgraph = h->vgraph.as<int>();
      fp.labels0 = h->labels0.as<int>(); fp.tile_vbeg = wb; fp.cta_tile = d_cta_tile;
      fp.barrier = d_barrier;
      fp.labels_all = labels_all; fp.sig_nbr = h->sig_nbr.as<int>(); fp.slot_of = h->slot_of.as<int>();
      fp.E = std::max<int64_t>(E, 1);
      {  // slot payloads (wl_fused2.cuh [A3]/[B]); GRAKEL_B200_WL_PAYLOAD=0: verify against the representative's CSR row
        const char* e = getenv("GRAKEL_B200_WL_PAYLOAD");
        if (!(e && atoi(e) == 0)) {
          GK_TRY(h->wl_payload.ensure(h->ht_cap * 32 * 2));
          fp.payload = h->wl_payload.as<int>();
        }
      }
      fp.frozen = h->wl_single.as<unsigned char>();
      fp.table = h->ht_keys.as<unsigned long long>();
      fp.ht_mask = (unsigned)(h->ht_cap - 1);
      fp.coo_keys = h->ft_keys.as<unsigned long long>(); fp.coo_cnt = h->ft_cnt.as<unsigned>();
      fp.seed = seed; fp.st = fst; fp.sc = sc;
      fp.diag_frozen = h->diag_frozen.as<unsigned long long>();
      if (const char* e = getenv("GRAKEL_B200_WL_DBG")) fp.dbg = atoi(e);
      if (prof) {
        GK_TRY(h->K_stage.ensure((size_t)G * L * 128));
        GK_CUDA(cudaMemsetAsync(h->K_stage.p, 0, (size_t)G * L * 128, h->stream));
        fp.prof = h->K_stage.as<long long>();
      }
      void* args[] = {&fp};
      GK_CUDA(cudaLaunchCooperativeKernel(fp.payload ? (void*)wl_fused2_kernel<true> : (void*)wl_fused2_kernel<false>, dim3(G), dim3(WLF_THREADS), args, WLF2_SMEM, h->stream));
      LAUNCH_CHECK(h);
  }
  return GK_OK;
}

extern "C" {

int gk_wl_features(gk_handle* h, int32_t n_iter, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->N <= 0) return fail(GK_ERR_STATE, "gk_wl_features: no graphs packed");
  if (!h->has_labels || h->V == 0) return fail(GK_ERR_ARG, "gk_wl_features: vertex labels are required");
  if (n_iter < 0 || n_iter + 1 >= MAX_LEVELS) return fail(GK_ERR_ARG, "gk_wl_features: n_iter out of range");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t V = h->V, E = h->E;
  const int L = n_iter + 1;
  h->n_levels = L;
  h->features_ready = false; h->feat_serial++;
  const int64_t launches0 = h->launches;

  WlPlan pl;
  GK_TRY(wl_setup(h, n_iter, &pl));
  const bool fused = pl.fused;
  const int G = pl.G, nb = pl.nb, n_tiles = pl.n_tiles;
  const size_t ft_level_cap = pl.ft_level_cap;
  (void)n_tiles;

  DevScalars* sc = h->scalars.as<DevScalars>();
  int* labels_all = h->labels_all.as<int>();
  int retries = 0;
  bool pro_enqueued = false, used_v2 = false;
  GK_CUDA(cudaEventRecord(h->tev[2], h->stream));
  for (;; ++retries) {
    pro_enqueued = false;
    if (retries > 8)
      return fail(GK_ERR_STATE, "gk_wl_features: repeated hash collisions (level mask 0x" +
                                    [&] { char b[16]; snprintf(b, sizeof(b), "%x", h->h_scalars.as<DevScalars>()->collision); return std::string(b); }() + ")");
    const unsigned long long seed = mix64(0x5851F42D4C957F2DULL + 0x9E3779B97F4A7C15ULL * (unsigned long long)retries);
    const char* e_v1 = getenv("GRAKEL_B200_WL_V1");
    const bool wl_v2 = fused && !(e_v1 && atoi(e_v1) != 0);
    FeatStats fst;
    if (!wl_v2) GK_TRY(init_scalars(h, h->n_labels0));
    GK_TRY(reset_feature_stats(h, (int64_t)h->n_labels0 + V * (int64_t)(L - 1) + 1, (int64_t)std::max(nb, G) * L, &fst, !wl_v2));
    h->wl_sparse_ids = false;
    used_v2 = wl_v2;
    if (wl_v2) {
      const bool prof = getenv("GRAKEL_B200_PROF") != nullptr;
      GK_TRY(wl_launch_v2(h, pl, seed, fst, prof));
      h->wl_sparse_ids = L > 1;
      GK_CUDA(cudaEventRecord(h->tev[3], h->stream));  // end of the feature stage
      if (!prof && !getenv("GRAKEL_B200_NO_PROLOGUE")) {
        // Gram prologue of the square (fit_transform) case, enqueued BEFORE this call's one host synchronisation:
        // self similarities + per-CTA partials (diag_finish) and the column histogram (col_hist).  gk_gram then
        // finds everything its host-side decisions need (threshold T, D_c, exactness bounds) already on the host
        // and launches without a synchronisation of its own (pro_serial).
        const int64_t D = (int64_t)h->n_labels0 + V * (int64_t)(L - 1);
        GK_TRY(h->diag_f64.ensure(h->N * 8));
        GK_TRY(h->colstats.ensure(sizeof(ColStats)));
        GK_TRY(h->h_colstats.ensure(sizeof(ColStats)));
        diag_finish<<<cdiv(h->N, 256), 256, 0, h->stream>>>((int)h->N, h->diag_u64.as<unsigned long long>(), h->diag_f64.as<double>(),
                                                            (int)h->n_part, h->part_max.as<unsigned>(), h->part_new.as<unsigned>(), sc);
        LAUNCH_CHECK(h);
        GK_CUDA(cudaMemsetAsync(h->colstats.p, 0, sizeof(ColStats), h->stream));
        col_hist<<<cdiv(std::max<int64_t>(D, 1), 256), 256, 0, h->stream>>>(std::max<int64_t>(D, 1), 1, (int)h->N, h->colcnt.as<unsigned>(),
                                                                          nullptr, nullptr, h->colstats.as<ColStats>());
        LAUNCH_CHECK(h);
        GK_CUDA(cudaMemcpyAsync(h->h_colstats.p, h->colstats.p, sizeof(ColStats), cudaMemcpyDeviceToHost, h->stream));
        pro_enqueued = true;
      }
      if (prof) {
        std::vector<long long> pr((size_t)G * L * 16);
        GK_CUDA(cudaMemcpyAsync(pr.data(), h->K_stage.p, pr.size() * 8, cudaMemcpyDeviceToHost, h->stream));
        GK_CUDA(cudaStreamSynchronize(h->stream));
        long long t0 = pr[0];
        for (int b = 0; b < G; ++b) t0 = std::min(t0, pr[(size_t)b * L * 16]);
        fprintf(stderr, "[wl_fused2 prof] us; per level: avg over CTAs of the phase duration (max)\n");
        for (int lv = 0; lv < L; ++lv) {
          double avg[4] = {0}, mxv[4] = {0}, sub[5] = {0};
          long long end_max = 0;
          for (int b = 0; b < G; ++b) {
            const long long* q = &pr[((size_t)b * L + lv) * 16];
            end_max = std::max(end_max, q[6] - t0);
            if (lv == 0) {
              avg[3] += (double)(q[6] - q[0]) / G; mxv[3] = std::max(mxv[3], (double)(q[6] - q[0]));
              sub[0] += (double)(q[1] - q[0]) / G; sub[1] += (double)(q[2] - q[1]) / G; sub[2] += (double)(q[3] - q[2]) / G; sub[3] += (double)(q[6] - q[3]) / G;
              continue;
            }
            const double d[4] = {(double)(q[1] - q[0]), (double)(q[2] - q[1]), (double)(q[3] - q[2]), (double)(q[6] - q[3])};
            for (int k = 0; k < 4; ++k) { avg[k] += d[k] / G; mxv[k] = std::max(mxv[k], d[k]); }
            sub[0] += (double)(q[10] - q[0]) / G; sub[1] += (double)(q[1] - q[10]) / G;   // A: signatures | insert + copy-out
            sub[2] += (double)(q[4] - q[2]) / G; sub[3] += (double)(q[5] - q[4]) / G; sub[4] += (double)(q[3] - q[5]) / G;  // B: verify | labels | emit
          }
          if (lv == 0) {
            fprintf(stderr, "  level 0: %.1f (%.1f) = stage %.1f + emit %.1f + table clear %.1f + flush %.1f | done at %.1f us\n", avg[3] / 1e3, mxv[3] / 1e3,
                    sub[0] / 1e3, sub[1] / 1e3, sub[2] / 1e3, sub[3] / 1e3, end_max / 1e3);
            continue;
          }
          fprintf(stderr, "  level %d: A %.1f (%.1f) wait %.1f (%.1f) B+emit %.1f (%.1f) clear+flush %.1f (%.1f) | A = sig %.1f + insert %.1f | B = verify %.1f + labels %.1f + emit %.1f | level done at %.1f us\n", lv,
                  avg[0] / 1e3, mxv[0] / 1e3, avg[1] / 1e3, mxv[1] / 1e3, avg[2] / 1e3, mxv[2] / 1e3, avg[3] / 1e3, mxv[3] / 1e3,
                  sub[0] / 1e3, sub[1] / 1e3, sub[2] / 1e3, sub[3] / 1e3, sub[4] / 1e3, end_max / 1e3);
        }
      }
    } else if (fused) {
      // one persistent cooperative kernel for all levels; it appends (graph, column, count) entries
      // to ft_keys / ft_cnt used as a compact COO list
      if (L > 1) GK_CUDA(cudaMemsetAsync(h->ht_keys.as<unsigned long long>() + h->ht_cap, 0xFF, h->ht_cap * 8, h->stream));
      int* wb = h->wlf_buf.as<int>();
      int* d_cta_tile = wb + n_tiles + 1;
      int* d_cta_count = d_cta_tile + G + 1;
      unsigned* d_barrier = reinterpret_cast<unsigned*>(d_cta_count + G);
      GK_CUDA(cudaMemsetAsync(d_barrier, 0, 4, h->stream));
      WlFusedParams fp;
      memset(&fp, 0, sizeof(fp));
      fp.V = (int)V; fp.L = L;
      fp.graph_ptr = h->graph_ptr.as<int>();
      fp.row_ptr = h->row_ptr.as<int>(); fp.col_idx = h->col_idx.as<int>(); fp.vgraph = h->vgraph.as<int>();
      fp.labels0 = h->labels0.as<int>(); fp.tile_vbeg = wb; fp.cta_tile = d_cta_tile; fp.cta_count = d_cta_count;
      fp.barrier = d_barrier;
      fp.labels_all = labels_all; fp.sig_nbr = h->sig_nbr.as<int>(); fp.slot_of = h->slot_of.as<int>();
      fp.rank_pack = h->flags.as<int>();
      // singleton shortcut (wl_fused.cuh, SKIP): 0.293 vs 0.336 ms for all six levels of config 2, full GPU suite green
      // with it (profiles/r01l_*); GRAKEL_B200_WL_SKIP=0 selects the kernel without it
      const char* e_skip = getenv("GRAKEL_B200_WL_SKIP");
      const bool wl_skip = !(e_skip && atoi(e_skip) == 0);
      if (wl_skip) {
        GK_TRY(h->wl_single.ensure((size_t)V));
        GK_CUDA(cudaMemsetAsync(h->wl_single.p, 0, (size_t)V, h->stream));
        fp.single = h->wl_single.as<unsigned char>();
      }
      fp.table = h->ht_keys.as<unsigned long long>();
      fp.ht_mask = (unsigned)(h->ht_cap - 1);
      fp.coo_keys = h->ft_keys.as<unsigned long long>(); fp.coo_cnt = h->ft_cnt.as<unsigned>();
      fp.seed = seed; fp.st = fst; fp.sc = sc;
      const bool prof = getenv("GRAKEL_B200_PROF") != nullptr;
      if (prof) {
        GK_TRY(h->K_stage.ensure((size_t)G * L * 128));
        GK_CUDA(cudaMemsetAsync(h->K_stage.p, 0, (size_t)G * L * 128, h->stream));
        fp.prof = h->K_stage.as<long long>();
      }
      void* args[] = {&fp};
      GK_CUDA(cudaLaunchCooperativeKernel(wl_skip ? (void*)wl_fused_kernel<true> : (void*)wl_fused_kernel<false>, dim3(G),
                                          dim3(WLF_THREADS), args, WLF_SMEM, h->stream));
      LAUNCH_CHECK(h);
      if (prof) {
        std::vector<long long> pr((size_t)G * L * 16);
        GK_CUDA(cudaMemcpyAsync(pr.data(), h->K_stage.p, pr.size() * 8, cudaMemcpyDeviceToHost, h->stream));
        GK_CUDA(cudaStreamSynchronize(h->stream));
        long long t0 = pr[0];
        for (int b = 0; b < G; ++b) t0 = std::min(t0, pr[(size_t)b * L * 16]);
        fprintf(stderr, "[wl_fused prof] ns since kernel start; per level: phase = avg over CTAs of its duration (max)\n");
        for (int lv = 0; lv < L; ++lv) {
          const char* names[6] = {"A", "wait1", "B", "clear", "wait2", "C"};
          double avg[6] = {0}, mx[6] = {0};
          long long end_max = 0;
          for (int b = 0; b < G; ++b) {
            const long long* q = &pr[((size_t)b * L + lv) * 16];
            end_max = std::max(end_max, q[6] - t0);
            if (lv == 0) { avg[5] += (double)(q[6] - q[0]) / G; mx[5] = std::max(mx[5], (double)(q[6] - q[0])); continue; }
            for (int k = 0; k < 6; ++k) { const double d = (double)(q[k + 1] - q[k]); avg[k] += d / G; mx[k] = std::max(mx[k], d); }
          }
          fprintf(stderr, "  level %d:", lv);
          for (int k = 0; k < 6; ++k) fprintf(stderr, " %s %.1f (%.1f)", names[k], avg[k] / 1e3, mx[k] / 1e3);
          if (lv) {  // split of phase A (last tile of each CTA): stage | thread-per-vertex | warp-per-vertex | copy-out
            double sa[4] = {0};
            for (int b = 0; b < G; ++b) {
              const long long* q = &pr[((size_t)b * L + lv) * 16];
              sa[0] += (double)(q[8] - q[0]) / G; sa[1] += (double)(q[9] - q[8]) / G;
              sa[2] += (double)(q[10] - q[9]) / G; sa[3] += (double)(q[1] - q[10]) / G;
            }
            fprintf(stderr, " | A = stage %.1f + thread %.1f + warp %.1f + out %.1f", sa[0] / 1e3, sa[1] / 1e3, sa[2] / 1e3, sa[3] / 1e3);
          }
          fprintf(stderr, " | level done at %.1f us\n", end_max / 1e3);
        }
      }
    } else {
    GK_CUDA(cudaMemsetAsync(h->ft_keys.p, 0xFF, h->ft_cap * 8, h->stream));
    GK_CUDA(cudaMemsetAsync(h->ft_cnt.p, 0, h->ft_cap * 4, h->stream));
    GK_CUDA(cudaMemcpyAsync(labels_all, h->labels0.p, V * 4, cudaMemcpyDeviceToDevice, h->stream));
    wl_insert_level0<<<nb, 256, 0, h->stream>>>((int)V, labels_all, h->vgraph.as<int>(),
                                                 h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(),
                                                 (unsigned)(ft_level_cap - 1), fst);
    LAUNCH_CHECK(h);
    for (int lv = 1; lv < L; ++lv) {
      const int* lab_in = labels_all + (size_t)(lv - 1) * V;
      int* lab_out = labels_all + (size_t)lv * V;
      GK_CUDA(cudaMemsetAsync(h->ht_keys.p, 0xFF, h->ht_cap * 8, h->stream));
      GK_CUDA(cudaMemsetAsync(h->ht_rep.p, 0x7F, h->ht_cap * 4, h->stream));
      if (h->group_width <= 8) {
        wl_sig_thread8<<<nb, 256, 0, h->stream>>>((int)V, h->row_ptr.as<int>(), h->col_idx.as<int>(), lab_in,
                                                  h->sig_nbr.as<int>(), seed, h->ht_keys.as<unsigned long long>(),
                                                  h->ht_rep.as<int>(), (unsigned)(h->ht_cap - 1), h->slot_of.as<int>());
      } else if (h->group_width == 16) {
        launch_sig_small<16>(h, lab_in, seed);
      } else {
        launch_sig_small<32>(h, lab_in, seed);
      }
      LAUNCH_CHECK(h);
      if (h->n_large) {
        wl_sig_large<<<cdiv(h->n_large * 32, 256), 256, 0, h->stream>>>(
            (int)h->n_large, h->large_list.as<int>(), h->row_ptr.as<int>(), h->col_idx.as<int>(), lab_in,
            h->sig_nbr.as<int>(), seed, h->ht_keys.as<unsigned long long>(), h->ht_rep.as<int>(),
            (unsigned)(h->ht_cap - 1), h->slot_of.as<int>());
        LAUNCH_CHECK(h);
      }
      wl_resolve<<<nb, 256, 0, h->stream>>>((int)V, h->row_ptr.as<int>(), lab_in, h->sig_nbr.as<int>(),
                                            h->ht_rep.as<int>(), h->slot_of.as<int>(), h->flags.as<int>(),
                                            h->block_sums.as<int>(), sc);
      LAUNCH_CHECK(h);
      wl_assign<<<nb, 256, 0, h->stream>>>((int)V, lv, h->flags.as<int>(), h->block_sums.as<int>(), lab_out, sc);
      LAUNCH_CHECK(h);
      wl_gather_insert<<<nb, 256, 0, h->stream>>>((int)V, lv, h->slot_of.as<int>(), lab_out, h->vgraph.as<int>(),
                                                   fst, h->ft_keys.as<unsigned long long>(),
                                                   h->ft_cnt.as<unsigned>(), (unsigned)(ft_level_cap - 1));
      LAUNCH_CHECK(h);
    }
    }  // multi-kernel path
    DevScalars* hs;
    GK_TRY(read_scalars(h, &hs));
    if (hs->ft_overflow) return fail(GK_ERR_STATE, "gk_wl_features: feature table overflow");
    if (!hs->collision) break;
  }
  if (!used_v2) {  // (wl_fused2 recorded the end of its stage right after the kernel; read_scalars synchronised)
    GK_CUDA(cudaEventRecord(h->tev[3], h->stream));
    GK_CUDA(cudaEventSynchronize(h->tev[3]));
  }
  DevScalars* hs = h->h_scalars.as<DevScalars>();
  h->n_columns = hs->level_base[L];
  h->features_ready = true; h->feat_serial++;
  h->feature_kind = 1;
  if (pro_enqueued) {
    HandleExtra* ex = extra_of(h);
    ex->pro_hist = *h->h_colstats.as<ColStats>();
    ex->pro_max_count = (long long)hs->max_count; ex->pro_max_diag = (long long)hs->max_diag; ex->pro_n_entries = (long long)hs->n_entries;
    h->pro_serial = h->feat_serial;
  }
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = h->N; stats->n_vertices = V; stats->n_edges = E;
    stats->n_levels = L;
    for (int i = 0; i < L; ++i) stats->level_dims[i] = hs->level_dims[i];
    stats->n_columns = h->n_columns;
    if (h->wl_sparse_ids) {  // the column space is sparse (n_labels0 + (L-1) V wide); report the number of classes
      stats->n_columns = 0;
      for (int i = 0; i < L; ++i) stats->n_columns += hs->level_dims[i];
    }
    stats->hash_retries = retries;
    stats->kernel_launches = h->launches - launches0;
    stats->ms_features = ev_ms(h->tev[2], h->tev[3]);
  }
  return GK_OK;
}

// WL-OA: the WL feature block, then its unary expansion (wl_oa.cuh); one gk_gram of the expanded
// block is the histogram-intersection matrix of weisfeiler_lehman_optimal_assignment.py:257-266.
int gk_wl_oa_features(gk_handle* h, int32_t n_iter, gk_stats* stats) {
  gk_stats local;
  gk_stats* st = stats ? stats : &local;
  GK_TRY(gk_wl_features(h, n_iter, st));
  h->features_ready = false; h->feat_serial++;
  const int64_t launches0 = h->launches;
  const int64_t D = std::max<int64_t>(h->n_columns, 1);
  const size_t out_cap = std::max<size_t>((size_t)h->V * (size_t)h->n_levels, 1);  // one entry per (vertex, level)
  if (out_cap > (1ULL << 31)) return fail(GK_ERR_ARG, "gk_wl_oa_features: feature block too large");
  GK_TRY(h->oa_keys.ensure(out_cap * 8));
  GK_TRY(h->oa_cnt.ensure(out_cap * 4));
  GK_TRY(h->oa_colcnt.ensure((out_cap + 1) * 4));
  GK_TRY(h->colmin.ensure(D * 4));  // scratch until the next gk_gram: largest count / first threshold column
  GK_TRY(h->colmax.ensure(D * 4));
  GK_TRY(h->colstats.ensure(std::max(sizeof(ColStats), sizeof(OaCursors))));
  GK_TRY(h->h_colstats.ensure(std::max(sizeof(ColStats), sizeof(OaCursors))));
  OaCursors* cur = h->colstats.as<OaCursors>();
  unsigned* colmaxcnt = h->colmin.as<unsigned>();
  unsigned* colbase = h->colmax.as<unsigned>();
  GK_CUDA(cudaMemsetAsync(cur, 0, sizeof(OaCursors), h->stream));
  GK_CUDA(cudaMemsetAsync(colmaxcnt, 0, D * 4, h->stream));
  GK_CUDA(cudaMemsetAsync(h->oa_keys.p, 0xFF, out_cap * 8, h->stream));
  GK_CUDA(cudaMemsetAsync(h->oa_colcnt.p, 0, (out_cap + 1) * 4, h->stream));
  GK_CUDA(cudaMemsetAsync(h->diag_u64.p, 0, h->N * 8, h->stream));
  oa_colmax<<<h->sm_count * 8, 256, 0, h->stream>>>(h->ft_cap, h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(),
                                                    colmaxcnt);
  LAUNCH_CHECK(h);
  oa_colbase<<<cdiv(D, OA_THREADS), OA_THREADS, 0, h->stream>>>(D, colmaxcnt, colbase, cur);
  LAUNCH_CHECK(h);
  oa_expand<<<cdiv((long long)h->ft_cap, OA_THREADS), OA_THREADS, 0, h->stream>>>(
      h->ft_cap, h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(), colbase, out_cap,
      h->oa_keys.as<unsigned long long>(), h->oa_cnt.as<unsigned>(), cur, h->oa_colcnt.as<unsigned>(),
      h->diag_u64.as<unsigned long long>(), h->scalars.as<DevScalars>());
  LAUNCH_CHECK(h);
  if (h->wl_sparse_ids) {  // frozen vertices wrote no entries: their (level) units of self similarity are kept aside
    add_u64<<<cdiv(h->N, 256), 256, 0, h->stream>>>((int)h->N, h->diag_frozen.as<unsigned long long>(), h->diag_u64.as<unsigned long long>());
    LAUNCH_CHECK(h);
  }
  h->n_part = 1;
  oa_finish<<<1, 1, 0, h->stream>>>(cur, h->part_max.as<unsigned>(), h->part_new.as<unsigned>(), h->scalars.as<DevScalars>(),
                                    h->wl_sparse_ids ? 1 : 0);
  LAUNCH_CHECK(h);
  GK_CUDA(cudaMemcpyAsync(h->h_colstats.p, cur, sizeof(OaCursors), cudaMemcpyDeviceToHost, h->stream));
  DevScalars* hs;
  GK_TRY(read_scalars(h, &hs));
  GK_CUDA(cudaEventRecord(h->tev[3], h->stream));
  GK_CUDA(cudaEventSynchronize(h->tev[3]));
  if (hs->ft_overflow) return fail(GK_ERR_STATE, "gk_wl_oa_features: expanded feature block overflow");
  const OaCursors hc = *h->h_colstats.as<OaCursors>();
  std::swap(h->ft_keys, h->oa_keys);
  std::swap(h->ft_cnt, h->oa_cnt);
  std::swap(h->colcnt, h->oa_colcnt);
  h->ft_cap = out_cap;
  h->col_cap = (int64_t)out_cap + 1;
  h->n_columns = (int64_t)hc.n_cols;
  h->features_ready = true; h->feat_serial++;
  st->n_columns = h->n_columns;
  st->kernel_launches += h->launches - launches0;
  st->ms_features = ev_ms(h->tev[2], h->tev[3]);
  return GK_OK;
}

// dense first-occurrence ids of level `level` (>= 1) of a wl_fused2 run into `dst` (device, V ints)
static int wl_densify(gk_handle* h, int level, int* dst) {
  const int V = (int)h->V;
  const int nb = cdiv(V, DENS_THREADS);
  GK_TRY(h->block_sums.ensure((size_t)nb * 4));
  GK_TRY(h->flags.ensure((size_t)V * 4));
  const int* lab = h->labels_all.as<int>() + (size_t)level * V;
  wl_dens_count<<<nb, DENS_THREADS, 0, h->stream>>>(V, lab, h->block_sums.as<int>());
  LAUNCH_CHECK(h);
  wl_dens_scan<<<1, DENS_THREADS, 0, h->stream>>>(nb, h->block_sums.as<int>());
  LAUNCH_CHECK(h);
  wl_dens_rank<<<nb, DENS_THREADS, 0, h->stream>>>(V, lab, h->block_sums.as<int>(), h->flags.as<int>());
  LAUNCH_CHECK(h);
  wl_dens_apply<<<cdiv(V, 256), 256, 0, h->stream>>>(V, lab, h->flags.as<int>(), dst);
  LAUNCH_CHECK(h);
  return GK_OK;
}

int gk_wl_labels(gk_handle* h, int32_t level, int32_t* out) {
  if (!h || !out) return fail(GK_ERR_ARG, "gk_wl_labels: null argument");
  if (h->feature_kind != 1 || level < 0 || level >= h->n_levels) return fail(GK_ERR_STATE, "gk_wl_labels: no such level");
  GK_CUDA(cudaSetDevice(h->dev));
  const int* src = h->labels_all.as<int>() + (size_t)level * h->V;
  if (h->wl_sparse_ids && level >= 1) {
    GK_TRY(wl_densify(h, level, h->slot_of.as<int>()));
    src = h->slot_of.as<int>();
  }
  GK_CUDA(cudaMemcpyAsync(out, src, h->V * 4, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

// ---------------------------------------------------------------------------
// NeighborhoodHash (nh.cuh).  gk_nh_features: the R relabel levels, then per level the histogram of the non-None
// labels (dense column ids of the labels present) and its unary expansion (wl_oa.cuh), kept for gk_nh_gram.
static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

int gk_nh_features(gk_handle* h, int32_t R, int32_t bits, int32_t flags, const int64_t* labels0, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->N <= 0) return fail(GK_ERR_STATE, "gk_nh_features: no graphs packed");
  if (R < 1 || R >= MAX_LEVELS) return fail(GK_ERR_ARG, "gk_nh_features: R out of range");
  if (bits < 1 || bits > 63) return fail(GK_ERR_ARG, "gk_nh_features: bits must be in 1 .. 63");
  const int64_t V = h->V, N = h->N;
  if (V > 0 && !labels0) return fail(GK_ERR_ARG, "gk_nh_features: labels0 is required");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t launches0 = h->launches;
  h->features_ready = false; h->feat_serial++;
  h->feature_kind = 0;
  const size_t Vs = (size_t)std::max<int64_t>(V, 1);
  const unsigned long long mask = (1ULL << bits) - 1ULL;
  const bool cs = flags & GK_NH_COUNT_SENSITIVE;
  GK_TRY(h->nh_labels.ensure((size_t)(R + 1) * Vs * 8));
  GK_TRY(h->nh_keys.ensure((size_t)R * Vs * 8));
  GK_TRY(h->nh_cnt.ensure((size_t)R * Vs * 4));
  GK_TRY(h->nh_colcnt.ensure((size_t)R * (Vs + 1) * 4));
  GK_TRY(h->nh_diag.ensure((size_t)R * N * 8));
  unsigned long long* lab = h->nh_labels.as<unsigned long long>();
  // scratch: sorted labels | sorted graph ids | flags | scan | count-block keys | counts | run starts | per-level
  // counters + cursors | CUB temporary storage
  size_t sort_tmp = 0, scan_tmp = 0;
  GK_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                          (const int*)nullptr, (int*)nullptr, (int)Vs, 0, 64, h->stream));
  GK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                        (int)Vs, h->stream));
  const size_t o_sg = align256(Vs * 8), o_flag = o_sg + align256(Vs * 4), o_pos = o_flag + align256(Vs * 8),
               o_ck = o_pos + align256(Vs * 8), o_cc = o_ck + align256(Vs * 8), o_first = o_cc + align256(Vs * 4),
               o_small = o_first + align256((Vs + 1) * 4),
               o_cub = o_small + align256((size_t)R * (sizeof(NhLevelCounts) + sizeof(OaCursors))),
               tmp_bytes = o_cub + std::max(sort_tmp, scan_tmp);
  GK_TRY(h->nh_tmp.ensure(tmp_bytes));
  char* tb = h->nh_tmp.as<char>();
  unsigned long long* sk = reinterpret_cast<unsigned long long*>(tb);
  int* sg = reinterpret_cast<int*>(tb + o_sg);
  unsigned long long* flag = reinterpret_cast<unsigned long long*>(tb + o_flag);
  unsigned long long* pos = reinterpret_cast<unsigned long long*>(tb + o_pos);
  unsigned long long* ck = reinterpret_cast<unsigned long long*>(tb + o_ck);
  unsigned* cc = reinterpret_cast<unsigned*>(tb + o_cc);
  int* first = reinterpret_cast<int*>(tb + o_first);
  NhLevelCounts* lc = reinterpret_cast<NhLevelCounts*>(tb + o_small);
  OaCursors* oc = reinterpret_cast<OaCursors*>(tb + o_small + (size_t)R * sizeof(NhLevelCounts));
  void* cub_tmp = tb + o_cub;
  GK_TRY(h->colmin.ensure(Vs * 4));  // largest count / first threshold column of every count-block column
  GK_TRY(h->colmax.ensure(Vs * 4));
  DevScalars* sc = h->scalars.as<DevScalars>();

  GK_CUDA(cudaEventRecord(h->tev[2], h->stream));
  if (V) GK_CUDA(cudaMemcpyAsync(lab, labels0, V * 8, cudaMemcpyHostToDevice, h->stream));  // -1 = all ones = None
  for (int r = 1; r <= R && V; ++r) {  // slot r = level r - 1 = NH_ applied r times (:196-198)
    const unsigned long long* in = lab + (size_t)(r - 1) * V;
    unsigned long long* out = lab + (size_t)r * V;
    const int width = h->group_width;  // wider rows are in the packed large list
    if (cs) nh_relabel<true><<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, width, h->row_ptr.as<int>(), h->col_idx.as<int>(), in, out, bits, mask);
    else nh_relabel<false><<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, width, h->row_ptr.as<int>(), h->col_idx.as<int>(), in, out, bits, mask);
    LAUNCH_CHECK(h);
    if (h->n_large) {
      const int grid = cdiv(h->n_large * 32, 256);
      if (cs) nh_relabel_warp<true><<<grid, 256, 0, h->stream>>>((int)h->n_large, h->large_list.as<int>(), h->row_ptr.as<int>(), h->col_idx.as<int>(), in, out, bits, mask);
      else nh_relabel_warp<false><<<grid, 256, 0, h->stream>>>((int)h->n_large, h->large_list.as<int>(), h->row_ptr.as<int>(), h->col_idx.as<int>(), in, out, bits, mask);
      LAUNCH_CHECK(h);
    }
  }
  GK_CUDA(cudaEventRecord(h->tev[3], h->stream));

  GK_CUDA(cudaMemsetAsync(tb + o_small, 0, (size_t)R * (sizeof(NhLevelCounts) + sizeof(OaCursors)), h->stream));
  GK_CUDA(cudaMemsetAsync(&sc->ft_overflow, 0, sizeof(unsigned), h->stream));
  GK_CUDA(cudaMemsetAsync(h->nh_keys.p, 0xFF, (size_t)R * Vs * 8, h->stream));
  GK_CUDA(cudaMemsetAsync(h->nh_colcnt.p, 0, (size_t)R * (Vs + 1) * 4, h->stream));
  GK_CUDA(cudaMemsetAsync(h->nh_diag.p, 0, (size_t)R * N * 8, h->stream));
  for (int r = 0; r < R && V; ++r) {
    size_t t1 = sort_tmp;
    GK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, t1, lab + (size_t)(r + 1) * V, sk, h->vgraph.as<int>(), sg, (int)V, 0, 64,
                                            h->stream));
    h->launches++;
    nh_mark<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, sk, sg, flag);
    LAUNCH_CHECK(h);
    size_t t2 = scan_tmp;
    GK_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, t2, flag, pos, (int)V, h->stream));
    h->launches++;
    GK_CUDA(cudaMemsetAsync(ck, 0xFF, (size_t)V * 8, h->stream));
    nh_emit<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, sk, sg, flag, pos, ck, first, lc + r);
    LAUNCH_CHECK(h);
    nh_counts<<<cdiv(V, 256), 256, 0, h->stream>>>((int)V, first, lc + r, cc);
    LAUNCH_CHECK(h);
    // unary expansion of the count block: one entry per non-None vertex (gk_wl_oa_features does the same for WL)
    unsigned* colmaxcnt = h->colmin.as<unsigned>();
    unsigned* colbase = h->colmax.as<unsigned>();
    GK_CUDA(cudaMemsetAsync(colmaxcnt, 0, (size_t)V * 4, h->stream));
    oa_colmax<<<h->sm_count * 8, 256, 0, h->stream>>>((size_t)V, ck, cc, colmaxcnt);
    LAUNCH_CHECK(h);
    oa_colbase<<<cdiv(V, OA_THREADS), OA_THREADS, 0, h->stream>>>(V, colmaxcnt, colbase, oc + r);
    LAUNCH_CHECK(h);
    oa_expand<<<cdiv(V, OA_THREADS), OA_THREADS, 0, h->stream>>>(
        (size_t)V, ck, cc, colbase, (size_t)V, h->nh_keys.as<unsigned long long>() + (size_t)r * Vs,
        h->nh_cnt.as<unsigned>() + (size_t)r * Vs, oc + r, h->nh_colcnt.as<unsigned>() + (size_t)r * (Vs + 1),
        h->nh_diag.as<unsigned long long>() + (size_t)r * N, sc);
    LAUNCH_CHECK(h);
  }
  GK_CUDA(cudaEventRecord(h->ev[13], h->stream));
  std::vector<NhLevelCounts> hl(R);
  std::vector<OaCursors> ho(R);
  GK_CUDA(cudaMemcpyAsync(hl.data(), lc, (size_t)R * sizeof(NhLevelCounts), cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaMemcpyAsync(ho.data(), oc, (size_t)R * sizeof(OaCursors), cudaMemcpyDeviceToHost, h->stream));
  DevScalars* hs;
  GK_TRY(read_scalars(h, &hs));
  if (hs->ft_overflow) return fail(GK_ERR_STATE, "gk_nh_features: expanded feature block overflow");
  HandleExtra* ex = extra_of(h);
  ex->nh_cols.assign(R, 0);
  ex->nh_entries.assign(R, 0);
  int64_t tot_cols = 0, tot_ent = 0;
  for (int r = 0; r < R; ++r) {
    ex->nh_cols[r] = (long long)ho[r].n_cols;
    ex->nh_entries[r] = (long long)ho[r].n_entries;
    tot_cols += ex->nh_cols[r];
    tot_ent += ex->nh_entries[r];
  }
  h->nh_R = R;
  h->n_levels = R;
  h->feature_kind = 4;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = N; stats->n_vertices = V; stats->n_edges = h->E;
    stats->n_levels = R;
    for (int r = 0; r < R; ++r) stats->level_dims[r] = (int64_t)hl[r].n_cols;
    stats->n_columns = tot_cols;
    stats->n_entries = tot_ent;
    stats->kernel_launches = h->launches - launches0;
    stats->ms_features = ev_ms(h->tev[2], h->tev[3]);
    stats->ms_panel = ev_ms(h->tev[3], h->ev[13]);
  }
  return GK_OK;
}

// gk_gram over level r's expanded block: the handle's feature-block buffers are pointed at the level's slices for the
// call and restored afterwards (gk_gram reads them, it never reallocates them)
static int nh_level_gram(gk_handle* h, int r, int64_t n_fit, int32_t flags, float* d_kf, int64_t ldf, gk_stats* gs) {
  const size_t Vs = (size_t)std::max<int64_t>(h->V, 1);
  HandleExtra* ex = extra_of(h);
  DevBuf lk, lc, lcc, ld;
  lk.p = h->nh_keys.as<unsigned long long>() + (size_t)r * Vs; lk.cap = Vs * 8;
  lc.p = h->nh_cnt.as<unsigned>() + (size_t)r * Vs; lc.cap = Vs * 4;
  lcc.p = h->nh_colcnt.as<unsigned>() + (size_t)r * (Vs + 1); lcc.cap = (Vs + 1) * 4;
  ld.p = h->nh_diag.as<unsigned long long>() + (size_t)r * h->N; ld.cap = (size_t)h->N * 8;
  GK_TRY(h->part_max.ensure(4));
  GK_TRY(h->part_new.ensure(4));
  nh_parts<<<1, 1, 0, h->stream>>>((unsigned long long)ex->nh_entries[r], h->part_max.as<unsigned>(), h->part_new.as<unsigned>());
  LAUNCH_CHECK(h);
  const size_t ft_cap0 = h->ft_cap;
  const int64_t col_cap0 = h->col_cap, n_columns0 = h->n_columns, n_part0 = h->n_part;
  std::swap(h->ft_keys, lk); std::swap(h->ft_cnt, lc); std::swap(h->colcnt, lcc); std::swap(h->diag_u64, ld);
  h->ft_cap = Vs; h->col_cap = (int64_t)Vs + 1; h->n_columns = ex->nh_cols[r]; h->n_part = 1;
  h->features_ready = true; h->feat_serial++;
  const int rc = gk_gram(h, n_fit, GK_OUT_DEVICE | (flags & (GK_GRAM_SIMT | GK_DENSE_ALL)), 0, -1, d_kf, GK_F32, ldf,
                         nullptr, nullptr, gs);
  std::swap(h->ft_keys, lk); std::swap(h->ft_cnt, lc); std::swap(h->colcnt, lcc); std::swap(h->diag_u64, ld);
  h->ft_cap = ft_cap0; h->col_cap = col_cap0; h->n_columns = n_columns0; h->n_part = n_part0;
  h->features_ready = false; h->feat_serial++;
  return rc;
}

int gk_nh_gram(gk_handle* h, int64_t n_fit, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->feature_kind != 4 || h->nh_R < 1) return fail(GK_ERR_STATE, "gk_nh_gram: no NeighborhoodHash levels (call gk_nh_features)");
  if (out_dtype != GK_F64) return fail(GK_ERR_UNSUPPORTED, "gk_nh_gram: the NeighborhoodHash Gram is fp64 only");
  if (h->n_rows > 0) return fail(GK_ERR_UNSUPPORTED, "gk_nh_gram: row map with NeighborhoodHash levels");
  if (flags & (GK_NORMALIZE | GK_DIST | GK_DIST_GATHER)) return fail(GK_ERR_UNSUPPORTED, "gk_nh_gram: unsupported flag");
  const int64_t N = h->N;
  if (n_fit <= 0 || n_fit > N) return fail(GK_ERR_ARG, "gk_nh_gram: n_fit out of range");
  // level intersections are fp32 integers: exact while every graph has fewer than 2^24 vertices
  if (h->max_graph_size >= (1 << 24)) return fail(GK_ERR_RANGE, "gk_nh_gram: a graph with 2^24 or more vertices");
  GK_CUDA(cudaSetDevice(h->dev));
  const bool square = n_fit == N;
  const int64_t rows = square ? N : N - n_fit, cols = n_fit;
  const int row0 = square ? 0 : (int)n_fit;
  const bool dev_out = flags & GK_OUT_DEVICE;
  if (dev_out && !K_out) return fail(GK_ERR_ARG, "gk_nh_gram: GK_OUT_DEVICE without a pointer");
  if (ld <= 0) ld = cols;
  if (ld < cols) return fail(GK_ERR_ARG, "gk_nh_gram: ld smaller than the row length");
  const int64_t launches0 = h->launches;
  const int64_t ldf = (cols + 7) / 8 * 8;  // 32-byte rows: TMA stores of the level Gram
  const int R = h->nh_R;
  const size_t level_stride = (size_t)std::max<int64_t>(rows, 1) * ldf;  // the R level Grams side by side
  GK_TRY(h->nh_kf.ensure((size_t)R * level_stride * 4));
  double* K64;
  int64_t ldk;
  if (dev_out) {
    K64 = reinterpret_cast<double*>(K_out);
    ldk = ld;
  } else {  // library-owned result (gk_result_device / gk_fetch)
    GK_TRY(h->K.ensure((size_t)std::max<int64_t>(rows, 1) * cols * 8));
    K64 = h->K.as<double>();
    ldk = cols;
    h->K_rows = rows; h->K_cols = cols; h->K_ld = cols; h->K_dtype = GK_F64;
  }
  gk_stats gs;
  memset(&gs, 0, sizeof(gs));
  float ms_gram = 0.f, ms_comb = 0.f;
  for (int r = 0; r < R && rows > 0; ++r) {
    memset(&gs, 0, sizeof(gs));
    GK_TRY(nh_level_gram(h, r, n_fit, flags, h->nh_kf.as<float>() + (size_t)r * level_stride, ldf, &gs));
    ms_gram += gs.ms_total;
  }
  if (rows > 0) {
    GK_CUDA(cudaEventRecord(h->tev[0], h->stream));
    nh_combine<<<h->sm_count * 8, 256, 0, h->stream>>>(rows, cols, row0, h->graph_ptr.as<int>(), h->nh_kf.as<float>(), ldf,
                                                       (long long)level_stride, R, K64, ldk);
    LAUNCH_CHECK(h);
    GK_CUDA(cudaEventRecord(h->tev[1], h->stream));
    GK_CUDA(cudaEventSynchronize(h->tev[1]));
    ms_comb = ev_ms(h->tev[0], h->tev[1]);
  }
  h->feature_kind = 4;  // the levels stay usable (a second gk_nh_gram, gk_nh_labels)
  GK_CUDA(cudaEventRecord(h->ev[14], h->stream));
  if (K_out && !dev_out && rows > 0)
    GK_CUDA(cudaMemcpy2DAsync(K_out, (size_t)ld * 8, K64, (size_t)ldk * 8, (size_t)cols * 8, (size_t)rows,
                              cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaEventRecord(h->ev[15], h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  if (stats) {
    const gk_stats last = gs;
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = N; stats->n_vertices = h->V; stats->n_edges = h->E;
    stats->n_levels = R;
    stats->n_dense_columns = last.n_dense_columns;
    stats->n_tail_columns = last.n_tail_columns;
    stats->threshold = last.threshold;
    stats->gram_path = last.gram_path;
    stats->max_diag = last.max_diag;
    stats->gemm_tiles = last.gemm_tiles;
    stats->kernel_launches = h->launches - launches0;
    stats->ms_gemm = ms_gram;
    stats->ms_tail = ms_comb;
    stats->ms_d2h = ev_ms(h->ev[14], h->ev[15]);
    stats->ms_total = ms_gram + ms_comb + stats->ms_d2h;
  }
  return GK_OK;
}

int gk_nh_labels(gk_handle* h, int32_t level, uint64_t* out) {
  if (!h || !out) return fail(GK_ERR_ARG, "gk_nh_labels: null argument");
  if (h->feature_kind != 4 || level < 0 || level >= h->nh_R) return fail(GK_ERR_STATE, "gk_nh_labels: no such level");
  GK_CUDA(cudaSetDevice(h->dev));
  if (h->V)
    GK_CUDA(cudaMemcpyAsync(out, h->nh_labels.as<unsigned long long>() + (size_t)(level + 1) * h->V, h->V * 8,
                            cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

// ---------------------------------------------------------------------------
// Shortest-path features.  wl_iter < 0: the ShortestPath kernel on the packed labels.
// wl_iter >= 0: WeisfeilerLehman(base_graph_kernel=ShortestPath) -- the graphs are relabelled for
// wl_iter rounds first (gk_wl_features), then the labelled path histogram of EVERY level goes into one
// feature block: label ids are made level-unique (id + first column of the level), so the levels use
// disjoint columns and one Gram equals the reference's sum of per-level matrices
// (weisfeiler_lehman.py:260-270 with shortest_path.py:370-410 as the base kernel).
static int sp_features_impl(gk_handle* h, int32_t flags, int32_t wl_iter, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->N <= 0) return fail(GK_ERR_STATE, "gk_sp_features: no graphs packed");
  GK_CUDA(cudaSetDevice(h->dev));
  const bool with_labels = flags & GK_SP_WITH_LABELS;
  if (with_labels && !h->has_labels) return fail(GK_ERR_ARG, "gk_sp_features: vertex labels are required");
  std::vector<long long> level_base(1, 0);  // first label id of each pass
  int n_pass = 1;
  long long n_labels_total = h->n_labels0;
  if (wl_iter >= 0) {
    if (!with_labels) return fail(GK_ERR_ARG, "gk_wl_sp_features: the base kernel needs vertex labels");
    gk_stats wst;
    GK_TRY(gk_wl_features(h, wl_iter, &wst));
    if (h->wl_sparse_ids) {  // the base kernel's counters are indexed by dense label ids
      for (int lv = 1; lv <= wl_iter; ++lv) GK_TRY(wl_densify(h, lv, h->labels_all.as<int>() + (size_t)lv * h->V));
      h->wl_sparse_ids = false;
    }
    n_pass = wl_iter + 1;
    level_base.assign(n_pass + 1, 0);
    for (int l = 0; l < n_pass; ++l) level_base[l + 1] = level_base[l] + wst.level_dims[l];
    n_labels_total = level_base[n_pass];
  }
  if (with_labels && n_labels_total >= (1 << 20)) return fail(GK_ERR_UNSUPPORTED, "gk_sp_features: more than 2^20 distinct labels");
  const bool use_u16 = (!h->has_weights || h->unit_weights) && h->max_graph_size < 16000;
  const size_t esz = use_u16 ? 2 : 8;
  HandleExtra* ex = extra_of(h);
  const int64_t N = h->N;
  const int64_t launches0 = h->launches;
  h->features_ready = false; h->feat_serial++;
  h->sp_flags = flags;

  // plan: graphs whose distance matrix fits the shared-memory budget vs the rest
  const size_t SMEM_DIST_MAX = 160 * 1024;
  std::vector<int> small, big;
  std::vector<int> bfs[4];  // unit weights: bitmask BFS with W = 1, 2, 4, 8 words (n <= 64 W)
  size_t max_small_nn = 0;
  ex->sp_goff.assign(N + 1, 0);
  const bool keep = flags & GK_SP_KEEP_DIST;
  long long off_big = 0, off_all = 0;
  std::vector<long long> goff_big(N, 0);
  for (int64_t g = 0; g < N; ++g) {
    const long long n = ex->graph_ptr[g + 1] - ex->graph_ptr[g];
    ex->sp_goff[g] = off_all;
    off_all += n * n;
    if (use_u16 && n <= 512) {
      bfs[n <= 64 ? 0 : n <= 128 ? 1 : n <= 256 ? 2 : 3].push_back((int)g);
    } else if ((size_t)(n * n) * esz <= SMEM_DIST_MAX) {
      small.push_back((int)g);
      max_small_nn = std::max(max_small_nn, (size_t)(n * n));
    } else {
      big.push_back((int)g);
      goff_big[g] = off_big;
      off_big += n * n;
    }
  }
  ex->sp_goff[N] = off_all;
  const size_t smem_small = SP_LOCAL_SLOTS * 12 + max_small_nn * esz + 16;
  const size_t smem_big = SP_LOCAL_SLOTS * 12 + 16;

  // device buffers
  gk::DevBuf& lists = h->sp_lists;  // [small list | big list | BFS classes]
  GK_TRY(lists.ensure((size_t)N * 4 + 16));
  std::vector<int> order(small);
  order.insert(order.end(), big.begin(), big.end());
  size_t bfs_off[4];
  for (int i = 0; i < 4; ++i) { bfs_off[i] = order.size(); order.insert(order.end(), bfs[i].begin(), bfs[i].end()); }
  GK_CUDA(cudaMemcpyAsync(lists.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, h->stream));
  GK_TRY(h->sp_graph_off.ensure((size_t)(N + 1) * 8 * 2));
  long long* d_goff_all = h->sp_graph_off.as<long long>();
  long long* d_goff_big = d_goff_all + (N + 1);
  GK_CUDA(cudaMemcpyAsync(d_goff_all, ex->sp_goff.data(), (N + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaMemcpyAsync(d_goff_big, goff_big.data(), N * 8, cudaMemcpyHostToDevice, h->stream));
  if (off_big) GK_TRY(h->sp_dist.ensure((size_t)off_big * esz));
  double* d_keep = nullptr;
  if (keep) {
    GK_TRY(h->K_stage.ensure((size_t)off_all * 8));
    d_keep = h->K_stage.as<double>();
  }
  GK_CUDA(cudaStreamSynchronize(h->stream));  // host vectors above go out of scope on retry

  if (use_u16) {
    GK_CUDA(cudaFuncSetAttribute(sp_apsp_hist<unsigned short>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(smem_small, smem_big)));
  } else {
    GK_CUDA(cudaFuncSetAttribute(sp_apsp_hist<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(smem_small, smem_big)));
  }

  size_t dict_cap = std::max<size_t>(h->sp_dict_cap, 1 << 16);
  size_t dkey_cap = 1 << 18;
  bool real_mode = false;
  size_t ft_cap = std::max<size_t>(next_pow2((size_t)std::max<int64_t>(h->V, 1024) * 16 * (size_t)std::min(n_pass, 4)), 1 << 20);
  DevScalars* sc = h->scalars.as<DevScalars>();
  GK_CUDA(cudaEventRecord(h->tev[2], h->stream));
  for (int attempt = 0;; ++attempt) {
    if (attempt > 6) return fail(GK_ERR_STATE, "gk_sp_features: tables keep overflowing");
    if (dict_cap > (1ULL << 28) || ft_cap > (1ULL << 31)) return fail(GK_ERR_STATE, "gk_sp_features: feature tables too large");
    GK_TRY(h->sp_dict_keys.ensure(dict_cap * 8));
    GK_TRY(h->ft_keys.ensure(ft_cap * 8));
    GK_TRY(h->ft_cnt.ensure(ft_cap * 4));
    h->sp_dict_cap = dict_cap;
    h->ft_cap = ft_cap;
    GK_TRY(init_scalars(h, 0));
    FeatStats fst;
    GK_TRY(reset_feature_stats(h, (int64_t)dict_cap, N, &fst));
    GK_CUDA(cudaMemsetAsync(h->sp_dict_keys.p, 0xFF, dict_cap * 8, h->stream));
    GK_CUDA(cudaMemsetAsync(h->ft_keys.p, 0xFF, ft_cap * 8, h->stream));
    GK_CUDA(cudaMemsetAsync(h->ft_cnt.p, 0, ft_cap * 4, h->stream));
    SpParams p;
    memset(&p, 0, sizeof(p));
    p.graph_ptr = h->graph_ptr.as<int>();
    p.row_ptr = h->row_ptr.as<int>();
    p.col_idx = h->col_idx.as<int>();
    p.weights = (h->has_weights && !use_u16) ? h->weights.as<double>() : nullptr;
    p.labels = with_labels ? h->labels0.as<int>() : nullptr;
    p.n_labels = with_labels ? (int)std::max<long long>(n_labels_total, 1) : 1;
    p.keep = d_keep;
    p.dict_keys = h->sp_dict_keys.as<unsigned long long>();
    p.dict_mask = (unsigned)(dict_cap - 1);
    p.ft_keys = h->ft_keys.as<unsigned long long>();
    p.ft_cnt = h->ft_cnt.as<unsigned>();
    p.ft_mask = (unsigned)(ft_cap - 1);
    p.sc = sc;
    p.st = fst;
    p.gdist = h->sp_dist.p;
    for (int pass = 0; pass < n_pass; ++pass) {
    if (wl_iter >= 0) {
      p.labels = h->labels_all.as<int>() + (size_t)pass * h->V;
      p.label_offset = (int)level_base[pass];
    }
    if (real_mode) {
      // non-integer path lengths: (1) fp64 Floyd-Warshall of every graph into global memory + a
      // dictionary of the distinct distance bit patterns, (2) histogram keyed by (lu, lv, id(d))
      GK_TRY(h->sp_dist.ensure((size_t)std::max<long long>(off_all, 1) * 8));
      GK_TRY(h->sp_dkeys.ensure(dkey_cap * 8));
      GK_CUDA(cudaMemsetAsync(h->sp_dkeys.p, 0xFF, dkey_cap * 8, h->stream));
      SpParams pa = p;
      pa.gdist = h->sp_dist.p;
      pa.goff = d_goff_all;
      pa.dict_keys = h->sp_dkeys.as<unsigned long long>();
      pa.dict_mask = (unsigned)(dkey_cap - 1);
      pa.keep = nullptr;
      const size_t smem_a = max_small_nn * 8 + 16;
      // path sums in the reference's order: Floyd-Warshall (adjacency input) or Dijkstra (edge dictionaries)
      const bool dj = flags & GK_SP_DIJKSTRA_ORDER;
      GK_CUDA(cudaFuncSetAttribute(spattr_apsp<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem_a, 16)));
      GK_CUDA(cudaFuncSetAttribute(sp_dijkstra_order_apsp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem_a, 16)));
      if (!small.empty()) {
        pa.glist = lists.as<int>();
        pa.dist_in_global = 0;
        if (dj) sp_dijkstra_order_apsp<<<(int)small.size(), SP_THREADS, smem_a, h->stream>>>(pa);
        else spattr_apsp<double><<<(int)small.size(), SP_THREADS, smem_a, h->stream>>>(pa);
        LAUNCH_CHECK(h);
      }
      if (!big.empty()) {
        pa.glist = lists.as<int>() + small.size();
        pa.dist_in_global = 1;
        if (dj) sp_dijkstra_order_apsp<<<(int)big.size(), SP_THREADS, 16, h->stream>>>(pa);
        else spattr_apsp<double><<<(int)big.size(), SP_THREADS, 16, h->stream>>>(pa);
        LAUNCH_CHECK(h);
      }
      SpParams pb = p;
      pb.gdist = h->sp_dist.p;
      pb.goff = d_goff_all;
      sp_hist_from_dist<<<(int)N, SP_THREADS, SP_LOCAL_SLOTS * 12, h->stream>>>(pb, h->sp_dkeys.as<unsigned long long>(),
                                                                              (unsigned)(dkey_cap - 1));
      LAUNCH_CHECK(h);
    } else {
    if (!small.empty()) {
      p.glist = lists.as<int>();
      p.n_list = (int)small.size();
      p.dist_in_global = 0;
      p.goff = d_goff_all;  // only used for `keep`
      if (use_u16) sp_apsp_hist<unsigned short><<<(int)small.size(), SP_THREADS, smem_small, h->stream>>>(p);
      else sp_apsp_hist<double><<<(int)small.size(), SP_THREADS, smem_small, h->stream>>>(p);
      LAUNCH_CHECK(h);
    }
    // the (up to four) word-width classes are independent: odd classes run on the side stream so
    // that the tail of one launch overlaps the next (they only share atomically updated tables)
    bool forked = false;
    for (int i = 0; i < 4; ++i) {
      if (bfs[i].empty()) continue;
      const int W = 1 << i;
      cudaStream_t st = h->stream;
      if (i & 1) {
        if (!forked) {
          GK_CUDA(cudaEventRecord(h->ev_fork, h->stream));
          GK_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
          forked = true;
        }
        st = h->stream2;
      }
      int nmax = 0;
      for (int g : bfs[i]) nmax = std::max(nmax, ex->graph_ptr[g + 1] - ex->graph_ptr[g]);
      const bool direct = p.n_labels <= SP_DIRECT_MAX_LABELS;
      const size_t smem = (direct ? SP_LOCAL_SLOTS * 4 : SP_LOCAL_SLOTS * 12) + (size_t)nmax * W * 8 + (size_t)16 * W * 8 +
                          (size_t)nmax * 4 + 16;
      p.glist = lists.as<int>() + bfs_off[i];
      p.n_list = (int)bfs[i].size();
      p.dist_in_global = 0;
      p.goff = d_goff_all;
      const int threads = nmax <= 32 ? 32 : nmax <= 64 ? 64 : 128;
      switch (W) {
        case 1: GK_CUDA(cudaFuncSetAttribute(sp_bfs_hist<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
        case 2: GK_CUDA(cudaFuncSetAttribute(sp_bfs_hist<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
        case 4: GK_CUDA(cudaFuncSetAttribute(sp_bfs_hist<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
        default: GK_CUDA(cudaFuncSetAttribute(sp_bfs_hist<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
      }
      switch (W) {
        case 1: sp_bfs_hist<1><<<(int)bfs[i].size(), threads, smem, st>>>(p); break;
        case 2: sp_bfs_hist<2><<<(int)bfs[i].size(), threads, smem, st>>>(p); break;
        case 4: sp_bfs_hist<4><<<(int)bfs[i].size(), threads, smem, st>>>(p); break;
        default: sp_bfs_hist<8><<<(int)bfs[i].size(), threads, smem, st>>>(p); break;
      }
      LAUNCH_CHECK(h);
    }
    if (forked) {
      GK_CUDA(cudaEventRecord(h->ev_join, h->stream2));
      GK_CUDA(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    }
    if (!big.empty()) {
      if (keep) return fail(GK_ERR_UNSUPPORTED, "gk_sp_features: KEEP_DIST with graphs beyond the shared-memory budget");
      p.glist = lists.as<int>() + small.size();
      p.n_list = (int)big.size();
      p.dist_in_global = 1;
      p.goff = d_goff_big;
      if (use_u16) sp_apsp_hist<unsigned short><<<(int)big.size(), SP_THREADS, smem_big, h->stream>>>(p);
      else sp_apsp_hist<double><<<(int)big.size(), SP_THREADS, smem_big, h->stream>>>(p);
      LAUNCH_CHECK(h);
    }
    }  // integer-distance mode
    }  // passes (WL levels)
    DevScalars* hs;
    GK_TRY(read_scalars(h, &hs));
    if (hs->sp_nonint && !real_mode) { real_mode = true; --attempt; continue; }  // switch to exact float keys
    if (real_mode && (hs->ft_overflow & 2u) && dkey_cap < (1u << 24)) {
      // either dictionary may have overflowed; grow the distance dictionary first
      dkey_cap *= 8;
      if (dkey_cap > (1u << 24)) dkey_cap = 1u << 24;
    }
    if (hs->ft_overflow & 2u) { dict_cap *= 8; continue; }
    if (hs->ft_overflow & 1u) { ft_cap *= 4; continue; }
    if ((size_t)hs->sp_dict_size * 2 > dict_cap) { dict_cap *= 4; continue; }  // keep probe chains short
    break;
  }
  GK_CUDA(cudaEventRecord(h->tev[3], h->stream));
  GK_CUDA(cudaEventSynchronize(h->tev[3]));
  DevScalars* hs = h->h_scalars.as<DevScalars>();
  h->n_columns = (int64_t)dict_cap;  // column id = dictionary slot
  h->features_ready = true; h->feat_serial++;
  h->feature_kind = 2;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = h->N; stats->n_vertices = h->V; stats->n_edges = h->E;
    stats->n_levels = 1;
    stats->level_dims[0] = hs->sp_dict_size;
    stats->n_columns = hs->sp_dict_size;
    stats->kernel_launches = h->launches - launches0;
    stats->ms_features = ev_ms(h->tev[2], h->tev[3]);
  }
  return GK_OK;
}

int gk_sp_features(gk_handle* h, int32_t flags, gk_stats* stats) { return sp_features_impl(h, flags, -1, stats); }

int gk_wl_sp_features(gk_handle* h, int32_t n_iter, int32_t flags, gk_stats* stats) {
  if (n_iter < 0) return fail(GK_ERR_ARG, "gk_wl_sp_features: n_iter out of range");
  return sp_features_impl(h, flags | GK_SP_WITH_LABELS, n_iter, stats);
}

int gk_sp_distances(gk_handle* h, int64_t g, double* out) {
  if (!h || !out) return fail(GK_ERR_ARG, "gk_sp_distances: null argument");
  if (h->feature_kind == 3 && h->sp_dist_esz) {
    // after gk_spattr_features: the APSP matrices of every graph are still in sp_dist (u16 with the saturated
    // value 0x3FFF for "no path", or fp64 with +inf)
    if (g < 0 || g >= h->N) return fail(GK_ERR_ARG, "gk_sp_distances: bad graph index");
    HandleExtra* ex = extra_of(h);
    const long long off = ex->sp_goff[g], cnt = ex->sp_goff[g + 1] - off;
    GK_CUDA(cudaSetDevice(h->dev));
    if (h->sp_dist_esz == 8) {
      GK_CUDA(cudaMemcpyAsync(out, h->sp_dist.as<double>() + off, cnt * 8, cudaMemcpyDeviceToHost, h->stream));
      GK_CUDA(cudaStreamSynchronize(h->stream));
    } else {
      std::vector<unsigned short> tmp((size_t)cnt);
      GK_CUDA(cudaMemcpyAsync(tmp.data(), h->sp_dist.as<unsigned short>() + off, cnt * 2, cudaMemcpyDeviceToHost, h->stream));
      GK_CUDA(cudaStreamSynchronize(h->stream));
      for (long long i = 0; i < cnt; ++i) out[i] = tmp[i] < 0x3FFF ? (double)tmp[i] : INFINITY;
    }
    return GK_OK;
  }
  if (h->feature_kind != 2 || !(h->sp_flags & GK_SP_KEEP_DIST)) return fail(GK_ERR_STATE, "gk_sp_distances: run gk_sp_features with GK_SP_KEEP_DIST (or gk_spattr_features) first");
  if (g < 0 || g >= h->N) return fail(GK_ERR_ARG, "gk_sp_distances: bad graph index");
  HandleExtra* ex = extra_of(h);
  const long long off = ex->sp_goff[g], cnt = ex->sp_goff[g + 1] - off;
  GK_CUDA(cudaSetDevice(h->dev));
  GK_CUDA(cudaMemcpyAsync(out, h->K_stage.as<double>() + off, cnt * 8, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

int gk_spattr_features(gk_handle* h, int32_t flags, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->N <= 0) return fail(GK_ERR_STATE, "gk_spattr_features: no graphs packed");
  if (!h->attrs.p || h->attr_dim <= 0) return fail(GK_ERR_ARG, "gk_spattr_features: node attributes are required");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t N = h->N;
  const int da = h->attr_dim, dd = da * da;
  if (dd > 1024) return fail(GK_ERR_UNSUPPORTED, "gk_spattr_features: attribute dimension above 32");
  const bool use_u16 = (!h->has_weights || h->unit_weights) && h->max_graph_size < 16000;
  const size_t esz = use_u16 ? 2 : 8;
  HandleExtra* ex = extra_of(h);
  const int64_t launches0 = h->launches;
  h->features_ready = false; h->feat_serial++;
  if ((size_t)h->max_graph_size * h->max_graph_size * 2 + (size_t)h->max_graph_size * da * 8 + (size_t)dd * 8 > 200 * 1024)
    return fail(GK_ERR_UNSUPPORTED, "gk_spattr_features: graph too large for the shared-memory feature kernel");

  // per-graph offsets of the distance matrices (all kept in global memory for phase C)
  std::vector<int> small, big;
  size_t max_small_nn = 0;
  ex->sp_goff.assign(N + 1, 0);
  long long off_all = 0;
  for (int64_t g = 0; g < N; ++g) {
    const long long n = ex->graph_ptr[g + 1] - ex->graph_ptr[g];
    ex->sp_goff[g] = off_all;
    off_all += n * n;
    if ((size_t)(n * n) * esz <= 160 * 1024) { small.push_back((int)g); max_small_nn = std::max(max_small_nn, (size_t)(n * n)); }
    else big.push_back((int)g);
  }
  ex->sp_goff[N] = off_all;
  std::vector<int> order(small);
  order.insert(order.end(), big.begin(), big.end());
  GK_TRY(h->sp_lists.ensure((size_t)N * 4 + 16));
  GK_CUDA(cudaMemcpyAsync(h->sp_lists.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, h->stream));
  GK_TRY(h->sp_graph_off.ensure((size_t)(N + 1) * 8));
  GK_CUDA(cudaMemcpyAsync(h->sp_graph_off.p, ex->sp_goff.data(), (N + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  GK_TRY(h->sp_dist.ensure((size_t)std::max<long long>(off_all, 1) * esz));
  const size_t dict_cap = 1 << 16;
  GK_TRY(h->sp_dict_keys.ensure(dict_cap * 8));
  GK_TRY(h->sp_dict_ids.ensure(dict_cap * 4));
  h->sp_dict_cap = dict_cap;
  GK_TRY(init_scalars(h, 0));
  GK_CUDA(cudaMemsetAsync(h->sp_dict_keys.p, 0xFF, dict_cap * 8, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));

  GK_CUDA(cudaEventRecord(h->tev[2], h->stream));
  SpParams p;
  memset(&p, 0, sizeof(p));
  p.graph_ptr = h->graph_ptr.as<int>();
  p.row_ptr = h->row_ptr.as<int>();
  p.col_idx = h->col_idx.as<int>();
  p.weights = (h->has_weights && !use_u16) ? h->weights.as<double>() : nullptr;
  p.gdist = h->sp_dist.p;
  p.goff = h->sp_graph_off.as<long long>();
  p.dict_keys = h->sp_dict_keys.as<unsigned long long>();
  p.dict_mask = (unsigned)(dict_cap - 1);
  p.sc = h->scalars.as<DevScalars>();
  const size_t smem_small = max_small_nn * esz + 16;
  const bool dj = !use_u16 && (flags & GK_SP_DIJKSTRA_ORDER);  // real-valued weights: path sums in Dijkstra's order
  if (use_u16) GK_CUDA(cudaFuncSetAttribute(spattr_apsp<unsigned short>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_small));
  else if (dj) GK_CUDA(cudaFuncSetAttribute(sp_dijkstra_order_apsp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_small));
  else GK_CUDA(cudaFuncSetAttribute(spattr_apsp<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_small));
  if (!small.empty()) {
    p.glist = h->sp_lists.as<int>();
    p.dist_in_global = 0;
    if (use_u16) spattr_apsp<unsigned short><<<(int)small.size(), SP_THREADS, smem_small, h->stream>>>(p);
    else if (dj) sp_dijkstra_order_apsp<<<(int)small.size(), SP_THREADS, smem_small, h->stream>>>(p);
    else spattr_apsp<double><<<(int)small.size(), SP_THREADS, smem_small, h->stream>>>(p);
    LAUNCH_CHECK(h);
  }
  if (!big.empty()) {
    p.glist = h->sp_lists.as<int>() + small.size();
    p.dist_in_global = 1;
    if (use_u16) spattr_apsp<unsigned short><<<(int)big.size(), SP_THREADS, 16, h->stream>>>(p);
    else if (dj) sp_dijkstra_order_apsp<<<(int)big.size(), SP_THREADS, 16, h->stream>>>(p);
    else spattr_apsp<double><<<(int)big.size(), SP_THREADS, 16, h->stream>>>(p);
    LAUNCH_CHECK(h);
  }
  // distinct distances -> block ids (ascending distance order, deterministic)
  std::vector<unsigned long long> keys(dict_cap);
  GK_CUDA(cudaMemcpyAsync(keys.data(), h->sp_dict_keys.p, dict_cap * 8, cudaMemcpyDeviceToHost, h->stream));
  DevScalars* hs;
  GK_TRY(read_scalars(h, &hs));
  if (hs->ft_overflow) return fail(GK_ERR_UNSUPPORTED, "gk_spattr_features: more than 32768 distinct path lengths");
  std::vector<std::pair<double, int>> found;
  for (size_t i = 0; i < dict_cap; ++i)
    if (keys[i] != EMPTY64) {
      double d;
      if (use_u16) d = (double)keys[i];
      else { long long b = (long long)keys[i]; memcpy(&d, &b, 8); }
      found.emplace_back(d, (int)i);
    }
  std::sort(found.begin(), found.end());
  const int n_blocks = (int)found.size();
  std::vector<int> slot_block(dict_cap, -1);
  for (int b = 0; b < n_blocks; ++b) slot_block[found[b].second] = b;
  GK_CUDA(cudaMemcpyAsync(h->sp_dict_ids.p, slot_block.data(), dict_cap * 4, cudaMemcpyHostToDevice, h->stream));
  const int64_t Dfeat = (int64_t)std::max(n_blocks, 1) * dd;
  if ((size_t)N * Dfeat * 8 > (size_t)64 << 30) return fail(GK_ERR_UNSUPPORTED, "gk_spattr_features: feature matrix above 64 GB");
  GK_TRY(h->fattr.ensure((size_t)N * Dfeat * 8));
  GK_CUDA(cudaMemsetAsync(h->fattr.p, 0, (size_t)N * Dfeat * 8, h->stream));
  h->fattr_dim = Dfeat;
  if (n_blocks > 0) {
    const size_t fixed = (size_t)h->max_graph_size * da * 8 + (size_t)h->max_graph_size * h->max_graph_size * 2 + 64;
    int chunk = (int)std::min<size_t>((size_t)n_blocks, (200 * 1024 - fixed) / ((size_t)dd * 8));
    if (chunk < 1) return fail(GK_ERR_UNSUPPORTED, "gk_spattr_features: shared memory budget exceeded");
    const size_t smem = (size_t)chunk * dd * 8 + fixed;
    if (use_u16) {
      GK_CUDA(cudaFuncSetAttribute(spattr_accumulate<unsigned short>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      spattr_accumulate<unsigned short><<<(int)N, 256, smem, h->stream>>>(
          h->graph_ptr.as<int>(), h->attrs.as<double>(), da, h->sp_dist.p, h->sp_graph_off.as<long long>(),
          h->sp_dict_keys.as<unsigned long long>(), (unsigned)(dict_cap - 1), h->sp_dict_ids.as<int>(), n_blocks, chunk,
          h->fattr.as<double>());
    } else {
      GK_CUDA(cudaFuncSetAttribute(spattr_accumulate<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      spattr_accumulate<double><<<(int)N, 256, smem, h->stream>>>(
          h->graph_ptr.as<int>(), h->attrs.as<double>(), da, h->sp_dist.p, h->sp_graph_off.as<long long>(),
          h->sp_dict_keys.as<unsigned long long>(), (unsigned)(dict_cap - 1), h->sp_dict_ids.as<int>(), n_blocks, chunk,
          h->fattr.as<double>());
    }
    LAUNCH_CHECK(h);
  }
  GK_TRY(h->diag_f64.ensure(N * 8));
  GK_TRY(h->fattr_exp.ensure(N * 4));
  rownorm_f64_kernel<<<(int)N, 256, 0, h->stream>>>(h->fattr.as<double>(), Dfeat, (int)N, h->diag_f64.as<double>(),
                                                    h->fattr_exp.as<int>());
  LAUNCH_CHECK(h);
  GK_CUDA(cudaEventRecord(h->tev[3], h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));  // host vectors above are sources of async copies
  h->n_columns = Dfeat;
  h->features_ready = true; h->feat_serial++;
  h->feature_kind = 3;
  h->sp_dist_esz = (int)esz;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = N; stats->n_vertices = h->V; stats->n_edges = h->E;
    stats->n_levels = 1;
    stats->level_dims[0] = n_blocks;
    stats->n_columns = Dfeat;
    stats->n_dense_columns = Dfeat;
    stats->kernel_launches = h->launches - launches0;
    stats->ms_features = ev_ms(h->tev[2], h->tev[3]);
  }
  return GK_OK;
}

static void build_tiles(std::vector<int2>& tiles, int a0, int a1, int b0, int b1, bool upper_only, int bm);

// Gram of the dense fp64 SP-attr feature matrix (feature_kind == 3).  Default: the tcgen05 kernel with tf32
// operands on a hi/lo split of the features (3xTF32: hi hi^T + hi lo^T + lo hi^T, fp32 accumulation in TMEM,
// k range processed in chunks and summed in fp64), self similarities exact in fp64.  Every row is scaled by a power
// of two before the split and K unscaled after it (spattr_split_tf32, unscale_gram_f64), so the range is fp64's and
// K(2^s a) = 2^(4s) K(a) bit for bit.  Error bound: |K - K_exact| <= 1e-5 * <|phi_i|, |phi_j|> -- relative for
// non-negative attributes (observed ~2e-6), normwise for signed ones, where cancelling entries can be far less
// accurate relatively.  GRAKEL_B200_SPATTR_F64=1 selects the fp64 CUDA-core Gram for elementwise accuracy.
static int gram_spattr(gk_handle* h, int64_t n_fit, int32_t flags, int64_t row_begin, int64_t row_end, void* K_out,
                       int32_t out_dtype, int64_t ld, double* xdiag, double* ydiag, gk_stats* stats) {
  if (out_dtype != GK_F64) return fail(GK_ERR_UNSUPPORTED, "ShortestPathAttr Gram is fp64 only");
  if (flags & GK_OUT_DEVICE) return fail(GK_ERR_UNSUPPORTED, "ShortestPathAttr Gram: device output not supported");
  const int64_t N = h->N;
  const bool square = n_fit == N;
  const int64_t k_rows_total = square ? N : N - n_fit, k_cols = n_fit;
  if (row_end < 0) row_end = k_rows_total;
  if (row_begin < 0 || row_begin > row_end || row_end > k_rows_total) return fail(GK_ERR_ARG, "gk_gram: bad row range");
  const int64_t k_rows = row_end - row_begin;
  if (ld <= 0) ld = k_cols;
  const int64_t launches0 = h->launches;
  GK_TRY(h->K.ensure((size_t)std::max<int64_t>(k_rows, 1) * k_cols * 8));
  h->K_rows = k_rows; h->K_cols = k_cols; h->K_ld = k_cols; h->K_dtype = GK_F64;
  const int a0 = (int)((square ? 0 : n_fit) + row_begin), a1 = (int)((square ? 0 : n_fit) + row_end);
  GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
  const char* e_f64 = getenv("GRAKEL_B200_SPATTR_F64");
  const bool use_f64 = e_f64 && atoi(e_f64) != 0;
  if (k_rows > 0 && !use_f64) {
    const long long D = h->fattr_dim, Dp = (D + BK_TF32 - 1) / BK_TF32 * BK_TF32, W = 3 * Dp;
    GK_TRY(h->panel.ensure((size_t)N * W * 4 * 2));
    float* P1 = h->panel.as<float>();
    float* P2 = P1 + (size_t)N * W;
    spattr_split_tf32<<<h->sm_count * 8, 256, 0, h->stream>>>(h->fattr.as<double>(), h->fattr_exp.as<int>(), D, Dp,
                                                              (int)N, P1, P2);
    LAUNCH_CHECK(h);
    const bool sym = square && row_begin == 0 && row_end == N;
    std::vector<int2> tiles;
    build_tiles(tiles, a0, a1, 0, (int)n_fit, sym, BM);
    GK_TRY(h->h_tiles.ensure(tiles.size() * sizeof(int2)));
    memcpy(h->h_tiles.p, tiles.data(), tiles.size() * sizeof(int2));
    GK_TRY(h->tiles.ensure(tiles.size() * sizeof(int2)));
    GK_CUDA(cudaMemcpyAsync(h->tiles.p, h->h_tiles.p, tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
    CUtensorMap tmA, tmB, tmC;
    memset(&tmC, 0, sizeof(tmC));
    GK_TRY(make_panel_map_f32(&tmA, P1, W, N, BM));
    GK_TRY(make_panel_map_f32(&tmB, P2, W, N, BN));
    GramParams p;
    memset(&p, 0, sizeof(p));
    p.tiles = h->tiles.as<int2>();
    p.n_tiles = (int)tiles.size();
    p.a_row_end = a1; p.b_row_end = (int)n_fit;
    p.c_row0 = a0; p.c_col0 = 0;
    p.out = h->K.p; p.ld = k_cols;
    p.mirror = 0;  // the symmetric case mirrors the upper triangle once, after all chunks (unscale_gram_f64)
    p.diag = h->diag_f64.as<double>();
    // The tensor core's fp32 accumulate truncates (measured: -1.8e-5 relative for 960 sequential MMAs on all-positive
    // data, profiles/r02e_spattr_err.txt), so no accumulator sums more than `chunk` k-blocks x 4 MMAs: the kernel
    // folds every chunk of a tile into the fp64 result itself (double-buffered TMEM accumulators: the MMAs of chunk
    // c+1 run while the epilogue adds chunk c).
    // Only the hi x hi third of the k range needs short chunks: the two cross thirds are 2^-11 of the sum, their
    // accumulated truncation is 2^-11 of the bound and they go through one accumulator.
    int chunk = 8;
    if (const char* e = getenv("GRAKEL_B200_SPATTR_CHUNK")) chunk = std::max(1, atoi(e));
    p.k_block0 = 0;
    p.num_k_blocks = (int)(W / BK_TF32);
    p.k_chunk = chunk;
    p.k_split = (int)(Dp / BK_TF32);
    p.accumulate = 0;
    const int grid = (int)std::min<size_t>(tiles.size(), h->sm_count);
    gram_tc_kernel<double, false, 1><<<grid, GEMM_THREADS, GEMM_SMEM, h->stream>>>(tmA, tmB, tmC, p);
    LAUNCH_CHECK(h);
    unscale_gram_f64<<<h->sm_count * 8, 256, 0, h->stream>>>(a0, k_rows, k_cols, h->fattr_exp.as<int>(),
                                                             h->K.as<double>(), k_cols, sym ? 1 : 0);
    LAUNCH_CHECK(h);
    if (square) {  // exact self similarities
      set_diag_f64<<<cdiv(k_rows, 256), 256, 0, h->stream>>>(a0, a1, 0, (int)n_fit, h->diag_f64.as<double>(), h->K.as<double>(), k_cols);
      LAUNCH_CHECK(h);
    }
  }
  if (k_rows > 0) {
    if (use_f64) {
      dim3 grid(cdiv(k_cols, 64), cdiv(k_rows, 64));
      gram_f64_kernel<<<grid, 256, 0, h->stream>>>(h->fattr.as<double>(), h->fattr_dim, a0, a1, 0, (int)n_fit,
                                                   h->K.as<double>(), k_cols);
      LAUNCH_CHECK(h);
    }
    if (flags & GK_NORMALIZE) {
      normalize_rows<double><<<h->sm_count * 8, 256, 0, h->stream>>>(k_rows, k_cols, h->K.as<double>(), k_cols,
                                                                      h->diag_f64.as<double>() + a0,
                                                                      h->diag_f64.as<double>(), (flags & GK_NAN_TO_NUM) ? 1 : 0);
      LAUNCH_CHECK(h);
    }
  }
  GK_CUDA(cudaEventRecord(h->tev[7], h->stream));
  if (K_out && k_rows > 0)
    GK_CUDA(cudaMemcpy2DAsync(K_out, (size_t)ld * 8, h->K.p, (size_t)k_cols * 8, (size_t)k_cols * 8, (size_t)k_rows,
                              cudaMemcpyDeviceToHost, h->stream));
  if (xdiag) GK_CUDA(cudaMemcpyAsync(xdiag, h->diag_f64.p, n_fit * 8, cudaMemcpyDeviceToHost, h->stream));
  if (ydiag && !square)
    GK_CUDA(cudaMemcpyAsync(ydiag, h->diag_f64.as<double>() + n_fit, (N - n_fit) * 8, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  if (stats) {
    stats->gram_path = 4;
    stats->gemm_launches = h->launches - launches0;
    stats->ms_gemm = ev_ms(h->tev[6], h->tev[7]);
  }
  return GK_OK;
}

// ---------------------------------------------------------------------------
}  // extern "C"

// ---------------------------------------------------------------------------
// Host delivery of an fp32 device matrix into the caller's float64 array (host_deliver.h): K is moved as
// fp32 -- for the symmetric square case only its upper triangle, in row bands of roughly equal area --
// through a ring of pinned staging buffers; host threads widen each band into the destination rows and
// write the mirrored half (8 x 8 register transposes) while the next bands are on the PCIe bus.
#include "host_deliver.h"

// Symmetric integer-valued fp32 result -> the caller's float64 host matrix: upper triangle over PCIe in the narrowest
// exact type (u16 when the largest self similarity is below 2^16, packed band by band on the device first; else fp32),
// widened and mirrored by the host pool (host_deliver.h).
static int deliver_square(gk_handle* h, const float* d_k, long long d_ld, int64_t k_rows, double* dst, int64_t ld, int64_t max_diag) {
  DeviceCopier cp{h};
  if (max_diag < 65536 && !getenv("GRAKEL_B200_NO_U16")) {
    const std::vector<long long> start = tri_bands(k_rows);
    const int nb = (int)start.size() - 1;
    std::vector<long long> tab(start);
    long long off = 0;
    for (int c = 0; c < nb; ++c) { tab.push_back(off); off += (start[c + 1] - start[c]) * (k_rows - start[c]); }
    GK_TRY(h->K_stage.ensure((size_t)off * 2 + tab.size() * 8 + 64));
    GK_TRY(h->h_bands.ensure(tab.size() * 8));
    memcpy(h->h_bands.p, tab.data(), tab.size() * 8);
    long long* d_tab = reinterpret_cast<long long*>(h->K_stage.as<char>() + (((size_t)off * 2 + 63) / 64 * 64));
    GK_CUDA(cudaMemcpyAsync(d_tab, h->h_bands.p, tab.size() * 8, cudaMemcpyHostToDevice, h->stream));
    pack_tri_u16<<<h->sm_count * 8, 256, 0, h->stream>>>(d_k, d_ld, k_rows, d_tab, d_tab + nb + 1, nb, h->K_stage.as<unsigned short>());
    LAUNCH_CHECK(h);
    return deliver_tri<uint16_t>(cp, h->K_stage.as<uint16_t>(), 0, k_rows, dst, ld);
  }
  return deliver_tri<float>(cp, d_k, d_ld, k_rows, dst, ld);
}

template <typename OutT, bool NORM>
static void launch_tc(gk_handle* h, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                      const GramParams& p, int grid) {
  gram_tc_kernel<OutT, NORM><<<grid, GEMM_THREADS, GEMM_SMEM, h->stream>>>(tmA, tmB, tmC, p);
}
template <typename OutT, bool NORM>
static void launch_simt(gk_handle* h, const unsigned* panel, long long ldp, int kdim, int a0, int a1, int b0, int b1,
                        const GramParams& p) {
  dim3 grid(cdiv(b1 - b0, 16), cdiv(a1 - a0, 16));
  gram_simt_kernel<OutT, NORM><<<grid, 256, 0, h->stream>>>(panel, ldp, kdim, a0, a1, b0, b1, p);
}
template <typename OutT, bool NORM>
static void launch_empty(gk_handle* h, int a0, int a1, int b0, int b1, const GramParams& p) {
  gram_empty_kernel<OutT, NORM><<<h->sm_count * 4, 256, 0, h->stream>>>(a0, a1, b0, b1, p);
}

// Build the tile list: bands of 12 row tiles, column-major inside a band, so that the
// ~148 tiles in flight cover a compact block of the output and share panel rows in L2.
static void build_tiles(std::vector<int2>& tiles, int a0, int a1, int b0, int b1, bool upper_only, int bm) {
  const int n_m = cdiv(a1 - a0, bm), n_n = cdiv(b1 - b0, BN);
  const int BAND = 12 * BM / bm;
  for (int m0 = 0; m0 < n_m; m0 += BAND) {
    const int m1 = std::min(n_m, m0 + BAND);
    for (int j = 0; j < n_n; ++j) {
      for (int i = m0; i < m1; ++i) {
        const int ar = a0 + i * bm, br = b0 + j * BN;
        if (upper_only && br + BN - 1 < ar) continue;  // tile entirely below the diagonal
        tiles.push_back(make_int2(ar, br));
      }
    }
  }
}

// ---- multi-GPU helpers (collective: every rank of the communicator calls them in the same order)
static int comm_barrier(gk_handle* h) {
  Comm* c = reinterpret_cast<Comm*>(h->comm);
  NcclApi* api = nccl_api();
  GK_NCCL(api, api->AllReduce(c->d_token, c->d_token, 1, ncclInt32, ncclSum, c->comm, h->stream));
  return GK_OK;
}

// Make h->K (>= bytes, the same request on every rank) visible to the peers: CUDA IPC handles travel through one
// ncclAllGather; mappings are renewed only when the buffer had to grow (the same call on every rank).
static int comm_share_K(gk_handle* h, size_t bytes) {
  Comm* c = reinterpret_cast<Comm*>(h->comm);
  NcclApi* api = nccl_api();
  if (c->exported && c->exported == h->K.p && h->K.cap >= bytes) return GK_OK;
  // peers unmap the old buffer before anybody frees it
  for (int r = 0; r < c->nranks; ++r)
    if (r != c->rank && c->peer_base[r]) { cudaIpcCloseMemHandle(c->peer_base[r]); c->peer_base[r] = nullptr; }
  GK_TRY(comm_barrier(h));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  GK_TRY(h->K.ensure(bytes));
  cudaIpcMemHandle_t mine;
  GK_CUDA(cudaIpcGetMemHandle(&mine, h->K.p));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
  unsigned char* d_mine = c->d_handles + (size_t)c->nranks * 64;
  GK_CUDA(cudaMemcpyAsync(d_mine, &mine, 64, cudaMemcpyHostToDevice, h->stream));
  GK_NCCL(api, api->AllGather(d_mine, c->d_handles, 64, ncclChar, c->comm, h->stream));
  std::vector<cudaIpcMemHandle_t> all(c->nranks);
  GK_CUDA(cudaMemcpyAsync(all.data(), c->d_handles, (size_t)c->nranks * 64, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  for (int r = 0; r < c->nranks; ++r) {
    if (r == c->rank) { c->peer_base[r] = h->K.p; continue; }
    GK_CUDA(cudaIpcOpenMemHandle(&c->peer_base[r], all[r], cudaIpcMemLazyEnablePeerAccess));
  }
  c->exported = h->K.p;
  c->exported_cap = h->K.cap;
  return GK_OK;
}

extern "C" {

int gk_gram(gk_handle* h, int64_t n_fit, int32_t flags, int64_t row_begin, int64_t row_end, void* K_out,
            int32_t out_dtype, int64_t ld, double* xdiag, double* ydiag, gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (!h->features_ready) return fail(GK_ERR_STATE, "gk_gram: no feature block (call gk_wl_features / gk_sp_features)");
  if (out_dtype != GK_F32 && out_dtype != GK_F64) return fail(GK_ERR_ARG, "gk_gram: bad out_dtype");
  const int64_t N = h->n_rows > 0 ? h->n_rows : h->N;  // rows of the feature block (gk_set_row_map)
  const int* d_row_map = h->n_rows > 0 ? h->row_map.as<int>() : nullptr;
  if (n_fit <= 0 || n_fit > N) return fail(GK_ERR_ARG, "gk_gram: n_fit out of range");
  if (h->feature_kind == 3) {
    if (d_row_map) return fail(GK_ERR_UNSUPPORTED, "gk_gram: row map with ShortestPathAttr features");
    GK_CUDA(cudaSetDevice(h->dev));
    return gram_spattr(h, n_fit, flags, row_begin, row_end, K_out, out_dtype, ld, xdiag, ydiag, stats);
  }
  const bool square = n_fit == N;
  const int64_t k_rows_total = square ? N : N - n_fit;
  const int64_t k_cols = n_fit;
  if (row_end < 0) row_end = k_rows_total;
  if (row_begin < 0 || row_begin > row_end || row_end > k_rows_total) return fail(GK_ERR_ARG, "gk_gram: bad row range");
  const int64_t k_rows = row_end - row_begin;
  if (ld <= 0) ld = k_cols;
  if (ld < k_cols) return fail(GK_ERR_ARG, "gk_gram: ld smaller than the row length");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t launches0 = h->launches;
  const bool normalize = flags & GK_NORMALIZE;
  const size_t esz = out_dtype == GK_F64 ? 8 : 4;
  DevScalars* sc = h->scalars.as<DevScalars>();

  GK_CUDA(cudaEventRecord(h->tev[4], h->stream));
  // ---- column statistics were maintained by the feature kernels; finish the self similarities
  const int64_t D = std::max<int64_t>(h->n_columns, 1);
  if (D > h->col_cap) return fail(GK_ERR_STATE, "gk_gram: column statistics missing");
  const int nbc = cdiv(D, 256);
  GK_TRY(h->colslot.ensure(D * 4));
  GK_TRY(h->colstats.ensure(sizeof(ColStats)));
  GK_TRY(h->h_colstats.ensure(sizeof(ColStats)));
  GK_TRY(h->diag_f64.ensure(N * 8));
  HandleExtra* hx = extra_of(h);
  const bool pro = square && !d_row_map && h->pro_serial == h->feat_serial && D <= h->col_cap;  // prologue already on the host
  if (!pro) GK_CUDA(cudaMemsetAsync(&sc->n_entries, 0, sizeof(unsigned long long) * 3 + sizeof(long long), h->stream));
  const unsigned long long* d_diag_u64 = h->diag_u64.as<unsigned long long>();
  if (d_row_map) {
    GK_TRY(h->diag_rows.ensure(N * 8));
    GK_CUDA(cudaMemsetAsync(h->diag_rows.p, 0, N * 8, h->stream));
    diag_remap<<<cdiv(h->N, 256), 256, 0, h->stream>>>((int)h->N, d_row_map, d_diag_u64, h->diag_rows.as<unsigned long long>());
    LAUNCH_CHECK(h);
    d_diag_u64 = h->diag_rows.as<unsigned long long>();
  }
  if (!pro) {
    diag_finish<<<cdiv(N, 256), 256, 0, h->stream>>>((int)N, d_diag_u64,
                                                     h->diag_f64.as<double>(), (int)h->n_part,
                                                     h->part_max.as<unsigned>(), h->part_new.as<unsigned>(), sc);
    LAUNCH_CHECK(h);
  }
  if (!square) {  // which columns occur on both the X and the Y side
    GK_TRY(h->colmin.ensure(D * 4));
    GK_TRY(h->colmax.ensure(D * 4));
    GK_CUDA(cudaMemsetAsync(h->colmin.p, 0x7F, D * 4, h->stream));
    GK_CUDA(cudaMemsetAsync(h->colmax.p, 0xFF, D * 4, h->stream));
    feat_minmax<<<h->sm_count * 16, 256, 0, h->stream>>>(h->ft_cap, h->ft_keys.as<unsigned long long>(), d_row_map,
                                                         h->colmin.as<int>(), h->colmax.as<int>());
    LAUNCH_CHECK(h);
  }

  // ---- head / tail split.  force_T: 1 = every contributing column dense.
  const double flops_per_col = square ? (double)k_rows * (double)(N + 1) : 2.0 * (double)k_rows * (double)k_cols;
  const double store_seconds = (double)k_rows * (double)k_cols * (double)esz / 6.5e12;  // K written once (debug print only)
  int force_T = (flags & (GK_GRAM_SIMT | GK_DENSE_ALL)) ? 1 : -1;
  if (force_T < 0) {  // testing knob: GRAKEL_B200_FORCE_T=<threshold>
    const char* e = getenv("GRAKEL_B200_FORCE_T");
    if (e && *e) force_T = std::max(1, atoi(e));
  }
  ColStats* cs = h->colstats.as<ColStats>();
  ColStats hc;
  DevScalars* hs = nullptr;
  int64_t max_count, max_diag, n_entries;
  if (pro) {  // gk_wl_features ran diag_finish + col_hist and brought the results back with its own synchronisation
    hc = hx->pro_hist;
    max_count = hx->pro_max_count; max_diag = hx->pro_max_diag; n_entries = hx->pro_n_entries;
  } else {
    GK_CUDA(cudaMemsetAsync(cs, 0, sizeof(ColStats), h->stream));
    col_hist<<<nbc, 256, 0, h->stream>>>(D, square ? 1 : 0, (int)n_fit, h->colcnt.as<unsigned>(), h->colmin.as<int>(),
                                         h->colmax.as<int>(), cs);
    LAUNCH_CHECK(h);
    GK_CUDA(cudaMemcpyAsync(h->h_colstats.p, cs, sizeof(ColStats), cudaMemcpyDeviceToHost, h->stream));
    GK_TRY(read_scalars(h, &hs));  // the one host synchronisation of gk_gram
    hc = *h->h_colstats.as<ColStats>();
    max_count = (int64_t)hs->max_count; max_diag = (int64_t)hs->max_diag; n_entries = (int64_t)hs->n_entries;
  }
  // ---- choose the Gram path and the head/tail threshold (host side, from the histogram)
  int path = 1;
  if ((flags & GK_GRAM_SIMT) || max_count > 256 || max_diag >= (1LL << 24)) { path = 2; force_T = 1; }
  int T = 1;
  {
    // T = 2^k minimising  head_cols * flops_per_col / rate + tail_updates * t_atomic
    // calibration (B200, profiles/r01b_*): dense mode sustains 1.5e15 flop/s; 4.36 M scattered fp32 atomics
    // take 152 us (random 32-byte sectors of a matrix that does not fit in L2: DRAM-bound)
    const double rate = 1.5e15;      // dense bf16 rate gram_tc_kernel sustains (flop/s)
    const double t_atomic = 3.5e-11; // amortised cost of one scattered pair update of K
    double best = -1.0;
    for (int k = 0; k <= HIST_BUCKETS - 2; ++k) {
      double head_cols = 0, tail_upd = 0;
      for (int b = 0; b < HIST_BUCKETS; ++b) {
        if (b > k) head_cols += (double)hc.hist_cols[b];
        else tail_upd += (double)hc.hist_work[b];
      }
      // measured (T = 64 vs 32 at config 2): the GEMM's time is additive in its store floor and its MMA
      // work -- operand loads and epilogue stores share the L2 -- so the constant store term does not
      // change the argmin and only the two variable terms are compared
      const double t_dense = head_cols * flops_per_col / rate;
      const double t = t_dense + tail_upd * t_atomic;
      if (best < 0 || t < best) { best = t; T = 1 << k; }
    }
    if (force_T >= 1) T = force_T;
  }
  int64_t Dc = 0, n_tail_cols = 0, n_tail_ent = 0;
  unsigned long long tail_work = 0;
  for (int b = 0; b < HIST_BUCKETS; ++b) {
    if (b < HIST_BUCKETS - 1 && (1LL << b) <= T) {
      n_tail_cols += (int64_t)hc.hist_cols[b];
      n_tail_ent += (int64_t)hc.hist_entries[b];
      tail_work += hc.hist_work[b];
    } else {
      Dc += (int64_t)hc.hist_cols[b];
    }
  }
  hc.T = T;
  if (getenv("GRAKEL_B200_DEBUG")) {
    fprintf(stderr, "[gk_gram] flops_per_col %.3g store_s %.3g T %d Dc %lld tail_cols %lld tail_ent %lld\n", flops_per_col,
            store_seconds, T, (long long)Dc, (long long)n_tail_cols, (long long)n_tail_ent);
    for (int b = 0; b < HIST_BUCKETS; ++b)
      fprintf(stderr, "  bucket %2d: cols %llu work %llu entries %llu\n", b, hc.hist_cols[b], hc.hist_work[b], hc.hist_entries[b]);
  }
  GK_TRY(h->tail_desc.ensure((size_t)std::max<int64_t>(n_tail_cols, 1) * sizeof(int2)));
  GK_TRY(h->tail_cur.ensure((size_t)std::max<int64_t>(n_tail_cols, 1) * 4));
  unsigned* col_counters = reinterpret_cast<unsigned*>(cs);  // the histogram has been read: reuse its first words
  GK_CUDA(cudaMemsetAsync(col_counters, 0, 16, h->stream));
  col_classify<<<nbc, 256, 0, h->stream>>>(D, square ? 1 : 0, (int)n_fit, h->colcnt.as<unsigned>(), h->colmin.as<int>(),
                                           h->colmax.as<int>(), T, h->colslot.as<int>(), h->tail_desc.as<int2>(),
                                           h->tail_cur.as<unsigned>(), col_counters);
  LAUNCH_CHECK(h);
  if (path == 1 && Dc == 0) path = 3;
  h->Dc = Dc;
  h->Dc_pad = (Dc + BK - 1) / BK * BK;
  if (force_T < 0 && path == 1 && square) hx->head_dc_pad = h->Dc_pad;

  // ---- transport type.  Tensor-core results are integers < 2^24 (checked above), i.e. exact in fp32: a float64
  // HOST result is produced and moved as fp32 (half the HBM writes; a quarter of the PCIe bytes for the
  // symmetric case, whose upper triangle alone is copied) and widened -- and, if asked, normalised in fp64 --
  // by host threads while the next band is in flight (host_deliver.h).  GRAKEL_B200_WIDEN=0 restores the
  // plain fp64 D2H copy of a device-side fp64 result.
  const char* widen_env = getenv("GRAKEL_B200_WIDEN");
  const bool widen_on_host = K_out && !(flags & GK_OUT_DEVICE) && out_dtype == GK_F64 && path != 2 &&
                             !(widen_env && atoi(widen_env) == 0);
  const bool host_norm = widen_on_host && normalize;
  const int32_t dev_dtype = widen_on_host ? GK_F32 : out_dtype;
  const size_t dev_esz = dev_dtype == GK_F64 ? 8 : 4;

  // multi-GPU row tiling (GK_DIST, collective): SYRK tiles shared between the ranks, mirrored halves stored into the
  // owner's row block over NVLink.  Needs the tensor path and fp32 device output; otherwise every rank computes its
  // row block with full tiles (the decision depends on replicated data only, so all ranks take the same branch).
  Comm* comm = reinterpret_cast<Comm*>(h->comm);
  const bool dist_req = (flags & (GK_DIST | GK_DIST_GATHER)) != 0;
  if (dist_req) {
    if (!comm) return fail(GK_ERR_STATE, "gk_gram: GK_DIST without gk_comm_init");
    if (!square || d_row_map) return fail(GK_ERR_UNSUPPORTED, "gk_gram: GK_DIST needs the square fit_transform case without a row map");
    if (flags & GK_OUT_DEVICE) return fail(GK_ERR_UNSUPPORTED, "gk_gram: GK_DIST results are library-owned (gk_result_device / gk_fetch / host K_out)");
    int64_t rb = 0, re = 0;
    GK_TRY(gk_comm_rows(h, N, &rb, &re));
    if (row_begin != rb || row_end != re) return fail(GK_ERR_ARG, "gk_gram: GK_DIST row range must be the one gk_comm_rows returns");
  }
  // GRAKEL_B200_DIST_SHARE=0: no tile sharing -- every rank computes its row block with full tiles (twice the SYRK
  // flops, no peer stores, no barriers): the round-1 scheme, kept for A/B measurements
  const char* e_share = getenv("GRAKEL_B200_DIST_SHARE");
  const bool dist = dist_req && path == 1 && dev_dtype == GK_F32 && !normalize && !(e_share && atoi(e_share) == 0);
  const bool gather = dist && (flags & GK_DIST_GATHER);
  const long long dist_per = dist_req ? dist_rows_per_rank(N, comm->nranks) : 0;


  // ---- output buffer
  void* d_out = nullptr;
  if (flags & GK_OUT_DEVICE) {
    if (!K_out) return fail(GK_ERR_ARG, "gk_gram: GK_OUT_DEVICE without a pointer");
    d_out = K_out;
  } else {
    // library-owned K: rows padded to a multiple of 8 elements so that every row is 32-byte aligned
    // (TMA / 256-bit stores in the GEMM epilogue for any n_fit, e.g. 14 142 graphs on 2 GPUs)
    h->K_ld = (k_cols + 7) / 8 * 8;
    if (dist_req) {
      // the same request on every rank: a block of dist_per rows (all comm->nranks of them for the gathered result)
      const size_t blk = (size_t)dist_per * h->K_ld * dev_esz;
      GK_TRY(comm_share_K(h, (flags & GK_DIST_GATHER) ? blk * comm->nranks : blk));
      d_out = (flags & GK_DIST_GATHER) ? (void*)(h->K.as<char>() + (size_t)comm->rank * blk) : h->K.p;
    } else {
      GK_TRY(h->K.ensure((size_t)std::max<int64_t>(k_rows, 1) * h->K_ld * dev_esz));
      d_out = h->K.p;
    }
    h->K_rows = k_rows; h->K_cols = k_cols; h->K_dtype = dev_dtype;
  }
  const long long d_ld = (flags & GK_OUT_DEVICE) ? ld : h->K_ld;

  // panel-row ranges: A rows index K rows, B rows index K columns
  const int a0 = (int)((square ? 0 : n_fit) + row_begin), a1 = (int)((square ? 0 : n_fit) + row_end);
  const int b0 = 0, b1 = (int)n_fit;
  const bool full_square = square && row_begin == 0 && row_end == N;
  const bool mirror = (full_square && !(flags & GK_FULL_TILES)) || dist;
  const bool has_tail = path != 2 && n_tail_cols > 0;
  const bool norm_in_epilogue = normalize && !has_tail && !host_norm;

  GramParams p;
  memset(&p, 0, sizeof(p));
  p.a_row_end = a1; p.b_row_end = b1;
  p.c_row0 = a0; p.c_col0 = b0;
  p.out = d_out; p.ld = d_ld;
  p.mirror = mirror ? 1 : 0;
  p.fix_diag = square ? 1 : 0;
  p.nan_to_num = (flags & GK_NAN_TO_NUM) ? 1 : 0;
  p.vec_ok = (((uintptr_t)d_out) % 32 == 0 && (d_ld * (long long)dev_esz) % 32 == 0) ? 1 : 0;
  p.diag = h->diag_f64.as<double>();
  if (dist) {
    const size_t blk = (size_t)dist_per * d_ld * 4;
    for (int r = 0; r < comm->nranks; ++r)
      p.peer[r] = (flags & GK_DIST_GATHER) ? (void*)((char*)comm->peer_base[r] + (size_t)r * blk) : comm->peer_base[r];
    p.n_peers = comm->nranks;
    p.peer_rows = (int)dist_per;
  }
  if (dist) GK_TRY(comm_barrier(h));  // nobody still reads the block a peer is about to overwrite

  GK_CUDA(cudaEventRecord(h->tev[5], h->stream));
  int64_t n_tiles = 0;
  if (k_rows > 0) {
    // (always at least a stub: gk_wl_gram's asynchronous pass sizes its tail by the capacity left here)
    GK_TRY(h->tail_ent.ensure((size_t)std::max<int64_t>(has_tail ? n_tail_ent : 0, 64) * sizeof(int2)));
    if (path == 1 || path == 3) {
      const size_t panel_bytes = (size_t)N * std::max<int64_t>(h->Dc_pad, BK) * 2;
      GK_TRY(h->panel.ensure(panel_bytes));
      if (Dc) GK_CUDA(cudaMemsetAsync(h->panel.p, 0, panel_bytes, h->stream));
      if (Dc || has_tail) {
        feat_scatter<<<cdiv((long long)h->ft_cap, 256), 256, 0, h->stream>>>(
            h->ft_cap, h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(), h->colslot.as<int>(), d_row_map,
            h->panel.as<__nv_bfloat16>(), h->Dc_pad, h->tail_cur.as<unsigned>(), h->tail_desc.as<int2>(),
            h->tail_ent.as<int2>());
        LAUNCH_CHECK(h);
      }
    }
    if (path == 1) {
      // CTA-pair kernel (gram_tc2.cuh: cta_group::2, 256 x 256 tiles) for fp32 un-normalised output through
      // TMA stores: 1 831 vs 1 515 TFLOP/s in dense mode, 0.201 vs 0.228 ms in head mode on the same box
      // (profiles/r01g_bench_cta{2,1}.json).  GRAKEL_B200_CTA2=0 selects the one-CTA kernel.
      const char* e_cta2 = getenv("GRAKEL_B200_CTA2");
      const bool cta2 = !(e_cta2 && atoi(e_cta2) == 0) && dev_dtype == GK_F32 && !norm_in_epilogue &&
                        ((uintptr_t)d_out) % 16 == 0 && (d_ld * 4) % 16 == 0 && !getenv("GRAKEL_B200_NO_TMA_STORE");
      if (dist && !cta2) return fail(GK_ERR_UNSUPPORTED, "gk_gram: GK_DIST needs the CTA-pair kernel (GRAKEL_B200_CTA2=0 is set?)");
      // the tile list depends on the shape of the request only: built and uploaded when that changes
      const long long tkey[8] = {dist ? 1 : 0, dist ? (long long)N : a0, dist ? comm->nranks : a1, dist ? comm->rank : b0, b1,
                                 mirror ? 1 : 0, cta2 ? BM2 : BM, 0};
      if (memcmp(tkey, hx->tiles_key, sizeof(tkey)) != 0 || !h->tiles.p) {
        std::vector<int2> tiles;
        if (dist) dist_tiles(N, comm->nranks, comm->rank, tiles);
        else build_tiles(tiles, a0, a1, b0, b1, mirror, cta2 ? BM2 : BM);
        GK_TRY(h->h_tiles.ensure(tiles.size() * sizeof(int2) + 16));
        memcpy(h->h_tiles.p, tiles.data(), tiles.size() * sizeof(int2));
        GK_TRY(h->tiles.ensure(tiles.size() * sizeof(int2) + 16));
        GK_CUDA(cudaMemcpyAsync(h->tiles.p, h->h_tiles.p, tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
        memcpy(hx->tiles_key, tkey, sizeof(tkey));
        hx->tiles_n = (long long)tiles.size();
      }
      n_tiles = hx->tiles_n;
      CUtensorMap tmA, tmB, tmC;
      PeerMaps peer_maps;
      memset(&peer_maps, 0, sizeof(peer_maps));
      GK_TRY(make_panel_map(&tmA, h->panel.p, h->Dc_pad, N, BM));
      GK_TRY(make_panel_map(&tmB, h->panel.p, h->Dc_pad, N, BN));
      memset(&tmC, 0, sizeof(tmC));
      p.tma_store = 0;
      if (dev_dtype == GK_F32 && !norm_in_epilogue && ((uintptr_t)d_out) % 16 == 0 && (d_ld * 4) % 16 == 0 &&
          !getenv("GRAKEL_B200_NO_TMA_STORE")) {
        GK_TRY(make_out_map(&tmC, d_out, k_cols, k_rows, d_ld));
        p.tma_store = 1;
        if (p.mirror && !dist) {  // full square: the mirrored half goes through the same tensor map
          const char* e = getenv("GRAKEL_B200_MIRROR_TMA");
          if (!e || atoi(e) != 0) p.mirror = 2;
        }
        if (dist) {  // mirrored blocks as bulk TMA stores into the owners' row blocks (else 32 row stores of 128 B per block)
          const char* e = getenv("GRAKEL_B200_DIST_TMA");
          if (e && atoi(e) != 0) {
            for (int r = 0; r < comm->nranks; ++r) {
              const long long r_rows = std::min<long long>(N, (long long)(r + 1) * dist_per) - std::min<long long>(N, (long long)r * dist_per);
              if (r_rows > 0) GK_TRY(make_out_map(&peer_maps.m[r], p.peer[r], k_cols, r_rows, d_ld));
            }
            p.mirror = 2;
          }
        }
      }
      p.tiles = h->tiles.as<int2>();
      p.n_tiles = (int)n_tiles;
      p.num_k_blocks = (int)(h->Dc_pad / BK);
      const int grid = cta2 ? 2 * (int)std::min<int64_t>(n_tiles, h->sm_count / 2) : (int)std::min<int64_t>(n_tiles, h->sm_count);
      const bool prof = !cta2 && getenv("GRAKEL_B200_PROF") != nullptr;
      if (prof) {
        GK_TRY(h->K_stage.ensure((size_t)grid * 64));
        GK_CUDA(cudaMemsetAsync(h->K_stage.p, 0, (size_t)grid * 64, h->stream));
        p.prof = h->K_stage.as<long long>();
      }
      GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
      if (n_tiles == 0) { /* a trailing rank without rows */ }
      else if (cta2) gram_tc2_kernel<<<grid, GEMM_THREADS, GEMM2_SMEM, h->stream>>>(tmA, tmC, p, peer_maps);
      else if (dev_dtype == GK_F64) { if (norm_in_epilogue) launch_tc<double, true>(h, tmA, tmB, tmC, p, grid); else launch_tc<double, false>(h, tmA, tmB, tmC, p, grid); }
      else { if (norm_in_epilogue) launch_tc<float, true>(h, tmA, tmB, tmC, p, grid); else launch_tc<float, false>(h, tmA, tmB, tmC, p, grid); }
      LAUNCH_CHECK(h);
      if (prof) {
        std::vector<long long> pr((size_t)grid * 8);
        GK_CUDA(cudaMemcpyAsync(pr.data(), h->K_stage.p, pr.size() * 8, cudaMemcpyDeviceToHost, h->stream));
        GK_CUDA(cudaStreamSynchronize(h->stream));
        double a[8] = {0};
        for (int b = 0; b < grid; ++b) for (int i = 0; i < 8; ++i) a[i] += (double)pr[(size_t)b * 8 + i] / grid;
        fprintf(stderr, "[gram_tc prof] tiles %lld kblocks %d grid %d | epi: wait_tfull %.0f work %.0f | mma: wait_tempty %.0f wait_full %.0f total %.0f | tma: wait_empty %.0f total %.0f (avg cycles per CTA)\n",
                (long long)n_tiles, p.num_k_blocks, grid, a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
      }
    } else if (path == 2) {
      const size_t panel_bytes = (size_t)N * std::max<int64_t>(Dc, 1) * 4;
      GK_TRY(h->panel.ensure(panel_bytes));
      GK_CUDA(cudaMemsetAsync(h->panel.p, 0, panel_bytes, h->stream));
      feat_fill_panel_u32<<<cdiv((long long)h->ft_cap, 256), 256, 0, h->stream>>>(
          h->ft_cap, h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(), h->colslot.as<int>(), d_row_map,
          h->panel.as<unsigned>(), std::max<int64_t>(Dc, 1));
      LAUNCH_CHECK(h);
      GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
      if (dev_dtype == GK_F64) { if (normalize) launch_simt<double, true>(h, h->panel.as<unsigned>(), std::max<int64_t>(Dc, 1), (int)Dc, a0, a1, b0, b1, p); else launch_simt<double, false>(h, h->panel.as<unsigned>(), std::max<int64_t>(Dc, 1), (int)Dc, a0, a1, b0, b1, p); }
      else { if (normalize) launch_simt<float, true>(h, h->panel.as<unsigned>(), std::max<int64_t>(Dc, 1), (int)Dc, a0, a1, b0, b1, p); else launch_simt<float, false>(h, h->panel.as<unsigned>(), std::max<int64_t>(Dc, 1), (int)Dc, a0, a1, b0, b1, p); }
      LAUNCH_CHECK(h);
    } else {
      GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
      if (dev_dtype == GK_F64) { if (norm_in_epilogue) launch_empty<double, true>(h, a0, a1, b0, b1, p); else launch_empty<double, false>(h, a0, a1, b0, b1, p); }
      else { if (norm_in_epilogue) launch_empty<float, true>(h, a0, a1, b0, b1, p); else launch_empty<float, false>(h, a0, a1, b0, b1, p); }
      LAUNCH_CHECK(h);
    }
    GK_CUDA(cudaEventRecord(h->tev[7], h->stream));
    if (dist) GK_TRY(comm_barrier(h));  // the peers' mirrored stores into this block precede the tail's atomics
    if (has_tail) {
      const int grid = cdiv(n_tail_cols * 32, 256);
      if (dev_dtype == GK_F64)
        tail_pairs<double><<<grid, 256, 0, h->stream>>>(n_tail_cols, h->tail_desc.as<int2>(), h->tail_ent.as<int2>(),
                                                        (int)n_fit, square ? 1 : 0, (int)row_begin, (int)row_end,
                                                        (double*)d_out, d_ld);
      else
        tail_pairs<float><<<grid, 256, 0, h->stream>>>(n_tail_cols, h->tail_desc.as<int2>(), h->tail_ent.as<int2>(),
                                                       (int)n_fit, square ? 1 : 0, (int)row_begin, (int)row_end,
                                                       (float*)d_out, d_ld);
      LAUNCH_CHECK(h);
      if (normalize && !host_norm) {
        const double* drow = h->diag_f64.as<double>() + a0;
        const double* dcol = h->diag_f64.as<double>() + b0;
        if (dev_dtype == GK_F64)
          normalize_rows<double><<<h->sm_count * 8, 256, 0, h->stream>>>(k_rows, k_cols, (double*)d_out, d_ld, drow, dcol, p.nan_to_num);
        else
          normalize_rows<float><<<h->sm_count * 8, 256, 0, h->stream>>>(k_rows, k_cols, (float*)d_out, d_ld, drow, dcol, p.nan_to_num);
        LAUNCH_CHECK(h);
      }
    }
  } else {
    GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
    GK_CUDA(cudaEventRecord(h->tev[7], h->stream));
    if (dist) GK_TRY(comm_barrier(h));
  }
  if (dist_req && (flags & GK_DIST_GATHER)) {
    // BASELINE config 4: every rank ends up with the full matrix -- one in-place all-gather of the finished row
    // blocks (NCCL over NVLink / NVSwitch); the library-owned result is reached through gk_result_device / gk_fetch
    NcclApi* api = nccl_api();
    const size_t cnt = (size_t)dist_per * d_ld;
    GK_CUDA(cudaEventRecord(h->ev[12], h->stream));
    GK_NCCL(api, api->AllGather(d_out, h->K.p, cnt, dev_dtype == GK_F64 ? ncclFloat64 : ncclFloat32, comm->comm, h->stream));
    h->K_rows = N;
  }
  GK_CUDA(cudaEventRecord(h->ev[13], h->stream));
  const int64_t launches_gram = h->launches - launches0;

  // ---- results to the host
  GK_CUDA(cudaEventRecord(h->ev[14], h->stream));
  if (K_out && !(flags & GK_OUT_DEVICE) && k_rows > 0) {
    if (widen_on_host) {
      const float* d_k = reinterpret_cast<const float*>(d_out);
      double* dst = reinterpret_cast<double*>(K_out);
      DeviceCopier cp{h};
      if (host_norm) {
        GK_TRY(h->h_diag.ensure((size_t)N * 8));
        GK_CUDA(cudaMemcpyAsync(h->h_diag.p, h->diag_f64.p, (size_t)N * 8, cudaMemcpyDeviceToHost, h->stream));
        GK_CUDA(cudaStreamSynchronize(h->stream));
        GK_TRY(deliver_rows(cp, d_k, d_ld, k_rows, k_cols, dst, ld, h->h_diag.as<double>() + a0, h->h_diag.as<double>() + b0,
                            p.nan_to_num));
      } else if (full_square && !getenv("GRAKEL_B200_NO_TRI")) {
        GK_TRY(deliver_square(h, d_k, d_ld, k_rows, dst, ld, max_diag));
      } else {
        GK_TRY(deliver_rows(cp, d_k, d_ld, k_rows, k_cols, dst, ld, nullptr, nullptr, 0));
      }
    } else {
      GK_CUDA(cudaMemcpy2DAsync(K_out, (size_t)ld * esz, d_out, (size_t)d_ld * esz, (size_t)k_cols * esz,
                                (size_t)k_rows, cudaMemcpyDeviceToHost, h->stream));
    }
  }
  if (xdiag) GK_CUDA(cudaMemcpyAsync(xdiag, h->diag_f64.p, n_fit * 8, cudaMemcpyDeviceToHost, h->stream));
  if (ydiag && !square)
    GK_CUDA(cudaMemcpyAsync(ydiag, h->diag_f64.as<double>() + n_fit, (N - n_fit) * 8, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaEventRecord(h->ev[15], h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  if (stats) {
    stats->n_graphs = N; stats->n_vertices = h->V; stats->n_edges = h->E;
    stats->n_entries = n_entries;
    stats->n_dense_columns = Dc;
    stats->n_tail_columns = n_tail_cols;
    stats->tail_updates = (int64_t)tail_work;
    stats->threshold = hc.T;
    stats->max_count = max_count;
    stats->max_diag = max_diag;
    stats->gram_path = path;
    stats->gemm_tiles = n_tiles;
    stats->gemm_launches = launches_gram;
    stats->ms_panel = ev_ms(h->tev[4], h->tev[6]);
    stats->ms_gemm = ev_ms(h->tev[6], h->tev[7]);
    stats->ms_tail = ev_ms(h->tev[7], h->ev[13]);
    stats->ms_d2h = ev_ms(h->ev[14], h->ev[15]);
    stats->ms_total = ev_ms(h->tev[4], h->ev[15]);
  }
  return GK_OK;
}

int gk_set_row_map(gk_handle* h, int64_t n_rows, const int32_t* row_of_graph) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (h->N <= 0) return fail(GK_ERR_STATE, "gk_set_row_map: no graphs packed");
  GK_CUDA(cudaSetDevice(h->dev));
  if (n_rows <= 0 || !row_of_graph) {  // back to the identity
    h->n_rows = 0;
    return GK_OK;
  }
  for (int64_t g = 0; g < h->N; ++g)
    if (row_of_graph[g] < 0 || row_of_graph[g] >= n_rows) return fail(GK_ERR_ARG, "gk_set_row_map: row index out of range");
  GK_TRY(h->row_map.ensure(h->N * 4));
  GK_CUDA(cudaMemcpyAsync(h->row_map.p, row_of_graph, h->N * 4, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  h->n_rows = n_rows;
  return GK_OK;
}

int gk_result_device(gk_handle* h, void** ptr, int64_t* rows, int64_t* cols, int64_t* ld, int32_t* dtype) {
  if (!h || !ptr) return fail(GK_ERR_ARG, "gk_result_device: null argument");
  if (!h->K.p || h->K_rows <= 0) return fail(GK_ERR_STATE, "gk_result_device: no device-resident result");
  *ptr = h->K.p;
  if (rows) *rows = h->K_rows;
  if (cols) *cols = h->K_cols;
  if (ld) *ld = h->K_ld;
  if (dtype) *dtype = h->K_dtype;
  return GK_OK;
}

int gk_fetch(gk_handle* h, void* K_out, int32_t out_dtype, int64_t ld) {
  if (!h || !K_out) return fail(GK_ERR_ARG, "gk_fetch: null argument");
  if (!h->K.p || h->K_rows <= 0) return fail(GK_ERR_STATE, "gk_fetch: no device-resident result");
  if (out_dtype != h->K_dtype) return fail(GK_ERR_ARG, "gk_fetch: dtype differs from the one gk_gram produced");
  const size_t esz = out_dtype == GK_F64 ? 8 : 4;
  if (ld <= 0) ld = h->K_cols;
  GK_CUDA(cudaSetDevice(h->dev));
  GK_CUDA(cudaMemcpy2DAsync(K_out, (size_t)ld * esz, h->K.p, (size_t)h->K_ld * esz, (size_t)h->K_cols * esz,
                            (size_t)h->K_rows, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  return GK_OK;
}

// --------------------------------------------------------------------------- TU files -> CSR (host only)
int gk_tu_open(const char* dir, const char* name, int32_t flags, gk_tu** out) {
  if (!dir || !name || !out) return fail(GK_ERR_ARG, "gk_tu_open: null argument");
  std::string err;
  const int r = gk::tu::open(dir, name, flags, out, &err);
  return r == GK_OK ? GK_OK : fail(r, "gk_tu_open: " + err);
}

int gk_tu_info(const gk_tu* t, int64_t* info) {
  if (!t || !info) return fail(GK_ERR_ARG, "gk_tu_info: null argument");
  info[0] = t->n_graphs; info[1] = t->n_nodes; info[2] = (int64_t)t->eu.size();
  info[3] = !t->node_label.empty(); info[4] = !t->el.empty(); info[5] = !t->classes.empty();
  info[6] = t->attr_dim; info[7] = 0;
  return GK_OK;
}

int gk_tu_pack(gk_tu* t, int32_t mode, int64_t* n_vertices, int64_t* n_edges) {
  if (!t) return fail(GK_ERR_ARG, "gk_tu_pack: null handle");
  std::string err;
  const int r = gk::tu::pack(t, mode, &err);
  if (r != GK_OK) return fail(r, "gk_tu_pack: " + err);
  if (n_vertices) *n_vertices = (int64_t)t->vnode.size();
  if (n_edges) *n_edges = (int64_t)t->col_idx.size();
  return GK_OK;
}

int gk_tu_fill(const gk_tu* t, int32_t* graph_ptr, int32_t* row_ptr, int32_t* col_idx, int32_t* node_labels,
               int32_t* edge_labels, double* attrs, int32_t* classes, int32_t* node_of_vertex) {
  if (!t) return fail(GK_ERR_ARG, "gk_tu_fill: null handle");
  if (t->mode < 0) return fail(GK_ERR_STATE, "gk_tu_fill: call gk_tu_pack first");
  const size_t V = t->vnode.size();
  if (graph_ptr) memcpy(graph_ptr, t->graph_ptr.data(), t->graph_ptr.size() * 4);
  if (row_ptr) memcpy(row_ptr, t->row_ptr.data(), t->row_ptr.size() * 4);
  if (col_idx && !t->col_idx.empty()) memcpy(col_idx, t->col_idx.data(), t->col_idx.size() * 4);
  if (node_labels) {
    if (t->vlabel.empty() && V) return fail(GK_ERR_STATE, "gk_tu_fill: the dataset has no node labels");
    if (V) memcpy(node_labels, t->vlabel.data(), V * 4);
  }
  if (edge_labels) {
    if (t->el.empty()) return fail(GK_ERR_STATE, "gk_tu_fill: the dataset has no edge labels");
    if (!t->elabel.empty()) memcpy(edge_labels, t->elabel.data(), t->elabel.size() * 4);
  }
  if (attrs) {
    if (!t->attr_dim) return fail(GK_ERR_STATE, "gk_tu_fill: node attributes were not loaded (GK_TU_ATTR_NODES)");
    for (size_t v = 0; v < V; ++v)
      memcpy(attrs + v * t->attr_dim, t->node_attr.data() + (size_t)t->vnode[v] * t->attr_dim, (size_t)t->attr_dim * 8);
  }
  if (classes) {
    if (t->classes.empty()) return fail(GK_ERR_STATE, "gk_tu_fill: the dataset has no graph classes");
    memcpy(classes, t->classes.data(), t->classes.size() * 4);
  }
  if (node_of_vertex)
    for (size_t v = 0; v < V; ++v) node_of_vertex[v] = t->vnode[v] + 1;
  return GK_OK;
}

int gk_tu_close(gk_tu* t) {
  delete t;
  return GK_OK;
}

// ---------------------------------------------------------------------------
}  // extern "C"

// ---------------------------------------------------------------------------
// The asynchronous WL pass: feature kernels, column statistics, the head/tail decision (gram_choose, ON THE DEVICE),
// panel, GEMM and tail are enqueued back to back -- the host synchronises once, at the end.  The synchronous route
// (gk_wl_features + gk_gram) needs the column histogram on the host between the two halves; here the host only sizes
// things by CAPACITY (the panel's row pitch, the tail buffers: what earlier passes on this handle allocated) and the
// device reports through GramDyn::bad when a capacity, an exactness bound or the WL hash check fails, in which case
// the caller repeats the pass through the synchronous route (which also grows the buffers).  Square fit_transform
// case with an fp32 device result: library-owned, caller's device buffer, or float64 host delivery.
static int wl_gram_async(gk_handle* h, int32_t n_iter, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld,
                         double* xdiag, gk_stats* stats, bool* done) {
  *done = false;
  for (const char* name : {"GRAKEL_B200_NO_ASYNC", "GRAKEL_B200_PROF", "GRAKEL_B200_NO_PROLOGUE", "GRAKEL_B200_WL_V1",
                           "GRAKEL_B200_WL_FUSED", "GRAKEL_B200_CTA2", "GRAKEL_B200_NO_TMA_STORE", "GRAKEL_B200_WIDEN",
                           "GRAKEL_B200_NO_TRI", "GRAKEL_B200_MIRROR_TMA", "GRAKEL_B200_DEBUG"})
    if (getenv(name)) return GK_OK;
  if (flags & ~(GK_OUT_DEVICE | GK_DENSE_ALL)) return GK_OK;
  if (h->N <= 0 || !h->has_labels || h->V == 0 || n_iter < 0 || n_iter + 1 >= MAX_LEVELS || h->n_rows > 0) return GK_OK;
  const int64_t N = h->N, V = h->V;
  const bool dev_out = (flags & GK_OUT_DEVICE) != 0;
  const bool host_out = K_out && !dev_out;
  if (host_out && out_dtype != GK_F64) return GK_OK;
  if (!host_out && out_dtype != GK_F32) return GK_OK;
  if (dev_out && !K_out) return GK_OK;
  if (ld > 0 && ld < N) return GK_OK;  // (the synchronous route reports the error)
  if (dev_out && (((uintptr_t)K_out) % 16 != 0 || ((ld > 0 ? ld : N) * 4) % 16 != 0)) return GK_OK;
  // capacities left by earlier passes
  int64_t S = (int64_t)(h->panel.cap / ((size_t)N * 2)) / BK * BK;
  {  // no wider than the last cost-model pass needed, plus a quarter (a dense-all pass may have left a much larger buffer,
     // and the whole pitch is zeroed: 466 MB in profiles/r03_full_summary.md before this cap)
    const long long want = extra_of(h)->head_dc_pad;
    if (!(flags & GK_DENSE_ALL) && !getenv("GRAKEL_B200_FORCE_T") && want > 0)
      S = std::min<int64_t>(S, (want + want / 4 + BK - 1) / BK * BK + BK);
  }
  if (S < BK || !h->tail_desc.p || !h->tail_cur.p || !h->tail_ent.p) return GK_OK;
  const long long cap_tail_cols = (long long)std::min(h->tail_desc.cap / sizeof(int2), h->tail_cur.cap / 4);
  const long long cap_tail_ent = (long long)(h->tail_ent.cap / sizeof(int2));
  GK_CUDA(cudaSetDevice(h->dev));
  const int L = n_iter + 1;
  h->n_levels = L;
  h->features_ready = false; h->feat_serial++;
  const int64_t launches0 = h->launches;
  WlPlan pl;
  GK_TRY(wl_setup(h, n_iter, &pl));
  if (!pl.fused) return GK_OK;
  HandleExtra* hx = extra_of(h);
  const int64_t D = (int64_t)h->n_labels0 + V * (int64_t)(L - 1);
  FeatStats fst;
  GK_TRY(reset_feature_stats(h, D + 1, (int64_t)std::max(pl.nb, pl.G) * L, &fst, false));
  GK_TRY(h->colstats.ensure(sizeof(ColStats)));
  if (!h->gram_dyn.p) {
    GK_TRY(h->gram_dyn.ensure(sizeof(GramDyn)));
    GK_CUDA(cudaMemsetAsync(h->gram_dyn.p, 0, sizeof(GramDyn), h->stream));  // the block ticket starts at zero
  }
  DevScalars* sc = h->scalars.as<DevScalars>();
  ColStats* cs = h->colstats.as<ColStats>();
  GramDyn* dyn = h->gram_dyn.as<GramDyn>();
  // ---- features first: everything else the host has to prepare overlaps the WL kernel
  GK_CUDA(cudaMemsetAsync(cs, 0, sizeof(ColStats), h->stream));
  GK_CUDA(cudaEventRecord(h->tev[2], h->stream));
  const unsigned long long seed = mix64(0x5851F42D4C957F2DULL);
  GK_TRY(wl_launch_v2(h, pl, seed, fst, false));
  h->wl_sparse_ids = L > 1;
  GK_CUDA(cudaEventRecord(h->tev[3], h->stream));
  // ---- the panel (full row pitch) is zeroed on the side stream while the column statistics run (the WL kernel itself
  // owns every register file: nothing can share an SM with it)
  GK_CUDA(cudaEventRecord(h->ev_fork, h->stream));
  GK_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
  panel_zero_rows<<<h->sm_count * 4, 256, 0, h->stream2>>>(h->panel.as<__nv_bfloat16>(), N, S, (int)(S / 8));
  LAUNCH_CHECK(h);
  GK_CUDA(cudaEventRecord(h->ev_stage[0], h->stream2));

  GK_TRY(h->colslot.ensure(std::max<int64_t>(D, 1) * 4));
  GK_TRY(h->h_dyn.ensure(sizeof(GramDyn) + 64));
  GK_TRY(h->diag_f64.ensure(N * 8));
  // output
  void* d_out;
  long long d_ld;
  if (dev_out) {
    d_out = K_out;
    d_ld = ld > 0 ? ld : N;
  } else {
    h->K_ld = (N + 7) / 8 * 8;
    GK_TRY(h->K.ensure((size_t)N * h->K_ld * 4));
    d_out = h->K.p;
    d_ld = h->K_ld;
    h->K_rows = N; h->K_cols = N; h->K_dtype = GK_F32;
  }
  // tile list (same key as gk_gram's)
  {
    const long long tkey[8] = {0, 0, (long long)N, 0, (long long)N, 1, BM2, 0};
    if (memcmp(tkey, hx->tiles_key, sizeof(tkey)) != 0 || !h->tiles.p) {
      std::vector<int2> tiles;
      build_tiles(tiles, 0, (int)N, 0, (int)N, true, BM2);
      GK_TRY(h->h_tiles.ensure(tiles.size() * sizeof(int2) + 16));
      memcpy(h->h_tiles.p, tiles.data(), tiles.size() * sizeof(int2));
      GK_TRY(h->tiles.ensure(tiles.size() * sizeof(int2) + 16));
      GK_CUDA(cudaMemcpyAsync(h->tiles.p, h->h_tiles.p, tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
      memcpy(hx->tiles_key, tkey, sizeof(tkey));
      hx->tiles_n = (long long)tiles.size();
    }
  }
  const int64_t n_tiles = hx->tiles_n;
  CUtensorMap tmA, tmC;
  PeerMaps peer_maps;
  memset(&peer_maps, 0, sizeof(peer_maps));
  GK_TRY(make_panel_map(&tmA, h->panel.p, S, N, BM));
  GK_TRY(make_out_map(&tmC, d_out, N, N, d_ld));
  int force_T = (flags & GK_DENSE_ALL) ? 1 : -1;
  if (force_T < 0) {
    const char* e = getenv("GRAKEL_B200_FORCE_T");
    if (e && *e) force_T = std::max(1, atoi(e));
  }
  // ---- columns: self similarities, histogram, the decision -- one launch, one copy back
  GK_CUDA(cudaEventRecord(h->tev[4], h->stream));
  const int64_t Dn = std::max<int64_t>(D, 1);
  const int nbc = cdiv(Dn, 256);
  {
    ColFusedParams q;
    q.D = Dn; q.N = (int)N; q.L = L;
    q.colcnt = h->colcnt.as<unsigned>();
    q.diag = h->diag_u64.as<unsigned long long>(); q.diag_f64 = h->diag_f64.as<double>();
    q.n_part = (int)h->n_part; q.part_max = h->part_max.as<unsigned>(); q.part_new = h->part_new.as<unsigned>();
    q.cs = cs; q.sc = sc; q.dyn = dyn;
    q.flops_per_col = (double)N * (double)(N + 1); q.rate = 1.5e15; q.t_atomic = 3.5e-11;
    q.force_T = force_T; q.stride_cap = (int)S; q.bk = BK;
    q.cap_tail_cols = cap_tail_cols; q.cap_tail_ent = cap_tail_ent;
    col_stats_fused<<<h->sm_count * 4, 256, 0, h->stream>>>(q);
    LAUNCH_CHECK(h);
  }
  // the copy back travels on the side stream: the main stream goes straight on to the classification
  GK_CUDA(cudaEventRecord(h->ev_stage[1], h->stream));
  GK_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_stage[1], 0));
  GK_CUDA(cudaMemcpyAsync(h->h_dyn.p, dyn, sizeof(GramDyn), cudaMemcpyDeviceToHost, h->stream2));
  GK_CUDA(cudaEventRecord(h->ev_join, h->stream2));  // the host waits for THIS, not for the GEMM behind it
  unsigned* col_counters = reinterpret_cast<unsigned*>(cs);  // cleared by the deciding block
  col_classify<<<nbc, 256, 0, h->stream>>>(Dn, 1, (int)N, h->colcnt.as<unsigned>(), nullptr, nullptr, 1, h->colslot.as<int>(),
                                           h->tail_desc.as<int2>(), h->tail_cur.as<unsigned>(), col_counters, dyn);
  LAUNCH_CHECK(h);
  GK_CUDA(cudaStreamWaitEvent(h->stream, h->ev_stage[0], 0));  // the zeroed panel
  feat_scatter<<<cdiv((long long)h->ft_cap, 256), 256, 0, h->stream>>>(
      h->ft_cap, h->ft_keys.as<unsigned long long>(), h->ft_cnt.as<unsigned>(), h->colslot.as<int>(), nullptr,
      h->panel.as<__nv_bfloat16>(), S, h->tail_cur.as<unsigned>(), h->tail_desc.as<int2>(), h->tail_ent.as<int2>());
  LAUNCH_CHECK(h);
  // ---- tail: bucketed by 32 x 32 block of K for the GEMM epilogue (GRAKEL_B200_TAIL_FUSED=0: the separate tail_pairs kernel)
  const char* e_tf = getenv("GRAKEL_B200_TAIL_FUSED");
  const bool tail_fused = !(e_tf && atoi(e_tf) == 0);
  const int nb32 = (int)((N + 31) / 32);
  const unsigned ovf_cap = 1u << 20;
  const char* e_sym = getenv("GRAKEL_B200_TB_SYM");
  const int tb_sym = (e_sym && atoi(e_sym) != 0) ? 1 : 0;  // symmetric lists (pairs with row < column only): half the atomics
  int tb_cap = TB_CAP;  // tests shrink it (GRAKEL_B200_TB_CAP) to drive updates through the overflow list
  if (const char* e = getenv("GRAKEL_B200_TB_CAP")) tb_cap = std::max(0, std::min(TB_CAP, atoi(e)));
  unsigned* d_ovf_n = nullptr;
  unsigned* d_tb_cnt_all = nullptr;
  if (tail_fused) {
    const size_t n_blk = (size_t)nb32 * nb32;
    // one buffer, one memset: [entry lines (n_blk x 128 B) | block counters | overflow counter]
    const size_t tb_words = n_blk * TB_CAP + n_blk + 16;
    GK_TRY(h->tb_ent.ensure(tb_words * 4));
    GK_TRY(h->tb_ovf.ensure((size_t)ovf_cap * sizeof(int4)));
    unsigned* d_tb_cnt = h->tb_ent.as<unsigned>() + n_blk * TB_CAP;
    d_tb_cnt_all = d_tb_cnt;
    d_ovf_n = d_tb_cnt + n_blk;
    GK_CUDA(cudaMemsetAsync(h->tb_ent.p, 0, tb_words * 4, h->stream));
    tail_bucket<<<h->sm_count * 16, 256, 0, h->stream>>>(h->tail_desc.as<int2>(), h->tail_ent.as<int2>(), dyn, nb32, tb_cap, TB_CAP, tb_sym,
                                                         d_tb_cnt, h->tb_ent.as<unsigned>(), h->tb_ovf.as<int4>(), ovf_cap, d_ovf_n);
    LAUNCH_CHECK(h);
    GK_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(h->h_dyn.p) + sizeof(GramDyn), d_ovf_n, 4, cudaMemcpyDeviceToHost, h->stream));
  }
  // ---- GEMM (k extent read from the device) + tail
  GramParams p;
  memset(&p, 0, sizeof(p));
  p.a_row_end = (int)N; p.b_row_end = (int)N;
  p.out = d_out; p.ld = d_ld;
  p.mirror = 2;
  p.fix_diag = 1;
  p.vec_ok = (((uintptr_t)d_out) % 32 == 0 && (d_ld * 4) % 32 == 0) ? 1 : 0;
  p.diag = h->diag_f64.as<double>();
  p.tma_store = 1;
  p.tiles = h->tiles.as<int2>();
  p.n_tiles = (int)n_tiles;
  p.num_k_blocks = 1;
  p.nkb_dev = &dyn->num_k_blocks;
  if (tail_fused) { p.tb_cnt = d_tb_cnt_all; p.tb_ent = h->tb_ent.as<unsigned>(); p.tb_nb32 = nb32; p.tb_cap = tb_cap; p.tb_sym = tb_sym; }
  const int grid = 2 * (int)std::min<int64_t>(n_tiles, h->sm_count / 2);
  GK_CUDA(cudaEventRecord(h->tev[6], h->stream));
  gram_tc2_kernel<<<grid, GEMM_THREADS, GEMM2_SMEM, h->stream>>>(tmA, tmC, p, peer_maps);
  LAUNCH_CHECK(h);
  GK_CUDA(cudaEventRecord(h->tev[7], h->stream));
  if (tail_fused)
    tail_overflow_apply<<<64, 256, 0, h->stream>>>(h->tb_ovf.as<int4>(), d_ovf_n, ovf_cap, (float*)d_out, d_ld, tb_sym);
  else
    tail_pairs<float><<<h->sm_count * 16, 256, 0, h->stream>>>(0, h->tail_desc.as<int2>(), h->tail_ent.as<int2>(), (int)N, 1, 0, (int)N,
                                                              (float*)d_out, d_ld, dyn);
  LAUNCH_CHECK(h);
  GK_CUDA(cudaEventRecord(h->ev[13], h->stream));
  const int64_t launches_all = h->launches - launches0;

  // ---- the decision reaches the host while the GEMM runs
  GK_CUDA(cudaEventSynchronize(h->ev_join));
  const GramDyn hd = *h->h_dyn.as<GramDyn>();
  if (hd.bad) {  // repeat through the synchronous route (it reports errors, retries hash seeds, grows buffers)
    GK_CUDA(cudaStreamSynchronize(h->stream));
    return GK_OK;
  }
  GK_CUDA(cudaEventRecord(h->ev[14], h->stream));
  if (host_out) GK_TRY(deliver_square(h, reinterpret_cast<const float*>(d_out), d_ld, N, reinterpret_cast<double*>(K_out), ld > 0 ? ld : N,
                                      (int64_t)hd.max_diag));
  if (xdiag) GK_CUDA(cudaMemcpyAsync(xdiag, h->diag_f64.p, N * 8, cudaMemcpyDeviceToHost, h->stream));
  GK_CUDA(cudaEventRecord(h->ev[15], h->stream));
  GK_CUDA(cudaStreamSynchronize(h->stream));
  if (tail_fused && *reinterpret_cast<const unsigned*>(reinterpret_cast<const char*>(h->h_dyn.p) + sizeof(GramDyn)) > ovf_cap)
    return GK_OK;  // more block overflows than the list holds (never seen): the synchronous route recomputes everything
  // ---- state as gk_wl_features + gk_gram leave it
  h->n_columns = hd.n_columns;
  h->features_ready = true; h->feat_serial++;
  h->feature_kind = 1;
  h->Dc = hd.Dc; h->Dc_pad = hd.Dc_pad;
  if (force_T < 0) hx->head_dc_pad = hd.Dc_pad;
  hx->pro_hist = hd.hist;
  hx->pro_max_count = (long long)hd.max_count; hx->pro_max_diag = (long long)hd.max_diag; hx->pro_n_entries = (long long)hd.n_entries;
  h->pro_serial = h->feat_serial;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_graphs = N; stats->n_vertices = V; stats->n_edges = h->E;
    stats->n_levels = L;
    for (int i = 0; i < L; ++i) { stats->level_dims[i] = hd.level_dims[i]; stats->n_columns += hd.level_dims[i]; }
    if (L == 1) stats->n_columns = h->n_columns;
    stats->hash_retries = 0;
    stats->kernel_launches = launches_all;
    stats->ms_features = ev_ms(h->tev[2], h->tev[3]);
    stats->n_entries = (int64_t)hd.n_entries;
    stats->n_dense_columns = hd.Dc;
    stats->n_tail_columns = hd.n_tail_cols;
    stats->tail_updates = (int64_t)hd.tail_work;
    stats->threshold = hd.T;
    stats->max_count = (int64_t)hd.max_count;
    stats->max_diag = (int64_t)hd.max_diag;
    stats->gram_path = 1;
    stats->gemm_tiles = n_tiles;
    stats->gemm_launches = 0;
    stats->ms_panel = ev_ms(h->tev[4], h->tev[6]);
    stats->ms_gemm = ev_ms(h->tev[6], h->tev[7]);
    stats->ms_tail = ev_ms(h->tev[7], h->ev[13]);
    stats->ms_d2h = ev_ms(h->ev[14], h->ev[15]);
    stats->ms_total = ev_ms(h->tev[2], h->ev[15]);
  }
  *done = true;
  return GK_OK;
}

extern "C" {

// WL features + square Gram in one call on the packed block (gk_wl_features followed by gk_gram(n_fit = N)): the
// asynchronous pass above when it applies, else the two synchronous calls.
int gk_wl_gram(gk_handle* h, int32_t n_iter, int32_t flags, void* K_out, int32_t out_dtype, int64_t ld, double* xdiag,
               gk_stats* stats) {
  if (!h) return fail(GK_ERR_ARG, "null handle");
  if (out_dtype != GK_F32 && out_dtype != GK_F64) return fail(GK_ERR_ARG, "gk_wl_gram: bad out_dtype");
  bool done = false;
  GK_TRY(wl_gram_async(h, n_iter, flags, K_out, out_dtype, ld, xdiag, stats, &done));
  if (done) return GK_OK;
  gk_stats s1, s2;
  memset(&s1, 0, sizeof(s1));
  GK_TRY(gk_wl_features(h, n_iter, &s1));
  s2 = s1;
  GK_TRY(gk_gram(h, h->N, flags, 0, -1, K_out, out_dtype, ld, xdiag, nullptr, &s2));
  if (stats) {
    *stats = s2;
    stats->kernel_launches = s1.kernel_launches;
  }
  return GK_OK;
}

int gk_wl_fit_transform(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr, const int32_t* row_ptr,
                        const int32_t* col_idx, const int32_t* labels, int32_t n_iter, int32_t flags, void* K_out,
                        int32_t out_dtype, int64_t ld, double* diag, gk_stats* stats) {
  gk_stats s1, s2;
  memset(&s1, 0, sizeof(s1));
  memset(&s2, 0, sizeof(s2));
  GK_TRY(gk_pack_csr(h, n_graphs, graph_ptr, row_ptr, col_idx, labels, nullptr, nullptr, 0));
  GK_TRY(gk_wl_gram(h, n_iter, flags, K_out, out_dtype, ld, diag, &s2));
  (void)s1;
  if (stats) {
    *stats = s2;
    stats->ms_h2d = ev_ms(h->tev[0], h->tev[1]);
  }
  return GK_OK;
}

int gk_sp_fit_transform(gk_handle* h, int64_t n_graphs, const int32_t* graph_ptr, const int32_t* row_ptr,
                        const int32_t* col_idx, const int32_t* labels, const double* weights, int32_t sp_flags,
                        int32_t flags, void* K_out, int32_t out_dtype, int64_t ld, double* diag, gk_stats* stats) {
  gk_stats s1, s2;
  memset(&s1, 0, sizeof(s1));
  GK_TRY(gk_pack_csr(h, n_graphs, graph_ptr, row_ptr, col_idx, labels, weights, nullptr, 0));
  GK_TRY(gk_sp_features(h, sp_flags, &s1));
  s2 = s1;
  GK_TRY(gk_gram(h, n_graphs, flags, 0, -1, K_out, out_dtype, ld, diag, nullptr, &s2));
  if (stats) {
    *stats = s2;
    stats->kernel_launches = s1.kernel_launches;
    stats->ms_h2d = ev_ms(h->tev[0], h->tev[1]);
  }
  return GK_OK;
}

// ---------------------------------------------------------------------------
// Dense self-test of the two Gram kernels (tests only): counts[n x d] -> K = C C^T.
int gk_selftest_gram(gk_handle* h, int64_t n, int64_t d, const uint16_t* counts, double* out_tc, double* out_simt) {
  if (!h || !counts || n <= 0 || d <= 0) return fail(GK_ERR_ARG, "gk_selftest_gram: bad arguments");
  GK_CUDA(cudaSetDevice(h->dev));
  const int64_t dpad = (d + BK - 1) / BK * BK;
  std::vector<__nv_bfloat16> pb((size_t)n * dpad, __float2bfloat16(0.f));
  std::vector<unsigned> pu((size_t)n * d, 0u);
  std::vector<double> dg(n, 0.0);
  for (int64_t i = 0; i < n; ++i)
    for (int64_t j = 0; j < d; ++j) {
      const unsigned c = counts[i * d + j];
      pb[i * dpad + j] = __float2bfloat16((float)c);
      pu[i * d + j] = c;
      dg[i] += (double)c * c;
    }
  gk::DevBuf dpb, dpu, ddg, dk1, dk2, dtl;
  GK_TRY(dpb.ensure(pb.size() * 2));
  GK_TRY(dpu.ensure(pu.size() * 4));
  GK_TRY(ddg.ensure(n * 8));
  GK_TRY(dk1.ensure((size_t)n * n * 8));
  GK_TRY(dk2.ensure((size_t)n * n * 8));
  GK_CUDA(cudaMemcpyAsync(dpb.p, pb.data(), pb.size() * 2, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaMemcpyAsync(dpu.p, pu.data(), pu.size() * 4, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaMemcpyAsync(ddg.p, dg.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
  GK_CUDA(cudaMemsetAsync(dk1.p, 0xFF, (size_t)n * n * 8, h->stream));  // NaN pattern: unwritten entries show up
  GK_CUDA(cudaMemsetAsync(dk2.p, 0xFF, (size_t)n * n * 8, h->stream));
  GramParams p;
  memset(&p, 0, sizeof(p));
  p.a_row_end = (int)n; p.b_row_end = (int)n;
  p.ld = n;
  p.diag = ddg.as<double>();
  p.vec_ok = (n * 8) % 32 == 0;
  int rc = GK_OK;
  if (out_tc) {
    std::vector<int2> tiles;
    build_tiles(tiles, 0, (int)n, 0, (int)n, true, BM);
    GK_TRY(dtl.ensure(tiles.size() * sizeof(int2)));
    GK_CUDA(cudaMemcpyAsync(dtl.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
    CUtensorMap tmA, tmB, tmC;
    memset(&tmC, 0, sizeof(tmC));
    GK_TRY(make_panel_map(&tmA, dpb.p, dpad, n, BM));
    GK_TRY(make_panel_map(&tmB, dpb.p, dpad, n, BN));
    p.tiles = dtl.as<int2>();
    p.n_tiles = (int)tiles.size();
    p.num_k_blocks = (int)(dpad / BK);
    p.out = dk1.p;
    p.mirror = 1;
    launch_tc<double, false>(h, tmA, tmB, tmC, p, (int)std::min<size_t>(tiles.size(), h->sm_count));
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) rc = fail(GK_ERR_CUDA, std::string("selftest tcgen05 kernel: ") + cudaGetErrorString(e));
    else {
      GK_CUDA(cudaMemcpy(out_tc, dk1.p, (size_t)n * n * 8, cudaMemcpyDeviceToHost));
    }
  }
  if (rc == GK_OK && out_simt) {
    p.out = dk2.p;
    p.mirror = 0;
    launch_simt<double, false>(h, dpu.as<unsigned>(), d, (int)d, 0, (int)n, 0, (int)n, p);
    GK_CUDA(cudaGetLastError());
    GK_CUDA(cudaStreamSynchronize(h->stream));
    GK_CUDA(cudaMemcpy(out_simt, dk2.p, (size_t)n * n * 8, cudaMemcpyDeviceToHost));
  }
  dpb.release(); dpu.release(); ddg.release(); dk1.release(); dk2.release(); dtl.release();
  return rc;
}

}  // extern "C"
