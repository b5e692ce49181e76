// Shortest-path kernel on node attributes (reference: shortest_path.py:16-164).
//
//   k(x,y) = sum_{i!=j} sum_{k!=m} [Sx[i,j] == Sy[k,m] < inf] <a_i,a_k> <a_j,a_m>      (:151-162)
//
// is bilinear in the attributes, so with F_x[d] = sum_{(i,j): i!=j, Sx[i,j]=d} a_i (x) a_j
// (a da x da matrix per distinct distance d) it equals sum_d <F_x[d], F_y[d]>: an explicit
// feature map of dimension da^2 * #distances and a plain Gram product (SURVEY 8a row a20;
// valid for the default metric=np.dot).  Everything here is fp64 -- the reference is.
#pragma once
#include "common.cuh"
#include "sp.cuh"

namespace gk {

// Phase A: APSP of every graph (shared-memory Floyd-Warshall as in sp_apsp_hist), the
// integer distance matrix is kept in global memory (u16 / f64 as computed) and every
// distinct finite distance is entered into the global dictionary.
template <typename T>
__global__ void __launch_bounds__(SP_THREADS)
spattr_apsp(SpParams p) {
  using DT = DistTraits<T>;
  extern __shared__ __align__(16) unsigned char sp_smem[];
  const int g = p.glist ? p.glist[blockIdx.x] : blockIdx.x;
  const int v0 = p.graph_ptr[g];
  const int n = p.graph_ptr[g + 1] - v0;
  if (n <= 0) return;
  T* gout = reinterpret_cast<T*>(p.gdist) + p.goff[g];
  T* dist = p.dist_in_global ? gout : reinterpret_cast<T*>(sp_smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int NW = SP_THREADS / 32;
  const long long nn = (long long)n * n;
  for (long long i = tid; i < nn; i += SP_THREADS) dist[i] = DT::inf();
  __syncthreads();
  for (int u = warp; u < n; u += NW) {
    const int b = p.row_ptr[v0 + u], e = p.row_ptr[v0 + u + 1];
    for (int k = b + lane; k < e; k += 32) {
      const int w = p.col_idx[k] - v0;
      if (w == u) continue;
      if constexpr (sizeof(T) == 2) dist[(long long)u * n + w] = 1;
      else dist[(long long)u * n + w] = p.weights ? (T)p.weights[k] : (T)1;
    }
    if (lane == 0) dist[(long long)u * n + u] = 0;
  }
  __syncthreads();
  for (int k = 0; k < n; ++k) {
    const T* rk = dist + (long long)k * n;
    for (int i = warp; i < n; i += NW) {
      if (i == k) continue;
      T* ri = dist + (long long)i * n;
      const T dik = ri[k];
      if (!DT::finite(dik)) continue;
      for (int j = lane; j < n; j += 32) {
        const T cand = DT::add(dik, rk[j]);
        if (cand < ri[j]) ri[j] = cand;
      }
    }
    __syncthreads();
  }
  for (long long i = tid; i < nn; i += SP_THREADS) {
    const T d = dist[i];
    if (!p.dist_in_global) gout[i] = d;
    const int u = (int)(i / n), w = (int)(i - (long long)u * n);
    if (u == w || !DT::finite(d)) continue;
    unsigned long long key;
    if constexpr (sizeof(T) == 2) key = (unsigned long long)d;
    else key = (unsigned long long)__double_as_longlong((double)d);  // exact-equality key (shortest_path.py:159)
    sp_dict_slot(p.dict_keys, p.dict_mask, key, p.sc);
  }
}

// Dijkstra semantics for real-valued weights (graph.py:1712-1764, tools.py:14-83).  The reference's Dijkstra sums a
// path left to right, dist[v] = fl(dist[u] + w(u, v)) with u the predecessor, where Floyd-Warshall adds two partial
// paths, so the two differ in the last bit on real weights -- and feature keys compare distances by exact float
// equality (shortest_path.py:472, 511).  With non-negative weights and monotone rounding, Dijkstra's result from a
// source s is the LEAST fixed point of  d[v] = min over edges (u, v) of fl(d[u] + w(u, v)),  d[s] = 0  (every walk's
// left-associated sum bounds it from above by induction, and it is attained), independent of the heap's tie
// breaking.  A chaotic Bellman-Ford iteration reaches the same fixed point: all sources of a graph at once, one CTA
// per graph, relaxations as 64-bit atomicMin on the bit patterns (order-preserving for non-negative doubles).
__global__ void __launch_bounds__(SP_THREADS)
sp_dijkstra_order_apsp(SpParams p) {
  extern __shared__ __align__(16) unsigned char sp_smem[];
  const int g = p.glist ? p.glist[blockIdx.x] : blockIdx.x;
  const int v0 = p.graph_ptr[g];
  const int n = p.graph_ptr[g + 1] - v0;
  if (n <= 0) return;
  double* gout = reinterpret_cast<double*>(p.gdist) + p.goff[g];
  unsigned long long* dist = reinterpret_cast<unsigned long long*>(p.dist_in_global ? (void*)gout : (void*)sp_smem);
  const int tid = threadIdx.x;
  const long long nn = (long long)n * n;
  const unsigned long long INF = 0x7ff0000000000000ULL;
  for (long long i = tid; i < nn; i += SP_THREADS) dist[i] = (i / n == i % n) ? 0ULL : INF;
  __shared__ int changed;
  if (tid == 0) changed = 1;
  __syncthreads();
  for (int round = 0; round < n + 1; ++round) {
    if (!changed) break;  // uniform: read after the barrier below
    __syncthreads();
    if (tid == 0) changed = 0;
    __syncthreads();
    // (source s, vertex u) pairs: relax the out-edges of u for source s
    for (long long i = tid; i < nn; i += SP_THREADS) {
      const int sidx = (int)(i / n), u = (int)(i - (long long)sidx * n);
      const unsigned long long du_bits = dist[i];
      if (du_bits >= INF) continue;
      const double du = __longlong_as_double((long long)du_bits);
      const int b = p.row_ptr[v0 + u], e = p.row_ptr[v0 + u + 1];
      for (int k = b; k < e; ++k) {
        const int w = p.col_idx[k] - v0;
        const double cand = du + (p.weights ? p.weights[k] : 1.0);
        const unsigned long long cb = (unsigned long long)__double_as_longlong(cand);
        unsigned long long* dst = &dist[(long long)sidx * n + w];
        if (cb < *dst) {
          const unsigned long long old = atomicMin(dst, cb);
          if (cb < old) changed = 1;
        }
      }
    }
    __syncthreads();
  }
  for (long long i = tid; i < nn; i += SP_THREADS) {
    const unsigned long long d = dist[i];
    if (!p.dist_in_global) gout[i] = __longlong_as_double((long long)d);
    const int u = (int)(i / n), w = (int)(i - (long long)u * n);
    if (u == w || d >= INF) continue;
    sp_dict_slot(p.dict_keys, p.dict_mask, d, p.sc);  // exact-equality key = the bit pattern
  }
}

// Real-valued edge weights: histogram of (l(u), l(v), id(d(u,v))) from distance matrices kept
// in global memory, where id() is the slot of the distance's bit pattern in the global distance
// dictionary filled by spattr_apsp<double> (exact float equality, shortest_path.py:472, 511).
__global__ void __launch_bounds__(SP_THREADS)
sp_hist_from_dist(SpParams p, const unsigned long long* __restrict__ dkeys, unsigned dmask) {
  extern __shared__ __align__(16) unsigned char sp_smem[];
  const int g = blockIdx.x;
  const int v0 = p.graph_ptr[g];
  const int n = p.graph_ptr[g + 1] - v0;
  if (n <= 0) return;
  unsigned long long* lkeys = reinterpret_cast<unsigned long long*>(sp_smem);
  unsigned* lcnt = reinterpret_cast<unsigned*>(sp_smem + SP_LOCAL_SLOTS * 8);
  const double* dist = reinterpret_cast<const double*>(p.gdist) + p.goff[g];
  const int tid = threadIdx.x;
  for (int i = tid; i < SP_LOCAL_SLOTS; i += SP_THREADS) { lkeys[i] = EMPTY64; lcnt[i] = 0; }
  __syncthreads();
  const long long nn = (long long)n * n;
  for (long long i = tid; i < nn; i += SP_THREADS) {
    const int u = (int)(i / n), w = (int)(i - (long long)u * n);
    const double d = dist[i];
    if (p.keep) p.keep[p.goff[g] + i] = d;
    if (u == w || !(d < 1.0e300)) continue;
    const unsigned long long dk = (unsigned long long)__double_as_longlong(d);
    unsigned slot = (unsigned)(mix64(dk) >> 13) & dmask;
    while (dkeys[slot] != dk) slot = (slot + 1) & dmask;
    const unsigned long long lu = p.labels ? (unsigned long long)(unsigned)(p.labels[v0 + u] + p.label_offset) : 0ULL;
    const unsigned long long lv = p.labels ? (unsigned long long)(unsigned)(p.labels[v0 + w] + p.label_offset) : 0ULL;
    sp_local_add(lkeys, lcnt, p, g, (lu << 44) | (lv << 24) | (unsigned long long)slot);
  }
  __syncthreads();
  for (int i = tid; i < SP_LOCAL_SLOTS; i += SP_THREADS) {
    const unsigned long long key = lkeys[i];
    if (key == EMPTY64) continue;
    const int col = sp_dict_slot(p.dict_keys, p.dict_mask, key, p.sc);
    sp_feature_add(p, g, col, lcnt[i]);
  }
}

// Phase C: F_g[blk] += a_i (x) a_j for every ordered pair at distance with block id blk.
// One CTA per graph, thread t owns element (t / da, t % da) of every block; F lives in
// shared memory (blocks processed in chunks of `chunk` distances if they do not fit).
template <typename T>
__global__ void __launch_bounds__(256)
spattr_accumulate(const int* __restrict__ graph_ptr, const double* __restrict__ attrs, int da,
                  const void* __restrict__ gdist, const long long* __restrict__ goff,
                  const unsigned long long* __restrict__ dict_keys, unsigned dict_mask,
                  const int* __restrict__ slot_block, int n_blocks, int chunk, double* __restrict__ phi) {
  using DT = DistTraits<T>;
  extern __shared__ __align__(16) unsigned char smem[];
  const int g = blockIdx.x;
  const int v0 = graph_ptr[g];
  const int n = graph_ptr[g + 1] - v0;
  const int dd = da * da;
  double* F = reinterpret_cast<double*>(smem);                 // [chunk][dd]
  double* A = F + (size_t)chunk * dd;                           // [n][da]
  short* blk = reinterpret_cast<short*>(A + (size_t)n * da);    // [n*n] block id or -1
  const T* dist = reinterpret_cast<const T*>(gdist) + goff[g];
  for (int i = threadIdx.x; i < n * da; i += blockDim.x) A[i] = attrs[(size_t)v0 * da + i];
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
    const int u = i / n, w = i - u * n;
    const T d = dist[i];
    int b = -1;
    if (u != w && DT::finite(d)) {
      unsigned long long key;
      if constexpr (sizeof(T) == 2) key = (unsigned long long)d;
      else key = (unsigned long long)__double_as_longlong((double)d);
      unsigned slot = (unsigned)(mix64(key) >> 13) & dict_mask;
      while (dict_keys[slot] != key) slot = (slot + 1) & dict_mask;
      b = slot_block[slot];
    }
    blk[i] = (short)b;
  }
  __syncthreads();
  double* out = phi + (size_t)g * n_blocks * dd;
  for (int c0 = 0; c0 < n_blocks; c0 += chunk) {
    const int c1 = min(n_blocks, c0 + chunk);
    for (int i = threadIdx.x; i < (c1 - c0) * dd; i += blockDim.x) F[i] = 0.0;
    __syncthreads();
    for (int e = threadIdx.x; e < dd; e += blockDim.x) {
      const int pi = e / da, qi = e - pi * da;
      for (int i = 0; i < n; ++i) {
        const double ai = A[i * da + pi];
        for (int j = 0; j < n; ++j) {
          const int b = blk[i * n + j];
          if (b >= c0 && b < c1) F[(size_t)(b - c0) * dd + e] += ai * A[j * da + qi];
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (c1 - c0) * dd; i += blockDim.x) out[(size_t)c0 * dd + i] = F[i];
    __syncthreads();
  }
}

// fp64 Gram  K[r][c] = <phi[a0 + r], phi[b0 + c]>  : 64x64 tile per CTA, 16x16 threads, 4x4 each
__global__ void __launch_bounds__(256)
gram_f64_kernel(const double* __restrict__ phi, long long D, int a0, int a1, int b0, int b1,
                double* __restrict__ out, long long ld) {
  __shared__ double As[16][65], Bs[16][65];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int ar0 = a0 + blockIdx.y * 64, br0 = b0 + blockIdx.x * 64;
  double acc[4][4] = {};
  for (long long k0 = 0; k0 < D; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      const int r = i >> 4, k = i & 15;
      const long long kk = k0 + k;
      As[k][r] = (ar0 + r < a1 && kk < D) ? phi[(long long)(ar0 + r) * D + kk] : 0.0;
      Bs[k][r] = (br0 + r < b1 && kk < D) ? phi[(long long)(br0 + r) * D + kk] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = ar0 + ty * 4 + i, c = br0 + tx * 4 + j;
      if (r < a1 && c < b1) out[(long long)(r - a0) * ld + (c - b0)] = acc[i][j];
    }
}

// Split of the fp64 feature matrix for the tensor-core Gram (3xTF32): x = hi + lo + O(2^-22 x) with hi, lo
// representable in tf32 (10 explicit mantissa bits: the low 13 bits of the fp32 pattern are zero after
// round-to-nearest-even on bit 13).  K = hi hi^T + hi lo^T + lo hi^T is ONE GEMM over the concatenated
// panels  P1 = [hi | hi | lo],  P2 = [hi | lo | hi]  (row pitch 3 * Dp floats, Dp = D rounded up to 32).
// Row r is split as phi[r] * 2^-rexp[r] (exact in fp64; rexp from rownorm_f64_kernel), so its largest entry lies
// in [1, 2) and hi, lo, their products and the fp32 chunk sums stay in fp32's normal range for any finite phi;
// unscale_gram_f64 multiplies K[r][c] by 2^(rexp[r] + rexp[c]) afterwards.
__device__ __forceinline__ float tf32_rne(float x) {
  unsigned u = __float_as_uint(x);
  u += 0x0FFFu + ((u >> 13) & 1u);
  u &= 0xFFFFE000u;
  return __uint_as_float(u);
}
__global__ void __launch_bounds__(256)
spattr_split_tf32(const double* __restrict__ phi, const int* __restrict__ rexp, long long D, long long Dp, int N,
                  float* __restrict__ P1, float* __restrict__ P2) {
  const long long total = (long long)N * Dp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / Dp, c = i - r * Dp;
    float hi = 0.f, lo = 0.f;
    if (c < D) {
      const double x = ldexp(phi[r * D + c], -rexp[r]);
      hi = tf32_rne((float)x);
      lo = tf32_rne((float)(x - (double)hi));
    }
    float* p1 = P1 + r * 3 * Dp;
    float* p2 = P2 + r * 3 * Dp;
    p1[c] = hi; p1[Dp + c] = hi; p1[2 * Dp + c] = lo;
    p2[c] = hi; p2[Dp + c] = lo; p2[2 * Dp + c] = hi;
  }
}
// K[r][c] *= 2^(rexp[a0 + r] + rexp[c]): undoes the row scaling of spattr_split_tf32 (exact unless the fp64 result
// itself leaves fp64's range).  mirror (square, all rows, a0 = 0): the upper triangle is scaled and copied to the lower
// one (tiles that straddle the diagonal are written from both sides with values that may differ in the last fp32
// rounding of the accumulator; the reference's matrix is exactly symmetric, kernel.py:277).
__global__ void __launch_bounds__(256)
unscale_gram_f64(int a0, long long rows, long long cols, const int* __restrict__ rexp, double* __restrict__ out,
                 long long ld, int mirror) {
  const long long total = rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols, c = i - r * cols;
    if (mirror && r > c) continue;
    const double v = ldexp(out[r * ld + c], rexp[a0 + r] + rexp[c]);
    out[r * ld + c] = v;
    if (mirror && r < c) out[c * ld + r] = v;
  }
}
// K[i][i] = diag[i] for the rows of a block (exact fp64 self similarities over the fp64 features)
__global__ void __launch_bounds__(256)
set_diag_f64(int a0, int a1, int b0, int b1, const double* __restrict__ diag, double* __restrict__ out, long long ld) {
  const int r = a0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (r < a1 && r >= b0 && r < b1) out[(long long)(r - a0) * ld + (r - b0)] = diag[r];
}

// per-row self similarity <phi[g], phi[g]>, and the row's scale exponent for spattr_split_tf32:
// rexp[g] = ilogb(max_k |phi[g][k]|), 0 for an all-zero row or one with a non-finite entry (left as it is)
__global__ void __launch_bounds__(256)
rownorm_f64_kernel(const double* __restrict__ phi, long long D, int N, double* __restrict__ diag, int* __restrict__ rexp) {
  const int g = blockIdx.x;
  if (g >= N) return;
  __shared__ double red[8], redm[8];
  __shared__ int redbad[8];
  double s = 0.0, m = 0.0;
  int bad = 0;
  for (long long k = threadIdx.x; k < D; k += 256) {
    const double x = phi[(long long)g * D + k];
    s += x * x;
    m = fmax(m, fabs(x));
    bad |= !isfinite(x);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, d);
    m = fmax(m, __shfl_xor_sync(0xffffffffu, m, d));
    bad |= __shfl_xor_sync(0xffffffffu, bad, d);
  }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s; redm[threadIdx.x >> 5] = m; redbad[threadIdx.x >> 5] = bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0, tm = 0.0;
    int tb = 0;
    for (int w = 0; w < 8; ++w) { t += red[w]; tm = fmax(tm, redm[w]); tb |= redbad[w]; }
    diag[g] = t;
    rexp[g] = (tb || tm == 0.0) ? 0 : ilogb(tm);
  }
}

}  // namespace gk
