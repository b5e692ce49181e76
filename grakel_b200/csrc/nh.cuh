// NeighborhoodHash (neighborhood_hash.py:14-570, Hido & Kashima) as R per-level histogram-intersection Grams.
//
// Labels are u64 on the device.  A label starts below 2^bits, but the count-sensitive hash XORs in l ^ occ unrotated
// whenever occ % bits == 0 (ROT, :384-390), so a label can outgrow the mask; NH_NONE (all ones) is the reference's
// None (a transform label unseen at fit time, :299-300), which spreads to a vertex and its in-neighbours' next level
// (:410-412, :439-441).
//
// Level r of a graph is the multiset of its non-None labels.  c_r(x, y) = sum_l min(cnt_x(l), cnt_y(l)) is the merge of
// nh_compare_labels (:531-570).  Per level the labels present get dense column ids (a stable sort of the labels with the
// graph id as payload: runs of a label are column ids, runs of (label, graph) are count entries), the count block goes
// through the unary expansion of wl_oa.cuh and the integer Gram of gram_tc.cuh, and nh_combine turns the R level Grams
// into the fp64 result with the reference's arithmetic.
#pragma once
#include "common.cuh"

namespace gk {

constexpr unsigned long long NH_NONE = ~0ULL;

// ROT(n, d) of :367-390: a rotation inside the low `bits` bits; d % bits == 0 returns n unmasked
__device__ __forceinline__ unsigned long long nh_rot(unsigned long long n, unsigned d, int bits, unsigned long long mask) {
  const unsigned m = d % (unsigned)bits;
  return m ? (((n << m) & mask) | ((n & mask) >> (bits - m))) : n;
}

// Contribution of neighbour slot i of the row [b, e) to radix_sort_rot (:449-504).  The reference sorts the neighbour
// labels stably by their low `bits` bits and XORs ROT(l ^ occ, occ) over the runs of equal adjacent labels.  For labels
// below 2^bits that is one term per distinct label; a label above the mask shares its key with other labels, and the
// runs then follow the stable order.  Slot i opens a run when the previous slot of its key holds another label; the
// run continues over the following slots of that key while they hold the same label.
__device__ __forceinline__ unsigned long long nh_cs_term(int b, int e, int i, const int* __restrict__ col_idx,
                                                          const unsigned long long* __restrict__ lab, int bits,
                                                          unsigned long long mask) {
  const unsigned long long l = lab[col_idx[i]], k = l & mask;
  for (int j = i - 1; j >= b; --j) {
    const unsigned long long lj = lab[col_idx[j]];
    if ((lj & mask) == k) {
      if (lj == l) return 0ULL;  // inside a run opened earlier
      break;
    }
  }
  unsigned occ = 1;
  for (int j = i + 1; j < e; ++j) {
    const unsigned long long lj = lab[col_idx[j]];
    if ((lj & mask) == k) {
      if (lj != l) break;
      ++occ;
    }
  }
  return nh_rot(l ^ (unsigned long long)occ, occ, bits, mask);
}

// XOR over the slots i0, i0 + step, ... of the row [b, e): the neighbour labels (simple, :414-416) or the radix terms
// (count-sensitive, :443-444); *none: a neighbour label is None
template <bool CS>
__device__ __forceinline__ unsigned long long nh_row_part(int b, int e, int i0, int step, const int* __restrict__ col_idx,
                                                           const unsigned long long* __restrict__ lab, int bits,
                                                           unsigned long long mask, bool* none) {
  unsigned long long acc = 0;
  bool nn = false;
  for (int i = b + i0; i < e; i += step) {
    const unsigned long long l = lab[col_idx[i]];
    if (l == NH_NONE) { nn = true; continue; }
    acc ^= CS ? nh_cs_term(b, e, i, col_idx, lab, bits, mask) : l;
  }
  *none = nn;
  return acc;
}

// one level, one thread per vertex of degree <= width (the others are in the packed large list)
template <bool CS>
__global__ void __launch_bounds__(256)
nh_relabel(int V, int width, const int* __restrict__ row_ptr, const int* __restrict__ col_idx,
           const unsigned long long* __restrict__ lab_in, unsigned long long* __restrict__ lab_out, int bits,
           unsigned long long mask) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const int b = row_ptr[v], e = row_ptr[v + 1];
  if (e - b > width) return;
  const unsigned long long lu = lab_in[v];
  bool none;
  const unsigned long long x = nh_row_part<CS>(b, e, 0, 1, col_idx, lab_in, bits, mask, &none);
  lab_out[v] = (lu == NH_NONE || none) ? NH_NONE : (nh_rot(lu, 1, bits, mask) ^ x);
}

// one level, one warp per high-degree vertex: the lanes split the row (the count-sensitive term of a slot scans the row,
// so a hub costs deg^2 / 32 steps per lane instead of deg^2 on one thread)
template <bool CS>
__global__ void __launch_bounds__(256)
nh_relabel_warp(int n_large, const int* __restrict__ large_list, const int* __restrict__ row_ptr,
                const int* __restrict__ col_idx, const unsigned long long* __restrict__ lab_in,
                unsigned long long* __restrict__ lab_out, int bits, unsigned long long mask) {
  const int w = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= n_large) return;
  const int v = large_list[w];
  const int b = row_ptr[v], e = row_ptr[v + 1];
  bool none;
  unsigned long long x = nh_row_part<CS>(b, e, lane, 32, col_idx, lab_in, bits, mask, &none);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, s);
  none = __any_sync(0xffffffffu, none);
  if (lane == 0) {
    const unsigned long long lu = lab_in[v];
    lab_out[v] = (lu == NH_NONE || none) ? NH_NONE : (nh_rot(lu, 1, bits, mask) ^ x);
  }
}

// Level histogram, after a stable sort of the labels (graph ids as payload, so every label run is ordered by graph):
// flag word of sorted slot i = (opens a column) << 32 | (opens a (graph, column) entry).  None sorts last and opens
// nothing.
__global__ void __launch_bounds__(256)
nh_mark(int V, const unsigned long long* __restrict__ sk, const int* __restrict__ sg, unsigned long long* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const unsigned long long k = sk[i];
  unsigned long long f = 0;
  if (k != NH_NONE) {
    const bool col = i == 0 || sk[i - 1] != k;
    const bool ent = col || sg[i - 1] != sg[i];
    f = ((unsigned long long)col << 32) | (unsigned long long)ent;
  }
  flag[i] = f;
}

struct NhLevelCounts {
  unsigned long long n_cols;     // distinct non-None labels of the level
  unsigned long long n_entries;  // (graph, label) entries
  unsigned long long n_valid;    // non-None vertices
};

// entry e = (graph, column) at its first sorted slot; the last valid slot closes the tally
__global__ void __launch_bounds__(256)
nh_emit(int V, const unsigned long long* __restrict__ sk, const int* __restrict__ sg,
        const unsigned long long* __restrict__ flag, const unsigned long long* __restrict__ pos,
        unsigned long long* __restrict__ keys, int* __restrict__ first, NhLevelCounts* cnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const unsigned long long f = flag[i];
  if (sk[i] == NH_NONE) return;
  const unsigned long long p = pos[i] + f;  // inclusive: (columns opened so far) << 32 | entries opened so far
  const unsigned col = (unsigned)(p >> 32) - 1u, ent = (unsigned)p - 1u;
  if (f & 1ULL) {
    keys[ent] = ((unsigned long long)(unsigned)sg[i] << 32) | col;
    first[ent] = i;
  }
  if (i == V - 1 || sk[i + 1] == NH_NONE) {
    cnt->n_cols = p >> 32;
    cnt->n_entries = (unsigned)p;
    cnt->n_valid = (unsigned long long)i + 1;
    first[(unsigned)p] = i + 1;  // sentinel: end of the last entry
  }
}

// count of entry e = length of its sorted run; slots past the last entry stay EMPTY64 (cleared by the host)
__global__ void __launch_bounds__(256)
nh_counts(int V, const int* __restrict__ first, const NhLevelCounts* __restrict__ cnt, unsigned* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= V || (unsigned long long)e >= cnt->n_entries) return;
  out[e] = (unsigned)(first[e + 1] - first[e]);
}

// partials of the expanded block as gk_gram's diag_finish folds them: one "CTA", largest count 1
__global__ void nh_parts(unsigned long long n_entries, unsigned* part_max, unsigned* part_new) {
  part_max[0] = n_entries ? 1u : 0u;
  part_new[0] = (unsigned)n_entries;
}

// K = sum over the levels of a_r = c_r / (n_row + n_col - c_r), divided by R (pairwise_operation, :340-341 with
// nh_compare_labels, :570).  The reference sums with the built-in sum(), which (CPython >= 3.12) adds floats with
// Neumaier's compensation: `0 + a_0` is a_0, every further term updates the running sum t and the compensation c, and
// c is added once at the end when it is non-zero and finite.  C holds the R level Grams (fp32 integers, exact), level r
// at C + r * level_stride.  Both halves of a square K are computed: the level Grams are mirrored, so K[i][j] and
// K[j][i] see the same operands and are equal.
__global__ void __launch_bounds__(256)
nh_combine(long long rows, long long cols, int row0, const int* __restrict__ graph_ptr, const float* __restrict__ C,
           long long ldc, long long level_stride, int R, double* __restrict__ K, long long ldk) {
  const long long n = rows * cols;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const long long r = t / cols, j = t - r * cols;
    const int gi = row0 + (int)r;
    const long long nn = (long long)(graph_ptr[gi + 1] - graph_ptr[gi]) + (graph_ptr[j + 1] - graph_ptr[j]);
    const float* cp = C + r * ldc + j;
    double f = 0.0, comp = 0.0;
    for (int lv = 0; lv < R; ++lv) {
      const double c = (double)__ldcs(cp + (size_t)lv * level_stride);
      const double a = __ddiv_rn(c, (double)(nn - (long long)c));
      if (lv == 0) { f = a; continue; }
      const double s = __dadd_rn(f, a);
      comp = fabs(f) >= fabs(a) ? __dadd_rn(comp, __dadd_rn(__dsub_rn(f, s), a))
                                : __dadd_rn(comp, __dadd_rn(__dsub_rn(a, s), f));
      f = s;
    }
    if (comp != 0.0 && isfinite(comp)) f = __dadd_rn(f, comp);
    __stcs(K + r * ldk + j, __ddiv_rn(f, (double)R));
  }
}

}  // namespace gk
