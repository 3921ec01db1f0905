// Order statistics and final top-k selection over per-row candidate lists.
//
// These replace the full per-row sorts of the reference -- np.argsort(errors[0])[:topK]
// (LINAS-engine/inference.py:79) and torch.argsort(tmp.cpu(), dim=-1) (MultiFusion/src/validate.py:74,92)
// -- with (a) a radix select that turns a score sample / candidate list into a threshold and
// (b) a shared-memory bitonic sort of the few hundred survivors.  K3 (the G-way merge after the
// multi-GPU all-gather) is the same sort over int64 global indices.
#include <math_constants.h>

#include "common.cuh"

namespace xmve {
namespace {

__device__ __forceinline__ uint32_t float_key(float x) {      // ascending key order == ascending float order
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// j-th largest (1-based) of get(0..n); -inf if n < j.  All threads of the block must call it.
// 4-pass radix select over the order-preserving float key.  (Scores of one row share their sign and most exponent
// bits, so the first passes hammer one or two histogram bins; warp-aggregating the adds with __match_any_sync was
// measured SLOWER -- 500 vs 320 us for 4096 rows x 8197 -- so small order statistics go through block_kth_pivot
// below instead, and this routine is the general fallback.)
template <typename Get>
__device__ float block_kth_largest_of(Get get, int64_t n, int j, uint32_t* hist, uint32_t* bcast) {
  if (j <= 0 || n < j) return -CUDART_INF_F;
  uint32_t prefix = 0, mask = 0;
  uint32_t remaining = static_cast<uint32_t>(j);
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
      const uint32_t k = float_key(get(i));
      if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 0xffu], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t cum = 0;
      int b = 255;
      for (; b > 0; --b) {
        if (cum + hist[b] >= remaining) break;
        cum += hist[b];
      }
      bcast[0] = static_cast<uint32_t>(b);
      bcast[1] = remaining - cum;
    }
    __syncthreads();
    prefix |= bcast[0] << shift;
    mask |= 0xffu << shift;
    remaining = bcast[1];
    __syncthreads();
  }
  return key_float(prefix);
}

// ---- small order statistics without histograms ---------------------------------------------------------------
// The j-th largest of a row for j <= PV_JMAX: find a pivot p with j <= #{x > p} <= PV_CAP by a safeguarded secant
// search on log-counts (the upper tail of a score row is close to log-linear; every probe is one contention-free
// counting pass that also collects the survivors while they fit), then rank the few survivors in shared memory.
// Typically: one pass for mean / deviation / max, two probes.  Rows with NaN / +inf / fewer than j finite values, and
// searches that do not settle, return false and the caller takes the radix path.
constexpr int PV_CAP = 1024, PV_JMAX = 256, PV_SMALL = 64;

struct PivotScratch {
  float buf[PV_CAP];
  float red[3 * 8];
  int cnt[8];
  int n_surv;
  int weird;
};

__device__ __forceinline__ float inv_normal_tail(float p) {           // z with P(Z > z) = p, p in (0, 0.5]
  const float t = sqrtf(-2.f * logf(p));
  return t - (2.515517f + 0.802853f * t + 0.010328f * t * t) / (1.f + 1.432788f * t + 0.189269f * t * t + 0.001308f * t * t * t);
}

// All 256 threads call it.  On success sc.buf[0 .. *n_out) holds every value above the pivot (>= j_max of them).
__device__ bool block_pivot_survivors(const float* __restrict__ row, int64_t n, int j_max, PivotScratch& sc, int* n_out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (n <= max(256, 3 * j_max) && n <= PV_CAP) {                       // short row: everything is a survivor
    int nan = 0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
      const float x = row[i];
      sc.buf[i] = x;
      nan |= (x != x) ? 1 : 0;
    }
    if (__syncthreads_or(nan)) return false;                           // NaN ordering is the radix path's business
    *n_out = static_cast<int>(n);
    return true;
  }
  // pass 1: finite count, mean, deviation, max
  float sum = 0.f, sq = 0.f, mx = -CUDART_INF_F;
  int nf = 0, weird = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float x = row[i];
    if (x != x || x == CUDART_INF_F) weird = 1;
    else if (x > -CUDART_INF_F) { sum += x; sq = fmaf(x, x, sq); mx = fmaxf(mx, x); ++nf; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    sq += __shfl_xor_sync(0xffffffffu, sq, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nf += __shfl_xor_sync(0xffffffffu, nf, o);
    weird |= __shfl_xor_sync(0xffffffffu, weird, o);
  }
  if (lane == 0) { sc.red[warp] = sum; sc.red[8 + warp] = sq; sc.red[16 + warp] = mx; sc.cnt[warp] = nf | (weird << 30); }
  __syncthreads();
  sum = sq = 0.f; mx = -CUDART_INF_F; nf = 0; weird = 0;
  for (int w = 0; w < 8; ++w) {
    sum += sc.red[w]; sq += sc.red[8 + w]; mx = fmaxf(mx, sc.red[16 + w]);
    nf += sc.cnt[w] & 0x3fffffff; weird |= sc.cnt[w] >> 30;
  }
  __syncthreads();
  if (weird || nf < j_max) return false;
  const float mean = sum / nf, sd = sqrtf(fmaxf(sq / nf - mean * mean, 0.f));
  const float target = fminf(2.5f * j_max, 0.5f * (j_max + PV_CAP));   // survivors aimed at
  const int c_ok = min(PV_CAP, max(384, 4 * j_max));                   // ... accepted (they are sorted afterwards)
  int c_best = 0;                                                      // a larger acceptable set seen on the way
  float lo = -CUDART_INF_F, hi = mx, c_lo = static_cast<float>(nf), c_hi = 0.5f;   // #{x > lo} >= j_max > #{x > hi}
  float p = mean + sd * inv_normal_tail(fminf(0.5f, target / nf));
  if (!(p < hi)) p = mean;                                             // degenerate spread
  float step = fmaxf(sd, 1e-30f);                                      // downward step while there is no lower bracket
  for (int it = 0; it < 16; ++it) {
    if (threadIdx.x == 0) sc.n_surv = 0;
    __syncthreads();
    // warp-aggregated compaction: one shared-memory add per warp and 32 elements, whatever the number of survivors
    // (truncated candidate lists, where most of the row survives a low pivot, made per-survivor adds the slow part)
    for (int64_t base = threadIdx.x - lane; base < n; base += blockDim.x) {
      const int64_t i = base + lane;
      const float x = i < n ? row[i] : -CUDART_INF_F;
      const bool hit = x > p;
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (m != 0) {
        int pos = 0;
        if (lane == 0) pos = atomicAdd(&sc.n_surv, __popc(m));
        pos = __shfl_sync(0xffffffffu, pos, 0);
        if (hit) {
          const int slot = pos + __popc(m & ((1u << lane) - 1u));
          if (slot < PV_CAP) sc.buf[slot] = x;
        }
      }
    }
    __syncthreads();
    const int c = sc.n_surv;
    __syncthreads();
    if (c >= j_max && c <= c_ok) { *n_out = c; return true; }
    c_best = (c >= j_max && c <= PV_CAP) ? c : 0;                      // usable if the search cannot do better
    if (c < j_max) { hi = p; c_hi = fmaxf(static_cast<float>(c), 0.5f); }
    else { lo = p; c_lo = static_cast<float>(c); }
    float next;
    if (lo > -CUDART_INF_F && (it % 3) != 2) {                         // secant on log-counts between the brackets
      const float f = (logf(c_lo) - logf(target)) / (logf(c_lo) - logf(c_hi));
      next = lo + (hi - lo) * fminf(fmaxf(f, 0.05f), 0.95f);
    } else if (lo > -CUDART_INF_F) {
      next = 0.5f * (lo + hi);                                         // every third probe: bisection
    } else {
      next = p - step;                                                 // no lower bracket yet: step down, doubling
      step *= 2.f;
      if (!(next > mean - 64.f * sd - 1e-30f)) return false;
    }
    if (!(next > lo && next < hi)) {                                   // brackets are adjacent floats: massive ties
      if (c_best) { *n_out = c_best; return true; }                    // (the buffer still holds that probe's survivors)
      return false;
    }
    p = next;
  }
  if (c_best) { *n_out = c_best; return true; }
  return false;
}

// Order statistics of the survivors (exact, ties counted).  A handful: rank by counting.  More: sort them once,
// descending, in shared memory (a bitonic network over <= 1024 floats costs ~1 us per block; counting ranks is
// O(c^2) and took 1.4 ms for 8192 rows of ~760 survivors).  All threads call these.
__device__ void block_sort_survivors(PivotScratch& sc, int c) {
  if (c <= PV_SMALL) return;
  int P = 1;
  while (P < c) P <<= 1;
  for (int i = c + threadIdx.x; i < P; i += blockDim.x) sc.buf[i] = -CUDART_INF_F;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int x = threadIdx.x; x < P; x += blockDim.x) {
        const int o = x ^ stride;
        if (o > x) {
          const bool desc = (x & size) == 0;
          const float a = sc.buf[x], b = sc.buf[o];
          if (desc ? (b > a) : (a > b)) { sc.buf[x] = b; sc.buf[o] = a; }
        }
      }
      __syncthreads();
    }
}

// after block_sort_survivors(sc, c)
__device__ float block_rank_select(const PivotScratch& sc, int c, int j, float* bcast) {
  if (j <= 0 || c < j) return -CUDART_INF_F;
  if (c > PV_SMALL) return sc.buf[j - 1];                              // sorted descending
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    const float v = sc.buf[i];
    int gt = 0, ge = 0;
    for (int k = 0; k < c; ++k) {
      const float w = sc.buf[k];
      gt += w > v ? 1 : 0;
      ge += w >= v ? 1 : 0;
    }
    if (gt < j && j <= ge) *bcast = v;                                 // every qualifying thread writes the same value
  }
  __syncthreads();
  return *bcast;
}

__device__ float block_kth_largest(const float* __restrict__ vals, int64_t n, int j, uint32_t* hist, uint32_t* bcast) {
  return block_kth_largest_of([vals](int64_t i) { return vals[i]; }, n, j, hist, bcast);
}

__global__ void __launch_bounds__(256)
row_kth_kernel(const float* __restrict__ vals, int64_t cols, int64_t ld, const int32_t* __restrict__ counts,
               int j1, float sub, const float* __restrict__ sub_dev, int j2, float* __restrict__ out) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bcast[2];
  __shared__ PivotScratch piv;
  __shared__ float pick;
  const int64_t r = blockIdx.x;
  int64_t n = cols;
  if (counts != nullptr) n = min(static_cast<int64_t>(counts[r]), cols);
  const float* row = vals + r * ld;
  if (sub_dev != nullptr) sub *= sub_dev[0];
  const int j_max = max(j1, j2);
  int c = 0;
  float res;
  if (j_max <= PV_JMAX && n >= j_max && block_pivot_survivors(row, n, j_max, piv, &c)) {
    block_sort_survivors(piv, c);
    res = block_rank_select(piv, c, j1, &pick) - sub;
    if (j2 > 0) res = fmaxf(res, block_rank_select(piv, c, j2, &pick));
  } else {
    __syncthreads();
    res = block_kth_largest(row, n, j1, hist, bcast) - sub;
    if (j2 > 0) res = fmaxf(res, block_kth_largest(row, n, j2, hist, bcast));
  }
  if (threadIdx.x == 0) out[r] = res;
}

// The J largest values of each row, descending, -inf padded.  Used to combine order statistics across corpus
// shards: the j-th largest of a union is among the per-shard top-j lists.
__global__ void __launch_bounds__(256)
row_topj_kernel(const float* __restrict__ vals, int64_t cols, int64_t ld, const int32_t* __restrict__ counts, int J,
                int P, float* __restrict__ out) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bcast[2];
  __shared__ int n_buf;
  __shared__ PivotScratch piv;
  extern __shared__ float topj_buf[];
  const int64_t r = blockIdx.x;
  int64_t n = cols;
  if (counts != nullptr) n = min(static_cast<int64_t>(counts[r]), cols);
  const float* row = vals + r * ld;
  // small J: the pivot search hands over every value above a pivot that at least J values exceed (<= 1024 of them);
  // sort those and keep the first J
  int c = 0;
  if (J <= PV_JMAX && n >= J && block_pivot_survivors(row, n, J, piv, &c)) {
    int Q = 1;
    while (Q < c) Q <<= 1;
    for (int i = c + threadIdx.x; i < Q; i += blockDim.x) piv.buf[i] = -CUDART_INF_F;
    __syncthreads();
    for (int size = 2; size <= Q; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int x = threadIdx.x; x < Q; x += blockDim.x) {
          const int o = x ^ stride;
          if (o > x) {
            const bool desc = (x & size) == 0;
            const float a = piv.buf[x], b = piv.buf[o];
            if (desc ? (b > a) : (a > b)) { piv.buf[x] = b; piv.buf[o] = a; }
          }
        }
        __syncthreads();
      }
    for (int i = threadIdx.x; i < J; i += blockDim.x) out[r * J + i] = piv.buf[i];
    return;
  }
  __syncthreads();
  if (threadIdx.x == 0) n_buf = 0;
  const float t = block_kth_largest(row, n, J, hist, bcast);       // -inf when the row has fewer than J values
  __syncthreads();
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = row[i];
    if (v > t) topj_buf[atomicAdd(&n_buf, 1)] = v;                  // strictly above the J-th largest: < J values
  }
  __syncthreads();
  const int cnt = n_buf;
  const int have = static_cast<int>(min(static_cast<int64_t>(J), n));
  for (int i = cnt + threadIdx.x; i < P; i += blockDim.x) topj_buf[i] = (i < have) ? t : -CUDART_INF_F;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int x = threadIdx.x; x < P; x += blockDim.x) {
        const int o = x ^ stride;
        if (o > x) {
          const bool desc = (x & size) == 0;
          const float a = topj_buf[x], b = topj_buf[o];
          if (desc ? (b > a) : (a > b)) {
            topj_buf[x] = b;
            topj_buf[o] = a;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < J; i += blockDim.x) out[r * J + i] = topj_buf[i];
}

// ---- bitonic top-k ------------------------------------------------------------------------------
template <typename IdxT>
__device__ __forceinline__ bool before(double sa, IdxT ia, double sb, IdxT ib) {
  return sa > sb || (sa == sb && ia < ib);                    // score descending, index ascending
}

template <typename IdxT>
struct IdxLimits;
template <>
struct IdxLimits<int32_t> {
  static __device__ int32_t max() { return 0x7fffffff; }
};
template <>
struct IdxLimits<int64_t> {
  static __device__ int64_t max() { return 0x7fffffffffffffffLL; }
};

// Bitonic sort of P (a power of two) (score, index) pairs by (score desc, index asc); all threads of the block call
// it.  keys / ids may live in shared or global memory (__syncthreads orders both within the block).
template <typename IdxT>
__device__ __forceinline__ void bitonic_sort_pairs(double* keys, IdxT* ids, int P) {
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < P; t += blockDim.x) {
        const int o = t ^ stride;
        if (o > t) {
          const bool asc = (t & size) == 0;                   // "before" order towards lower indices
          const double sa = keys[t], sb = keys[o];
          const IdxT ia = ids[t], ib = ids[o];
          const bool swap = asc ? before<IdxT>(sb, ib, sa, ia) : before<IdxT>(sa, ia, sb, ib);
          if (swap) {
            keys[t] = sb; keys[o] = sa;
            ids[t] = ib; ids[o] = ia;
          }
        }
      }
      __syncthreads();
    }
  }
}

// Segmented input of the selection kernel (K3 after ONE all-gather of packed per-rank blocks): n segments, each a
// [rows, len] block `stride` elements after the previous one; overflow flags [rows] per segment, flag_stride apart.
struct Segments {
  int n;
  int64_t len, stride, flag_stride;
};

template <typename IdxT>
__global__ void __launch_bounds__(1024)
select_topk_kernel(const double* __restrict__ score, const IdxT* __restrict__ idx, int64_t cols,
                   const int32_t* __restrict__ counts, int64_t idx_offset, const int64_t* __restrict__ exclude, int k,
                   const float* __restrict__ thr, float eps, const float* __restrict__ eps_dev,
                   const float* __restrict__ bound, const int32_t* __restrict__ overflow, Segments seg, int pmax,
                   double* __restrict__ out_score, int64_t* __restrict__ out_idx, int32_t* __restrict__ out_valid,
                   int32_t* __restrict__ cert, float* __restrict__ thr_next, int32_t* __restrict__ n_uncertified) {
  extern __shared__ __align__(16) uint8_t sel_smem[];
  double* keys = reinterpret_cast<double*>(sel_smem);
  IdxT* ids = reinterpret_cast<IdxT*>(keys + pmax);
  __shared__ int n_valid_s;
  const int64_t r = blockIdx.x;
  int64_t n_in = cols;
  bool cand_overflow = false;
  if (counts != nullptr) {
    cand_overflow = counts[r] > cols;
    n_in = min(static_cast<int64_t>(counts[r]), cols);
  }
  if (eps_dev != nullptr) eps *= eps_dev[0];
  if (overflow != nullptr)                                             // a shard's candidate list overflowed
    for (int g = 0; g < seg.n; ++g)
      if (overflow[g * seg.flag_stride + r] != 0) cand_overflow = true;
  __shared__ uint32_t sel_hist[256];
  __shared__ uint32_t sel_bcast[2];
  if (threadIdx.x == 0) n_valid_s = 0;
  __syncthreads();
  const int64_t excl = exclude ? exclude[r] : -1;
  // entry i of row r: contiguous [rows, cols], or (segmented) the per-rank blocks of an all-gathered buffer --
  // segment g = i / seg.len holds its [rows, seg.len] block at g * seg.stride elements
  auto at = [&](int64_t i) -> int64_t {
    if (seg.n <= 1) return r * cols + i;
    const int64_t g = i / seg.len;
    return g * seg.stride + r * seg.len + (i - g * seg.len);
  };
  // valid entry i -> its score, anything else -> -inf
  auto value = [&](int64_t i) -> double {
    const double s = score[at(i)];
    const IdxT id = idx ? idx[at(i)] : static_cast<IdxT>(i);          // idx == NULL: column number
    return (s > -CUDART_INF && !(exclude && static_cast<int64_t>(id) + idx_offset == excl)) ? s : -CUDART_INF;
  };
  {                                                                    // one shared-memory add per warp
    int mine = 0;
    for (int64_t i = threadIdx.x; i < n_in; i += blockDim.x) mine += value(i) > -CUDART_INF ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine != 0) atomicAdd(&n_valid_s, mine);
  }
  __syncthreads();
  const int n_all = n_valid_s;                                         // every valid entry of the row
  // More valid entries than the sort holds (dense neighbourhoods: thousands of items within eps of the k-th
  // best): keep only those whose score, rounded to float, reaches the k-th largest rounded score.  Rounding is
  // monotone, so the kept set contains the exact top-k; it can exceed the capacity only through > pmax scores
  // that agree to float precision with the k-th.
  float floor_f = -CUDART_INF_F;
  if (n_all > pmax)
    floor_f = block_kth_largest_of([&](int64_t i) { return __double2float_rn(value(i)); }, n_in, k, sel_hist, sel_bcast);
  __syncthreads();
  if (threadIdx.x == 0) n_valid_s = 0;
  __syncthreads();
  for (int64_t base = threadIdx.x & ~31; base < n_in; base += blockDim.x) {   // warp-aggregated compaction
    const int64_t i = base + (threadIdx.x & 31);
    const double s = i < n_in ? value(i) : -CUDART_INF;
    const bool keep = s > -CUDART_INF && __double2float_rn(s) >= floor_f;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (m != 0) {
      int pos = 0;
      if ((threadIdx.x & 31) == 0) pos = atomicAdd(&n_valid_s, __popc(m));
      pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
      if (keep && pos < pmax) {
        keys[pos] = s;
        ids[pos] = idx ? idx[at(i)] : static_cast<IdxT>(i);
      }
    }
  }
  __syncthreads();
  const int n_valid = n_valid_s;                                       // entries kept for the sort
  const int n = min(n_valid, pmax);
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = n + threadIdx.x; i < P; i += blockDim.x) {
    keys[i] = -CUDART_INF;
    ids[i] = IdxLimits<IdxT>::max();
  }
  __syncthreads();
  bitonic_sort_pairs<IdxT>(keys, ids, P);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const bool ok = i < n;
    out_score[r * k + i] = ok ? keys[i] : -CUDART_INF;
    out_idx[r * k + i] = ok ? static_cast<int64_t>(ids[i]) + idx_offset : -1;
  }
  if (threadIdx.x == 0) {
    if (out_valid) out_valid[r] = n_all;
    if (cert != nullptr && thr == nullptr) {
      // no threshold (a shard's local list before the merge): report only whether the list is exact -- no candidate
      // overflow, and every entry that can belong to the top-k fit the sort (else it holds an arbitrary subset of
      // more than pmax float-tied scores)
      cert[r] = (!cand_overflow && n_valid <= pmax) ? 1 : 0;
      if (n_uncertified != nullptr && cert[r] == 0) atomicAdd(n_uncertified, 1);
    } else if (cert != nullptr) {
      const float t = thr[r];
      const bool enough = n >= k && n_valid <= pmax;
      const double kth = enough ? keys[k - 1] : -CUDART_INF;
      const bool complete = (t == -CUDART_INF_F) || (kth - static_cast<double>(eps) >= static_cast<double>(t));
      cert[r] = (!cand_overflow && enough && complete) ? 1 : 0;
      if (n_uncertified != nullptr && cert[r] == 0) atomicAdd(n_uncertified, 1);
      if (thr_next != nullptr) {
        float nx;
        if (cand_overflow || n_valid > pmax) nx = bound ? bound[r] : t;          // approx kth of retained - 2 eps
        else if (enough) nx = static_cast<float>(kth) - 1.0001f * eps - 1e-7f;   // provably complete
        else nx = t - fmaxf(8.f * eps, 0.25f * fabsf(t));                        // too few found: lower and retry
        thr_next[r] = nx;
      }
    }
  }
}

int pow2_ceil(int64_t x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// ---- range search: every rescored candidate whose exact score reaches a per-row minimum ---------------------------
// Entry c < min(counts[r], cap) of row r matches iff exact > -inf, exact >= min_score[r] (NaN never does) and its
// global row idx + idx_offset is not exclude[r]; with kAfter (similar pairs) its global row must also exceed
// after[r].  Counting and filling apply the same test, so the fill finds exactly the number of entries the count gave.
constexpr int RANGE_SMEM_MAX = 16384;                       // entries sorted in shared memory (12 B each)

template <bool kAfter>
__device__ __forceinline__ bool range_hit(double s, int64_t row, double lo, int64_t excl, int64_t floor) {
  return s > -CUDART_INF && s >= lo && row != excl && (!kAfter || row > floor);
}

template <bool kAfter>
__global__ void __launch_bounds__(256)
range_count_kernel(const double* __restrict__ exact, const int32_t* __restrict__ idx, const int32_t* __restrict__ counts,
                   int cap, int64_t idx_offset, const int64_t* __restrict__ exclude, const double* __restrict__ min_score,
                   int64_t* __restrict__ out, const int64_t* __restrict__ after) {
  __shared__ int part[8];
  const int64_t r = blockIdx.x;
  const int n = min(counts[r], cap);
  const double lo = min_score[r];
  const int64_t excl = exclude ? exclude[r] : -1;
  const int64_t floor = kAfter ? after[r] : 0;
  int mine = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    mine += range_hit<kAfter>(exact[r * cap + i], static_cast<int64_t>(idx[r * cap + i]) + idx_offset, lo, excl, floor)
                ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t t = 0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += part[w];
    out[r] = t;
  }
}

// Row r's m = len[r] matches are compacted, sorted by (score desc, row asc) with bitonic_sort_pairs and written to
// [off[r], off[r] + m).  Rows of up to smem_cap entries sort in shared memory; longer rows in the caller's scratch, row
// r at byte 24 * off[r]: 2m fp64 keys then 2m int32 rows (room for the power-of-two padding, P < 2m).
template <bool kAfter>
__global__ void __launch_bounds__(1024)
range_fill_kernel(const double* __restrict__ exact, const int32_t* __restrict__ idx, const int32_t* __restrict__ counts,
                  int cap, int64_t idx_offset, const int64_t* __restrict__ exclude, const double* __restrict__ min_score,
                  const int64_t* __restrict__ off, const int64_t* __restrict__ len, int smem_cap, uint8_t* scratch,
                  double* __restrict__ out_score, int64_t* __restrict__ out_idx, const int64_t* __restrict__ after) {
  extern __shared__ __align__(16) uint8_t range_smem[];
  __shared__ int n_s;
  const int64_t r = blockIdx.x;
  const int64_t m = len[r];
  if (m == 0) return;
  const int64_t o = off[r];
  double* keys;
  int32_t* ids;
  if (m <= smem_cap) {
    keys = reinterpret_cast<double*>(range_smem);
    ids = reinterpret_cast<int32_t*>(keys + smem_cap);
  } else {
    keys = reinterpret_cast<double*>(scratch + 24 * o);
    ids = reinterpret_cast<int32_t*>(scratch + 24 * o + 16 * m);
  }
  const int n = min(counts[r], cap);
  const double lo = min_score[r];
  const int64_t excl = exclude ? exclude[r] : -1;
  const int64_t floor = kAfter ? after[r] : 0;
  if (threadIdx.x == 0) n_s = 0;
  __syncthreads();
  for (int base = threadIdx.x & ~31; base < n; base += blockDim.x) {          // warp-aggregated compaction
    const int i = base + (threadIdx.x & 31);
    const double s = i < n ? exact[r * cap + i] : -CUDART_INF;
    const int32_t v = i < n ? idx[r * cap + i] : 0;
    const bool keep = i < n && range_hit<kAfter>(s, static_cast<int64_t>(v) + idx_offset, lo, excl, floor);
    const unsigned mk = __ballot_sync(0xffffffffu, keep);
    if (mk != 0) {
      int pos = 0;
      if ((threadIdx.x & 31) == 0) pos = atomicAdd(&n_s, __popc(mk));
      pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(mk & ((1u << (threadIdx.x & 31)) - 1u));
      if (keep && pos < m) { keys[pos] = s; ids[pos] = v; }
    }
  }
  __syncthreads();
  const int got = static_cast<int>(min(static_cast<int64_t>(n_s), m));
  int P = 1;
  while (P < got) P <<= 1;
  for (int i = got + threadIdx.x; i < P; i += blockDim.x) {
    keys[i] = -CUDART_INF;
    ids[i] = IdxLimits<int32_t>::max();
  }
  __syncthreads();
  bitonic_sort_pairs<int32_t>(keys, ids, P);
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const bool ok = i < got;
    out_score[o + i] = ok ? keys[i] : -CUDART_INF;
    out_idx[o + i] = ok ? static_cast<int64_t>(ids[i]) + idx_offset : -1;
  }
}

// Merge of n_seg sorted runs per row: an entry's output position is its position in its own run plus, for every other
// run, the number of entries there that precede it (binary search) -- no sort, no scratch, any run length.
__global__ void __launch_bounds__(256)
range_merge_kernel(const double* __restrict__ score, const int64_t* __restrict__ idx, int n_seg,
                   const int64_t* __restrict__ seg_off, int64_t rows, const int64_t* __restrict__ off,
                   double* __restrict__ out_score, int64_t* __restrict__ out_idx) {
  const int64_t r = blockIdx.x;
  const int64_t o = off[r], total = off[r + 1] - o;
  for (int64_t j = static_cast<int64_t>(blockIdx.y) * blockDim.x + threadIdx.x; j < total;
       j += static_cast<int64_t>(gridDim.y) * blockDim.x) {
    int s = 0;
    int64_t i = j;
    for (; s < n_seg; ++s) {
      const int64_t len = seg_off[s * (rows + 1) + r + 1] - seg_off[s * (rows + 1) + r];
      if (i < len) break;
      i -= len;
    }
    if (s == n_seg) break;                                   // the runs hold fewer entries than off says
    const int64_t p = seg_off[s * (rows + 1) + r] + i;
    const double x = score[p];
    const int64_t v = idx[p];
    int64_t pos = i;
    for (int h = 0; h < n_seg; ++h) {
      if (h == s) continue;
      const int64_t b = seg_off[h * (rows + 1) + r];
      int64_t lo = b, hi = seg_off[h * (rows + 1) + r + 1];
      while (lo < hi) {
        const int64_t mid = lo + (hi - lo) / 2;
        if (before<int64_t>(score[mid], idx[mid], x, v)) lo = mid + 1;
        else hi = mid;
      }
      pos += lo - b;
    }
    out_score[o + pos] = x;
    out_idx[o + pos] = v;
  }
}

// ---- two-round rescore: the pilot ------------------------------------------------------------------
// Round one rescores each shard's m best approximate candidates exactly.  pilot_top extracts the (up to) m largest
// of those exact scores per row, descending, -inf padded (the entry of the query's excluded item is skipped); the
// lists of all shards are gathered and pilot_bound turns the k-th largest exact score of the union -- a LOWER bound
// on the true k-th best score, whatever subset was rescored -- into the second-round window: a candidate whose
// approximate score is below kth1 - eps cannot reach the top-k (exact <= approx + eps < kth1 <= true k-th).
constexpr int PILOT_MAX = 1024;

__global__ void __launch_bounds__(1024)
pilot_top_kernel(const double* __restrict__ exact, const int32_t* __restrict__ idx, const int32_t* __restrict__ counts,
                 int cap, int64_t idx_offset, const int64_t* __restrict__ exclude, int m, double* __restrict__ out) {
  __shared__ double buf[PILOT_MAX];
  __shared__ int n_s;
  const int64_t r = blockIdx.x;
  const int n_in = min(counts[r], cap);
  const int64_t excl = exclude ? exclude[r] : -1;
  if (threadIdx.x == 0) n_s = 0;
  __syncthreads();
  for (int base = threadIdx.x & ~31; base < n_in; base += blockDim.x) {          // warp-aggregated compaction
    const int i = base + (threadIdx.x & 31);
    const double s = i < n_in ? exact[r * cap + i] : -CUDART_INF;
    const bool keep = s > -CUDART_INF && !(exclude && static_cast<int64_t>(idx[r * cap + i]) + idx_offset == excl);
    const unsigned mk = __ballot_sync(0xffffffffu, keep);
    if (mk != 0) {
      int pos = 0;
      if ((threadIdx.x & 31) == 0) pos = atomicAdd(&n_s, __popc(mk));
      pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(mk & ((1u << (threadIdx.x & 31)) - 1u));
      if (keep && pos < PILOT_MAX) buf[pos] = s;  // more than PILOT_MAX (ties at the round-one bound): any subset is valid
    }
  }
  __syncthreads();
  const int n = min(n_s, PILOT_MAX);
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = n + threadIdx.x; i < P; i += blockDim.x) buf[i] = -CUDART_INF;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < P; t += blockDim.x) {
        const int o = t ^ stride;
        if (o > t) {
          const bool desc = (t & size) == 0;
          const double a = buf[t], b = buf[o];
          if (desc ? (b > a) : (a > b)) { buf[t] = b; buf[o] = a; }
        }
      }
      __syncthreads();
    }
  for (int i = threadIdx.x; i < m; i += blockDim.x) out[r * m + i] = i < n ? buf[i] : -CUDART_INF;
}

// lists [n_seg, rows, m] -> bound[r] = round_down(kth largest of the union - eps), -inf when the union holds fewer
// than k finite scores.  One segment (one shard): the list is already sorted, the answer is its k-th entry -- one warp
// per row.  Several: one block per row sorts the union (at most 8192 values) in shared memory.
__global__ void __launch_bounds__(256)
pilot_bound_single_kernel(const double* __restrict__ lists, int64_t rows, int m, int k, float eps,
                          const float* __restrict__ eps_dev, float* __restrict__ bound) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  if (eps_dev != nullptr) eps *= eps_dev[0];
  const double kth = k <= m ? lists[r * m + (k - 1)] : -CUDART_INF;
  bound[r] = kth > -CUDART_INF ? __double2float_rd(kth - static_cast<double>(eps)) : -CUDART_INF_F;
}

__global__ void __launch_bounds__(256)
pilot_bound_kernel(const double* __restrict__ lists, int n_seg, int64_t rows, int m, int k, float eps,
                   const float* __restrict__ eps_dev, int P, float* __restrict__ bound) {
  extern __shared__ double pb_buf[];
  const int64_t r = blockIdx.x;
  if (eps_dev != nullptr) eps *= eps_dev[0];
  const int total = n_seg * m;
  for (int i = threadIdx.x; i < P; i += blockDim.x)
    pb_buf[i] = i < total ? lists[(static_cast<int64_t>(i / m) * rows + r) * m + (i % m)] : -CUDART_INF;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < P; t += blockDim.x) {
        const int o = t ^ stride;
        if (o > t) {
          const bool desc = (t & size) == 0;
          const double a = pb_buf[t], b = pb_buf[o];
          if (desc ? (b > a) : (a > b)) { pb_buf[t] = b; pb_buf[o] = a; }
        }
      }
      __syncthreads();
    }
  if (threadIdx.x == 0) {
    const double kth = k <= total ? pb_buf[k - 1] : -CUDART_INF;
    bound[r] = kth > -CUDART_INF ? __double2float_rd(kth - static_cast<double>(eps)) : -CUDART_INF_F;
  }
}

// ---- the error bound eps on the device (engine.measured_eps without a host round trip) ---------------------------
// dq2 = max over queries of sum_s q_resid[s][q]; eps = dq*vn + qn*dv + k_len*2^-22*qn*vn + 1e-6 with
// qn = sqrt(sum w^2) + dq, vn = sqrt(S)*(1 + 2^-8); NaN / non-positive -> fallback.  One block.
__global__ void __launch_bounds__(1024)
eps_bound_kernel(const float* __restrict__ q_resid, int n_space, int64_t nq, const float* __restrict__ dv2,
                 double w_norm, int k_len, float fallback, float* __restrict__ eps_out) {
  __shared__ float red[32];
  __shared__ int bad_s;
  if (threadIdx.x == 0) bad_s = 0;
  __syncthreads();
  float mx = 0.f;
  bool bad = false;
  for (int64_t q = threadIdx.x; q < nq; q += blockDim.x) {
    float t = 0.f;
    for (int s = 0; s < n_space; ++s) t += q_resid[static_cast<int64_t>(s) * nq + q];
    if (!(t == t)) bad = true;
    mx = fmaxf(mx, t);
  }
  if (bad) bad_s = 1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < static_cast<int>(blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
    const float dv2v = dv2[0];
    double e = -1.0;
    if (!bad_s && dv2v == dv2v) {
      const double dq = sqrt(static_cast<double>(mx)), dv = sqrt(static_cast<double>(dv2v));
      const double qn = w_norm + dq, vn = sqrt(static_cast<double>(n_space)) * (1.0 + 0.00390625);
      e = dq * vn + qn * dv + static_cast<double>(k_len) * 2.384185791015625e-07 * qn * vn + 1e-6;
    }
    eps_out[0] = (e > 0.0 && e < CUDART_INF) ? __double2float_ru(e) : fallback;
  }
}

template <typename IdxT>
int launch_select(const double* score, const IdxT* idx, int64_t rows, int64_t cols, const int32_t* counts,
                  int64_t idx_offset, const int64_t* exclude, int32_t k, const float* thr, float eps,
                  const float* eps_dev, const float* bound, const int32_t* overflow, Segments seg, double* out_score,
                  int64_t* out_idx, int32_t* out_valid, int32_t* cert, float* thr_next, int32_t* n_uncertified,
                  cudaStream_t st) {
  XMVE_REQUIRE(score && out_score && out_idx && rows >= 0 && cols > 0 && k > 0, "select_topk: bad arguments");
  XMVE_REQUIRE(thr_next == nullptr || thr != nullptr, "select_topk: thr_next needs thr");
  if (rows == 0) return XMVE_OK;
  int pmax = pow2_ceil(cols);
  if (pmax > 16384) pmax = 16384;
  // Many rows: a modest sort capacity keeps several blocks resident per SM (the full 16384-entry buffer is 196 KB:
  // one block per SM, 1.7 ms for 8192 rows of ~500 valid entries each).  Rows with more valid entries than the
  // capacity are first cut at their k-th largest rounded score (see the kernel); the rows that still do not fit come
  // back uncertified (without thr: cert = 0) and the engine re-runs them in batches of fewer than 512 rows, which get
  // the full capacity.
  if (rows >= 512) {
    int small = pow2_ceil(4 * static_cast<int64_t>(k));
    if (small < 2048) small = 2048;
    if (pmax > small) pmax = small;
  }
  if (pmax < k) return fail(XMVE_ERR_LIMIT, "select_topk: k=%d exceeds the %d-entry sort capacity", k, pmax);
  const int smem = pmax * static_cast<int>(sizeof(double) + sizeof(IdxT));
  if (smem > 220 * 1024) {
    pmax = 8192;                                            // int64 indices: 16 B per entry
    if (pmax < k) return fail(XMVE_ERR_LIMIT, "select_topk: k too large");
  }
  const int smem_bytes = pmax * static_cast<int>(sizeof(double) + sizeof(IdxT));
  static int attr_bytes[MAX_DEVICES] = {};                 // per <IdxT> instantiation and per device
  const int dev = current_device();
  if (dev < 0) return fail(XMVE_ERR_DEVICE, "select_topk: no current device");
  if (smem_bytes > attr_bytes[dev]) {
    XMVE_CUDA(cudaFuncSetAttribute(select_topk_kernel<IdxT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    attr_bytes[dev] = smem_bytes;
  }
  // small sorts: 256 threads, so that eight rows are resident per SM (the kernel is a chain of short dependent phases)
  // ... and a handful of rows (AVS: 60 queries): one block per row cannot fill the chip, so each block gets 1024
  // threads and its sort phases are four times shorter
  const int threads = pmax <= 2048 ? (rows <= 148 && pmax >= 1024 ? 1024 : 256) : (rows <= 296 ? 1024 : 512);
  select_topk_kernel<IdxT><<<static_cast<unsigned>(rows), threads, smem_bytes, st>>>(
      score, idx, cols, counts, idx_offset, exclude, k, thr, eps, eps_dev, bound, overflow, seg, pmax, out_score,
      out_idx, out_valid, cert, thr_next, n_uncertified);
  return launch_status("select_topk_kernel");
}

}  // namespace
}  // namespace xmve

extern "C" int xmve_row_kth(const float* vals, int64_t rows, int64_t cols, int64_t ld, const int32_t* counts,
                            int32_t j1, float sub, const float* sub_dev, int32_t j2, float* out, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(vals && out && rows >= 0 && cols > 0 && ld >= cols && j1 > 0, "row_kth: bad arguments");
  if (rows == 0) return XMVE_OK;
  row_kth_kernel<<<static_cast<unsigned>(rows), 256, 0, static_cast<cudaStream_t>(stream)>>>(vals, cols, ld, counts,
                                                                                            j1, sub, sub_dev, j2, out);
  return launch_status("row_kth_kernel");
}

extern "C" int xmve_select_topk_i32(const double* score, const int32_t* idx, int64_t rows, int64_t cols,
                                    const int32_t* counts, int64_t idx_offset, const int64_t* exclude, int32_t k,
                                    const float* thr, float eps, const float* eps_dev, const float* bound,
                                    double* out_score, int64_t* out_idx, int32_t* out_valid, int32_t* cert,
                                    float* thr_next, int32_t* n_uncertified, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  return launch_select<int32_t>(score, idx, rows, cols, counts, idx_offset, exclude, k, thr, eps, eps_dev, bound,
                                nullptr, Segments{1, cols, 0, 0}, out_score, out_idx, out_valid, cert, thr_next,
                                n_uncertified, static_cast<cudaStream_t>(stream));
}

extern "C" int xmve_select_topk_i64(const double* score, const int64_t* idx, int64_t rows, int64_t cols,
                                    const int64_t* exclude, int32_t k, const float* thr, float eps,
                                    const float* eps_dev, const int32_t* overflow, double* out_score, int64_t* out_idx,
                                    int32_t* out_valid, int32_t* cert, float* thr_next, int32_t* n_uncertified,
                                    void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  return launch_select<int64_t>(score, idx, rows, cols, nullptr, 0, exclude, k, thr, eps, eps_dev, nullptr, overflow,
                                Segments{1, cols, 0, rows}, out_score, out_idx, out_valid, cert, thr_next,
                                n_uncertified, static_cast<cudaStream_t>(stream));
}

extern "C" int xmve_merge_topk_packed(const void* packed, int32_t n_seg, int64_t seg_bytes, int64_t rows, int32_t len,
                                      const int64_t* exclude, int32_t k, const float* thr, float eps,
                                      const float* eps_dev, double* out_score, int64_t* out_idx, int32_t* cert,
                                      float* thr_next, int32_t* n_uncertified, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(packed != nullptr && n_seg >= 1 && rows >= 0 && len > 0, "merge_topk_packed: bad arguments");
  const int64_t need = xmve_packed_topk_bytes(rows, len);
  XMVE_REQUIRE(seg_bytes >= need && seg_bytes % 8 == 0, "merge_topk_packed: seg_bytes %lld < %lld or not a multiple of 8",
               static_cast<long long>(seg_bytes), static_cast<long long>(need));
  const uint8_t* base = static_cast<const uint8_t*>(packed);
  const double* score = reinterpret_cast<const double*>(base);
  const int64_t* idx = reinterpret_cast<const int64_t*>(base + rows * len * 8);
  const int32_t* flags = reinterpret_cast<const int32_t*>(base + rows * len * 16);
  return launch_select<int64_t>(score, idx, rows, static_cast<int64_t>(n_seg) * len, nullptr, 0, exclude, k, thr, eps,
                                eps_dev, nullptr, flags, Segments{n_seg, len, seg_bytes / 8, seg_bytes / 4}, out_score,
                                out_idx, nullptr, cert, thr_next, n_uncertified, static_cast<cudaStream_t>(stream));
}

extern "C" int64_t xmve_packed_topk_bytes(int64_t rows, int32_t len) {
  const int64_t b = rows * len * 16 + rows * 4;
  return (b + 15) / 16 * 16;
}

namespace {
// count / fill of xmve_range_select (kAfter false) and xmve_pair_select (kAfter true)
template <bool kAfter>
int range_select(const char* name, const double* exact, const int32_t* cand_idx, const int32_t* cand_count,
                 int64_t rows, int32_t cap, int64_t idx_offset, const int64_t* exclude, const double* min_score,
                 int64_t* counts, const int64_t* off, int64_t max_len, void* scratch, double* out_score,
                 int64_t* out_idx, const int64_t* after, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(exact && cand_idx && cand_count && min_score && counts && rows >= 0 && cap > 0 && (!kAfter || after),
               "%s: bad arguments", name);
  if (rows == 0) return XMVE_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (off == nullptr) {
    range_count_kernel<kAfter><<<static_cast<unsigned>(rows), 256, 0, st>>>(exact, cand_idx, cand_count, cap,
                                                                              idx_offset, exclude, min_score, counts,
                                                                              after);
    return launch_status("range_count_kernel");
  }
  XMVE_REQUIRE(out_score && out_idx && max_len >= 0 && max_len <= cap, "%s: fill needs outputs, 0 <= max_len <= cap",
               name);
  if (max_len > RANGE_SMEM_MAX && scratch == nullptr)
    return fail(XMVE_ERR_LIMIT, "%s: a row has %lld entries (> %d): pass scratch (24 bytes per output entry)", name,
                static_cast<long long>(max_len), RANGE_SMEM_MAX);
  const int smem_cap = pow2_ceil(max_len < 1 ? 1 : (max_len > RANGE_SMEM_MAX ? RANGE_SMEM_MAX : max_len));
  const int smem_bytes = smem_cap * static_cast<int>(sizeof(double) + sizeof(int32_t));
  static int attr_bytes[MAX_DEVICES] = {};
  const int dev = current_device();
  if (dev < 0) return fail(XMVE_ERR_DEVICE, "%s: no current device", name);
  if (smem_bytes > attr_bytes[dev]) {
    XMVE_CUDA(cudaFuncSetAttribute(range_fill_kernel<kAfter>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    attr_bytes[dev] = smem_bytes;
  }
  range_fill_kernel<kAfter><<<static_cast<unsigned>(rows), max_len > 2048 ? 1024 : 256, smem_bytes, st>>>(
      exact, cand_idx, cand_count, cap, idx_offset, exclude, min_score, off, counts, smem_cap,
      static_cast<uint8_t*>(scratch), out_score, out_idx, after);
  return launch_status("range_fill_kernel");
}
}  // namespace

extern "C" int xmve_range_select(const double* exact, const int32_t* cand_idx, const int32_t* cand_count, int64_t rows,
                                 int32_t cap, int64_t idx_offset, const int64_t* exclude, const double* min_score,
                                 int64_t* counts, const int64_t* off, int64_t max_len, void* scratch,
                                 double* out_score, int64_t* out_idx, void* stream) {
  return range_select<false>("range_select", exact, cand_idx, cand_count, rows, cap, idx_offset, exclude, min_score,
                             counts, off, max_len, scratch, out_score, out_idx, nullptr, stream);
}

extern "C" int xmve_pair_select(const double* exact, const int32_t* cand_idx, const int32_t* cand_count, int64_t rows,
                                int32_t cap, int64_t idx_offset, const int64_t* exclude, const double* min_score,
                                int64_t* counts, const int64_t* off, int64_t max_len, void* scratch,
                                double* out_score, int64_t* out_idx, const int64_t* after, void* stream) {
  return range_select<true>("pair_select", exact, cand_idx, cand_count, rows, cap, idx_offset, exclude, min_score,
                            counts, off, max_len, scratch, out_score, out_idx, after, stream);
}

extern "C" int xmve_range_merge(const double* score, const int64_t* idx, int32_t n_seg, const int64_t* seg_off,
                                int64_t rows, const int64_t* off, int64_t max_len, double* out_score, int64_t* out_idx,
                                void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(seg_off && off && out_score && out_idx && n_seg >= 1 && rows >= 0 && max_len >= 0,
               "range_merge: bad arguments");
  if (rows == 0 || max_len == 0) return XMVE_OK;
  XMVE_REQUIRE(score && idx, "range_merge: bad arguments");
  int64_t gy = (max_len + 4095) / 4096;
  if (gy > 65535) gy = 65535;
  range_merge_kernel<<<dim3(static_cast<unsigned>(rows), static_cast<unsigned>(gy)), 256, 0,
                       static_cast<cudaStream_t>(stream)>>>(score, idx, n_seg, seg_off, rows, off, out_score, out_idx);
  return launch_status("range_merge_kernel");
}

extern "C" int xmve_row_topj(const float* vals, int64_t rows, int64_t cols, int64_t ld, const int32_t* counts,
                             int32_t j, float* out, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(vals && out && rows >= 0 && cols > 0 && ld >= cols && j > 0, "row_topj: bad arguments");
  if (j > 4096) return fail(XMVE_ERR_LIMIT, "row_topj: j=%d exceeds 4096", j);
  if (rows == 0) return XMVE_OK;
  const int P = pow2_ceil(j);
  row_topj_kernel<<<static_cast<unsigned>(rows), 256, P * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      vals, cols, ld, counts, j, P, out);
  return launch_status("row_topj_kernel");
}

extern "C" int xmve_pilot_top(const double* exact, const int32_t* idx, const int32_t* counts, int64_t rows, int32_t cap,
                              int64_t idx_offset, const int64_t* exclude, int32_t m, double* out, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(exact && idx && counts && out && rows >= 0 && cap > 0 && m > 0, "pilot_top: bad arguments");
  if (m > PILOT_MAX) return fail(XMVE_ERR_LIMIT, "pilot_top: m=%d exceeds %d", m, PILOT_MAX);
  if (rows == 0) return XMVE_OK;
  pilot_top_kernel<<<static_cast<unsigned>(rows), (rows <= 296 && m > 256) ? 1024 : 256, 0, static_cast<cudaStream_t>(stream)>>>(
      exact, idx, counts, cap, idx_offset, exclude, m, out);
  return launch_status("pilot_top_kernel");
}

extern "C" int xmve_pilot_bound(const double* lists, int32_t n_seg, int64_t rows, int32_t m, int32_t k, float eps,
                                const float* eps_dev, float* bound, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(lists && bound && n_seg >= 1 && rows >= 0 && m > 0 && k > 0, "pilot_bound: bad arguments");
  if (rows == 0) return XMVE_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_seg == 1) {
    pilot_bound_single_kernel<<<static_cast<unsigned>((rows + 255) / 256), 256, 0, st>>>(lists, rows, m, k, eps, eps_dev,
                                                                                       bound);
    return launch_status("pilot_bound_single_kernel");
  }
  const int64_t total = static_cast<int64_t>(n_seg) * m;
  if (total > 4096) return fail(XMVE_ERR_LIMIT, "pilot_bound: %lld pilot scores per row exceed 4096", (long long)total);
  const int P = pow2_ceil(total);
  pilot_bound_kernel<<<static_cast<unsigned>(rows), 256, P * sizeof(double), st>>>(lists, n_seg, rows, m, k, eps,
                                                                                  eps_dev, P, bound);
  return launch_status("pilot_bound_kernel");
}

extern "C" int xmve_eps_bound(const float* q_resid, int32_t n_space, int64_t nq, const float* dv2, double w_norm,
                              int32_t k_len, float fallback, float* eps_out, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(q_resid && dv2 && eps_out && n_space >= 1 && nq >= 0 && k_len > 0, "eps_bound: bad arguments");
  eps_bound_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(q_resid, n_space, nq, dv2, w_norm, k_len,
                                                                      fallback, eps_out);
  return launch_status("eps_bound_kernel");
}
