// K4: bit-exact rank / metric kernels over a caller-supplied errors matrix, and norm_score.
//
// The reference finds the rank of every ground-truth item by fully sorting every row (and every
// strided column) and searching the permutation in Python (LINAS-engine/util/metrics.py:61-102,
// 124-157; 78 s of the 122 s at the MSR-VTT full-test shape).  A rank is just a count:
//   rank(g) = 1 + #{m : x[m] < x[g]} + #{m < g : x[m] == x[g]}
// (the position of g in a stable ascending argsort), so one streaming pass over the matrix gives
// all ranks exactly; R@K, MedR (histogram), MeanR (integer sum) and AP (double-precision sums in
// rank order, basic/metric.py:31-46) follow without any floating-point freedom.
#include <math_constants.h>

#include "common.cuh"

namespace xmve {
namespace {

// axis 0: query = row i.  One WARP per (row, group of G ground-truth entries): lanes stride over the row with four
// independent loads in flight, so a 24 KB row of doubles is read at memory speed (a block per row with a dozen
// elements per thread was latency-bound: 1.3 TB/s at the MSR-VTT full-test shape).
template <typename T, int G>
__global__ void __launch_bounds__(256)
gt_ranks_rows_kernel(const T* __restrict__ x, int64_t n_query, int64_t n_col, int64_t ld, int n_groups,
                     const int64_t* __restrict__ gt_off, const int32_t* __restrict__ gt_ids,
                     int32_t* __restrict__ ranks) {
  const int lane = threadIdx.x & 31;
  const int64_t unit = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const int64_t q = unit / n_groups;
  if (q >= n_query) return;
  const int64_t e0 = gt_off[q] + (unit - q * n_groups) * G;
  const int64_t e1 = min(gt_off[q + 1], e0 + G);
  if (e0 >= e1) return;
  const int ng = static_cast<int>(e1 - e0);
  const T* __restrict__ row = x + q * ld;
  T gv[G];
  int gi[G], cnt[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    gi[g] = g < ng ? gt_ids[e0 + g] : 0;
    gv[g] = row[gi[g]];
    cnt[g] = 0;
  }
  int64_t m = lane;
  for (; m + 96 < n_col; m += 128) {
    const T v0 = row[m], v1 = row[m + 32], v2 = row[m + 64], v3 = row[m + 96];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      cnt[g] += (v0 < gv[g] || (v0 == gv[g] && m < gi[g])) ? 1 : 0;
      cnt[g] += (v1 < gv[g] || (v1 == gv[g] && m + 32 < gi[g])) ? 1 : 0;
      cnt[g] += (v2 < gv[g] || (v2 == gv[g] && m + 64 < gi[g])) ? 1 : 0;
      cnt[g] += (v3 < gv[g] || (v3 == gv[g] && m + 96 < gi[g])) ? 1 : 0;
    }
  }
  for (; m < n_col; m += 32) {
    const T v = row[m];
#pragma unroll
    for (int g = 0; g < G; ++g) cnt[g] += (v < gv[g] || (v == gv[g] && m < gi[g])) ? 1 : 0;
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
    int c = cnt[g];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0 && g < ng) ranks[e0 + g] = 1 + c;
  }
}

// axis 1: query = column i, memories = rows.  A block owns 32 adjacent columns (lane <-> column, so every row read
// is one coalesced line) and a slice of the rows; partial counts are added atomically into ranks[] (zeroed by the
// host wrapper; slice 0 adds the leading 1).  Up to CG ground-truth entries per column are ranked in one pass over
// the data (the 20 captions per video of MSR-VTT).
//
// rank(g) - 1 = #{m : (x[m], m) < (x[g], g)} lexicographically.  The column's ground-truth keys are sorted once
// (shared memory, one lane per column); an element then needs ONE branch-free binary search (five steps) for
// p = #{g : key_g <= (x[m], m)} and one private histogram bump -- the count of entry g is the prefix sum of the
// histogram up to g.  The first version compared every element with all 24 entries (~100 instructions and 96 live
// registers per element: 16 warps per SM, 0.37 TB/s over the 1.43 GB matrix of the C2 shape).
constexpr int CG = 31;                                   // entries per pass (the sorted list is padded to 32)
template <typename T>
__global__ void __launch_bounds__(256)
gt_ranks_cols_kernel(const T* __restrict__ x, int64_t n_row, int64_t n_col, int64_t ld,
                     const int64_t* __restrict__ gt_off, const int32_t* __restrict__ gt_ids, int max_gt,
                     int rows_per_slice, int32_t* __restrict__ ranks) {
  __shared__ T s_key[32][32];                            // [sorted position][column of the block]
  __shared__ int s_row[32][32];                          // ... its row (the tie rule) ...
  __shared__ int s_ent[32][32];                          // ... and its place in the column's CSR list
  __shared__ int s_hist[32][256];                        // [p][thread]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t col = static_cast<int64_t>(blockIdx.x) * 32 + lane;
  const bool col_ok = col < n_col;
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * rows_per_slice;
  const int64_t r1 = min(n_row, r0 + rows_per_slice);
  const int64_t e_lo = col_ok ? gt_off[col] : 0, e_hi = col_ok ? gt_off[col + 1] : 0;
  const T inf = static_cast<T>(CUDART_INF);
  for (int base = 0; base < max_gt; base += CG) {
    if (warp == 0) {                                     // one lane per column: gather and insertion-sort its keys
      int ng = 0;
      for (int g = 0; g < CG; ++g) {
        if (e_lo + base + g >= e_hi) break;
        const int gi = gt_ids[e_lo + base + g];
        T gv = x[static_cast<int64_t>(gi) * ld + col];
        int gr = gi;
        if (gv != gv) { gv = -inf; gr = -1; }           // NaN ground truth: ranked by gt_ranks_nan_kernel afterwards
        int pos = ng;
        while (pos > 0 && (s_key[pos - 1][lane] > gv || (s_key[pos - 1][lane] == gv && s_row[pos - 1][lane] > gr))) {
          s_key[pos][lane] = s_key[pos - 1][lane];
          s_row[pos][lane] = s_row[pos - 1][lane];
          s_ent[pos][lane] = s_ent[pos - 1][lane];
          --pos;
        }
        s_key[pos][lane] = gv;
        s_row[pos][lane] = gr;
        s_ent[pos][lane] = base + g;
        ++ng;
      }
      for (int g = ng; g < 32; ++g) {                    // padding: above every element
        s_key[g][lane] = inf;
        s_row[g][lane] = 0x7fffffff;
        s_ent[g][lane] = -1;
      }
    }
#pragma unroll
    for (int p = 0; p < 32; ++p) s_hist[p][threadIdx.x] = 0;
    __syncthreads();
    if (col_ok) {
      auto bump = [&](T v, int64_t m) {
        if (v != v) return;                              // NaN elements are below nothing
        int lo = 0;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
          const T k = s_key[lo + step - 1][lane];
          const bool le = k < v || (k == v && static_cast<int64_t>(s_row[lo + step - 1][lane]) <= m);
          lo += le ? step : 0;
        }
        ++s_hist[lo][threadIdx.x];                       // lo = #{g : key_g <= (v, m)}  (<= 31)
      };
      int64_t m = r0 + warp;
      for (; m + 24 < r1; m += 32) {                     // four independent row reads in flight
        const T va = x[m * ld + col], vb = x[(m + 8) * ld + col], vc = x[(m + 16) * ld + col],
                vd = x[(m + 24) * ld + col];
        bump(va, m);
        bump(vb, m + 8);
        bump(vc, m + 16);
        bump(vd, m + 24);
      }
      for (; m < r1; m += 8) bump(x[m * ld + col], m);
    }
    // entry at sorted position g is preceded by every element whose p is <= g
    int run = 0;
    for (int g = 0; g < 32; ++g) {
      run += s_hist[g][threadIdx.x];
      const int ent = s_ent[g][lane];
      if (ent >= 0) {
        const int add = run + ((blockIdx.y == 0 && warp == 0) ? 1 : 0);
        if (add != 0) atomicAdd(&ranks[e_lo + ent], add);
      }
    }
    __syncthreads();                                     // the sorted lists are rebuilt by the next pass
  }
}

// NaN ground truths.  NumPy's argsort (the reference's ranking) places every NaN after every number, NaNs in index
// order, so an entry whose value is NaN has rank 1 + #{non-NaN elements of the line} + #{NaN elements m < g}.  The two
// kernels above order numbers only; this pass runs after either of them and overwrites the ranks of those entries.
// One warp per CSR entry: it leaves at once unless the entry's value is NaN, else its lanes scan the line.  Query q's
// line is x[q * q_step + m * m_step], m < n_mem.
template <typename T>
__global__ void __launch_bounds__(256)
gt_ranks_nan_kernel(const T* __restrict__ x, int64_t n_mem, int64_t q_step, int64_t m_step,
                    const int64_t* __restrict__ gt_off, const int32_t* __restrict__ gt_ids, int64_t n_query,
                    int64_t n_entries, int32_t* __restrict__ ranks) {
  const int64_t e = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= n_entries) return;
  int64_t lo = 0, hi = n_query;                                 // owner: the last q with gt_off[q] <= e
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (gt_off[mid] <= e) lo = mid; else hi = mid;
  }
  const T* line = x + lo * q_step;
  const int64_t g = gt_ids[e];
  const T gv = line[g * m_step];
  if (gv == gv) return;
  int64_t c = 0;
  for (int64_t m = lane; m < n_mem; m += 32) {
    const T v = line[m * m_step];
    c += (v == v || m < g) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) ranks[e] = static_cast<int32_t>(1 + c);
}

// One block per query: sort the query's ranks, reduce to best rank / AP, bump the global tallies.
// The sort is a bitonic network whose compare-exchanges are ALL ascending (the first step of every merge mirrors its
// block), so a list of any length n is sorted as if padded with +inf: exchanges with a partner >= n are skipped.
// Lists of up to smem_cap entries are sorted in shared memory, longer ones in the caller's global scratch.
__global__ void __launch_bounds__(128)
rank_metrics_kernel(const int32_t* __restrict__ ranks, const int64_t* __restrict__ gt_off, int64_t n_mem,
                    int first_only, int ap_k, int smem_cap, int32_t* __restrict__ scratch,
                    int32_t* __restrict__ best, double* __restrict__ ap,
                    unsigned long long* __restrict__ recall_counts, unsigned long long* __restrict__ rank_sum,
                    int32_t* __restrict__ hist) {
  extern __shared__ int32_t s_rank_smem[];
  const int64_t q = blockIdx.x;
  const int64_t e0 = gt_off[q], e1 = gt_off[q + 1];
  const int n = static_cast<int>(e1 - e0);
  int32_t* s_rank = n <= smem_cap ? s_rank_smem : scratch + e0;
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s_rank[i] = ranks[e0 + i];
  __syncthreads();
  const int first_rank = n > 0 ? s_rank[0] : 0;               // rank of the FIRST ground-truth entry
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    const int half = size >> 1;
    for (int pr = threadIdx.x; pr < (P >> 1); pr += blockDim.x) {           // mirror step
      const int blk = pr / half, j = pr - blk * half;
      const int t = blk * size + j, o = blk * size + size - 1 - j;
      if (o < n) {
        const int a = s_rank[t], b = s_rank[o];
        if (b < a) { s_rank[t] = b; s_rank[o] = a; }
      }
    }
    __syncthreads();
    for (int stride = half >> 1; stride > 0; stride >>= 1) {
      for (int pr = threadIdx.x; pr < (P >> 1); pr += blockDim.x) {
        const int t = 2 * stride * (pr / stride) + (pr % stride), o = t + stride;
        if (o < n) {
          const int a = s_rank[t], b = s_rank[o];
          if (b < a) { s_rank[t] = b; s_rank[o] = a; }
        }
      }
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) {
    const int64_t length = (ap_k > 0 && ap_k <= n_mem) ? ap_k : n_mem;      // MetricScorer.getLength
    const int b = n > 0 ? s_rank[0] : static_cast<int>(n_mem + 1);
    double a = 0.0;
    if (n > 0) {
      if (first_only) {
        if (first_rank <= length) a += 1.0 / static_cast<double>(first_rank);
        a /= 1.0;
      } else {
        for (int j = 0; j < n && s_rank[j] <= length; ++j) a += static_cast<double>(j + 1) / static_cast<double>(s_rank[j]);
        a /= static_cast<double>(n);
      }
    }
    if (best) best[q] = b;
    if (ap) ap[q] = a;
    if (recall_counts) {
      if (b <= 1) atomicAdd(&recall_counts[0], 1ull);
      if (b <= 5) atomicAdd(&recall_counts[1], 1ull);
      if (b <= 10) atomicAdd(&recall_counts[2], 1ull);
    }
    if (rank_sum) atomicAdd(rank_sum, static_cast<unsigned long long>(b));
    if (hist) atomicAdd(&hist[b], 1);
  }
}

// ---- norm_score ----------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long dkey(double x) {        // order-preserving key
  const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(x));
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_d(unsigned long long k) {
  return __longlong_as_double(static_cast<long long>((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

__global__ void minmax_init_kernel(unsigned long long* keys) {
  keys[0] = ~0ull;   // running min key
  keys[1] = 0ull;    // running max key
}

template <typename T>
__global__ void __launch_bounds__(256)
minmax_kernel(const T* __restrict__ x, int64_t n_row, int64_t n_col, int64_t ld, unsigned long long* keys) {
  double mn = CUDART_INF, mx = -CUDART_INF;
  bool nan = false;
  const int64_t total = n_row * n_col;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double s = -static_cast<double>(x[(i / n_col) * ld + (i % n_col)]);   // score = -error
    nan |= s != s;
    mn = fmin(mn, s);
    mx = fmax(mx, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  nan = __any_sync(0xffffffffu, nan);
  if ((threadIdx.x & 31) == 0) {
    // np.min / np.max are NaN if any element is, while fmin / fmax skip NaN.  A NaN's own key is no help: its sign is
    // arbitrary (s = -x flips it) and a negative NaN's key sorts below -inf.  So the flag stores the extreme keys 0 and
    // ~0, which both decode to NaN.
    atomicMin(&keys[0], nan ? 0ull : dkey(mn));
    atomicMax(&keys[1], nan ? ~0ull : dkey(mx));
  }
}

// out = -(((-E) - min) / max(-E - min)) in the input's own precision (validate.py:8-11)
template <typename T>
__global__ void __launch_bounds__(256)
norm_apply_kernel(const T* __restrict__ x, int64_t n_row, int64_t n_col, int64_t ld, T* __restrict__ out,
                  int64_t out_ld, const unsigned long long* __restrict__ keys) {
  const T mn = static_cast<T>(key_d(keys[0]));
  // max(s - min) == max(s) - min (rounding is monotone).  With an infinite min NumPy's max(s - min) is NaN and this
  // one may be inf, but then every s - min is +-inf or NaN and every output NaN either way.
  const T mx = static_cast<T>(key_d(keys[1])) - mn;
  const int64_t total = n_row * n_col;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / n_col, c = i % n_col;
    const T s = -x[r * ld + c];
    out[r * out_ld + c] = -((s - mn) / mx);
  }
}

}  // namespace
}  // namespace xmve

extern "C" int xmve_gt_ranks(const void* errors, int dtype, int64_t n_row, int64_t n_col, int64_t ld, int axis,
                             const int64_t* gt_off, const int32_t* gt_ids, int64_t n_query, int64_t n_entries,
                             int32_t max_gt, int32_t* ranks, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(errors && gt_off && gt_ids && ranks && n_row > 0 && n_col > 0 && ld >= n_col, "gt_ranks: bad arguments");
  XMVE_REQUIRE(dtype == XMVE_F32 || dtype == XMVE_F64, "gt_ranks: dtype must be f32 or f64");
  XMVE_REQUIRE(axis == 0 || axis == 1, "gt_ranks: axis must be 0 or 1");
  XMVE_REQUIRE(n_query == (axis == 0 ? n_row : n_col), "gt_ranks: n_query must match the query axis");
  XMVE_REQUIRE(n_entries >= 0 && max_gt >= 0, "gt_ranks: negative CSR sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_entries == 0 || max_gt == 0) return XMVE_OK;
  const int64_t nan_blocks = (n_entries + 7) / 8;               // gt_ranks_nan_kernel: one warp per entry
  if (nan_blocks > 2147483647LL) return fail(XMVE_ERR_LIMIT, "gt_ranks: too many entries");
  if (axis == 0) {
    const int G = max_gt == 1 ? 1 : 8;
    const int n_groups = (max_gt + G - 1) / G;
    const int64_t units = n_query * n_groups;
    const unsigned grid = static_cast<unsigned>((units + 7) / 8);
    if ((units + 7) / 8 > 2147483647LL) return fail(XMVE_ERR_LIMIT, "gt_ranks: too many (query, ground-truth) units");
#define XMVE_ROWS(T, GG)                                                                                          \
  gt_ranks_rows_kernel<T, GG><<<grid, 256, 0, st>>>(static_cast<const T*>(errors), n_query, n_col, ld, n_groups, gt_off, \
                                                    gt_ids, ranks)
    if (dtype == XMVE_F32) { if (G == 1) XMVE_ROWS(float, 1); else XMVE_ROWS(float, 8); }
    else { if (G == 1) XMVE_ROWS(double, 1); else XMVE_ROWS(double, 8); }
#undef XMVE_ROWS
  } else {
    XMVE_CUDA(cudaMemsetAsync(ranks, 0, static_cast<size_t>(n_entries) * sizeof(int32_t), st));
    const int col_blocks = static_cast<int>((n_col + 31) / 32);
    int slices = (4 * sm_count() + col_blocks - 1) / col_blocks;
    if (slices < 1) slices = 1;
    int rows_per_slice = static_cast<int>((n_row + slices - 1) / slices);
    rows_per_slice = (rows_per_slice + 15) / 16 * 16;
    slices = static_cast<int>((n_row + rows_per_slice - 1) / rows_per_slice);
    dim3 grid(static_cast<unsigned>(col_blocks), static_cast<unsigned>(slices));
    if (dtype == XMVE_F32)
      gt_ranks_cols_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(errors), n_row, n_col, ld, gt_off,
                                                        gt_ids, max_gt, rows_per_slice, ranks);
    else
      gt_ranks_cols_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double*>(errors), n_row, n_col, ld, gt_off,
                                                         gt_ids, max_gt, rows_per_slice, ranks);
  }
  const int64_t n_mem = axis == 0 ? n_col : n_row, q_step = axis == 0 ? ld : 1, m_step = axis == 0 ? 1 : ld;
  if (dtype == XMVE_F32)
    gt_ranks_nan_kernel<float><<<static_cast<unsigned>(nan_blocks), 256, 0, st>>>(
        static_cast<const float*>(errors), n_mem, q_step, m_step, gt_off, gt_ids, n_query, n_entries, ranks);
  else
    gt_ranks_nan_kernel<double><<<static_cast<unsigned>(nan_blocks), 256, 0, st>>>(
        static_cast<const double*>(errors), n_mem, q_step, m_step, gt_off, gt_ids, n_query, n_entries, ranks);
  return launch_status("gt_ranks kernels");
}

namespace xmve {
namespace {
// One warp per CSR entry e: the 1-based position of wanted[e] in the ranked list of the query that owns e
// (first occurrence), `absent` when it is not in the list.  The lanes scan the list with coalesced loads.
__global__ void __launch_bounds__(256)
list_ranks_kernel(const int64_t* __restrict__ lists, int64_t n_query, int64_t len, int64_t ld,
                  const int64_t* __restrict__ off, const int64_t* __restrict__ wanted, int64_t n_entries, int32_t absent,
                  int32_t* __restrict__ rank) {
  const int64_t e = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= n_entries) return;
  int64_t lo = 0, hi = n_query;                                 // owner: the last q with off[q] <= e
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (off[mid] <= e) lo = mid; else hi = mid;
  }
  const int64_t* row = lists + lo * ld;
  const int64_t w = wanted[e];
  int32_t found = absent;
  for (int64_t p0 = 0; p0 < len; p0 += 32) {
    const int64_t p = p0 + lane;
    const unsigned hit = __ballot_sync(0xffffffffu, p < len && row[p] == w);
    if (hit != 0) {
      found = static_cast<int32_t>(p0 + (__ffs(hit) - 1) + 1);
      break;
    }
  }
  if (lane == 0) rank[e] = found;
}
}  // namespace
}  // namespace xmve

extern "C" int xmve_list_ranks(const int64_t* lists, int64_t n_query, int64_t len, int64_t ld, const int64_t* off,
                               const int64_t* wanted, int64_t n_entries, int32_t absent, int32_t* rank, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(lists && off && rank && n_query > 0 && len > 0 && ld >= len && n_entries >= 0, "list_ranks: bad arguments");
  if (n_entries == 0) return XMVE_OK;
  XMVE_REQUIRE(wanted != nullptr, "list_ranks: wanted is null");
  const int64_t blocks = (n_entries + 7) / 8;
  if (blocks > 2147483647LL) return fail(XMVE_ERR_LIMIT, "list_ranks: too many entries");
  list_ranks_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      lists, n_query, len, ld, off, wanted, n_entries, absent, rank);
  return launch_status("list_ranks_kernel");
}

namespace xmve {
namespace {
// Rank of a ground-truth item from a candidate list (corpora whose score matrix cannot exist): entry e owns the
// exact scores of the candidates whose approximate score fell into the guard band around its ground truth's score.
// before[e] += #{c : exact[e, c] > s_gt[e]  or  (exact[e, c] == s_gt[e] and global index of c < g[e])} -- the
// candidates that precede the ground truth in a stable ascending argsort of the errors (util/metrics.py:139-145).
// One warp per entry.
__global__ void __launch_bounds__(256)
count_before_kernel(const double* __restrict__ exact, const int32_t* __restrict__ idx,
                    const int32_t* __restrict__ counts, int cap, int64_t idx_offset,
                    const double* __restrict__ s_gt, const int64_t* __restrict__ g, int64_t n_entries,
                    long long* __restrict__ before) {
  const int64_t e = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= n_entries) return;
  const int n = min(counts[e], cap);
  const double s = s_gt[e];
  const int64_t gi = g[e];
  int c = 0;
  for (int i = lane; i < n; i += 32) {
    const double x = exact[e * cap + i];
    const int64_t id = static_cast<int64_t>(idx[e * cap + i]) + idx_offset;
    c += (x > s || (x == s && id < gi)) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0 && c != 0) atomicAdd(reinterpret_cast<unsigned long long*>(&before[e]), static_cast<unsigned long long>(c));
}

// The same question against a chunk of an exact fp64 score matrix (the fallback for ground truths so deep that the
// guard band of the tensor-core pass overflows): scores [n_entries, cols] cover global columns col0 .. col0+cols.
// Values above s_gt + delta are counted; the few inside |x - s_gt| <= delta (delta ~ 1e-13: the two fp64 summation
// orders agree to ~1e-15) are appended to a per-entry list and settled by the rescore kernel's own arithmetic.
__global__ void __launch_bounds__(256)
count_band_f64_kernel(const double* __restrict__ scores, int64_t cols, int64_t ld, int64_t col0,
                      const double* __restrict__ s_gt, double delta, int64_t n_entries,
                      long long* __restrict__ above, int32_t* __restrict__ band_count, int32_t* __restrict__ band_idx,
                      int band_cap) {
  const int64_t e = blockIdx.y;
  const double s = s_gt[e];
  const double* row = scores + e * ld;
  int c = 0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < cols;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double x = row[i];
    if (x > s + delta) {
      ++c;
    } else if (x >= s - delta) {
      const int slot = atomicAdd(&band_count[e], 1);
      if (slot < band_cap) band_idx[e * band_cap + slot] = static_cast<int32_t>(i);   // column within the chunk
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c != 0)
    atomicAdd(reinterpret_cast<unsigned long long*>(&above[e]), static_cast<unsigned long long>(c));
}
}  // namespace
}  // namespace xmve

extern "C" int xmve_count_before(const double* exact, const int32_t* idx, const int32_t* counts, int64_t n_entries,
                                 int32_t cap, int64_t idx_offset, const double* s_gt, const int64_t* g,
                                 int64_t* before, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(exact && idx && counts && s_gt && g && before && n_entries >= 0 && cap > 0, "count_before: bad arguments");
  if (n_entries == 0) return XMVE_OK;
  const int64_t blocks = (n_entries + 7) / 8;
  if (blocks > 2147483647LL) return fail(XMVE_ERR_LIMIT, "count_before: too many entries");
  count_before_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      exact, idx, counts, cap, idx_offset, s_gt, g, n_entries, reinterpret_cast<long long*>(before));
  return launch_status("count_before_kernel");
}

extern "C" int xmve_count_band_f64(const double* scores, int64_t n_entries, int64_t cols, int64_t ld, int64_t col0,
                                   const double* s_gt, double delta, int64_t* above, int32_t* band_count,
                                   int32_t* band_idx, int32_t band_cap, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(scores && s_gt && above && band_count && band_idx && n_entries >= 0 && cols > 0 && ld >= cols &&
                   band_cap > 0 && delta >= 0.0, "count_band_f64: bad arguments");
  if (n_entries == 0) return XMVE_OK;
  if (n_entries > 65535) return fail(XMVE_ERR_LIMIT, "count_band_f64: more than 65535 entries per call; chunk it");
  (void)col0;
  int bx = static_cast<int>((cols + 2047) / 2048);
  if (bx > 64) bx = 64;
  dim3 grid(static_cast<unsigned>(bx), static_cast<unsigned>(n_entries));
  count_band_f64_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      scores, cols, ld, col0, s_gt, delta, n_entries, reinterpret_cast<long long*>(above), band_count, band_idx,
      band_cap);
  return launch_status("count_band_f64_kernel");
}

extern "C" int xmve_rank_metrics(const int32_t* ranks, const int64_t* gt_off, int64_t n_query, int64_t n_mem,
                                 int first_only, int ap_k, int32_t max_gt, int32_t* sort_scratch, int32_t* best,
                                 double* ap, int64_t* recall_counts, int64_t* rank_sum, int32_t* hist, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(ranks && gt_off && n_query >= 0 && n_mem > 0 && max_gt >= 0, "rank_metrics: bad arguments");
  if (n_query == 0) return XMVE_OK;
  constexpr int SMEM_MAX = 16384;                                  // entries sorted in shared memory
  if (max_gt > SMEM_MAX && sort_scratch == nullptr)
    return fail(XMVE_ERR_LIMIT, "rank_metrics: a query has %d entries (> %d): pass sort_scratch (n_entries int32)",
                max_gt, SMEM_MAX);
  int cap = 32;
  while (cap < max_gt && cap < SMEM_MAX) cap <<= 1;
  const int smem = cap * static_cast<int>(sizeof(int32_t));
  if (smem > 48 * 1024) {
    static bool attr_set[MAX_DEVICES] = {};
    const int dev = current_device();
    if (dev < 0) return fail(XMVE_ERR_DEVICE, "rank_metrics: no current device");
    if (!attr_set[dev]) {
      XMVE_CUDA(cudaFuncSetAttribute(rank_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     SMEM_MAX * static_cast<int>(sizeof(int32_t))));
      attr_set[dev] = true;
    }
  }
  rank_metrics_kernel<<<static_cast<unsigned>(n_query), 128, smem, static_cast<cudaStream_t>(stream)>>>(
      ranks, gt_off, n_mem, first_only, ap_k, cap, sort_scratch, best, ap,
      reinterpret_cast<unsigned long long*>(recall_counts), reinterpret_cast<unsigned long long*>(rank_sum), hist);
  return launch_status("rank_metrics_kernel");
}

namespace xmve {
namespace {
// acc = w * e (first) or acc + w * e, each operation rounded separately like NumPy's (no fused multiply-add)
template <typename T>
__global__ void __launch_bounds__(256)
fuse_kernel(T* __restrict__ acc, int64_t acc_ld, const T* __restrict__ e, int64_t e_ld, int64_t n_row, int64_t n_col,
            T w, int first) {
  const int64_t total = n_row * n_col;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / n_col, c = i % n_col;
    const T x = e[r * e_ld + c];
    T y;
    if (sizeof(T) == 8) {
      const double t = __dmul_rn(static_cast<double>(w), static_cast<double>(x));
      y = static_cast<T>(first ? t : __dadd_rn(static_cast<double>(acc[r * acc_ld + c]), t));
    } else {
      const float t = __fmul_rn(static_cast<float>(w), static_cast<float>(x));
      y = static_cast<T>(first ? t : __fadd_rn(static_cast<float>(acc[r * acc_ld + c]), t));
    }
    acc[r * acc_ld + c] = y;
  }
}
}  // namespace
}  // namespace xmve

extern "C" int xmve_fuse_accumulate(void* acc, int64_t acc_ld, const void* e, int64_t e_ld, int dtype, int64_t n_row,
                                    int64_t n_col, double w, int first, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(acc && e && n_row >= 0 && n_col >= 0 && acc_ld >= n_col && e_ld >= n_col, "fuse_accumulate: bad arguments");
  XMVE_REQUIRE(dtype == XMVE_F32 || dtype == XMVE_F64, "fuse_accumulate: dtype must be f32 or f64");
  if (n_row == 0 || n_col == 0) return XMVE_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = 8 * sm_count();
  if (dtype == XMVE_F32)
    fuse_kernel<float><<<grid, 256, 0, st>>>(static_cast<float*>(acc), acc_ld, static_cast<const float*>(e), e_ld, n_row,
                                             n_col, static_cast<float>(w), first);
  else
    fuse_kernel<double><<<grid, 256, 0, st>>>(static_cast<double*>(acc), acc_ld, static_cast<const double*>(e), e_ld,
                                              n_row, n_col, w, first);
  return launch_status("fuse_kernel");
}

extern "C" int xmve_norm_score(const void* errors, int dtype, int64_t n_row, int64_t n_col, int64_t ld, void* out,
                               int64_t out_ld, double* minmax_scratch, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(errors && out && minmax_scratch && n_row > 0 && n_col > 0 && ld >= n_col && out_ld >= n_col,
               "norm_score: bad arguments");
  XMVE_REQUIRE(dtype == XMVE_F32 || dtype == XMVE_F64, "norm_score: dtype must be f32 or f64");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(minmax_scratch);
  const int grid = 8 * sm_count();
  minmax_init_kernel<<<1, 1, 0, st>>>(keys);
  if (dtype == XMVE_F32) {
    minmax_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(errors), n_row, n_col, ld, keys);
    norm_apply_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(errors), n_row, n_col, ld,
                                                   static_cast<float*>(out), out_ld, keys);
  } else {
    minmax_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double*>(errors), n_row, n_col, ld, keys);
    norm_apply_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double*>(errors), n_row, n_col, ld,
                                                    static_cast<double*>(out), out_ld, keys);
  }
  return launch_status("norm_score kernels");
}
