// Exact (double precision) scoring: the candidate rescore after the bf16 tensor-core filter pass,
// and a tiled fp64 score matrix for small problems.
//
// The reference's natural dtype on this path is float64: encode_vid / encode_text store fp32 model
// outputs into np.zeros (float64) arrays (LINAS-engine/evaluation.py:102-105,134,157) and cal_error
// normalises and multiplies them in double (:19-21).  Both kernels below reproduce that arithmetic
// (fp32-valued inputs, fp64 products and sums) up to summation order, which is what makes the
// returned top-k order and the ground-truth ranks identical to the reference's.
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"

namespace xmve {
namespace {

constexpr int RS_WARPS = 8;
constexpr int MAX_SPACES = 8;

struct SpaceDesc {
  int n_space;
  int off[MAX_SPACES + 1];
  double w[MAX_SPACES];
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// gridDim.y blocks per query row (more when there are few rows) share the row's candidate slots evenly.  A block
// works through its slots 1024 at a time in two phases: (A) all threads read the approximate scores, mark what is below
// the bound and COMPACT the slots that need an exact score into a shared-memory list (one shared-memory add per warp
// and 32 slots); (B) the warps take list entries round-robin, one warp-wide dot product each.  Without the list a
// warp owned 32 fixed slots and the rows to rescore -- one slot in ten, Poisson-distributed -- left some warps with
// twice the work of others; with 60 query rows (AVS) that imbalance was the kernel's duration.
// The query row is widened to fp64 ONCE into shared memory: the inner loop then costs one F2F (corpus element) and
// one DFMA per element -- the fp32->fp64 conversions, not HBM, were what bounded the first version (86 F2F vs 60 DFMA
// in its SASS, 3.2 TB/s of gather); four 16-byte loads per lane are kept in flight.
constexpr int RS_CHUNK = 1024;
__global__ void __launch_bounds__(RS_WARPS * 32, 6)
rescore_kernel(const float* __restrict__ q_raw, int64_t nq, int64_t q_ld, const double* __restrict__ q_norm,
               const float* __restrict__ v_raw, int64_t nv, int64_t v_ld, const double* __restrict__ v_norm,
               const __grid_constant__ SpaceDesc sp, int norm_mode, const float* __restrict__ cand_score,
               const int32_t* __restrict__ cand_idx, const int32_t* __restrict__ cand_count, int cap,
               const float* __restrict__ bound, const float* __restrict__ bound_hi, double* __restrict__ exact) {
  extern __shared__ __align__(16) double q_s[];
  __shared__ int todo_list[RS_CHUNK];                                // slots that need an exact score ...
  __shared__ int todo_row[RS_CHUNK];                                 // ... and their corpus rows
  __shared__ int todo_n;
  const int64_t q = blockIdx.x;
  const int dtot = sp.off[sp.n_space];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = min(cand_count[q], cap);
  // this block's share of the slots, in whole groups of 32
  const int per = ((n + 31) / 32 + static_cast<int>(gridDim.y) - 1) / static_cast<int>(gridDim.y) * 32;
  const int s0 = static_cast<int>(blockIdx.y) * per, s1 = min(n, s0 + per);
  if (s0 >= n) return;                                             // nothing for this block (uniform: before any barrier)
  for (int i = threadIdx.x; i < dtot; i += blockDim.x) q_s[i] = static_cast<double>(q_raw[q * q_ld + i]);
  const float bnd = bound ? bound[q] : -CUDART_INF_F;
  // second round: slots at or above bound_hi hold the exact scores of the first round and are left alone
  const float bnd_hi = bound_hi ? bound_hi[q] : CUDART_INF_F;
  const bool vec = (v_ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(v_raw) & 15u) == 0);
  for (int c0 = s0; c0 < s1; c0 += RS_CHUNK) {
    if (threadIdx.x == 0) todo_n = 0;
    __syncthreads();                                               // (also: q_s is complete)
    const int c1 = min(s1, c0 + RS_CHUNK);
    for (int base = c0 + warp * 32; base < c1; base += RS_WARPS * 32) {
      const int c = base + lane;                                   // slots >= n are never read downstream
      const float approx = c < c1 ? cand_score[q * cap + c] : -CUDART_INF_F;
      const bool mine = c < c1 && approx >= bnd && approx < bnd_hi;
      const int row = mine ? cand_idx[q * cap + c] : 0;
      if (c < c1 && approx < bnd) exact[q * cap + c] = -CUDART_INF;
      const unsigned m = __ballot_sync(0xffffffffu, mine);
      if (m != 0) {
        int pos = 0;
        if (lane == 0) pos = atomicAdd(&todo_n, __popc(m));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(m & ((1u << lane) - 1u));
        if (mine) {
          todo_list[pos] = c;
          todo_row[pos] = row;
        }
      }
    }
    __syncthreads();
    const int n_todo = todo_n;
    // One warp-wide dot product per list entry; the row number comes from the list (read coalesced in phase A) and
    // the row's norm is requested before the row, so the row data is the only dependent global load.  Variants
    // measured and not kept (profiles/r2_summary.md section 8): two rows per warp (-11 % at D = 2048, +5 % at
    // D = 640) and six or eight loads in flight per lane (+30 %: fewer resident warps, spilled registers).
    for (int e = warp; e < n_todo; e += RS_WARPS) {
      const int slot = todo_list[e];
      const int64_t v = todo_row[e];
      const float* __restrict__ vr = v_raw + v * v_ld;
      double res = 0.0;
      for (int s = 0; s < sp.n_space; ++s) {
        const int lo = sp.off[s], hi = sp.off[s + 1];
        double nvv = v_norm[static_cast<int64_t>(s) * nv + v];
        double nqv = q_norm[static_cast<int64_t>(s) * nq + q];
        double acc = 0.0;
        if (vec && (lo % 4 == 0) && ((hi - lo) % 4 == 0)) {
          const float4* v4 = reinterpret_cast<const float4*>(vr + lo);
          const double* qd = q_s + lo;
          const int n4 = (hi - lo) / 4;
          int i = lane;
          for (; i + 96 < n4; i += 128) {                      // 4 independent 16-byte loads in flight per lane
            const float4 b0 = __ldg(v4 + i), b1 = __ldg(v4 + i + 32), b2 = __ldg(v4 + i + 64), b3 = __ldg(v4 + i + 96);
            const double2 a00 = *reinterpret_cast<const double2*>(qd + 4 * i);
            const double2 a01 = *reinterpret_cast<const double2*>(qd + 4 * i + 2);
            const double2 a10 = *reinterpret_cast<const double2*>(qd + 4 * (i + 32));
            const double2 a11 = *reinterpret_cast<const double2*>(qd + 4 * (i + 32) + 2);
            const double2 a20 = *reinterpret_cast<const double2*>(qd + 4 * (i + 64));
            const double2 a21 = *reinterpret_cast<const double2*>(qd + 4 * (i + 64) + 2);
            const double2 a30 = *reinterpret_cast<const double2*>(qd + 4 * (i + 96));
            const double2 a31 = *reinterpret_cast<const double2*>(qd + 4 * (i + 96) + 2);
            acc = fma(a00.x, static_cast<double>(b0.x), acc);
            acc = fma(a00.y, static_cast<double>(b0.y), acc);
            acc = fma(a01.x, static_cast<double>(b0.z), acc);
            acc = fma(a01.y, static_cast<double>(b0.w), acc);
            acc = fma(a10.x, static_cast<double>(b1.x), acc);
            acc = fma(a10.y, static_cast<double>(b1.y), acc);
            acc = fma(a11.x, static_cast<double>(b1.z), acc);
            acc = fma(a11.y, static_cast<double>(b1.w), acc);
            acc = fma(a20.x, static_cast<double>(b2.x), acc);
            acc = fma(a20.y, static_cast<double>(b2.y), acc);
            acc = fma(a21.x, static_cast<double>(b2.z), acc);
            acc = fma(a21.y, static_cast<double>(b2.w), acc);
            acc = fma(a30.x, static_cast<double>(b3.x), acc);
            acc = fma(a30.y, static_cast<double>(b3.y), acc);
            acc = fma(a31.x, static_cast<double>(b3.z), acc);
            acc = fma(a31.y, static_cast<double>(b3.w), acc);
          }
          for (; i < n4; i += 32) {
            const float4 b0 = __ldg(v4 + i);
            const double2 a0 = *reinterpret_cast<const double2*>(qd + 4 * i);
            const double2 a1 = *reinterpret_cast<const double2*>(qd + 4 * i + 2);
            acc = fma(a0.x, static_cast<double>(b0.x), acc);
            acc = fma(a0.y, static_cast<double>(b0.y), acc);
            acc = fma(a1.x, static_cast<double>(b0.z), acc);
            acc = fma(a1.y, static_cast<double>(b0.w), acc);
          }
        } else {
          for (int i = lo + lane; i < hi; i += 32) acc = fma(q_s[i], static_cast<double>(vr[i]), acc);
        }
        acc = warp_sum(acc);
        if (norm_mode == XMVE_NORM_EPS) {
          nqv = fmax(nqv, 1e-12);
          nvv = fmax(nvv, 1e-12);
        }
        res += sp.w[s] * (acc / (nqv * nvv));
      }
      if (lane == 0) exact[q * cap + slot] = res;
    }
    __syncthreads();                                               // the list is reused by the next chunk
  }
}

// ---- tiled fp64 score matrix: out = alpha * A * B^T ----------------------------------------------
// 128 x 64 output tile, 256 threads with 8 x 4 outputs each (32 DFMA per 6 shared-memory loads of 16 bytes), the next
// k-slab is fetched into registers while the current one is multiplied.
constexpr int TM = 128, TN = 64, TK = 16;

__global__ void __launch_bounds__(256, 2)
score_f64_kernel(const double* __restrict__ a, int64_t nq, int64_t a_ld, const double* __restrict__ b, int64_t nv,
                 int64_t b_ld, int k, double alpha, double* __restrict__ out, int64_t out_ld) {
  __shared__ __align__(16) double as[TK][TM + 2];
  __shared__ __align__(16) double bs[TK][TN + 2];
  const int64_t q0 = static_cast<int64_t>(blockIdx.y) * TM, v0 = static_cast<int64_t>(blockIdx.x) * TN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  // global -> registers: A slab 128 x 16 (8 doubles per thread), B slab 64 x 16 (4 per thread); k fastest
  const int lr = threadIdx.x >> 2, lc = (threadIdx.x & 3) * 4;         // row 0..63, k offset 0,4,8,12
  double ra[2][4], rb[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int64_t r = q0 + lr + 64 * h;
        ra[h][e] = (r < nq && k0 + lc + e < k) ? a[r * a_ld + k0 + lc + e] : 0.0;
      }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t r = v0 + lr;
      rb[e] = (r < nv && k0 + lc + e < k) ? b[r * b_ld + k0 + lc + e] : 0.0;
    }
  };
  double acc[8][4] = {};
  fetch(0);
  for (int k0 = 0; k0 < k; k0 += TK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      as[lc + e][lr] = ra[0][e];
      as[lc + e][lr + 64] = ra[1][e];
      bs[lc + e][lr] = rb[e];
    }
    __syncthreads();
    if (k0 + TK < k) fetch(k0 + TK);                                    // in flight during the multiply
#pragma unroll
    for (int c = 0; c < TK; ++c) {
      double av[8], bv[4];
#pragma unroll
      for (int i = 0; i < 8; i += 2) {
        const double2 t = *reinterpret_cast<const double2*>(&as[c][ty * 8 + i]);
        av[i] = t.x;
        av[i + 1] = t.y;
      }
#pragma unroll
      for (int j = 0; j < 4; j += 2) {
        const double2 t = *reinterpret_cast<const double2*>(&bs[c][tx * 4 + j]);
        bv[j] = t.x;
        bv[j + 1] = t.y;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t q = q0 + ty * 8 + i, v = v0 + tx * 4 + j;
      if (q < nq && v < nv) out[q * out_ld + v] = alpha * acc[i][j];
    }
}

// ---- the same matrix on the FP64 tensor-core path (DMMA) -------------------------------------------------------
// mma.sync.m8n8k4.f64: one warp multiplies an 8 x 4 by a 4 x 8 fp64 tile (IEEE fused multiply-adds).  Block tile
// 128 queries x 64 corpus rows, 4 warps of 64 x 32 (8 x 4 MMA tiles, 64 accumulators per thread): per k-step of 4 a
// warp reads 12 doubles per lane for 32 MMAs -- 0.4 bytes of shared memory per FMA against 3 for the register-tiled
// FMA kernel above, which is what held that one at 17 TFLOP/s.  Operands arrive through a cp.async ring
// (16-byte copies, zero-filled past the matrix edges); rows are padded by 4 doubles so that the 8 x 4 fragment loads
// of a half-warp fall into 16 different bank pairs.
// Two shapes of the ring: <BK = 32, 2 stages> (default: half as many block barriers per flop; 2 x 54 KB per block, two
// blocks per SM) and <BK = 16, 3 stages> (XMVE_F64_BK=16).
constexpr int DM_BM = 128, DM_BN = 64;
template <int BK, int STAGES>
struct DmCfg {
  static constexpr int LD = BK + 4;                            // (BK + 4) % 16 == 4: conflict-free fragment loads
  static constexpr int STAGE_DOUBLES = (DM_BM + DM_BN) * LD;
  static constexpr int SMEM_BYTES = STAGES * STAGE_DOUBLES * 8;
  static constexpr int PIECES = BK / 2;                        // 16-byte pieces per row and k-block
  static constexpr int ROWS_PASS = 128 / PIECES;               // rows covered by the 128 threads in one pass
  static constexpr int A_PASSES = DM_BM / ROWS_PASS, B_PASSES = DM_BN / ROWS_PASS;
};

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma_884(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

template <int DM_BK, int DM_STAGES>
__global__ void __launch_bounds__(128, 2)
score_f64_mma_kernel(const double* __restrict__ a, int64_t nq, int64_t a_ld, const double* __restrict__ b, int64_t nv,
                     int64_t b_ld, int k, double alpha, double w, int fuse, double* __restrict__ out, int64_t out_ld) {
  // fuse: 0 -> out = alpha * S;  1 -> out = w * (alpha * S);  2 -> out = out + w * (alpha * S), every product and sum
  // rounded on its own (what NumPy's `acc + w * e` does): the multi-space fusion of section 8a row F in the epilogue
  using C = DmCfg<DM_BK, DM_STAGES>;
  constexpr int DM_LD = C::LD, DM_STAGE_DOUBLES = C::STAGE_DOUBLES;
  extern __shared__ __align__(16) double dm_smem[];
  const int64_t q0 = static_cast<int64_t>(blockIdx.y) * DM_BM, v0 = static_cast<int64_t>(blockIdx.x) * DM_BN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 1, wn = warp & 1;                     // 2 x 2 warps of 64 x 32
  const int n_kb = (k + DM_BK - 1) / DM_BK;

  // One k-block of both operands -> stage: (128 + 64) rows x BK/2 sixteen-byte pieces.  Piece `it` of a thread is
  // row it * ROWS_PASS + tid / PIECES (A rows first, B rows after) at the thread's FIXED k offset
  // c2 = 2 * (tid % PIECES): every address is a loop-invariant base plus it * (ROWS_PASS rows), so the producer costs
  // a handful of instructions per piece.  (The first version recomputed row / matrix / pointer per piece: 1.3 G integer
  // instructions against 1.1 G DMMAs, and the warps that feed the tensor pipe spent a third of their time there.)
  constexpr int RP = C::ROWS_PASS;
  const int r8 = threadIdx.x / C::PIECES, c2 = (threadIdx.x % C::PIECES) * 2;
  const double* a_src = a + (q0 + r8) * a_ld + c2;
  const double* b_src = b + (v0 + r8) * b_ld + c2;
  const int64_t a_step = RP * a_ld, b_step = RP * b_ld;
  // pieces whose row lies inside the matrix: it < a_rows_it (A), it < b_rows_it (B)
  int64_t a_it = (nq - q0 - r8 + RP - 1) / RP, b_it = (nv - v0 - r8 + RP - 1) / RP;
  const int a_rows_it = static_cast<int>(a_it < 0 ? 0 : (a_it > C::A_PASSES ? C::A_PASSES : a_it));
  const int b_rows_it = static_cast<int>(b_it < 0 ? 0 : (b_it > C::B_PASSES ? C::B_PASSES : b_it));
  const uint32_t smem0 = static_cast<uint32_t>(__cvta_generic_to_shared(dm_smem)) + (r8 * DM_LD + c2) * 8;
  auto load_stage = [&](int kb, int stage) {
    const int k0 = kb * DM_BK;
    const int left = k - k0 - c2;                               // doubles of this thread's column pair inside k
    const int kbytes = left >= 2 ? 16 : (left == 1 ? 8 : 0);
    const uint32_t dst0 = smem0 + stage * DM_STAGE_DOUBLES * 8;
    const double* pa = a_src + k0;
    const double* pb = b_src + k0;
#pragma unroll
    for (int it = 0; it < C::A_PASSES; ++it) {
      const int bytes = it < a_rows_it ? kbytes : 0;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + it * RP * DM_LD * 8),
                   "l"(bytes ? pa + it * a_step : a), "r"(bytes) : "memory");
    }
#pragma unroll
    for (int it = 0; it < C::B_PASSES; ++it) {
      const int bytes = it < b_rows_it ? kbytes : 0;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (DM_BM + it * RP) * DM_LD * 8),
                   "l"(bytes ? pb + it * b_step : b), "r"(bytes) : "memory");
    }
  };

  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < DM_STAGES - 1; ++s) {
    if (s < n_kb) load_stage(s, s);
    cp_async_commit();
  }
  for (int kb = 0; kb < n_kb; ++kb) {
    cp_async_wait<DM_STAGES - 2>();
    __syncthreads();                                           // stage kb has landed; stage kb-1 is free again
    if (kb + DM_STAGES - 1 < n_kb) load_stage(kb + DM_STAGES - 1, (kb + DM_STAGES - 1) % DM_STAGES);
    cp_async_commit();
    const double* as = dm_smem + (kb % DM_STAGES) * DM_STAGE_DOUBLES + (wm * 64 + (lane >> 2)) * DM_LD + (lane & 3);
    const double* bs = dm_smem + (kb % DM_STAGES) * DM_STAGE_DOUBLES + DM_BM * DM_LD + (wn * 32 + (lane >> 2)) * DM_LD +
                       (lane & 3);
#pragma unroll
    for (int kk = 0; kk < DM_BK; kk += 4) {
      double af[8], bf[4];
#pragma unroll
      for (int i = 0; i < 8; ++i) af[i] = as[i * 8 * DM_LD + kk];
#pragma unroll
      for (int j = 0; j < 4; ++j) bf[j] = bs[j * 8 * DM_LD + kk];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma_884(acc[i][j], af[i], bf[j]);
    }
  }
  cp_async_wait<0>();
  // C fragment: row = lane / 4, columns 2 * (lane % 4) + {0, 1}
  const bool vec = (out_ld % 2 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t q = q0 + wm * 64 + i * 8 + (lane >> 2);
    if (q >= nq) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t v = v0 + wn * 32 + j * 8 + (lane & 3) * 2;
      double* dst = out + q * out_ld + v;
      double e0 = __dmul_rn(alpha, acc[i][j][0]), e1 = __dmul_rn(alpha, acc[i][j][1]);
      if (fuse != 0) {
        e0 = __dmul_rn(w, e0);
        e1 = __dmul_rn(w, e1);
      }
      if (vec && v + 1 < nv) {
        if (fuse == 2) {
          const double2 old = *reinterpret_cast<const double2*>(dst);
          e0 = __dadd_rn(old.x, e0);
          e1 = __dadd_rn(old.y, e1);
        }
        *reinterpret_cast<double2*>(dst) = make_double2(e0, e1);
      } else {
        if (v < nv) dst[0] = fuse == 2 ? __dadd_rn(dst[0], e0) : e0;
        if (v + 1 < nv) dst[1] = fuse == 2 ? __dadd_rn(dst[1], e1) : e1;
      }
    }
  }
}

constexpr int PTM = 64, PTN = 64, PTK = 16;   // pairwise measures: 256 threads, 4 x 4 outputs each

// ---- non-cosine measures of cal_error (evaluation.py:22-35): tiled pairwise distances on the CUDA cores --------
// out[q, v] = alpha * f(a_q, b_v) + beta with f = sum|a-b| (L1), sqrt(sum (a-b)^2) (L2) or sum min / sum max (jaccard).
template <int MEASURE>
__global__ void __launch_bounds__(256)
pairwise_kernel(const double* __restrict__ a, int64_t nq, int64_t a_ld, const double* __restrict__ b, int64_t nv,
                int64_t b_ld, int k, double alpha, double beta, double* __restrict__ out, int64_t out_ld) {
  __shared__ double as[PTK][PTM + 1];
  __shared__ double bs[PTK][PTN + 1];
  const int64_t q0 = static_cast<int64_t>(blockIdx.y) * PTM, v0 = static_cast<int64_t>(blockIdx.x) * PTN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4] = {};
  double acc2[MEASURE == XMVE_MEASURE_JACCARD ? 4 : 1][4] = {};
  for (int k0 = 0; k0 < k; k0 += PTK) {
    for (int e = threadIdx.x; e < PTM * PTK; e += 256) {
      const int r = e / PTK, c = e % PTK;
      as[c][r] = (q0 + r < nq && k0 + c < k) ? a[(q0 + r) * a_ld + k0 + c] : 0.0;
      bs[c][r] = (v0 + r < nv && k0 + c < k) ? b[(v0 + r) * b_ld + k0 + c] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < PTK; ++c) {
      double av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        av[i] = as[c][ty * 4 + i];
        bv[i] = bs[c][tx * 4 + i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (MEASURE == XMVE_MEASURE_L1) {
            acc[i][j] += fabs(av[i] - bv[j]);
          } else if (MEASURE == XMVE_MEASURE_L2 || MEASURE == XMVE_MEASURE_SQL2) {
            const double t = av[i] - bv[j];
            acc[i][j] = fma(t, t, acc[i][j]);
          } else if (MEASURE == XMVE_MEASURE_DOT) {
            acc[i][j] = fma(av[i], bv[j], acc[i][j]);
          } else if (MEASURE == XMVE_MEASURE_ORDER) {
            const double t = fmax(bv[j] - av[i], 0.0);
            acc[i][j] = fma(t, t, acc[i][j]);
          } else {
            acc[i][j] += fmin(av[i], bv[j]);
            acc2[MEASURE == XMVE_MEASURE_JACCARD ? i : 0][j] += fmax(av[i], bv[j]);
          }
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t q = q0 + ty * 4 + i, v = v0 + tx * 4 + j;
      if (q < nq && v < nv) {
        double f = acc[i][j];
        if (MEASURE == XMVE_MEASURE_L2 || MEASURE == XMVE_MEASURE_ORDER) f = sqrt(f);
        if (MEASURE == XMVE_MEASURE_JACCARD) f = f / acc2[MEASURE == XMVE_MEASURE_JACCARD ? i : 0][j];
        out[q * out_ld + v] = alpha * f + beta;
      }
    }
}

}  // namespace
}  // namespace xmve

namespace xmve {
namespace {
// Triplet ranking cost of a square score matrix (LINAS-engine/loss.py:112-153): block i owns row i and column i.
//   cost_s [i, j] = max(0, margin + scores[i, j] - scores[i, i])   (compare the diagonal with its ROW:    v2t)
//   cost_im[i, j] = max(0, margin + scores[i, j] - scores[j, j])   (compare the diagonal with its COLUMN: t2v)
// with the diagonal cleared; max_violation keeps the largest entry of each row (cost_s) / column (cost_im).
// out[0] += sum over the kept cost_s entries, out[1] += the same for cost_im (fp64 atomics).
__global__ void __launch_bounds__(256)
triplet_cost_kernel(const double* __restrict__ scores, int64_t n, int64_t ld, double margin, int max_violation,
                    double* __restrict__ out) {
  __shared__ double red[2][8];
  const int64_t i = blockIdx.x;
  const double dii = scores[i * ld + i];
  double a_s = 0.0, a_im = 0.0;                                 // running sum or max (costs are >= 0)
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    if (j == i) continue;
    const double cs = fmax(margin + scores[i * ld + j] - dii, 0.0);                       // row i
    const double cm = fmax(margin + scores[j * ld + i] - dii, 0.0);                       // column i: diag of column i
    if (max_violation) { a_s = fmax(a_s, cs); a_im = fmax(a_im, cm); }
    else { a_s += cs; a_im += cm; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double t_s = __shfl_xor_sync(0xffffffffu, a_s, o), t_im = __shfl_xor_sync(0xffffffffu, a_im, o);
    if (max_violation) { a_s = fmax(a_s, t_s); a_im = fmax(a_im, t_im); }
    else { a_s += t_s; a_im += t_im; }
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a_s; red[1][threadIdx.x >> 5] = a_im; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) {
      if (max_violation) { a_s = fmax(a_s, red[0][w]); a_im = fmax(a_im, red[1][w]); }
      else { a_s += red[0][w]; a_im += red[1][w]; }
    }
    atomicAdd(&out[0], a_s);
    atomicAdd(&out[1], a_im);
  }
}
}  // namespace
}  // namespace xmve

extern "C" int xmve_triplet_cost(const double* scores, int64_t n, int64_t ld, double margin, int max_violation,
                                 double* out, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(scores && out && n >= 0 && ld >= n, "triplet_cost: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  XMVE_CUDA(cudaMemsetAsync(out, 0, 2 * sizeof(double), st));
  if (n == 0) return XMVE_OK;
  triplet_cost_kernel<<<static_cast<unsigned>(n), 256, 0, st>>>(scores, n, ld, margin, max_violation, out);
  return launch_status("triplet_cost_kernel");
}

extern "C" int xmve_pairwise_f64(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld,
                                 int k, int measure, double alpha, double beta, double* out, int64_t out_ld,
                                 void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(a && b && out && nq >= 0 && nv >= 0 && k > 0 && a_ld >= k && b_ld >= k && out_ld >= nv,
               "pairwise_f64: bad arguments");
  XMVE_REQUIRE(measure >= XMVE_MEASURE_L1 && measure <= XMVE_MEASURE_ORDER, "pairwise_f64: unknown measure %d", measure);
  if (nq == 0 || nv == 0) return XMVE_OK;
  dim3 grid(static_cast<unsigned>((nv + PTN - 1) / PTN), static_cast<unsigned>((nq + PTM - 1) / PTM));
  if (grid.y > 65535) return fail(XMVE_ERR_LIMIT, "pairwise_f64: more than %d query rows; chunk the call", 65535 * PTM);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (measure == XMVE_MEASURE_L1)
    pairwise_kernel<XMVE_MEASURE_L1><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  else if (measure == XMVE_MEASURE_L2)
    pairwise_kernel<XMVE_MEASURE_L2><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  else if (measure == XMVE_MEASURE_SQL2)
    pairwise_kernel<XMVE_MEASURE_SQL2><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  else if (measure == XMVE_MEASURE_DOT)
    pairwise_kernel<XMVE_MEASURE_DOT><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  else if (measure == XMVE_MEASURE_ORDER)
    pairwise_kernel<XMVE_MEASURE_ORDER><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  else
    pairwise_kernel<XMVE_MEASURE_JACCARD><<<grid, 256, 0, st>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, beta, out, out_ld);
  return launch_status("pairwise_kernel");
}

extern "C" int xmve_rescore(const float* q_raw, int64_t nq, int64_t q_ld, const double* q_norm, const float* v_raw,
                            int64_t nv, int64_t v_ld, const double* v_norm, int n_space, const int32_t* space_off,
                            const double* weights, int norm_mode, const float* cand_score, const int32_t* cand_idx,
                            const int32_t* cand_count, int32_t cap, const float* bound, const float* bound_hi,
                            double* exact, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(q_raw && q_norm && v_raw && v_norm && space_off && weights && cand_score && cand_idx && cand_count &&
                   exact, "rescore: null pointer");
  XMVE_REQUIRE(n_space >= 1 && n_space <= MAX_SPACES, "rescore: n_space must be in [1, %d]", MAX_SPACES);
  XMVE_REQUIRE(nq >= 0 && nv > 0 && cap > 0, "rescore: bad sizes");
  SpaceDesc sp;
  sp.n_space = n_space;
  for (int s = 0; s <= n_space; ++s) sp.off[s] = space_off[s];      // host arrays (tiny)
  for (int s = 0; s < n_space; ++s) {
    sp.w[s] = weights[s];
    XMVE_REQUIRE(sp.off[s + 1] > sp.off[s], "rescore: space offsets must increase");
  }
  const int dtot = sp.off[n_space];
  XMVE_REQUIRE(sp.off[0] == 0 && dtot <= q_ld && dtot <= v_ld, "rescore: offsets exceed the raw row length");
  if (dtot > 6000) return fail(XMVE_ERR_LIMIT, "rescore: total raw dim %d > 6000 (48 KB of shared memory)", dtot);
  if (nq == 0) return XMVE_OK;
  // few query rows (AVS: 60): split every row's candidates over several blocks so that all SMs gather
  // (blocks whose share of the row's actual candidate count is empty leave at once).  The grid is kept within ONE
  // wave of resident blocks: 900 blocks on 740 slots ran as 1.2 waves, i.e. at 60 % of the gather bandwidth.
  const size_t dyn_smem = dtot * sizeof(double);
  static int resident[MAX_DEVICES][2] = {};                         // per device: [dynamic bytes it was queried for, blocks]
  const int dev = current_device();
  if (dev < 0) return fail(XMVE_ERR_DEVICE, "rescore: no current device");
  if (resident[dev][1] == 0 || resident[dev][0] != static_cast<int>(dyn_smem)) {
    int per_sm = 0;
    // from about 5 000 dims the query row and the static lists exceed the 48 KB a launch gets without opting in
    XMVE_CUDA(cudaFuncSetAttribute(rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(dyn_smem)));
    XMVE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rescore_kernel, RS_WARPS * 32, dyn_smem));
    const int sms = sm_count();
    if (per_sm <= 0 || sms <= 0) return fail(XMVE_ERR_DEVICE, "rescore: cannot query the occupancy");
    resident[dev][0] = static_cast<int>(dyn_smem);
    resident[dev][1] = per_sm * sms;
  }
  int64_t split = resident[dev][1] / nq;
  if (split > 64) split = 64;
  if (split > (cap + RS_WARPS * 32 - 1) / (RS_WARPS * 32)) split = (cap + RS_WARPS * 32 - 1) / (RS_WARPS * 32);
  if (split < 1) split = 1;
  if (nq > 2147483647) return fail(XMVE_ERR_LIMIT, "rescore: too many query rows");
  const dim3 grid(static_cast<unsigned>(nq), static_cast<unsigned>(split));
  rescore_kernel<<<grid, RS_WARPS * 32, dyn_smem, static_cast<cudaStream_t>(stream)>>>(
      q_raw, nq, q_ld, q_norm, v_raw, nv, v_ld, v_norm, sp, norm_mode, cand_score, cand_idx, cand_count, cap, bound,
      bound_hi, exact);
  return launch_status("rescore_kernel");
}

namespace xmve {
namespace {
int launch_score_f64(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld, int k,
                     double alpha, double w, int fuse, double* out, int64_t out_ld, void* stream) {
  XMVE_REQUIRE(a && b && out && nq >= 0 && nv >= 0 && k > 0 && a_ld >= k && b_ld >= k && out_ld >= nv,
               "score_f64: bad arguments");
  if (nq == 0 || nv == 0) return XMVE_OK;
  dim3 grid(static_cast<unsigned>((nv + TN - 1) / TN), static_cast<unsigned>((nq + TM - 1) / TM));
  if (grid.y > 65535) return fail(XMVE_ERR_LIMIT, "score_f64: more than %d query rows; chunk the call", 65535 * TM);
  // FP64 tensor-core path: needs 16-byte aligned operand rows (cp.async); XMVE_F64_KERNEL=fma forces the FMA kernel
  const bool aligned = aligned16(a) && aligned16(b) && a_ld % 2 == 0 && b_ld % 2 == 0;
  const char* force = getenv("XMVE_F64_KERNEL");
  if (aligned && !(force != nullptr && force[0] == 'f')) {
    static bool attr_set[MAX_DEVICES] = {};
    const int dev = current_device();
    if (dev < 0) return fail(XMVE_ERR_DEVICE, "score_f64: no current device");
    if (!attr_set[dev]) {
      XMVE_CUDA(cudaFuncSetAttribute(score_f64_mma_kernel<32, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     DmCfg<32, 2>::SMEM_BYTES));
      XMVE_CUDA(cudaFuncSetAttribute(score_f64_mma_kernel<16, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     DmCfg<16, 3>::SMEM_BYTES));
      attr_set[dev] = true;
    }
    static_assert(DM_BM == TM && DM_BN == TN, "both fp64 kernels share one grid");
    const char* bk = getenv("XMVE_F64_BK");
    if (bk != nullptr && atoi(bk) == 16)
      score_f64_mma_kernel<16, 3><<<grid, 128, DmCfg<16, 3>::SMEM_BYTES, static_cast<cudaStream_t>(stream)>>>(
          a, nq, a_ld, b, nv, b_ld, k, alpha, w, fuse, out, out_ld);
    else
      score_f64_mma_kernel<32, 2><<<grid, 128, DmCfg<32, 2>::SMEM_BYTES, static_cast<cudaStream_t>(stream)>>>(
          a, nq, a_ld, b, nv, b_ld, k, alpha, w, fuse, out, out_ld);
    return launch_status("score_f64_mma_kernel");
  }
  if (fuse != 0) return fail(XMVE_ERR_ARG, "score_f64_fused: operand rows must be 16-byte aligned (even row strides)");
  score_f64_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a, nq, a_ld, b, nv, b_ld, k, alpha, out,
                                                                       out_ld);
  return launch_status("score_f64_kernel");
}
}  // namespace
}  // namespace xmve

extern "C" int xmve_score_f64(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld,
                              int k, double alpha, double* out, int64_t out_ld, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  return launch_score_f64(a, nq, a_ld, b, nv, b_ld, k, alpha, 1.0, 0, out, out_ld, stream);
}

extern "C" int xmve_score_f64_fused(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv,
                                    int64_t b_ld, int k, double alpha, double w, int first, double* out,
                                    int64_t out_ld, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  return launch_score_f64(a, nq, a_ld, b, nv, b_ld, k, alpha, w, first ? 1 : 2, out, out_ld, stream);
}
