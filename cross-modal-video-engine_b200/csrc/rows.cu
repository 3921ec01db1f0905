// K1: row normalise + cast.  HBM-bound: one warp per embedding row, the row is read from HBM once
// (the second pass hits L1/L2), norms are accumulated in fp64.
//
// Replaces evaluation.l2norm (LINAS-engine/evaluation.py:10-14), which cal_error re-runs over the
// whole corpus on every call (:19-20), F.normalize(index).float() (MultiFusion/src/validate.py:55)
// and Combiner.time_process (mean over frames, MultiFusion/src/combiner.py:140-143).
#include <cuda_bf16.h>

#include "common.cuh"

namespace xmve {
namespace {

constexpr int WARPS = 8;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// (frame-pooled) raw value of element i of one row, as fp32
template <typename T>
__device__ __forceinline__ float pooled(const T* __restrict__ r, int i, int d, int frames) {
  if (frames == 1) return static_cast<float>(r[i]);
  float s = 0.f;
  for (int f = 0; f < frames; ++f) s += static_cast<float>(r[static_cast<int64_t>(f) * d + i]);
  return s / static_cast<float>(frames);
}

__device__ __forceinline__ void write_planes(__nv_bfloat16* __restrict__ op, int i, int dpad, int layout, float y) {
  const __nv_bfloat16 hi = __float2bfloat16_rn(y);
  if (layout == XMVE_OP_X1) {
    op[i] = hi;
    return;
  }
  const __nv_bfloat16 lo = __float2bfloat16_rn(y - __bfloat162float(hi));
  op[i] = hi;
  if (layout == XMVE_OP_X3_QUERY) {          // [hi | hi | lo]
    op[dpad + i] = hi;
    op[2 * dpad + i] = lo;
  } else {                                   // [hi | lo | hi]
    op[dpad + i] = lo;
    op[2 * dpad + i] = hi;
  }
}

template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
prepare_rows_kernel(const T* __restrict__ src, int64_t n, int d, int frames, int64_t src_ld,
                    float* __restrict__ raw_out, int64_t raw_ld, int64_t raw_off, double* __restrict__ norm_out,
                    float* __restrict__ resid_out, __nv_bfloat16* __restrict__ op_out, int64_t op_ld, int64_t op_off, int layout, int dpad,
                    float weight, int norm_mode, int vec4) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const T* __restrict__ r = src + row * src_ld;
  float* __restrict__ raw = raw_out ? raw_out + row * raw_ld + raw_off : nullptr;

  double ss = 0.0;
  if (vec4) {                                // fp32, frames == 1, 16-byte aligned rows, d % 4 == 0
    const float4* r4 = reinterpret_cast<const float4*>(r);
    for (int i = lane; i < d / 4; i += 32) {
      const float4 x = r4[i];
      ss += static_cast<double>(x.x) * x.x + static_cast<double>(x.y) * x.y + static_cast<double>(x.z) * x.z +
            static_cast<double>(x.w) * x.w;
      if (raw) reinterpret_cast<float4*>(raw)[i] = x;
    }
  } else {
    for (int i = lane; i < d; i += 32) {
      const float x = pooled(r, i, d, frames);
      ss += static_cast<double>(x) * static_cast<double>(x);
      if (raw) raw[i] = x;
    }
  }
  ss = warp_sum(ss);
  const double nrm = sqrt(ss);
  if (lane == 0 && norm_out) norm_out[row] = nrm;
  if (op_out == nullptr) return;

  const double den = (norm_mode == XMVE_NORM_EPS) ? fmax(nrm, 1e-12) : nrm;
  __nv_bfloat16* __restrict__ op = op_out + row * op_ld + op_off;
  const int planes = (layout == XMVE_OP_X1) ? 1 : 3;
  double rs = 0.0;                           // || w * x_hat - bf16(w * x_hat) ||^2 of this row (x1 operand)
  for (int i = lane; i < d; i += 32) {
    const float x = pooled(r, i, d, frames);
    const double xd = static_cast<double>(x) / den;
    const float y = weight * static_cast<float>(xd);
    write_planes(op, i, dpad, layout, y);
    const double delta = static_cast<double>(weight) * xd - static_cast<double>(__bfloat162float(__float2bfloat16_rn(y)));
    rs += delta * delta;
  }
  if (resid_out != nullptr) {
    rs = warp_sum(rs);
    if (lane == 0) resid_out[row] = __double2float_ru(rs);
  }
  for (int pl = 0; pl < planes; ++pl)
    for (int i = d + lane; i < dpad; i += 32) op[pl * dpad + i] = __float2bfloat16_rn(0.f);
}

// Fast path (fp32 rows, d % 4 == 0, d <= 128 * MAXV, 16-byte aligned): the (frame-pooled) row lives in registers --
// MAXV independent 16-byte loads per lane up front, one pass over HBM in and out, 8-byte packed bf16 stores.  The
// scale is applied as a multiplication by 1/||x|| in double (identical to the division after rounding to float
// except within 2^-53 of a rounding boundary); the bf16 residual is accumulated in fp32 and inflated by 1e-3,
// which covers the fp32 roundings of y (2^-23 |y| against a residual of ~2^-9 |y|) -- it only has to be an upper
// bound.  The first version of K1 re-read the row element by element with a double division each: 3.3-3.8 TB/s.
template <int MAXV>
__global__ void __launch_bounds__(WARPS * 32)
prepare_rows_fast_kernel(const float* __restrict__ src, int64_t n, int d, int frames, int64_t src_ld,
                         float* __restrict__ raw_out, int64_t raw_ld, int64_t raw_off, double* __restrict__ norm_out,
                         float* __restrict__ resid_out, __nv_bfloat16* __restrict__ op_out, int64_t op_ld,
                         int64_t op_off, int layout, int dpad, float weight, int norm_mode) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const float4* __restrict__ r4 = reinterpret_cast<const float4*>(src + row * src_ld);
  const int n4 = d >> 2;                     // float4 per (pooled) row
  float4 v[MAXV];
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int i = lane + 32 * j;
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n4) {
      if (frames == 1) {
        v[j] = __ldcs(r4 + i);               // streamed: read exactly once
      } else {                               // Combiner.time_process: sum over the frames, then / frames
        float4 s = __ldcs(r4 + i);
        for (int f = 1; f < frames; ++f) {
          const float4 t = __ldcs(r4 + static_cast<int64_t>(f) * n4 + i);
          s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
        }
        const float fr = static_cast<float>(frames);
        v[j] = make_float4(s.x / fr, s.y / fr, s.z / fr, s.w / fr);
      }
    }
  }
  double ss = 0.0;
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    ss = fma(static_cast<double>(v[j].x), static_cast<double>(v[j].x), ss);
    ss = fma(static_cast<double>(v[j].y), static_cast<double>(v[j].y), ss);
    ss = fma(static_cast<double>(v[j].z), static_cast<double>(v[j].z), ss);
    ss = fma(static_cast<double>(v[j].w), static_cast<double>(v[j].w), ss);
  }
  if (raw_out != nullptr) {
    float4* __restrict__ raw4 = reinterpret_cast<float4*>(raw_out + row * raw_ld + raw_off);
#pragma unroll
    for (int j = 0; j < MAXV; ++j) {
      const int i = lane + 32 * j;
      if (i < n4) raw4[i] = v[j];
    }
  }
  ss = warp_sum(ss);
  const double nrm = sqrt(ss);
  if (lane == 0 && norm_out) norm_out[row] = nrm;
  if (op_out == nullptr) return;

  const double inv = 1.0 / ((norm_mode == XMVE_NORM_EPS) ? fmax(nrm, 1e-12) : nrm);
  __nv_bfloat16* __restrict__ op = op_out + row * op_ld + op_off;
  const int planes = (layout == XMVE_OP_X1) ? 1 : 3;
  float rs = 0.f;
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int i = lane + 32 * j;
    if (i < n4) {
      const float x[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
      __nv_bfloat16 hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float y = weight * static_cast<float>(static_cast<double>(x[e]) * inv);
        hi[e] = __float2bfloat16_rn(y);
        const float dlt = y - __bfloat162float(hi[e]);           // exact in fp32
        lo[e] = __float2bfloat16_rn(dlt);
        rs = fmaf(dlt, dlt, rs);
      }
      uint2 ph, pl;
      ph.x = static_cast<uint32_t>(__bfloat16_as_ushort(hi[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi[1])) << 16);
      ph.y = static_cast<uint32_t>(__bfloat16_as_ushort(hi[2])) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi[3])) << 16);
      *reinterpret_cast<uint2*>(op + 4 * i) = ph;
      if (planes == 3) {
        pl.x = static_cast<uint32_t>(__bfloat16_as_ushort(lo[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(lo[1])) << 16);
        pl.y = static_cast<uint32_t>(__bfloat16_as_ushort(lo[2])) | (static_cast<uint32_t>(__bfloat16_as_ushort(lo[3])) << 16);
        const bool q_side = layout == XMVE_OP_X3_QUERY;           // [hi | hi | lo]  vs  [hi | lo | hi]
        *reinterpret_cast<uint2*>(op + dpad + 4 * i) = q_side ? ph : pl;
        *reinterpret_cast<uint2*>(op + 2 * dpad + 4 * i) = q_side ? pl : ph;
      }
    }
  }
  for (int pl_ = 0; pl_ < planes; ++pl_)
    for (int i = d + lane; i < dpad; i += 32) op[pl_ * dpad + i] = __float2bfloat16_rn(0.f);
  if (resid_out != nullptr) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
    if (lane == 0) resid_out[row] = rs * 1.001f;
  }
}

template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
normalize_f64_kernel(const T* __restrict__ src, int64_t n, int d, int64_t src_ld, double* __restrict__ dst,
                     int64_t dst_ld, int norm_mode) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const T* __restrict__ r = src + row * src_ld;
  double ss = 0.0;
  for (int i = lane; i < d; i += 32) {
    const double x = static_cast<double>(r[i]);
    ss += x * x;
  }
  ss = warp_sum(ss);
  double nrm = sqrt(ss);
  if (norm_mode == XMVE_NORM_EPS) nrm = fmax(nrm, 1e-12);
  double* __restrict__ o = dst + row * dst_ld;
  for (int i = lane; i < d; i += 32) o[i] = static_cast<double>(r[i]) / nrm;   // 1.0 * X / norm
}

// One thread per column: its label is read once, then the column is masked in every row (grid-stride over rows).
template <typename T>
__global__ void __launch_bounds__(256)
mask_scores_kernel(T* __restrict__ scores, int64_t rows, int64_t cols, int64_t ld, const uint8_t* __restrict__ labels,
                   int64_t label_step, const uint64_t* __restrict__ allow) {
  const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const uint32_t lab = labels[c * label_step];
  for (int64_t r = blockIdx.y; r < rows; r += gridDim.y)
    if (((allow[r] >> lab) & 1ull) == 0) scores[r * ld + c] = -INFINITY;
}

}  // namespace
}  // namespace xmve

extern "C" int xmve_prepare_rows(const void* src, int src_dtype, int64_t n, int d, int frames, int64_t src_ld,
                                 float* raw_out, int64_t raw_ld, int64_t raw_off, double* norm_out, float* resid_out,
                                 void* op_out, int64_t op_ld, int64_t op_off, int op_layout, float weight,
                                 int norm_mode, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(src != nullptr && n >= 0 && d > 0 && frames >= 1, "prepare_rows: bad src / n / d / frames");
  XMVE_REQUIRE(src_ld >= static_cast<int64_t>(frames) * d, "prepare_rows: src_ld < frames * d");
  XMVE_REQUIRE(src_dtype == XMVE_F32 || src_dtype == XMVE_F64, "prepare_rows: src_dtype must be f32 or f64");
  XMVE_REQUIRE(op_layout >= XMVE_OP_X1 && op_layout <= XMVE_OP_X3_CORPUS, "prepare_rows: bad op_layout");
  const int dpad = (d + 63) / 64 * 64;
  const int planes = op_layout == XMVE_OP_X1 ? 1 : 3;
  XMVE_REQUIRE(op_out == nullptr || op_ld >= op_off + static_cast<int64_t>(planes) * dpad,
               "prepare_rows: operand row too short for %d plane(s) of %d", planes, dpad);
  XMVE_REQUIRE(raw_out == nullptr || raw_ld >= raw_off + d, "prepare_rows: raw row too short");
  XMVE_REQUIRE(resid_out == nullptr || op_out != nullptr, "prepare_rows: resid_out needs op_out");
  if (n == 0) return XMVE_OK;
  const unsigned grid = static_cast<unsigned>((n + WARPS - 1) / WARPS);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* op = static_cast<__nv_bfloat16*>(op_out);
  const bool fast = src_dtype == XMVE_F32 && d % 4 == 0 && d <= 2048 && src_ld % 4 == 0 && aligned16(src) &&
                    (raw_out == nullptr || (raw_ld % 4 == 0 && raw_off % 4 == 0 && aligned16(raw_out))) &&
                    (op_out == nullptr || (op_ld % 4 == 0 && op_off % 4 == 0 && dpad % 4 == 0 &&
                                           (reinterpret_cast<uintptr_t>(op_out) & 7u) == 0));
  if (fast) {
    const float* sp = static_cast<const float*>(src);
    if (d <= 1024)
      prepare_rows_fast_kernel<8><<<grid, WARPS * 32, 0, st>>>(sp, n, d, frames, src_ld, raw_out, raw_ld, raw_off,
                                                               norm_out, resid_out, op, op_ld, op_off, op_layout, dpad,
                                                               weight, norm_mode);
    else
      prepare_rows_fast_kernel<16><<<grid, WARPS * 32, 0, st>>>(sp, n, d, frames, src_ld, raw_out, raw_ld, raw_off,
                                                                norm_out, resid_out, op, op_ld, op_off, op_layout, dpad,
                                                                weight, norm_mode);
    return launch_status("prepare_rows_fast_kernel");
  }
  if (src_dtype == XMVE_F32) {
    const int vec4 = (frames == 1 && d % 4 == 0 && src_ld % 4 == 0 && aligned16(src) &&
                      (raw_out == nullptr || (raw_ld % 4 == 0 && raw_off % 4 == 0 && aligned16(raw_out))))
                         ? 1 : 0;
    prepare_rows_kernel<float><<<grid, WARPS * 32, 0, st>>>(static_cast<const float*>(src), n, d, frames, src_ld,
                                                            raw_out, raw_ld, raw_off, norm_out, resid_out, op, op_ld,
                                                            op_off, op_layout, dpad, weight, norm_mode, vec4);
  } else {
    prepare_rows_kernel<double><<<grid, WARPS * 32, 0, st>>>(static_cast<const double*>(src), n, d, frames, src_ld,
                                                             raw_out, raw_ld, raw_off, norm_out, resid_out, op, op_ld,
                                                             op_off, op_layout, dpad, weight, norm_mode, 0);
  }
  return launch_status("prepare_rows_kernel");
}

extern "C" int xmve_normalize_f64(const void* src, int src_dtype, int64_t n, int d, int64_t src_ld, double* dst,
                                  int64_t dst_ld, int norm_mode, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(src != nullptr && dst != nullptr && n >= 0 && d > 0 && src_ld >= d && dst_ld >= d,
               "normalize_f64: bad arguments");
  XMVE_REQUIRE(src_dtype == XMVE_F32 || src_dtype == XMVE_F64, "normalize_f64: src_dtype must be f32 or f64");
  if (n == 0) return XMVE_OK;
  const unsigned grid = static_cast<unsigned>((n + WARPS - 1) / WARPS);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_dtype == XMVE_F32)
    normalize_f64_kernel<float><<<grid, WARPS * 32, 0, st>>>(static_cast<const float*>(src), n, d, src_ld, dst,
                                                             dst_ld, norm_mode);
  else
    normalize_f64_kernel<double><<<grid, WARPS * 32, 0, st>>>(static_cast<const double*>(src), n, d, src_ld, dst,
                                                              dst_ld, norm_mode);
  return launch_status("normalize_f64_kernel");
}

extern "C" int xmve_mask_scores(void* scores, int dtype, int64_t rows, int64_t cols, int64_t ld,
                                const uint8_t* labels, int64_t label_step, const uint64_t* allow, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  XMVE_REQUIRE(scores != nullptr && labels != nullptr && allow != nullptr && rows >= 0 && cols >= 0 && ld >= cols &&
                   label_step >= 1,
               "mask_scores: bad arguments");
  XMVE_REQUIRE(dtype == XMVE_F32 || dtype == XMVE_F64, "mask_scores: dtype must be f32 or f64");
  if (rows == 0 || cols == 0) return XMVE_OK;
  const dim3 grid(static_cast<unsigned>((cols + 255) / 256), static_cast<unsigned>(rows < 65535 ? rows : 65535));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == XMVE_F32)
    mask_scores_kernel<float><<<grid, 256, 0, st>>>(static_cast<float*>(scores), rows, cols, ld, labels, label_step,
                                                    allow);
  else
    mask_scores_kernel<double><<<grid, 256, 0, st>>>(static_cast<double*>(scores), rows, cols, ld, labels,
                                                     label_step, allow);
  return launch_status("mask_scores_kernel");
}
