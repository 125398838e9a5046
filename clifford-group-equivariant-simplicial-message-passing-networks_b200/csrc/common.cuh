// Shared helpers for the csmpn_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <stdio.h>

#include "../../include/csmpn_b200.h"
#include "algebra_gen.cuh"

namespace csmpn {

constexpr float kEps = 1e-6f;        // EPS of cegnn_utils.py:5
constexpr float kSmoothEps = 1e-16f; // eps of CliffordAlgebra._smooth_abs_sqrt (cliffordalgebra.py:148-149)

// last CUDA error text (per thread) for csmpn_last_cuda_error()
inline char* last_error_buf() {
  static thread_local char buf[256] = "";
  return buf;
}

// process-wide count of kernels launched by this library (bench.py reports it as gpu_launches)
unsigned long long& launch_counter();

inline int cuda_fail(cudaError_t e, const char* what) {
  snprintf(last_error_buf(), 256, "%s: %s", what, cudaGetErrorString(e));
  return CSMPN_ERR_CUDA;
}

#define CSMPN_CUDA_TRY(expr)                                  \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return ::csmpn::cuda_fail(_e, #expr); \
  } while (0)

// every kernel launch is followed by this macro: it also counts launches (csmpn_launch_count())
#define CSMPN_LAUNCH_CHECK(name)                              \
  do {                                                        \
    ++::csmpn::launch_counter();                              \
    cudaError_t _e = cudaGetLastError();                      \
    if (_e != cudaSuccess) return ::csmpn::cuda_fail(_e, name); \
  } while (0)

// Per-call metric description handed to kernels by value (lives in the constant bank).
struct MetricParams {
  float mf[32];  // indexed by BITMAP: product of metric entries over the set bits
  float qs[32];  // indexed by BLADE: beta_i * c[i,0,i]  (sign of x_i^2 in the quadratic form)
  int euclid;    // 1 if every metric entry is exactly 1
};

// Metric operand of the fused block kernels: the Euclidean instantiations (MET = false) take an empty struct whose
// null tables are never read (the generated products and the quadratic forms fold them out at compile time), the
// non-Euclidean ones take MetricParams by value.
struct NoMetric {
  static constexpr const float* mf = nullptr;
  static constexpr const float* qs = nullptr;
};
template <bool MET> struct MetricArgT { using type = NoMetric; };
template <> struct MetricArgT<true> { using type = MetricParams; };
template <bool MET> using MetricArg = typename MetricArgT<MET>::type;

// qs_i x_i (MET) or x_i: one factor of the quadratic-form term qs_i x_i^2 and of its derivative 2 qs_i x_i
template <bool MET>
__device__ __forceinline__ float qs_x(const float* qs, int i, float x) {
  if constexpr (MET) return qs[i] * x;
  else return x;
}

// bitmap of blade `idx` in short-lex order, host side
inline void host_blade_bitmaps(int dim, int* bitmap_of_index) {
  int n = 0;
  for (int g = 0; g <= dim; ++g) {
    // lexicographic order of ascending index tuples == ascending order of the bit-reversed... enumerate directly
    // combinations of size g of {0..dim-1} in lexicographic order
    int idx[8];
    for (int i = 0; i < g; ++i) idx[i] = i;
    while (true) {
      int bm = 0;
      for (int i = 0; i < g; ++i) bm |= 1 << idx[i];
      bitmap_of_index[n++] = bm;
      int i = g - 1;
      while (i >= 0 && idx[i] == dim - g + i) --i;
      if (i < 0) break;
      ++idx[i];
      for (int j = i + 1; j < g; ++j) idx[j] = idx[j - 1] + 1;
    }
  }
}

inline int make_metric_params(int dim, const float* metric, MetricParams* mp) {
  if (dim < 1 || dim > 5) return CSMPN_ERR_BAD_DIM;
  if (!metric) return CSMPN_ERR_BAD_ARG;
  int B = 1 << dim;
  memset(mp, 0, sizeof(*mp));
  mp->euclid = 1;
  for (int i = 0; i < dim; ++i)
    if (metric[i] != 1.0f) mp->euclid = 0;
  for (int bm = 0; bm < B; ++bm) {
    float f = 1.f;
    for (int v = 0; v < dim; ++v)
      if (bm >> v & 1) f *= metric[v];
    mp->mf[bm] = f;
  }
  int bitmaps[32];
  host_blade_bitmaps(dim, bitmaps);
  // beta_i * c[i,0,i] = beta_i * reorder_sign(b,b) * mf[b]; beta_i * reorder_sign(b,b) == +1 for every blade
  for (int i = 0; i < B; ++i) mp->qs[i] = mp->mf[bitmaps[i]];
  return CSMPN_OK;
}

// metric of a fused block call (csmpn_block_desc.metric, NULL = Euclidean): true, with *mp filled, when the
// non-Euclidean kernels must run
inline bool block_metric(int dim, const csmpn_block_desc& d, MetricParams* mp) {
  return d.metric && make_metric_params(dim, d.metric, mp) == CSMPN_OK && !mp->euclid;
}

// dispatch a runtime dim (1..5) to a compile-time template argument
#define CSMPN_DISPATCH_DIM(dim, D, ...)                  \
  switch (dim) {                                         \
    case 1: { constexpr int D = 1; __VA_ARGS__; } break; \
    case 2: { constexpr int D = 2; __VA_ARGS__; } break; \
    case 3: { constexpr int D = 3; __VA_ARGS__; } break; \
    case 4: { constexpr int D = 4; __VA_ARGS__; } break; \
    case 5: { constexpr int D = 5; __VA_ARGS__; } break; \
    default: return CSMPN_ERR_BAD_DIM;                   \
  }

// ---------------------------------------------------------------- device helpers
template <int N>
__device__ __forceinline__ void load_vec(float* dst, const float* __restrict__ src) {
  if constexpr (N % 4 == 0) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
      float4 v = *reinterpret_cast<const float4*>(src + 4 * q);
      dst[4 * q] = v.x; dst[4 * q + 1] = v.y; dst[4 * q + 2] = v.z; dst[4 * q + 3] = v.w;
    }
  } else if constexpr (N % 2 == 0) {
#pragma unroll
    for (int q = 0; q < N / 2; ++q) {
      float2 v = *reinterpret_cast<const float2*>(src + 2 * q);
      dst[2 * q] = v.x; dst[2 * q + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int q = 0; q < N; ++q) dst[q] = src[q];
  }
}

template <int N>
__device__ __forceinline__ void store_vec(float* __restrict__ dst, const float* src) {
  if constexpr (N % 4 == 0) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q)
      *reinterpret_cast<float4*>(dst + 4 * q) = make_float4(src[4 * q], src[4 * q + 1], src[4 * q + 2], src[4 * q + 3]);
  } else if constexpr (N % 2 == 0) {
#pragma unroll
    for (int q = 0; q < N / 2; ++q) *reinterpret_cast<float2*>(dst + 2 * q) = make_float2(src[2 * q], src[2 * q + 1]);
  } else {
#pragma unroll
    for (int q = 0; q < N; ++q) dst[q] = src[q];
  }
}

__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + expf(-v)); }

// (q^2 + 1e-16)^(1/4)   -- CliffordAlgebra._smooth_abs_sqrt
__device__ __forceinline__ float smooth_abs_sqrt(float q) { return sqrtf(sqrtf(fmaf(q, q, kSmoothEps))); }

// per-grade quadratic forms q_g = sum_{i in g} qs_i x_i^2   (cliffordalgebra.py:143-146)
template <int DIM>
__device__ __forceinline__ void grade_q(const float* x, const float* qs, float* q) {
  using A = Alg<DIM>;
#pragma unroll
  for (int g = 0; g < A::G; ++g) q[g] = 0.f;
#pragma unroll
  for (int i = 0; i < A::B; ++i) q[A::grade_of(i)] = fmaf(qs[i] * x[i], x[i], q[A::grade_of(i)]);
}

// ---------------------------------------------------------------- fixed-order reduction of per-CTA partials
// One job of final_reduce_kernel (tc_block_bwd.cu), the last kernel of both block engines' backward; a job with out =
// NULL is skipped (a gradient the caller does not want).
struct FinalJob {
  const float* in;   // partials
  float* out;
  int parts;         // number of partials
  int64_t stride;    // floats between partials
  int kind;          // 0: out[i] = sum in[p][i] (n = count);  1: weight gradient from [G][M][N] partials
  int n;             // kind 0: element count; kind 1: c_out * c_in * G
  int G, M, N, m0, co, ci;  // kind 1: out[((o0 + o)*ci_tot + i0 + i)*G + g] = sum_p in[p][(g*M + m0 + o)*N + i], i < ci
  int ci_tot, i0, o0;
};

// final_reduce_kernel over jobs[0, count), split into launches of at most kFinalJobs jobs each
int launch_final_reduce(const FinalJob* jobs, size_t count, cudaStream_t stream);

inline int sm_count_cached() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

}  // namespace csmpn
