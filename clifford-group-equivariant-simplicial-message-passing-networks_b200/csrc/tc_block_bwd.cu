// Tensor-core backward of one CEMLP block (autograd of cegnn_utils.py:180-207) for Euclidean Cl(2,0) / Cl(3,0).
//
// All intermediates are BPT tensors (tc_block.cuh).  Saved by the forward: y1 (pre-SiLU), y2 (post-SiLU), xr
// (pre-normalisation), o (pre-LayerNorm), and x0 (the assembled input row) when the input was not already BPT.
//
//   tc_b1_kernel  (FP32 pipe)   MVLayerNorm + weighted-geometric-product + normalisation adjoints:
//                               grad_y, o, xr, y2 -> d (grad of the product sum), dxr, dy2p; grads of la, wp, na, bl
//   tc_bgemm      (tensor pipe) dy2 = dy2p + d * WL + dxr * WR                     (K = 2C, transposed weights)
//   tc_b3_kernel  (FP32 pipe)   MVSiLU adjoint: dy2, y1 -> dy1; grads of sa, sb, b1
//   tc_bgemm      (tensor pipe) grad_x = dy1 * W1                                    (BPT or reference layout)
//   tc_dw_kernel  (tensor pipe) weight gradients [d | dxr]^T y2 and dy1^T x0: MN-major TF32 operands, K = rows,
//                               accumulated over blades of a grade and over all tiles of a CTA in TMEM
//   tc_final_kernel             fixed-order sum of the per-CTA partials -> reference parameter layouts
//
// The elementwise kernels keep one channel per thread for the whole kernel (warp = 4 channels x 8 rows), so every
// per-channel parameter gradient is a register accumulator and every BPT access of a warp is one 128-byte line.
#include <utility>
#include <vector>

#include "tc_block.cuh"

namespace csmpn {
namespace tcb {

// =====================================================================================================================
// B1 / B3: elementwise adjoints
struct EwArgs {
  int64_t rows;
  int tiles, C, Cp;
  const float* gy;  // grad_y: BPT [Cp] or reference layout [rows, C, B]
  int gy_bpt;
  const int32_t* gy_rows;  // reference layout only: block row r reads grad_y row gy_rows[r] (NULL: r) ...
  int64_t gy_stride;       // ... at this row pitch in floats (the aggregation's adjoint folded into the gather)
  const float *o, *xr, *y2, *y1, *dy2;
  const float *la, *wp, *na, *sa, *sb;
  float *d, *dxr, *dy2p, *dy1;
  float* partial;  // [grid][C][NP]
};

template <int DIM>
__device__ __forceinline__ void load_mv_bpt(float* v, const float* t, int Cp, int64_t tile, int c4, int r, int j) {
  constexpr int B = Alg<DIM>::B;
#pragma unroll
  for (int b = 0; b < B; ++b) v[b] = t[bpt_off(B, Cp, tile, b, c4, r) + j];
}
template <int DIM>
__device__ __forceinline__ void store_mv_bpt(float* t, const float* v, int Cp, int64_t tile, int c4, int r, int j) {
  constexpr int B = Alg<DIM>::B;
#pragma unroll
  for (int b = 0; b < B; ++b) t[bpt_off(B, Cp, tile, b, c4, r) + j] = v[b];
}

// ---- register-free prefetch: every thread streams ITS OWN elements of the next iteration into a private column of a
// shared-memory stage with 4-byte cp.async (LDGSTS), two stages deep, and reads them back with LDS.  No cross-thread
// traffic, so no barrier: cp.async.wait_group orders a thread's own copies.  The loads of iteration i+1 are in flight
// during the ~900 instructions of iteration i, which the 128-register budget (2 CTAs per SM) cannot do with registers.
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(dst_smem)), "l"(src) : "memory");
}
// Stage of one warp and one tensor: [blade][8 rows][4 channels] floats = the warp's 8 rows x 4 channels of an iteration.
// The warp fills it COOPERATIVELY with 16-byte copies (8 B copies per tensor, B / 4 per lane, a quarter of the 4-byte
// copies a thread-private stage needs: the kernel was throttled by its memory-instruction queue); thread (row rr,
// channel j) = lane 4 rr + j then reads word lane of every blade row.  Cross-lane: __syncwarp after cp.async.wait_group.
template <int DIM>
__device__ __forceinline__ void prefetch_mv_bpt(float* st, const float* t, int Cp, int64_t tile, int c4, int r0, int lane) {
  constexpr int B = Alg<DIM>::B;
#pragma unroll
  for (int k = lane; k < B * 8; k += 32) {
    const int b = k >> 3, row = k & 7;
    cp_async16(st + (b * 8 + row) * 4, t + bpt_off(B, Cp, tile, b, c4, r0 + row));
  }
}
template <int DIM>
__device__ __forceinline__ void read_stage(float* v, const float* st, int lane) {
#pragma unroll
  for (int b = 0; b < Alg<DIM>::B; ++b) v[b] = st[b * 32 + lane];
}

// CP (channel padding) is a template constant: thread count, BPT blade stride and stage strides become immediates, which
// removes the 64-bit address arithmetic (17 % of the executed instructions when they were runtime values).
// CP channels per CTA (CP * 8 threads); CPT = padded channel count of the tensors.  Wide blocks (CPT > CP = 64) run one
// CTA per (work unit, 64-channel slab = blockIdx.y); the row statistics of the layer norm need every channel, so each
// CTA walks phase 1 over all slabs and phase 2 over its own.
template <int DIM, int CP, int CPT>
__global__ void __launch_bounds__(CP * 8, CP <= 32 ? 2 : 1) tc_b1_kernel(EwArgs a) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, P = A::P, NP = P + G + 2;
  constexpr int NSLAB = CPT / CP;
  static_assert(CPT % CP == 0, "wide blocks are whole slabs");
  extern __shared__ float sm[];
  constexpr int nw = CP >> 2, nt = CP * 8;
  float* part1 = sm;                 // [nw][128]
  float* part2 = part1 + nw * kTile; // [nw][128]
  float* inv_mu_s = part2 + nw * kTile;
  float* dmu_s = inv_mu_s + kTile;
  float* stage = dmu_s + kTile;      // [2 stages][4 tensors][B][nt]
  const int tid = threadIdx.x, c4l = tid >> 5, lane = tid & 31, j = lane & 3, rr = lane >> 2;
  const int c4 = (NSLAB > 1 ? (int)blockIdx.y * nw : 0) + c4l;  // channel group of phase 2 (own slab)
  const int ch = c4 * 4 + j, C = a.C;
  constexpr int Cp = CPT;
  const bool ch_ok = ch < C;
  float la = ch_ok ? a.la[ch] : 0.f, wv[P], sn[G];
#pragma unroll
  for (int q = 0; q < P; ++q) wv[q] = ch_ok ? a.wp[ch * P + q] : 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) sn[g] = ch_ok ? sigmoidf_(a.na[ch * G + g]) : 0.f;
  float g_w[P], g_na[G], g_la = 0.f, g_bl = 0.f;
#pragma unroll
  for (int q = 0; q < P; ++q) g_w[q] = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) g_na[g] = 0.f;

  // iteration it of a unit: it < 8 -> phase 1 (row statistics: o, grad_y), it >= 8 -> phase 2 (adjoints: + y2, xr);
  // 8 rows of the unit per iteration
  constexpr int kIt = kTile / 16;
  constexpr int kIt1 = NSLAB * kIt;  // phase-1 iterations of a unit: 8 rows each, slab after slab
  // warp-private stages: [stage s][tensor][blade][8 rows][4 channels]
  float* stage_w = stage + (size_t)c4l * (2 * 4 * B * 32);
  auto stage_of = [&](int s, int tensor) { return stage_w + (size_t)(s * 4 + tensor) * B * 32; };
  auto prefetch = [&](int64_t unit, int it, int s) {
    const int64_t tile = unit >> 1;
    const int r0 = (int)(unit & 1) * (kTile / 2) + (it & (kIt - 1)) * 8, r = r0 + rr;
    const int c4x = it < kIt1 ? (it / kIt) * nw + c4l : c4;  // phase 1 walks every slab, phase 2 the own one
    const int chx = c4x * 4 + j;
    __syncwarp();  // every lane has finished reading this stage (iteration before last)
    prefetch_mv_bpt<DIM>(stage_of(s, 0), a.o, Cp, tile, c4x, r0, lane);
    if (a.gy_bpt) {
      prefetch_mv_bpt<DIM>(stage_of(s, 1), a.gy, Cp, tile, c4x, r0, lane);
    } else {
      float* dst = stage_of(s, 1) + lane;  // reference layout: every thread fetches its own multivector
      if (chx < C && tile * kTile + r < a.rows) {
        // the row indices of a tile are 512 contiguous bytes: L1 hits after the first touch of each line
        const int64_t grow = a.gy_rows ? (int64_t)__ldg(a.gy_rows + tile * kTile + r) : tile * kTile + r;
        const float* src = a.gy + (size_t)grow * a.gy_stride + (size_t)chx * B;
#pragma unroll
        for (int b = 0; b < B; ++b) cp_async4(dst + b * 32, src + b);
      } else {
#pragma unroll
        for (int b = 0; b < B; ++b) dst[b * 32] = 0.f;
      }
    }
    if (it >= kIt1) {
      prefetch_mv_bpt<DIM>(stage_of(s, 2), a.y2, Cp, tile, c4, r0, lane);
      prefetch_mv_bpt<DIM>(stage_of(s, 3), a.xr, Cp, tile, c4, r0, lane);
    }
    cp_async_commit();
  };

  // work unit = half a tile (64 rows): finer units balance the persistent CTAs when there are only a few tiles per SM
  const int64_t n_units = 2 * (int64_t)a.tiles;
  int seq = 0;  // global iteration counter of this thread: stage = seq & 1
  if ((int64_t)blockIdx.x < n_units) prefetch(blockIdx.x, 0, 0);
  for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
    const int64_t tile = unit >> 1;
    const int rbase = (int)(unit & 1) * (kTile / 2);
    const int64_t row0 = tile * kTile;
#pragma unroll 1
    for (int it = 0; it < kIt1 + kIt; ++it, ++seq) {
      // stream the next iteration (possibly the first one of this CTA's next unit), then wait for the current one
      if (it + 1 < kIt1 + kIt) prefetch(unit, it + 1, (seq + 1) & 1);
      else if (unit + gridDim.x < n_units) prefetch(unit + gridDim.x, 0, (seq + 1) & 1);
      else cp_async_commit();
      cp_async_wait<1>();
      __syncwarp();  // the copies of all lanes of this warp have landed
      const int s = seq & 1;
      const int r = rbase + (it & (kIt - 1)) * 8 + rr;
      const bool ok = ch_ok && row0 + r < a.rows;
      if (it < kIt1) {
        // ---- phase 1: row statistics of the layer norm (channel group of slab it / kIt)
        const int chx = ((it / kIt) * nw + c4l) * 4 + j;
        const bool okx = chx < C && row0 + r < a.rows;
        const float lax = NSLAB > 1 ? (chx < C ? a.la[chx] : 0.f) : la;
        float o[B], dy[B];
        read_stage<DIM>(o, stage_of(s, 0), lane);
        read_stage<DIM>(dy, stage_of(s, 1), lane);
        float dot = 0.f;
#pragma unroll
        for (int b = 0; b < B; ++b) dot = fmaf(dy[b], o[b], dot);
        float nu = okx ? fast_sas(mv_sumsq<DIM>(o)) : 0.f;
        float dt = okx ? lax * dot : 0.f;
        nu += __shfl_xor_sync(0xffffffffu, nu, 1); dt += __shfl_xor_sync(0xffffffffu, dt, 1);
        nu += __shfl_xor_sync(0xffffffffu, nu, 2); dt += __shfl_xor_sync(0xffffffffu, dt, 2);
        if (j == 0) {
          if (NSLAB > 1 && it >= kIt) { part1[c4l * kTile + r] += nu; part2[c4l * kTile + r] += dt; }
          else { part1[c4l * kTile + r] = nu; part2[c4l * kTile + r] = dt; }
        }
        if (it == kIt1 - 1) {
          __syncthreads();
          if (tid < kTile / 2) {
            const int r2 = rbase + tid;
            float s1 = 0.f, s2 = 0.f;
            for (int w = 0; w < nw; ++w) { s1 += part1[w * kTile + r2]; s2 += part2[w * kTile + r2]; }
            const float inv_mu = 1.f / (s1 / (float)C + kEps);
            inv_mu_s[r2] = inv_mu;
            dmu_s[r2] = -s2 * inv_mu * inv_mu / (float)C;
          }
          __syncthreads();
        }
        continue;
      }
      // ---- phase 2: adjoints
      float dd[B];
      {
        float o[B];
        read_stage<DIM>(o, stage_of(s, 0), lane);
        read_stage<DIM>(dd, stage_of(s, 1), lane);
        const float inv_mu = inv_mu_s[r];
        float dot = 0.f;
#pragma unroll
        for (int b = 0; b < B; ++b) dot = fmaf(dd[b], o[b], dot);
        if (ok) g_la = fmaf(dot, inv_mu, g_la);
        const float Q = mv_sumsq<DIM>(o);
        const float nu = fast_sas(Q);
        const float k1 = la * inv_mu * kInvSqrt2;
        const float k2 = dmu_s[r] * Q * fast_rcp(nu * nu * nu) * kInvSqrt2;
#pragma unroll
        for (int b = 0; b < B; ++b) dd[b] = ok ? fmaf(k1, dd[b], k2 * o[b]) : 0.f;  // d = do / sqrt2
      }
      store_mv_bpt<DIM>(a.d, dd, Cp, tile, c4, r, j);
      g_bl += dd[0];
      float y2[B], xr[B];
      read_stage<DIM>(y2, stage_of(s, 2), lane);
      read_stage<DIM>(xr, stage_of(s, 3), lane);
      float q[G], nrm[G], rinv[G], xn[B], dxn[B], dy2[B];
      norm_factors<DIM>(xr, sn, q, nrm, rinv);
#pragma unroll
      for (int b = 0; b < B; ++b) { xn[b] = xr[b] * rinv[A::grade_of(b)]; dy2[b] = 0.f; dxn[b] = 0.f; }
      A::template wgp_bwd<false>(y2, xn, wv, dd, nullptr, dy2, dxn, g_w);
      store_mv_bpt<DIM>(a.dy2p, dy2, Cp, tile, c4, r, j);
      float t[G], coef[G];
#pragma unroll
      for (int g = 0; g < G; ++g) t[g] = 0.f;
#pragma unroll
      for (int b = 0; b < B; ++b) t[A::grade_of(b)] = fmaf(dxn[b], xr[b], t[A::grade_of(b)]);
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const float ddn = -t[g] * rinv[g] * rinv[g];
        g_na[g] = fmaf(ddn * (nrm[g] - 1.f), sn[g] * (1.f - sn[g]), g_na[g]);
        coef[g] = ddn * sn[g] * q[g] * fast_rcp(nrm[g] * nrm[g] * nrm[g]);
      }
#pragma unroll
      for (int b = 0; b < B; ++b) dxn[b] = fmaf(dxn[b], rinv[A::grade_of(b)], coef[A::grade_of(b)] * xr[b]);
      store_mv_bpt<DIM>(a.dxr, dxn, Cp, tile, c4, r, j);
    }
  }
  cp_async_wait<0>();
  // ---- fixed-order reduction over the 8 row lanes of a channel, one partial per CTA
  auto red = [&](float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
  };
  float* out = a.partial + ((size_t)blockIdx.x * C + (ch_ok ? ch : 0)) * NP;
#pragma unroll
  for (int q = 0; q < P; ++q) { const float v = red(g_w[q]); if (rr == 0 && ch_ok) out[q] = v; }
#pragma unroll
  for (int g = 0; g < G; ++g) { const float v = red(g_na[g]); if (rr == 0 && ch_ok) out[P + g] = v; }
  { const float v = red(g_la); if (rr == 0 && ch_ok) out[P + G] = v; }
  { const float v = red(g_bl); if (rr == 0 && ch_ok) out[P + G + 1] = v; }
}

template <int DIM, int CP, int CPT>
__global__ void __launch_bounds__(CP * 8, CP <= 32 ? 2 : 1) tc_b3_kernel(EwArgs a) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, NP = 2 * G + 1;
  extern __shared__ float sm[];
  constexpr int nt = CP * 8;
  float* stage = sm;  // [2 stages][2 tensors][B][nt]
  const int tid = threadIdx.x, c4l = tid >> 5, lane = tid & 31, j = lane & 3, rr = lane >> 2;
  const int c4 = (CPT > CP ? (int)blockIdx.y * (CP >> 2) : 0) + c4l;  // wide blocks: 64-channel slab blockIdx.y
  const int ch = c4 * 4 + j, C = a.C;
  constexpr int Cp = CPT;
  const bool ch_ok = ch < C;
  float sa[G], sb[G], g_sa[G], g_sb[G], g_b1 = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    sa[g] = ch_ok ? a.sa[ch * G + g] : 0.f;
    sb[g] = ch_ok ? a.sb[ch * G + g] : 0.f;
    g_sa[g] = 0.f; g_sb[g] = 0.f;
  }
  constexpr int kIt = kTile / 16;
  float* stage_w = stage + (size_t)c4l * (2 * 2 * B * 32);
  auto stage_of = [&](int s, int tensor) { return stage_w + (size_t)(s * 2 + tensor) * B * 32; };
  auto prefetch = [&](int64_t unit, int it, int s) {
    const int64_t tile = unit >> 1;
    const int r0 = (int)(unit & 1) * (kTile / 2) + it * 8;
    __syncwarp();
    prefetch_mv_bpt<DIM>(stage_of(s, 0), a.y1, Cp, tile, c4, r0, lane);
    prefetch_mv_bpt<DIM>(stage_of(s, 1), a.dy2, Cp, tile, c4, r0, lane);
    cp_async_commit();
  };
  const int64_t n_units = 2 * (int64_t)a.tiles;
  int seq = 0;
  if ((int64_t)blockIdx.x < n_units) prefetch(blockIdx.x, 0, 0);
  for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
    const int64_t tile = unit >> 1;
    const int rbase = (int)(unit & 1) * (kTile / 2);
    const int64_t row0 = tile * kTile;
#pragma unroll 1
    for (int it = 0; it < kIt; ++it, ++seq) {
      if (it + 1 < kIt) prefetch(unit, it + 1, (seq + 1) & 1);
      else if (unit + gridDim.x < n_units) prefetch(unit + gridDim.x, 0, (seq + 1) & 1);
      else cp_async_commit();
      cp_async_wait<1>();
      __syncwarp();
      const int s = seq & 1;
      const int r = rbase + it * 8 + rr;
      const bool ok = ch_ok && row0 + r < a.rows;
      float y1[B], dy[B], sg[G], inv[G], t[G], ds[G];
      read_stage<DIM>(y1, stage_of(s, 0), lane);
      read_stage<DIM>(dy, stage_of(s, 1), lane);
      silu_gates<DIM>(y1, sa, sb, sg, inv);
#pragma unroll
      for (int g = 0; g < G; ++g) t[g] = 0.f;
#pragma unroll
      for (int b = 0; b < B; ++b) t[A::grade_of(b)] = fmaf(dy[b], y1[b], t[A::grade_of(b)]);
#pragma unroll
      for (int g = 0; g < G; ++g) {
        ds[g] = ok ? t[g] * sg[g] * (1.f - sg[g]) : 0.f;
        g_sa[g] = fmaf(ds[g], inv[g], g_sa[g]);
        g_sb[g] += ds[g];
      }
#pragma unroll
      for (int b = 0; b < B; ++b) {
        const int g = A::grade_of(b);
        const float dinv = (g == 0) ? 1.f : 2.f * y1[b];
        dy[b] = ok ? fmaf(sg[g], dy[b], ds[g] * sa[g] * dinv) : 0.f;
      }
      g_b1 += dy[0];
      store_mv_bpt<DIM>(a.dy1, dy, Cp, tile, c4, r, j);
    }
  }
  cp_async_wait<0>();
  auto red = [&](float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
  };
  float* out = a.partial + ((size_t)blockIdx.x * C + (ch_ok ? ch : 0)) * NP;
#pragma unroll
  for (int g = 0; g < G; ++g) { const float v = red(g_sa[g]); if (rr == 0 && ch_ok) out[g] = v; }
#pragma unroll
  for (int g = 0; g < G; ++g) { const float v = red(g_sb[g]); if (rr == 0 && ch_ok) out[G + g] = v; }
  { const float v = red(g_b1); if (rr == 0 && ch_ok) out[2 * G] = v; }
}

// =====================================================================================================================
// transposed-weight GEMM:  out[r, n] = addend[r, n] + sum_s sum_k src_s[r, k] * W_s[k, n]     (W_s global [K_s, N_s, G])
// The kernels index src / cp / w / wk with runtime values, so they take the arguments as __grid_constant__: without it
// nvcc copies the whole struct to a local-memory stack frame first.
struct GemmArgs {
  int64_t rows;
  int tiles;
  const float* src[2];  // BPT sources, channel padding cp[s], nk[s] K chunks each
  int cp[2], nk[2];
  const float* w[2];    // weights [wk[s]][wn][G] (c_out = K side, c_in = N side)
  int wk[2], wn;
  int n16;              // N padded to 16 (image rows)
  int kmax;             // max nk * 8 (image columns)
  const float* addend;  // BPT [n16] or NULL
  float* out;
  int out_bpt;          // 1: BPT [n16]; 0: reference layout [rows, wn, B]
  // streamed-weights mode (wide blocks): pre-split images in global memory, np = output channels per pass
  const float* wimg;
  int np;
};

// Store channel group gc4 of row r of `tile` to a.out: BPT (rows past the end as zeros) or the reference layout, one
// 32-byte store per (row, channel) when B == 8 and the output is 32-byte aligned (wide_ok).
template <int DIM>
__device__ __forceinline__ void store_gemm_group(const GemmArgs& a, const float (&v)[Alg<DIM>::B][4], int64_t tile, int gc4, int r,
                                                 bool wide_ok) {
  constexpr int B = Alg<DIM>::B;
  const int64_t row0 = tile * kTile;
  const bool row_ok = row0 + r < a.rows;
  if (a.out_bpt) {
#pragma unroll
    for (int b = 0; b < B; ++b) {
      float4 x = make_float4(v[b][0], v[b][1], v[b][2], v[b][3]);
      if (!row_ok) x = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(a.out + bpt_off(B, a.n16, tile, b, gc4, r)) = x;
    }
  } else if (row_ok) {
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int n = gc4 * 4 + jj;
      if (n >= a.wn) continue;
      float* dst = a.out + ((size_t)(row0 + r) * a.wn + n) * B;
      if constexpr (B == 8) {
        if (wide_ok) {
          float w8[8];
#pragma unroll
          for (int b = 0; b < 8; ++b) w8[b] = v[b][jj];
          st_global_v8(dst, w8);
          continue;
        }
      }
#pragma unroll
      for (int h = 0; h < B / 4; ++h)
        *reinterpret_cast<float4*>(dst + 4 * h) = make_float4(v[4 * h][jj], v[4 * h + 1][jj], v[4 * h + 2][jj], v[4 * h + 3][jj]);
    }
  }
}

// TERMS: numeric mode (tc_block.cuh, n_images)
template <int DIM, bool ST, int TERMS = 3>
__global__ void __launch_bounds__(kThreads, 1) tc_bgemm_kernel(const __grid_constant__ GemmArgs a) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, NI = n_images(TERMS);
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int nmax = ST ? a.np : (512 / B) / 16 * 16;            // output channels per pass (TMEM columns / blades)
  const uint32_t wunit = ST ? wunit_bytes<DIM>(nmax, NI) : 0u;
  const uint32_t half = B * kPS + wunit;
  const uint32_t img = ST ? (uint32_t)nmax * 32u : (uint32_t)a.n16 * a.kmax * 4;
  const uint32_t set_bytes = ST ? 0u : G * NI * img;
  uint8_t* wimg = smem + (size_t)kRing * half + B * kPS;
  const int nsets = a.src[1] ? 2 : 1;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wimg + (size_t)nsets * set_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
  Pipe p;
  p.init(smem, bars, half);
  const int npass = (a.n16 + nmax - 1) / nmax;
  const int nk = a.nk[0] + a.nk[1];
  const int per_tile = npass * nk;
  const int my_tiles = cta_tiles(a.tiles);
  auto load = [&](int qq) {
    // = cta_tile(qq / per_tile); called through the helper, nvcc gives tc_bgemm_kernel<3, true> 4 more registers
    const int64_t tile = (int64_t)blockIdx.x + (int64_t)(qq / per_tile) * gridDim.x;
    const int kc = (qq % per_tile) % nk;
    const int s = kc < a.nk[0] ? 0 : 1;
    if constexpr (ST) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.wimg) + (size_t)(qq % per_tile) * wunit;
      issue_chunk_load_w<B>(p, qq, a.src[s], a.cp[s], tile, s ? kc - a.nk[0] : kc, wsrc, wunit);
    } else {
      issue_chunk_load<B>(p, qq, a.src[s], a.cp[s], tile, s ? kc - a.nk[0] : kc);
    }
  };
  ChunkFeed<> feed{p, my_tiles * per_tile};
  int q = 0;
  if (warp == 0) feed.prime(load);
  const uint32_t tcols = tmem_cols((uint32_t)B * (a.n16 < nmax ? a.n16 : nmax));
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  if (!ST) {
    const WJob wj[2] = {{wimg, a.w[0], a.wk[0], a.wn, 0}, {wimg + set_bytes, a.w[nsets - 1], a.wk[nsets - 1], a.wn, 0}};
    stage_weight_jobs<DIM, true, 2, TERMS>(wj, nsets, img, a.n16, a.kmax, wimg, (uint32_t)nsets * set_bytes);
  }
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t lane_base = (warp & 3) * 32;
  const bool wide_ok = aligned32(a.out);
  for (int t = 0; t < my_tiles; ++t) {
    const int64_t tile = cta_tile(t);
    for (int ps = 0; ps < npass; ++ps) {
      const int n0 = ps * nmax;
      const int Np = (a.n16 - n0) < nmax ? (a.n16 - n0) : nmax;
      const uint32_t idesc = idesc_tf32(kTile, Np, false, false);
      for (int kc = 0; kc < nk; ++kc, ++q) {
        if (warp == 0) {  // issuer
          p.wait_full(q);
          feed.refill(q, load);
          if constexpr (ST) {
            p.wait_landed(q);  // the weight unit of this chunk
            issue_chunk_mma<DIM, TERMS>(p, q, tbase, Np, kc > 0, p.slot(q) + B * kPS, img, 0, 1, 0, nmax, 0, 0, idesc);
          } else {
            const int s = kc < a.nk[0] ? 0 : 1;
            issue_chunk_mma<DIM, TERMS>(p, q, tbase, Np, kc > 0, wimg, img, s, 1, set_bytes, a.n16, s ? kc - a.nk[0] : kc, n0, idesc);
          }
        } else {          // converters
          p.wait_landed(q);
          split_chunk<B, TERMS>(p, q);
        }
      }
      // ---- epilogue of this pass: output channels [n0, n0 + Np).  The addend rows of the first channel group are
      // requested before waiting for the MMAs, those of the next group while the current one is processed.
      const int r = lane_base + lane;
      float4 ad[B];
      if (a.addend && (warp >> 2) < (Np >> 2)) {
#pragma unroll
        for (int b = 0; b < B; ++b) ad[b] = *reinterpret_cast<const float4*>(a.addend + bpt_off(B, a.n16, tile, b, (n0 >> 2) + (warp >> 2), r));
      }
      p.wait_mmas(q - 1);
      if (warp == 0) feed.refill_all(q, load);
      for (int c4 = warp >> 2; c4 < (Np >> 2); c4 += 4) {
        float v[B][4];
#pragma unroll
        for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tbase, lane_base, b * Np + c4 * 4), v[b]);
        tmem_wait_ld();
        const int gc4 = (n0 >> 2) + c4;
        if (a.addend) {
#pragma unroll
          for (int b = 0; b < B; ++b) {
            v[b][0] += ad[b].x; v[b][1] += ad[b].y; v[b][2] += ad[b].z; v[b][3] += ad[b].w;
          }
          if (c4 + 4 < (Np >> 2)) {
#pragma unroll
            for (int b = 0; b < B; ++b) ad[b] = *reinterpret_cast<const float4*>(a.addend + bpt_off(B, a.n16, tile, b, gc4 + 4, r));
          }
        }
        store_gemm_group<DIM>(a, v, tile, gc4, r, wide_ok);
      }
      fence_before_sync();
    }
  }
  tmem_teardown(warp, tbase, tcols);
}

// =====================================================================================================================
// The same GEMM with an OVERLAPPED epilogue (resident weights, one pass, B * n16 <= 256 TMEM columns): accumulators
// alternate between two TMEM buffers by tile and the epilogue of tile t-1 runs as channel-group units between the chunks
// of tile t's K loop (PendingEpilogue, see tc_f1db_kernel).  Warp 0 issues; warps 1-15 convert; warps 4-15 own the
// epilogue.  Bit-identical outputs.
template <int DIM, int TERMS = 3>
__global__ void __launch_bounds__(kThreads, 1) tc_bgemmdb_kernel(const __grid_constant__ GemmArgs a) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, NI = n_images(TERMS);
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const uint32_t img = (uint32_t)a.n16 * a.kmax * 4;
  const uint32_t set_bytes = G * NI * img;
  uint8_t* wimg = smem + (kRing + 1) * B * kPS;
  const int nsets = a.src[1] ? 2 : 1;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wimg + (size_t)nsets * set_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
  Pipe p;
  p.init(smem, bars, B * kPS);
  const int nk = a.nk[0] + a.nk[1];
  const int my_tiles = cta_tiles(a.tiles);
  auto load = [&](int qq) {
    const int kc = qq % nk;
    const int s = kc < a.nk[0] ? 0 : 1;
    issue_chunk_load<B>(p, qq, a.src[s], a.cp[s], cta_tile(qq / nk), s ? kc - a.nk[0] : kc);
  };
  ChunkFeed<> feed{p, my_tiles * nk};
  int q = 0;
  if (warp == 0) feed.prime(load);
  const int Np = a.n16;
  const uint32_t bufcols = (uint32_t)B * Np;  // <= 256 (host)
  const uint32_t tcols = tmem_cols(2 * bufcols);
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  {
    const WJob wj[2] = {{wimg, a.w[0], a.wk[0], a.wn, 0}, {wimg + set_bytes, a.w[nsets - 1], a.wk[nsets - 1], a.wn, 0}};
    stage_weight_jobs<DIM, true, 2, TERMS>(wj, nsets, img, a.n16, a.kmax, wimg, (uint32_t)nsets * set_bytes);
  }
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t idesc = idesc_tf32(kTile, Np, false, false);
  const uint32_t lane_base = (warp & 3) * 32;
  const int r = lane_base + lane;
  const bool wide_ok = aligned32(a.out);
  const int n_c4 = Np >> 2;

  auto epilogue_unit = [&](int64_t tile, int c4, uint32_t tb) {
    float v[B][4];
#pragma unroll
    for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tb, lane_base, b * Np + c4 * 4), v[b]);
    if (a.addend) {
      float4 ad[B];
#pragma unroll
      for (int b = 0; b < B; ++b) ad[b] = *reinterpret_cast<const float4*>(a.addend + bpt_off(B, a.n16, tile, b, c4, r));
      tmem_wait_ld();
#pragma unroll
      for (int b = 0; b < B; ++b) {
        v[b][0] += ad[b].x; v[b][1] += ad[b].y; v[b][2] += ad[b].z; v[b][3] += ad[b].w;
      }
    } else {
      tmem_wait_ld();
    }
    store_gemm_group<DIM>(a, v, tile, c4, r, wide_ok);
  };
  PendingEpilogue pend;

  for (int t = 0; t < my_tiles; ++t) {
    const int64_t tile = cta_tile(t);
    const uint32_t tb = tbase + (uint32_t)(t & 1) * bufcols;
    for (int kc = 0; kc < nk; ++kc, ++q) {
      if (warp == 0) {  // issuer
        p.wait_full(q);
        feed.refill(q, load);
        const int s = kc < a.nk[0] ? 0 : 1;
        issue_chunk_mma<DIM, TERMS>(p, q, tb, Np, kc > 0, wimg, img, s, 1, set_bytes, a.n16, s ? kc - a.nk[0] : kc, 0, idesc);
      } else {
        p.wait_landed(q);
        split_chunk<B, TERMS>(p, q);
        pend.step(p, n_c4, epilogue_unit);
      }
    }
    pend.drain(p, n_c4, epilogue_unit);
    pend.start(warp, tile, q - 1, tb);
  }
  pend.drain(p, n_c4, epilogue_unit);
  tmem_teardown(warp, tbase, tcols);
}

// =====================================================================================================================
// weight-gradient GEMM:  D_g[m, n] += sum_{tiles, blades b of grade g, rows r} Acat[r, m, b] * Bsrc[r, n, b]
// Acat = channels of a0 followed by the channels of a1 (BPT, cpa each); operands MN-major (K = rows).
struct DwArgs {
  int64_t rows;
  int tiles;
  const float *a0, *a1, *bsrc;
  int cpa, cpb;   // channels of a0 / a1 and of bsrc used by this launch (multiples of 16)
  int cpa_total;  // channel padding of the a0 / a1 tensors
  int a_c4;       // first 4-channel group of a0 / a1 used by this launch
  int cpb_total;  // channel padding of the bsrc tensor
  int b_c4;       // first 4-channel group of bsrc used by this launch
  int M;          // 64 or 128, >= channels of Acat
  float* partial; // [grid][G][M][cpb]
  long long* dbg; // optional timeline buffer (csmpn_tc_debug_buffer): CTA 0, threads 0 (issuer) and 32 (converter)
};
long long*& debug_buffer();  // tc_block_fwd.cu
#ifdef CSMPN_DEBUG_TOOLS
#define DW_STAMP(code)                                                                       \
  do {                                                                                       \
    if (TL && a.dbg && blockIdx.x == 0 && (tid == 0 || tid == 32) && dbg_n < 250) {          \
      a.dbg[(tid ? 512 : 0) + 2 * dbg_n] = (code);                                           \
      a.dbg[(tid ? 512 : 0) + 2 * dbg_n + 1] = clock64();                                    \
      ++dbg_n;                                                                               \
    }                                                                                        \
  } while (0)
#else
#define DW_STAMP(code) do { } while (0)
#endif

// Step = (tile, blade, half of the tile's rows): 64 rows = 8 K steps.  A landing unit = (tile, blade) = two steps: the
// blade slabs of the operand tensors ([channels/4][128 rows][4], contiguous in a BPT tensor) arrive with 2-3 large bulk
// copies into one of kDwLand landing slots (the next unit loads while the current one is converted); a conversion pass
// splits a step into hi / lo and re-lays it out as [row][32 channels] operand groups (SWIZZLE_128B_BASE32B),
// double-buffered so that the conversion of step s+1 overlaps the MMAs of step s.
// TERMS = 1 (single-pass TF32): the conversion writes only the operands rounded to nearest TF32 (the hi groups; the lo
// groups keep the zeros of the prologue) and the issuer runs one MMA per K step (see `merged` for M = 64).
constexpr int kDwRows = 64;
constexpr int kDwLand = 2;                 // landing slots; a slot holds one (tile, blade) = both row halves = two steps
constexpr uint32_t kLand = kTile * 16;     // landing stride of one 4-channel column: [128 rows][4 channels], as in global memory

template <int DIM, bool TL, int TERMS = 3>
__global__ void __launch_bounds__(256, 1) tc_dw_kernel(DwArgs a) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  [[maybe_unused]] int dbg_n = 0;
  const int ca4 = a.cpa >> 2;
  const int na4 = (a.a1 ? 2 : 1) * ca4;  // 4-channel groups of Acat
  const int nb4 = a.cpb >> 2;
  const int n4 = na4 + nb4;
  const int ga = a.M / 32, gb = (a.cpb + 31) / 32;  // 32-channel operand groups
  const uint32_t grp = kDwRows * 128;               // bytes of one operand group [64 rows][32 ch]
  const uint32_t op_bytes = 2u * (ga + gb) * grp;   // one operand buffer: A hi, A lo, B hi, B lo
  uint8_t* ops = smem;                              // 2 operand buffers
  uint8_t* land = ops + 2 * (size_t)op_bytes;       // kDwLand landing slots
  const uint32_t land_bytes = (uint32_t)n4 * kLand;
  uint64_t* bars = reinterpret_cast<uint64_t*>(land + (size_t)kDwLand * land_bytes);
  // A (tile, blade) of a BPT tensor is contiguous ([channel/4][128 rows][4]), so a landing unit is 2-3 bulk copies of
  // 8-32 KB.  (cp.async.bulk is a uniform-datapath instruction: per-lane addresses are serialised at ~70 cycles per copy,
  // and the 24 one-KB copies per step of the first version took 72 % of the issuer's time.)
  uint64_t* load_bar = bars;                 // [kDwLand] the bulk copies of a step have landed
  uint64_t* op_bar = bars + kDwLand;         // [2] the MMAs reading an operand buffer have completed
  uint64_t* full_bar = bars + kDwLand + 2;   // [2] every converter warp has written its part of an operand buffer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kDwLand + 4);
  constexpr int kConvWarps = 7;              // warps 1..7 convert, warp 0 only issues copies and MMAs
  for (uint32_t i = tid; i < (2 * op_bytes) >> 4; i += 256) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tid == 0) {
    for (int i = 0; i < kDwLand + 2; ++i) mbar_init(&bars[i], 1);
    mbar_init(&full_bar[0], kConvWarps);
    mbar_init(&full_bar[1], kConvWarps);
    mbar_fence_init();
  }
  // M == 64 ("merged"): the hi and lo operand groups are contiguous in shared memory, so ONE instruction per K step of
  // shape 128 x (2 * 32 gb) x 8 multiplies [A_hi; A_lo] by [B_hi | B_lo] and yields all four split products at once
  // (lanes 0-63: A_hi rows, lanes 64-127: A_lo rows; first column half: B_hi, second: B_lo) instead of three M = 64
  // instructions.  The epilogue adds the two column halves and writes the two lane halves as two partials.
  // TERMS = 1 keeps the M = 128 instruction, now 128 x (32 gb) x 8 on [A; 0] x B: lanes 64-127 multiply the zero lo
  // groups and their partial is zero.  The M = 64 shape would read half the A rows, but its TMEM accumulator layout
  // differs from the M = 128 one every other kernel here uses; one instruction per K step either way.
  const bool merged = a.M == 64;
  const uint32_t ncol = merged ? (TERMS == 1 ? 1u : 2u) * gb * 32u : (uint32_t)a.cpb;  // accumulator columns per grade
  const uint32_t tcols = tmem_cols((uint32_t)G * ncol);
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t idesc = merged ? idesc_tf32(128, (int)ncol, true, true) : idesc_tf32(a.M, a.cpb, true, true);
  const int steps = cta_tiles(a.tiles) * B * 2;  // step = (tile, blade, row half)
  // The producer/issuer warp and the converter warps are decoupled by mbarriers (no CTA-wide barrier in the loop): the
  // conversion of step st+1 runs while warp 0 issues the MMAs of step st and the copies of step st+kDwLand.
  if (warp == 0) {
    const int units = steps >> 1;        // landing units = (tile, blade)
    auto issue = [&](int lu) {           // all lanes of warp 0
      const int64_t tile = cta_tile(lu / B);
      const int b = lu % B;
      uint8_t* dst = land + (size_t)(lu % kDwLand) * land_bytes;
      uint64_t* bar = &load_bar[lu % kDwLand];
      if (lane == 0) {
        mbar_arrive_expect_tx(bar, (uint32_t)n4 * kLand);
        bulk_g2s(dst, a.a0 + bpt_off(B, a.cpa_total, tile, b, a.a_c4, 0), (uint32_t)ca4 * kLand, bar);
        if (a.a1) bulk_g2s(dst + (size_t)ca4 * kLand, a.a1 + bpt_off(B, a.cpa_total, tile, b, a.a_c4, 0), (uint32_t)ca4 * kLand, bar);
        bulk_g2s(dst + (size_t)na4 * kLand, a.bsrc + bpt_off(B, a.cpb_total, tile, b, a.b_c4, 0), (uint32_t)nb4 * kLand, bar);
      }
      __syncwarp();
    };
    int loaded = 0;
    for (; loaded < kDwLand && loaded < units; ++loaded) issue(loaded);
    uint32_t grade_used = 0;
    for (int st = 0; st < steps; ++st) {
      const int b = (st >> 1) % B, g = A::grade_of(b);
      DW_STAMP(30);
      mbar_wait(&full_bar[st & 1], (st >> 1) & 1);
      fence_after_sync();
      DW_STAMP(31);
      const uint8_t* op_a = ops + (size_t)(st & 1) * op_bytes;
      const uint8_t* op_b = op_a + 2 * (size_t)ga * grp;
      const uint64_t a_hi = desc_mn32b(smem_addr(op_a), grp, 0), a_lo = a_hi + ((uint64_t)ga * grp >> 4);
      const uint64_t b_hi = desc_mn32b(smem_addr(op_b), grp, 0), b_lo = b_hi + ((uint64_t)gb * grp >> 4);
      const uint32_t dcol = tbase + (uint32_t)g * ncol;
      const uint32_t acc = (grade_used >> g) & 1;
      if (merged || TERMS == 1) {
#pragma unroll
        for (int ks = 0; ks < kDwRows / 8; ++ks) mma_tf32_w(dcol, a_hi + ks * 64, b_hi + ks * 64, idesc, ks == 0 ? acc : 1u);
      } else {
#pragma unroll
        for (int ks = 0; ks < kDwRows / 8; ++ks) {  // one K step = 8 rows = 1024 bytes = 64 descriptor units
          mma_tf32_w(dcol, a_hi + ks * 64, b_hi + ks * 64, idesc, ks == 0 ? acc : 1u);
          mma_tf32_w(dcol, a_hi + ks * 64, b_lo + ks * 64, idesc, 1);
          mma_tf32_w(dcol, a_lo + ks * 64, b_hi + ks * 64, idesc, 1);
        }
      }
      mma_commit_w(&op_bar[st & 1]);
      __syncwarp();
      DW_STAMP(32);
      // both row halves of the landing unit st >> 1 have been converted (full_bar observed above): refill its slot
      if ((st & 1) && loaded < units) { issue(loaded); ++loaded; }
      DW_STAMP(33);
      grade_used |= 1u << g;
    }
  } else {
    const int ct = tid - 32, nconv = kConvWarps * 32;
    for (int st = 0; st < steps; ++st) {
      const int lu = st >> 1, rh = st & 1;
      DW_STAMP(40);
      mbar_wait(&load_bar[lu % kDwLand], (lu / kDwLand) & 1);
      DW_STAMP(41);
      if (st >= 2) mbar_wait(&op_bar[st & 1], ((st - 2) >> 1) & 1);  // the MMAs of step st-2 released this operand buffer
      DW_STAMP(42);
      const uint8_t* src = land + (size_t)(lu % kDwLand) * land_bytes + (uint32_t)rh * (kDwRows * 16);
      uint8_t* op_a = ops + (size_t)(st & 1) * op_bytes;  // A hi groups, A lo groups
      uint8_t* op_b = op_a + 2 * (size_t)ga * grp;        // B hi groups, B lo groups
      // Item -> (column u, row r): every aligned group of 8 threads (one 128-bit shared-memory phase) takes rows
      // rb .. rb+7 of a column PAIR, four rows from each column.  The reads then cover eight distinct 16-byte bank
      // groups (r mod 8; columns are 2 KB apart) and so do the swizzled writes ((c/8 ^ r%4, c%8/4) differs in all 8).
      for (int it = ct; it < kDwRows * n4; it += nconv) {
        const int pr = it >> 7, w = it & 127, q = w & 7, g8 = w >> 3;
        const int swap = g8 >> 3, r = ((g8 & 7) << 3) + q;
        const int u = 2 * pr + ((q >> 2) ^ swap);
        const float4 x = *reinterpret_cast<const float4*>(src + (uint32_t)u * kLand + r * 16);
        const bool isb = u >= na4;
        const int cc = (isb ? u - na4 : u) * 4;  // channel inside its operand
        uint8_t* base = isb ? op_b : op_a;
        const int ng = isb ? gb : ga;
        const uint32_t off = (uint32_t)(cc >> 5) * grp + mn32b_off(r, cc & 31);
        if constexpr (TERMS == 1) {
          *reinterpret_cast<float4*>(base + off) = tf32_rna4(x);
        } else {
          float4 h, l;
          split4(x, h, l);
          *reinterpret_cast<float4*>(base + off) = h;
          *reinterpret_cast<float4*>(base + (size_t)ng * grp + off) = l;
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full_bar[st & 1]);
      DW_STAMP(43);
    }
  }
  uint32_t grade_used = 0;
  for (int st = 0; st < steps; ++st) grade_used |= 1u << A::grade_of((st >> 1) % B);
  if (steps > 0) mbar_wait(&op_bar[(steps - 1) & 1], ((steps - 1) >> 1) & 1);
  fence_after_sync();
  // ---- epilogue: D_g -> per-CTA partial [G][M][cpb]; grades this CTA never touched are written as zeros
  if (warp < 4 && merged) {
    // lane R = 32 warp + lane: rows R < 64 are A_hi products, R >= 64 A_lo products -> partial 2 * blockIdx + (R >> 6)
    const int R = warp * 32 + lane, m = R & 63;
    float* out = a.partial + ((size_t)blockIdx.x * 2 + (R >> 6)) * G * 64 * a.cpb;
    for (int g = 0; g < G; ++g) {
      const bool used = steps > 0 && ((grade_used >> g) & 1);
      for (int n = 0; n < a.cpb; n += 4) {
        float v[4] = {0.f, 0.f, 0.f, 0.f}, w[4] = {0.f, 0.f, 0.f, 0.f};
        if (used) {
          tmem_ld4(tmem_at(tbase, warp * 32, g * ncol + n), v);
          if (TERMS == 3) tmem_ld4(tmem_at(tbase, warp * 32, g * ncol + gb * 32 + n), w);
          tmem_wait_ld();
        }
        *reinterpret_cast<float4*>(out + ((size_t)g * 64 + m) * a.cpb + n) = make_float4(v[0] + w[0], v[1] + w[1], v[2] + w[2], v[3] + w[3]);
      }
    }
  } else if (warp < 4) {
    float* out = a.partial + (size_t)blockIdx.x * G * a.M * a.cpb;
    const int m = warp * 32 + lane;
    for (int g = 0; g < G; ++g) {
      const bool used = steps > 0 && ((grade_used >> g) & 1);
      for (int n = 0; n < a.cpb; n += 4) {
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (used) {
          tmem_ld4(tmem_at(tbase, warp * 32, g * a.cpb + n), v);
          tmem_wait_ld();
        }
        *reinterpret_cast<float4*>(out + ((size_t)g * a.M + m) * a.cpb + n) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  }
  tmem_teardown(warp, tbase, tcols);
}

// =====================================================================================================================
// fixed-order reduction of per-CTA partials
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
constexpr int kFinalJobs = 14;
struct FinalJobs { FinalJob j[kFinalJobs]; int count; };

// 16 consecutive elements per CTA x 16 partial groups: thread (e, pg) sums partials pg, pg+16, ... in order (independent
// loads, 64 contiguous bytes per partial row), then the 16 group sums are combined in a fixed order (bit-reproducible).
// Elements are enumerated in SOURCE order (i fastest).
__global__ void __launch_bounds__(256) tc_final_kernel(FinalJobs jobs) {
  __shared__ float red[16][17];
  const int e = threadIdx.x & 15, pg = threadIdx.x >> 4;
  int64_t idx = (int64_t)blockIdx.x * 16 + e;
  float s = 0.f;
  float* outp = nullptr;
  for (int k = 0; k < jobs.count; ++k) {
    const FinalJob& jb = jobs.j[k];
    if (idx < jb.n) {
      if (jb.out) {
        size_t src, dst;
        if (jb.kind == 0) {
          src = dst = (size_t)idx;
        } else {
          const int i = (int)(idx % jb.ci), o = (int)((idx / jb.ci) % jb.co), g = (int)(idx / ((int64_t)jb.ci * jb.co));
          src = ((size_t)g * jb.M + jb.m0 + o) * jb.N + i;
          dst = ((size_t)(jb.o0 + o) * jb.ci_tot + jb.i0 + i) * jb.G + g;
        }
        const float* in = jb.in + src;
#pragma unroll 4
        for (int p = pg; p < jb.parts; p += 16) s += in[(size_t)p * jb.stride];
        outp = jb.out + dst;
      }
      break;
    }
    idx -= jb.n;
  }
  red[pg][e] = s;
  __syncthreads();
  if (pg == 0 && outp) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) t += red[i][e];
    *outp = t;
  }
}

// =====================================================================================================================
// host side
template <int DIM>
size_t gemm_smem(int nsets, int n16, int kmax, int nimg = 2) {
  constexpr int B = Alg<DIM>::B, G = Alg<DIM>::G;
  const size_t s = (size_t)(kRing + 1) * B * kPS + (size_t)nsets * G * nimg * n16 * kmax * 4 + 128;
  return nimg == 2 ? s : one_cta_per_sm(s);
}
template <int DIM>
size_t dw_smem(int M, int na4, int cpb) {
  const int ga = M / 32, gb = (cpb + 31) / 32;
  return (size_t)2 * 2 * (ga + gb) * kDwRows * 128 + (size_t)kDwLand * (na4 + cpb / 4) * kLand + 128;  // kLand = 2 KB
}

struct BwdPlan {
  int Cp, cin, n16, tiles;
  int grid_ew, grid_dw;
  int M1, M2;  // dW GEMM heights: [d|dxr] and dy1
  int nbw;       // input channels per column pass of the W1 gradient (64 or 32)
  int dw_split;  // the [d|dxr] weight-gradient GEMM does not fit shared memory as one job: run d and dxr separately
  // wide blocks (the resident plan does not fit): GEMM weights streamed with the K chunks in passes of np output channels;
  // weight gradients as one launch per (64-channel slab of d / dxr / dy1, 32-channel slab of y2 / x0)
  int wide, np, n_dwa, n_dwb;
  int64_t img_dy2, img_gx;  // floats of the pre-split weight images of the two GEMMs
  size_t dw_part;           // floats of the partials of one slab launch
  // workspace layout (float offsets)
  size_t o_d, o_dxr, o_dy2p, o_dy2, o_dy1, o_p1, o_p3, o_dwa, o_dwb, o_img, total;
};
constexpr int kSlabA = 64, kSlabB = 32;  // wide weight-gradient launches: A rows (merged M = 64) x B columns
template <int DIM>
size_t gemm_smem_streamed(int np, int nimg = 2) {
  constexpr int B = Alg<DIM>::B;
  const size_t s = (size_t)kRing * (B * kPS + wunit_bytes<DIM>(np, nimg)) + (size_t)B * kPS + 128;
  return nimg == 2 ? s : one_cta_per_sm(s);
}

// The plan is chosen for the default (split) weight images, so both numeric modes run a shape the same way;
// single-pass TF32 (d.tf32) only halves the streamed image buffers.
template <int DIM>
int make_bwd_plan(const csmpn_block_desc& d, BwdPlan* p) {
  constexpr int B = Alg<DIM>::B, G = Alg<DIM>::G, P = Alg<DIM>::P;
  p->Cp = round_up(d.c, 16);
  p->cin = d.c0 + d.c1 + d.c2;
  p->n16 = round_up(p->cin, 16);
  p->tiles = (int)((d.rows + kTile - 1) / kTile);
  p->wide = 0; p->np = 0; p->n_dwa = p->n_dwb = 0; p->img_dy2 = p->img_gx = 0; p->dw_part = 0;
  const int sms = sm_count_cached();
  p->grid_ew = 2 * p->tiles < 2 * sms ? (p->tiles > 0 ? 2 * p->tiles : 1) : 2 * sms;
  p->grid_dw = p->tiles < sms ? (p->tiles > 0 ? p->tiles : 1) : sms;
  bool resident = 2 * B * p->Cp <= 512 && p->Cp <= 64;
  if (resident) {
    p->M1 = 2 * p->Cp <= 64 ? 64 : 128;
    p->M2 = 64;
    p->dw_split = 0;
    if (dw_smem<DIM>(p->M1, 2 * p->Cp / 4, p->Cp) > kSmemMax) { p->dw_split = 1; p->M1 = 64; }
    if (gemm_smem<DIM>(2, p->Cp, p->Cp) > kSmemMax || gemm_smem<DIM>(1, p->n16, p->Cp) > kSmemMax) resident = false;
  }
  if (resident) {
    // the W1 gradient runs in column passes of <= nbw input channels
    p->nbw = dw_smem<DIM>(p->M2, p->Cp / 4, p->n16 < 64 ? p->n16 : 64) <= kSmemMax ? 64 : 32;
    const int nb = p->n16 < p->nbw ? p->n16 : p->nbw;
    if (dw_smem<DIM>(p->M1, (p->dw_split ? 1 : 2) * p->Cp / 4, p->Cp) > kSmemMax || dw_smem<DIM>(p->M2, p->Cp / 4, nb) > kSmemMax ||
        p->n16 > 4 * p->nbw)
      resident = false;
  }
  if (!resident) {
    // wide plan: elementwise kernels exist for Cp <= 64 and for whole 64-channel slabs up to 256
    if (!(p->Cp <= 64 || p->Cp == 128 || p->Cp == 256)) return CSMPN_ERR_UNSUPPORTED;
    p->wide = 1;
    p->np = (512 / B) / 16 * 16;
    if (gemm_smem_streamed<DIM>(p->np) > kSmemMax || dw_smem<DIM>(kSlabA, kSlabA / 4, kSlabB) > kSmemMax) return CSMPN_ERR_UNSUPPORTED;
    const int sa = (p->Cp + kSlabA - 1) / kSlabA;
    p->n_dwa = 2 * sa * ((p->Cp + kSlabB - 1) / kSlabB);
    p->n_dwb = sa * ((p->n16 + kSlabB - 1) / kSlabB);
    p->dw_part = (size_t)p->grid_dw * 2 * G * kSlabA * kSlabB;
    const int nimg = d.tf32 ? 1 : 2;
    p->img_dy2 = weight_image_floats<DIM>(0, p->np, (p->Cp + p->np - 1) / p->np, 2 * (p->Cp / 8), nimg);
    p->img_gx = weight_image_floats<DIM>(0, p->np, (p->n16 + p->np - 1) / p->np, p->Cp / 8, nimg);
  }
  const size_t t = (size_t)bpt_floats(B, d.rows, p->Cp);
  size_t o = 0;
  p->o_d = o; o += t;
  p->o_dxr = o; o += t;
  p->o_dy2p = o; o += t;
  p->o_dy2 = o; o += t;
  p->o_dy1 = o; o += t;
  auto al = [](size_t x) { return (x + 31) / 32 * 32; };  // keep every segment 128-byte aligned
  p->o_p1 = o; o = al(o + (size_t)p->grid_ew * d.c * (P + G + 2));
  p->o_p3 = o; o = al(o + (size_t)p->grid_ew * d.c * (2 * G + 1));
  // M == 64 launches write two partials per CTA (hi and lo operand halves, see tc_dw_kernel)
  if (p->wide) {
    p->o_dwa = o; o += (size_t)p->n_dwa * p->dw_part;
    p->o_dwb = o; o += (size_t)p->n_dwb * p->dw_part;
    p->o_img = o; o += (size_t)((p->img_dy2 + 31) / 32 * 32 + (p->img_gx + 31) / 32 * 32);
  } else {
    p->o_dwa = o; o += (size_t)p->grid_dw * (p->M1 == 64 ? 2 : 1) * G * p->M1 * p->Cp * (p->dw_split ? 2 : 1);
    p->o_dwb = o; o += (size_t)p->grid_dw * 2 * G * p->M2 * p->n16;
    p->o_img = o;
  }
  p->total = o;
  return CSMPN_OK;
}

// TERMS: numeric mode (csmpn_block_desc.tf32 = 1 -> 1, else 3); the elementwise kernels do not depend on it
template <int DIM, int TERMS>
int launch_bwd(const csmpn_block_desc& d, const csmpn_block_grads& g, void* workspace, int64_t bytes, cudaStream_t stream) {
  constexpr int B = Alg<DIM>::B, G = Alg<DIM>::G, P = Alg<DIM>::P, NI = n_images(TERMS);
  BwdPlan p;
  int st = make_bwd_plan<DIM>(d, &p);
  if (st) return st;
  if (!workspace || bytes < (int64_t)(p.total * 4)) return CSMPN_ERR_WORKSPACE;
  if (!d.save_y1 || !d.save_y2 || !d.save_xr || !d.save_o) return CSMPN_ERR_BAD_ARG;
  const float* x0 = d.in_bpt ? d.p0 : d.save_x0;
  if (!x0) return CSMPN_ERR_BAD_ARG;
  if (p.tiles == 0) {  // no rows: every parameter gradient is zero (the header promises they are all overwritten)
    const size_t c = d.c, cin = p.cin;
    const std::pair<float*, size_t> outs[] = {{g.g_w1, c * cin * G}, {d.has_b1 ? g.g_b1 : nullptr, c}, {g.g_sa, c * G}, {g.g_sb, c * G},
                                              {g.g_wr, c * c * G}, {g.g_na, c * G}, {g.g_wl, c * c * G}, {g.g_bl, c}, {g.g_wp, c * P}, {g.g_la, c}};
    for (const auto& o : outs)
      if (o.first) CSMPN_CUDA_TRY(cudaMemsetAsync(o.first, 0, o.second * sizeof(float), stream));
    return CSMPN_OK;
  }
  float* ws = (float*)workspace;
  const int C = d.c, Cp = p.Cp;
  // ---- B1
  EwArgs e;
  memset(&e, 0, sizeof(e));
  e.rows = d.rows; e.tiles = p.tiles; e.C = C; e.Cp = Cp;
  e.gy = g.grad_y; e.gy_bpt = g.gy_bpt;
  e.gy_rows = g.gy_bpt ? nullptr : g.gy_rows;
  e.gy_stride = (!g.gy_bpt && g.gy_row_stride > 0) ? g.gy_row_stride : (int64_t)C * Alg<DIM>::B;
  e.o = d.save_o; e.xr = d.save_xr; e.y2 = d.save_y2; e.y1 = d.save_y1;
  e.la = d.la; e.wp = d.wp; e.na = d.na; e.sa = d.sa; e.sb = d.sb;
  e.d = ws + p.o_d; e.dxr = ws + p.o_dxr; e.dy2p = ws + p.o_dy2p; e.dy2 = ws + p.o_dy2; e.dy1 = ws + p.o_dy1;
  e.partial = ws + p.o_p1;
  const int cps = Cp <= 64 ? Cp : 64;           // channels per elementwise CTA (wide blocks: 64-channel slabs)
  const int nslab = Cp / cps;
  const int ew_threads = (cps / 4) * 32;
  const dim3 ew_grid(p.grid_ew, nslab);
  const int mask = d.stage_mask ? d.stage_mask : ~0;
  if (mask & 1) {
    const size_t sm1 = (size_t)(2 * (cps / 4) * kTile + 2 * kTile) * 4 + (size_t)2 * 4 * B * ew_threads * 4;
    auto run = [&](auto kern) -> int {
      CSMPN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1));
      kern<<<ew_grid, ew_threads, sm1, stream>>>(e);
      return CSMPN_OK;
    };
    int rc = Cp == 16 ? run(tc_b1_kernel<DIM, 16, 16>) : Cp == 32 ? run(tc_b1_kernel<DIM, 32, 32>)
             : Cp == 48 ? run(tc_b1_kernel<DIM, 48, 48>) : Cp == 64 ? run(tc_b1_kernel<DIM, 64, 64>)
             : Cp == 128 ? run(tc_b1_kernel<DIM, 64, 128>) : run(tc_b1_kernel<DIM, 64, 256>);
    if (rc) return rc;
    CSMPN_LAUNCH_CHECK("tc_b1_kernel");
  }
  // ---- dy2 = dy2p + d WL + dxr WR
  const int grid = p.tiles < sm_count_cached() ? p.tiles : sm_count_cached();
  float* img_dy2 = ws + p.o_img;
  float* img_gx = img_dy2 + (p.img_dy2 + 31) / 32 * 32;
  GemmArgs ga;
  memset(&ga, 0, sizeof(ga));
  ga.rows = d.rows; ga.tiles = p.tiles;
  ga.src[0] = ws + p.o_d; ga.src[1] = ws + p.o_dxr; ga.cp[0] = ga.cp[1] = Cp; ga.nk[0] = ga.nk[1] = Cp / 8;
  ga.w[0] = d.wl; ga.w[1] = d.wr; ga.wk[0] = ga.wk[1] = C; ga.wn = C;
  ga.n16 = Cp; ga.kmax = Cp;
  ga.addend = ws + p.o_dy2p; ga.out = ws + p.o_dy2; ga.out_bpt = 1;
  CSMPN_CUDA_TRY(cudaFuncSetAttribute(tc_bgemm_kernel<DIM, false, TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CSMPN_CUDA_TRY(cudaFuncSetAttribute(tc_bgemm_kernel<DIM, true, TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  CSMPN_CUDA_TRY(cudaFuncSetAttribute(tc_bgemmdb_kernel<DIM, TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  if (mask & 2) {
    if (p.wide) {
      WPrepArgs w{d.wl, d.wr, 0, 1, C, C, C, p.np, (Cp + p.np - 1) / p.np, Cp / 8, Cp / 8, img_dy2};
      int rc = launch_weight_images<DIM, TERMS>(w, p.img_dy2, stream);
      if (rc) return rc;
      ga.wimg = img_dy2; ga.np = p.np;
      tc_bgemm_kernel<DIM, true, TERMS><<<grid, kThreads, gemm_smem_streamed<DIM>(p.np, NI), stream>>>(ga);
    } else if (use_overlapped_epilogue(B, ga.n16)) {
      tc_bgemmdb_kernel<DIM, TERMS><<<grid, kThreads, gemm_smem<DIM>(2, ga.n16, ga.kmax, NI), stream>>>(ga);
    } else {
      tc_bgemm_kernel<DIM, false, TERMS><<<grid, kThreads, gemm_smem<DIM>(2, ga.n16, ga.kmax, NI), stream>>>(ga);
    }
    CSMPN_LAUNCH_CHECK("tc_bgemm_kernel(dy2)");
  }
  // ---- B3
  e.partial = ws + p.o_p3;
  if (mask & 4) {
    const size_t sm3 = (size_t)2 * 2 * B * ew_threads * 4;
    auto run = [&](auto kern) -> int {
      CSMPN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm3));
      kern<<<ew_grid, ew_threads, sm3, stream>>>(e);
      return CSMPN_OK;
    };
    int rc = Cp == 16 ? run(tc_b3_kernel<DIM, 16, 16>) : Cp == 32 ? run(tc_b3_kernel<DIM, 32, 32>)
             : Cp == 48 ? run(tc_b3_kernel<DIM, 48, 48>) : Cp == 64 ? run(tc_b3_kernel<DIM, 64, 64>)
             : Cp == 128 ? run(tc_b3_kernel<DIM, 64, 128>) : run(tc_b3_kernel<DIM, 64, 256>);
    if (rc) return rc;
    CSMPN_LAUNCH_CHECK("tc_b3_kernel");
  }
  // ---- grad_x = dy1 W1
  if (g.grad_x && (mask & 8)) {
    memset(&ga, 0, sizeof(ga));
    ga.rows = d.rows; ga.tiles = p.tiles;
    ga.src[0] = ws + p.o_dy1; ga.cp[0] = Cp; ga.nk[0] = Cp / 8;
    ga.w[0] = d.w1; ga.wk[0] = C; ga.wn = p.cin;
    ga.n16 = p.n16; ga.kmax = Cp;
    ga.out = g.grad_x; ga.out_bpt = g.gx_bpt;
    if (p.wide) {
      WPrepArgs w{d.w1, nullptr, 0, 1, p.cin, C, 0, p.np, (p.n16 + p.np - 1) / p.np, Cp / 8, 0, img_gx};
      int rc = launch_weight_images<DIM, TERMS>(w, p.img_gx, stream);
      if (rc) return rc;
      ga.wimg = img_gx; ga.np = p.np;
      tc_bgemm_kernel<DIM, true, TERMS><<<grid, kThreads, gemm_smem_streamed<DIM>(p.np, NI), stream>>>(ga);
    } else if (use_overlapped_epilogue(B, ga.n16)) {
      tc_bgemmdb_kernel<DIM, TERMS><<<grid, kThreads, gemm_smem<DIM>(1, ga.n16, ga.kmax, NI), stream>>>(ga);
    } else {
      tc_bgemm_kernel<DIM, false, TERMS><<<grid, kThreads, gemm_smem<DIM>(1, ga.n16, ga.kmax, NI), stream>>>(ga);
    }
    CSMPN_LAUNCH_CHECK("tc_bgemm_kernel(grad_x)");
  }
  // ---- weight gradients
  DwArgs da;
  memset(&da, 0, sizeof(da));
  da.dbg = debug_buffer();
#ifdef CSMPN_DEBUG_TOOLS
  auto dw_kernel = da.dbg ? tc_dw_kernel<DIM, true, TERMS> : tc_dw_kernel<DIM, false, TERMS>;
#else
  auto dw_kernel = tc_dw_kernel<DIM, false, TERMS>;
#endif
  CSMPN_CUDA_TRY(cudaFuncSetAttribute(dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
  da.rows = d.rows; da.tiles = p.tiles;
  std::vector<FinalJob> jobs;
  auto wjob = [&](const float* in, float* out, int parts, int M, int N, int m0, int co, int ci, int ci_tot, int i0, int o0) {
    if (co <= 0 || ci <= 0 || !out) return;
    FinalJob jb;
    memset(&jb, 0, sizeof(jb));
    jb.in = in; jb.out = out; jb.parts = parts; jb.stride = (int64_t)G * M * N; jb.kind = 1; jb.n = co * ci * G;
    jb.G = G; jb.M = M; jb.N = N; jb.m0 = m0; jb.co = co; jb.ci = ci; jb.ci_tot = ci_tot; jb.i0 = i0; jb.o0 = o0;
    jobs.push_back(jb);
  };
  auto clampi = [](int v, int hi) { return v < 0 ? 0 : (v > hi ? hi : v); };
  if (p.wide) {
    // one launch per (64-channel slab of an A tensor, 32-channel slab of the B tensor); merged M = 64: two partials per CTA
    const size_t smw = dw_smem<DIM>(kSlabA, kSlabA / 4, kSlabB);
    da.M = kSlabA; da.a1 = nullptr;
    int li = 0;
    for (int which = 0; which < 2; ++which) {  // d -> g_wl, dxr -> g_wr
      for (int ma = 0; ma < Cp; ma += kSlabA) {
        const int ca = (Cp - ma) < kSlabA ? (Cp - ma) : kSlabA;
        for (int nb = 0; nb < Cp; nb += kSlabB, ++li) {
          float* part = ws + p.o_dwa + (size_t)li * p.dw_part;
          if (mask & 16) {
            da.a0 = ws + (which ? p.o_dxr : p.o_d); da.cpa = ca; da.cpa_total = Cp; da.a_c4 = ma / 4;
            da.bsrc = d.save_y2; da.cpb = kSlabB; da.cpb_total = Cp; da.b_c4 = nb / 4;
            da.partial = part;
            dw_kernel<<<p.grid_dw, 256, smw, stream>>>(da);
            CSMPN_LAUNCH_CHECK("tc_dw_kernel(wl,wr slab)");
          }
          wjob(part, which ? g.g_wr : g.g_wl, p.grid_dw * 2, kSlabA, kSlabB, 0, clampi(C - ma, ca), clampi(C - nb, kSlabB), C, nb, ma);
        }
      }
    }
    li = 0;
    for (int ma = 0; ma < Cp; ma += kSlabA) {
      const int ca = (Cp - ma) < kSlabA ? (Cp - ma) : kSlabA;
      for (int nb = 0; nb < p.n16; nb += kSlabB, ++li) {
        const int cb = (p.n16 - nb) < kSlabB ? (p.n16 - nb) : kSlabB;
        float* part = ws + p.o_dwb + (size_t)li * p.dw_part;
        if (mask & 32) {
          da.a0 = ws + p.o_dy1; da.cpa = ca; da.cpa_total = Cp; da.a_c4 = ma / 4;
          da.bsrc = x0; da.cpb = cb; da.cpb_total = p.n16; da.b_c4 = nb / 4;
          da.partial = part;
          dw_kernel<<<p.grid_dw, 256, dw_smem<DIM>(kSlabA, kSlabA / 4, cb), stream>>>(da);
          CSMPN_LAUNCH_CHECK("tc_dw_kernel(w1 slab)");
        }
        wjob(part, g.g_w1, p.grid_dw * 2, kSlabA, cb, 0, clampi(C - ma, ca), clampi(p.cin - nb, cb), p.cin, nb, ma);
      }
    }
  } else {
    da.a0 = ws + p.o_d; da.a1 = ws + p.o_dxr; da.cpa = Cp; da.cpa_total = Cp; da.a_c4 = 0;
    da.bsrc = d.save_y2; da.cpb = Cp; da.cpb_total = Cp; da.b_c4 = 0;
    da.M = p.M1;
    da.partial = ws + p.o_dwa;
    const int pa = p.M1 == 64 ? 2 : 1;  // partials per CTA
    const size_t dwa_part = (size_t)p.grid_dw * pa * G * p.M1 * Cp;
    if (!(mask & 16)) {
    } else if (!p.dw_split) {
      dw_kernel<<<p.grid_dw, 256, dw_smem<DIM>(da.M, 2 * Cp / 4, Cp), stream>>>(da);
      CSMPN_LAUNCH_CHECK("tc_dw_kernel(wl,wr)");
    } else {
      da.a1 = nullptr;
      dw_kernel<<<p.grid_dw, 256, dw_smem<DIM>(da.M, Cp / 4, Cp), stream>>>(da);
      CSMPN_LAUNCH_CHECK("tc_dw_kernel(wl)");
      da.a0 = ws + p.o_dxr;
      da.partial = ws + p.o_dwa + dwa_part;
      dw_kernel<<<p.grid_dw, 256, dw_smem<DIM>(da.M, Cp / 4, Cp), stream>>>(da);
      CSMPN_LAUNCH_CHECK("tc_dw_kernel(wr)");
    }
    for (int i0 = 0; i0 < p.n16 && (mask & 32); i0 += p.nbw) {
      const int nb = (p.n16 - i0) < p.nbw ? (p.n16 - i0) : p.nbw;
      da.a0 = ws + p.o_dy1; da.a1 = nullptr; da.cpa = Cp; da.cpa_total = Cp; da.a_c4 = 0;
      da.bsrc = x0; da.cpb = nb; da.cpb_total = p.n16; da.b_c4 = i0 / 4;
      da.M = p.M2;
      da.partial = ws + p.o_dwb + (size_t)p.grid_dw * 2 * G * p.M2 * i0;
      dw_kernel<<<p.grid_dw, 256, dw_smem<DIM>(da.M, Cp / 4, nb), stream>>>(da);
      CSMPN_LAUNCH_CHECK("tc_dw_kernel(w1)");
    }
    wjob(ws + p.o_dwa, g.g_wl, p.grid_dw * pa, p.M1, Cp, 0, C, C, C, 0, 0);
    if (!p.dw_split) wjob(ws + p.o_dwa, g.g_wr, p.grid_dw * pa, p.M1, Cp, Cp, C, C, C, 0, 0);
    else wjob(ws + p.o_dwa + dwa_part, g.g_wr, p.grid_dw * pa, p.M1, Cp, 0, C, C, C, 0, 0);
    for (int i0 = 0; i0 < p.cin; i0 += p.nbw) {
      const int nb = (p.n16 - i0) < p.nbw ? (p.n16 - i0) : p.nbw;
      const int ci = (p.cin - i0) < p.nbw ? (p.cin - i0) : p.nbw;
      wjob(ws + p.o_dwb + (size_t)p.grid_dw * 2 * G * p.M2 * i0, g.g_w1, p.grid_dw * 2, p.M2, nb, 0, C, ci, p.cin, i0, 0);
    }
  }
  // ---- final reduction
  // small per-channel gradients: partial rows [C][NP]; viewed as kind-1 jobs with G := 1, "N" := NP, one column range each
  auto cjob = [&](const float* in, float* out, int parts, int NPk, int col0, int width) {
    // out[ch*width + q] = sum_p in[p][ch*NPk + col0 + q]  ==  kind 1 with G = 1, M = C, N = NPk, co = C, ci = width, offset col0
    FinalJob jb;
    memset(&jb, 0, sizeof(jb));
    jb.in = in + col0; jb.out = out; jb.parts = parts; jb.stride = (int64_t)C * NPk; jb.kind = 1; jb.n = C * width;
    jb.G = 1; jb.M = C; jb.N = NPk; jb.m0 = 0; jb.co = C; jb.ci = width; jb.ci_tot = width; jb.i0 = 0; jb.o0 = 0;
    jobs.push_back(jb);
  };
  const int NP1 = P + G + 2, NP3 = 2 * G + 1;
  cjob(ws + p.o_p1, g.g_wp, p.grid_ew, NP1, 0, P);
  cjob(ws + p.o_p1, g.g_na, p.grid_ew, NP1, P, G);
  cjob(ws + p.o_p1, g.g_la, p.grid_ew, NP1, P + G, 1);
  cjob(ws + p.o_p1, g.g_bl, p.grid_ew, NP1, P + G + 1, 1);
  cjob(ws + p.o_p3, g.g_sa, p.grid_ew, NP3, 0, G);
  cjob(ws + p.o_p3, g.g_sb, p.grid_ew, NP3, G, G);
  cjob(ws + p.o_p3, d.has_b1 ? g.g_b1 : nullptr, p.grid_ew, NP3, 2 * G, 1);
  if (mask & 64) {
    for (size_t j0 = 0; j0 < jobs.size(); j0 += kFinalJobs) {  // wide blocks have more jobs than one launch takes
      FinalJobs fj;
      memset(&fj, 0, sizeof(fj));
      int64_t total = 0;
      for (size_t k = j0; k < jobs.size() && k < j0 + kFinalJobs; ++k) {
        fj.j[fj.count++] = jobs[k];
        total += jobs[k].n;
      }
      tc_final_kernel<<<(unsigned)((total + 15) / 16), 256, 0, stream>>>(fj);
      CSMPN_LAUNCH_CHECK("tc_final_kernel");
    }
  }
  return CSMPN_OK;
}

template <int DIM>
int64_t bwd_ws_bytes(const csmpn_block_desc& d) {
  BwdPlan p;
  if (make_bwd_plan<DIM>(d, &p)) return -1;
  return (int64_t)(p.total * 4);
}

}  // namespace tcb

int tc_block_bwd(int dim, const csmpn_block_desc* d, const csmpn_block_grads* g, void* ws, int64_t bytes, cudaStream_t stream) {
  if (dim == 2) return d->tf32 ? tcb::launch_bwd<2, 1>(*d, *g, ws, bytes, stream) : tcb::launch_bwd<2, 3>(*d, *g, ws, bytes, stream);
  if (dim == 3) return d->tf32 ? tcb::launch_bwd<3, 1>(*d, *g, ws, bytes, stream) : tcb::launch_bwd<3, 3>(*d, *g, ws, bytes, stream);
  return CSMPN_ERR_UNSUPPORTED;
}
// the backward of a block of this shape fits (shared memory / TMEM plans of every backward kernel)
bool tc_block_bwd_supported(int dim, int c_in, int c) {
  csmpn_block_desc d;
  memset(&d, 0, sizeof(d));
  d.c0 = c_in; d.c = c; d.rows = 128;
  tcb::BwdPlan p;
  if (dim == 2) return tcb::make_bwd_plan<2>(d, &p) == CSMPN_OK;
  if (dim == 3) return tcb::make_bwd_plan<3>(d, &p) == CSMPN_OK;
  return false;
}
int tc_block_bwd_wide(int dim, int c_in, int c) {
  csmpn_block_desc d;
  memset(&d, 0, sizeof(d));
  d.c0 = c_in; d.c = c; d.rows = 128;
  tcb::BwdPlan p;
  const int st = dim == 2 ? tcb::make_bwd_plan<2>(d, &p) : dim == 3 ? tcb::make_bwd_plan<3>(d, &p) : -1;
  return st == CSMPN_OK && p.wide;
}
int64_t tc_block_bwd_workspace(int dim, const csmpn_block_desc* d) {
  if (dim == 2) return tcb::bwd_ws_bytes<2>(*d);
  if (dim == 3) return tcb::bwd_ws_bytes<3>(*d);
  return -1;
}

}  // namespace csmpn
