// Fused CEMLP-block kernels (forward and backward) for non-degenerate diagonal metrics of dimension 2, 3 and 5.
// MET instantiations fold the metric into the elementwise stages (common.cuh MetricArg); the GEMMs do not depend on it.
//
// One block = MVLinear -> MVSiLU -> SteerableGeometricProductLayer -> MVLayerNorm  (cegnn_utils.py:180-207).
//
// Execution model (B200): persistent CTAs, one per SM, each looping over tiles of TR rows.  Every stage reads and
// writes shared-memory tiles (no register-resident state crosses a stage), which keeps the instruction footprint
// small enough for the instruction cache and lets the elementwise stages use a thread-per-(row, channel) mapping:
//  * The three weight matrices of the block stay RESIDENT in shared memory for the life of the CTA (natural
//    [n][m][g] layout, row stride = 4 mod 32 words, which serves both the forward and the transposed GEMMs
//    conflict-free).  When they do not fit (wide layers) they are staged per GEMM in K-chunks instead.
//  * The input rows of a tile are fetched by TMA: one cp.async.bulk per (row, source) into shared memory,
//    completion on an mbarrier.  For the EGCL message block the receiver rows h[dst] land in bufA and the sender
//    rows h[src] in bufB, and one shared-memory pass forms h[dst] - h[src]; the [E, C+2T, B] message input of the
//    reference (cegnn_utils.py:254-259) is never materialised in HBM.
//  * The three per-grade channel GEMMs read their K operand from shared memory and keep their outputs in registers,
//    where bias, MVSiLU, normalisation, the table-driven weighted geometric product and the layer norm are applied.
//
// Backward uses three saved [rows, C, B] tensors (pre-SiLU y1, pre-normalisation xr, pre-LayerNorm o) instead of
// recomputing the forward GEMMs: the layer is bound by the FP32 pipe, not by HBM, so three extra tensors of traffic
// are cheaper than a third of the backward FLOPs.  Weight gradients are tile-local GEMMs accumulated into per-CTA
// global accumulators; the small per-channel parameter gradients are reduced with fixed-order warp shuffles.  A last
// kernel sums the per-CTA partials in a fixed order, so every gradient is bit-reproducible run to run.
#include "gemm.cuh"

namespace csmpn {

constexpr float kInvSqrt2 = 0.70710678118654752440f;
constexpr int kMaxSmem = 220 * 1024;

// fused-kernel GEMM thread tile: RB rows x NCH channels x B blades = 32 accumulators
template <int DIM> struct FCfg;
template <> struct FCfg<2> { static constexpr int RB = 2, NCH = 4; };
template <> struct FCfg<3> { static constexpr int RB = 1, NCH = 4; };
template <> struct FCfg<5> { static constexpr int RB = 1, NCH = 1; };

struct FusedPlan {
  int tr, rg, nc, threads;   // per group
  int ng;                    // thread groups per CTA (1 or 2); CTA size = ng * threads
  int tile_words;            // shared-memory words owned by one group (tiles + statistics)
  int ew_rows;         // rows handled per elementwise pass (= threads / C); thread t owns channel t % C
  int s1, s2, s3;      // tile row strides (words): s1 = pad(max(C, gathered c0) B), s2 = pad(C B), s3 = pad(max(c_in, C) B)
  int resident;        // weights resident in shared memory
  int sw1, swc;        // resident row strides: pad(c_in*GP), pad(c*GP)
  int off_w1, off_wr, off_wl;  // word offsets of the resident weights inside the weight area
  int kc1, kcc, kt1, ktc;      // staged mode: K-chunks (forward GEMM1 / CxC, transposed W1 / CxC)
  int wbuf;            // words of the weight area
  size_t smem;
  int grid;
  int ks;              // max row splits of the weight-gradient GEMMs
};

// Shared-memory layout (words):  forward  [A: tr*s3][B: tr*s1][C: tr*s2][weights][nu: tr*c][mu: 2*tr][barriers]
//                                backward [T1: tr*s1][T2: tr*s2][T3: tr*s3][T4: tr*s2][weights][nu][dt][mu: 2*tr][barriers]
template <int DIM>
inline int make_fused_plan(const csmpn_block_desc& d, bool backward, FusedPlan* out) {
  using Cfg = FCfg<DIM>;
  constexpr int B = Alg<DIM>::B, GP = GemmCfg<DIM>::GP;
  FusedPlan p;
  memset(&p, 0, sizeof(p));
  const int c = d.c, cin = d.c0 + d.c1 + d.c2;
  if (c > 256) return CSMPN_ERR_UNSUPPORTED;
  p.nc = (c + Cfg::NCH - 1) / Cfg::NCH;
  const int wide = cin > c ? cin : c;
  const int bwide = (d.mode == 1 && d.c0 > c) ? d.c0 : c;
  p.s1 = pad_stride(bwide * B);
  p.s2 = pad_stride(c * B);
  p.s3 = pad_stride(wide * B);
  p.sw1 = pad_stride(cin * GP);
  p.swc = pad_stride(c * GP);
  const int res_words = c * p.sw1 + 2 * c * p.swc;
  auto tile_words = [&](int tr) {
    size_t t = backward ? (size_t)tr * (p.s1 + 2 * p.s2 + p.s3) : (size_t)tr * (p.s1 + p.s2 + p.s3);
    return t + 2 * (size_t)tr * c + 2 * tr + 16;
  };
  // two half-size groups (same shared memory as one tile twice the size) when the whole CTA fits 256 threads
  auto two_groups = [&](int tr) { return (tr % (2 * Cfg::RB) == 0) && tr >= 16; };
  auto threads_for = [&](int tr) { return (((tr / Cfg::RB) * p.nc + 31) / 32) * 32; };
  static const int cand[] = {64, 48, 32, 24, 16, 12, 8, 6, 4, 2, 1};
  int best = 0;
  for (int tr : cand) {
    if (tr % Cfg::RB || threads_for(tr) > 256) continue;
    if ((tile_words(tr) + res_words) * 4 <= (size_t)kMaxSmem) { best = tr; break; }
  }
  if (best) {
    p.resident = 1;
    p.tr = best;
    p.off_w1 = 0;
    p.off_wr = c * p.sw1;
    p.off_wl = p.off_wr + c * p.swc;
    p.wbuf = res_words;
  } else {
    p.resident = 0;
    const int wb_words = 5632;  // 22 KB staging area
    for (int tr : cand) {
      if (tr % Cfg::RB || threads_for(tr) > 256) continue;
      if ((tile_words(tr) + wb_words) * 4 <= (size_t)kMaxSmem) { best = tr; break; }
    }
    if (!best) return CSMPN_ERR_UNSUPPORTED;
    p.tr = best;
    auto fit_fwd = [&](int odim, int kdim) {
      int kc = (wb_words / odim - 4) / GP;
      if (kc > kdim) kc = kdim;
      return kc < 1 ? 1 : kc;
    };
    auto fit_trans = [&](int odim, int kdim) {
      int kc = wb_words / pad_stride(odim * GP);
      if (kc > kdim) kc = kdim;
      return kc < 1 ? 1 : kc;
    };
    p.kc1 = fit_fwd(c, cin);
    p.kcc = fit_fwd(c, c);
    p.kt1 = fit_trans(cin, c);
    p.ktc = fit_trans(c, c);
    int w1 = c * pad_stride(p.kc1 * GP), w2 = c * pad_stride(p.kcc * GP);
    int w3 = p.kt1 * pad_stride(cin * GP), w4 = p.ktc * pad_stride(c * GP);
    p.wbuf = w1 > w2 ? w1 : w2;
    if (w3 > p.wbuf) p.wbuf = w3;
    if (w4 > p.wbuf) p.wbuf = w4;
    if ((tile_words(p.tr) + p.wbuf) * 4 > (size_t)kMaxSmem) return CSMPN_ERR_UNSUPPORTED;
  }
  p.ng = 1;
  if (p.resident && two_groups(p.tr) && threads_for(p.tr / 2) >= c && threads_for(p.tr / 2) * 2 <= 256 &&
      (2 * tile_words(p.tr / 2) + res_words) * 4 <= (size_t)kMaxSmem) {
    p.ng = 2;
    p.tr /= 2;
  }
  p.rg = p.tr / Cfg::RB;
  p.threads = threads_for(p.tr);
  if (p.threads < c) p.threads = ((c + 31) / 32) * 32;  // the elementwise stages need one thread per channel
  if (p.threads * p.ng > 256) return CSMPN_ERR_UNSUPPORTED;
  p.ew_rows = p.threads / c;
  if (p.ew_rows > p.tr) p.ew_rows = p.tr;
  p.tile_words = (int)tile_words(p.tr);
  p.smem = ((size_t)p.ng * tile_words(p.tr) + p.wbuf) * sizeof(float);
  int64_t tiles = (d.rows + (int64_t)p.tr * p.ng - 1) / ((int64_t)p.tr * p.ng);
  int per_sm = (int)((size_t)(226 * 1024) / (p.smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  if (per_sm * p.threads * p.ng > 512) per_sm = 512 / (p.threads * p.ng) > 0 ? 512 / (p.threads * p.ng) : 1;
  int64_t cap = (int64_t)sm_count_cached() * per_sm;
  p.grid = (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
  const int NA = Alg<DIM>::G <= 4 ? 4 : 2;
  int tc = ((c + NA - 1) / NA) * ((c + 3) / 4);
  p.ks = p.threads / tc > 0 ? p.threads / tc : 1;  // per group
  if (p.ks > 16) p.ks = 16;
  while (p.ks > 1 && p.tr % p.ks) --p.ks;
  *out = p;
  return CSMPN_OK;
}

// ---------------------------------------------------------------------------------------------------
// mbarrier / TMA (bulk async copy) helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_row_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------
// thread-local multivector math: quadratic forms q_g = sum_{i in g} qs_i x_i^2 (MET), sums of squares (Euclidean)
template <int DIM, bool MET>
__device__ __forceinline__ void silu_gates(const float* y1, const float* a, const float* b, float* sg, float* inv, const float* qs) {
  using A = Alg<DIM>;
#pragma unroll
  for (int g = 0; g < A::G; ++g) inv[g] = 0.f;
#pragma unroll
  for (int i = 0; i < A::B; ++i) inv[A::grade_of(i)] = fmaf(qs_x<MET>(qs, i, y1[i]), y1[i], inv[A::grade_of(i)]);
  inv[0] = y1[0];
#pragma unroll
  for (int g = 0; g < A::G; ++g) sg[g] = sigmoidf_(fmaf(a[g], inv[g], b[g]));
}

// normalisation: xn_i = xr_i * rinv[g];  den_g = s_g (nrm_g - 1) + 1 + eps
template <int DIM, bool MET>
__device__ __forceinline__ void norm_factors(const float* xr, const float* s, float* q, float* nrm, float* rinv, const float* qs) {
  using A = Alg<DIM>;
#pragma unroll
  for (int g = 0; g < A::G; ++g) q[g] = 0.f;
#pragma unroll
  for (int i = 0; i < A::B; ++i) q[A::grade_of(i)] = fmaf(qs_x<MET>(qs, i, xr[i]), xr[i], q[A::grade_of(i)]);
#pragma unroll
  for (int g = 0; g < A::G; ++g) {
    nrm[g] = smooth_abs_sqrt(q[g]);
    rinv[g] = 1.f / (fmaf(s[g], nrm[g] - 1.f, 1.f) + kEps);
  }
}

// full quadratic form Q = sum_i qs_i x_i^2 (MVLayerNorm)
template <int DIM, bool MET>
__device__ __forceinline__ float mv_q(const float* x, const float* qs) {
  float Q = 0.f;
#pragma unroll
  for (int i = 0; i < Alg<DIM>::B; ++i) Q = fmaf(qs_x<MET>(qs, i, x[i]), x[i], Q);
  return Q;
}

// ---------------------------------------------------------------------------------------------------
// A CTA runs NG (1 or 2) independent thread groups.  Each group owns its own tiles in shared memory, its own
// mbarriers and its own stream of row tiles, and synchronises with a named barrier, so one group's TMA waits,
// barriers and elementwise stages overlap the other group's GEMMs while both share the resident weights.
struct Grp {
  int tid, nthr, id;
  __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, %1;" ::"r"(id + 1), "r"(nthr) : "memory"); }
};

// ---------------------------------------------------------------------------------------------------
// TMA row loaders.  Every thread of the CTA issues at most a few cp.async.bulk row copies (one per (row, piece)
// item, so the dependent index loads of the gather are spread over all threads); thread 0 arrives on the mbarrier
// (initialised with one arrival) with the total byte count, which is known arithmetically.
struct RowPiece {
  float* tile; int stride; int col;   // destination: tile row r, word offset col
  const float* src; int ch;           // source tensor [*, ch, B]
  const int32_t* idx;                 // row index array (NULL: dense rows row0 + r)
};

template <int DIM, int NP>
__device__ __forceinline__ void tma_issue_pieces(const Grp& g, const RowPiece (&pc)[NP], int npieces, int64_t row0,
                                                 int valid, uint64_t* bar) {
  constexpr int B = Alg<DIM>::B;
  if (g.tid == 0) {
    uint32_t per_row = 0;
    for (int k = 0; k < npieces; ++k) per_row += (uint32_t)pc[k].ch * B * 4;
    mbar_arrive_expect_tx(bar, per_row * (uint32_t)valid);
  }
  for (int item = g.tid; item < valid * npieces; item += g.nthr) {
    const int r = item / npieces, k = item - r * npieces;
    const RowPiece& q = pc[k];
    const int64_t srow = q.idx ? (int64_t)__ldg(q.idx + row0 + r) : row0 + r;
    tma_row_g2s(q.tile + r * q.stride + q.col, q.src + srow * (int64_t)q.ch * B, (uint32_t)q.ch * B * 4, bar);
  }
}

// pieces of the assembled input row of the block into `tile` (stride s3); sender rows of the gather go to `tmp`
template <int DIM>
__device__ __forceinline__ int input_pieces(RowPiece* pc, float* tile, int s3, float* tmp, int s1, const csmpn_block_desc& d) {
  constexpr int B = Alg<DIM>::B;
  int n = 0;
  if (d.mode == 0) {
    pc[n++] = RowPiece{tile, s3, 0, d.p0, d.c0, nullptr};
    if (d.c1) pc[n++] = RowPiece{tile, s3, d.c0 * B, d.p1, d.c1, nullptr};
    if (d.c2) pc[n++] = RowPiece{tile, s3, (d.c0 + d.c1) * B, d.p2, d.c2, nullptr};
  } else {
    pc[n++] = RowPiece{tile, s3, 0, d.p0, d.c0, d.dst};
    pc[n++] = RowPiece{tmp, s1, 0, d.p0, d.c0, d.src};
    if (d.c1 && d.pair_attr) {  // extra channels = (table[src] | table[dst]), table = p1 [n_nodes, c1/2, B]
      pc[n++] = RowPiece{tile, s3, d.c0 * B, d.p1, d.c1 / 2, d.src};
      pc[n++] = RowPiece{tile, s3, (d.c0 + d.c1 / 2) * B, d.p1, d.c1 / 2, d.dst};
    } else if (d.c1) {
      pc[n++] = RowPiece{tile, s3, d.c0 * B, d.p1, d.c1, d.eid};
    }
  }
  return n;
}

// after the wait: gather mode forms h[dst] - h[src]; missing rows of a tail tile are zeroed
template <int DIM>
__device__ __forceinline__ void finish_input_rows(const Grp& g, float* tile, int s3, const float* tmp, int s1,
                                                  const csmpn_block_desc& d, int tr, int valid) {
  constexpr int B = Alg<DIM>::B;
  if (d.mode == 1) {
    const int v0 = d.c0 * B / 4;
    for (int idx = g.tid; idx < valid * v0; idx += g.nthr) {
      const int r = idx / v0, v = idx - r * v0;
      float4 a = *reinterpret_cast<const float4*>(tile + r * s3 + 4 * v);
      const float4 b = *reinterpret_cast<const float4*>(tmp + r * s1 + 4 * v);
      a.x -= b.x; a.y -= b.y; a.z -= b.z; a.w -= b.w;
      *reinterpret_cast<float4*>(tile + r * s3 + 4 * v) = a;
    }
  }
  if (valid < tr) {
    const int vpr = (d.c0 + d.c1 + d.c2) * B / 4;
    for (int idx = g.tid; idx < (tr - valid) * vpr; idx += g.nthr) {
      const int r = valid + idx / vpr, v = idx % vpr;
      *reinterpret_cast<float4*>(tile + r * s3 + 4 * v) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

__device__ __forceinline__ void zero_tail_rows(const Grp& g, float* tile, int stride, int words, int tr, int valid) {
  const int vpr = words / 4;
  for (int idx = g.tid; idx < (tr - valid) * vpr; idx += g.nthr) {
    const int r = valid + idx / vpr, v = idx % vpr;
    *reinterpret_cast<float4*>(tile + r * stride + 4 * v) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// weight operand of a GEMM stage: resident in shared memory, or staged from global in K-chunks
struct WRef {
  const float* g;   // global [c_out][c_in][G]
  float* s;         // shared: resident matrix, or the staging area
  int c_out, c_in;
  int sw;           // resident row stride
  int kchunk;       // staged mode
  int resident;
};

// acc += buf[:, 0:kdim] * W   for output channels  obase + c + a * nco  (a < NCHT), masked by owidth.
// The leading barrier publishes the shared-memory writes of the previous stage.
template <int DIM, bool TRANS, int NCHT>
__device__ __forceinline__ void gemm_run(const Grp& g, float (&acc)[FCfg<DIM>::RB][NCHT][Alg<DIM>::B],
                                         const float* __restrict__ buf_rows, int stride, const WRef& w, bool active, int c,
                                         int nco, int obase, int owidth, bool lead_sync = true) {
  constexpr int B = Alg<DIM>::B, GP = GemmCfg<DIM>::GP, RB = FCfg<DIM>::RB;
  const int kdim = TRANS ? w.c_out : w.c_in;
  const int odim = TRANS ? w.c_in : w.c_out;
  if (w.resident) {
    if (lead_sync) g.sync();
    if (active) {
      const float* wp[NCHT];
#pragma unroll
      for (int a = 0; a < NCHT; ++a) {
        int ol = c + a * nco;
        int o = obase + (ol < owidth ? ol : 0);
        wp[a] = TRANS ? w.s + o * GP : w.s + o * w.sw;
      }
      gemm_accumulate<DIM, NCHT, RB>(acc, buf_rows, stride, wp, TRANS ? w.sw : GP, kdim);
    }
    return;
  }
  for (int k0 = 0; k0 < kdim; k0 += w.kchunk) {
    const int kc = (kdim - k0) < w.kchunk ? (kdim - k0) : w.kchunk;
    const int sw = TRANS ? pad_stride(odim * GP) : pad_stride(kc * GP);
    g.sync();
    stage_weights<DIM, TRANS>(w.s, sw, w.g, w.c_out, w.c_in, Alg<DIM>::G, k0, kc);
    g.sync();
    if (active) {
      const float* wp[NCHT];
#pragma unroll
      for (int a = 0; a < NCHT; ++a) {
        int ol = c + a * nco;
        int o = obase + (ol < owidth ? ol : 0);
        wp[a] = TRANS ? w.s + o * GP : w.s + o * sw;
      }
      gemm_accumulate<DIM, NCHT, RB>(acc, buf_rows + k0 * B, stride, wp, TRANS ? sw : GP, kc);
    }
  }
}

template <int DIM>
__device__ __forceinline__ void setup_weights(const csmpn_block_desc& d, const FusedPlan& p, float* wsm, WRef& w1, WRef& wr,
                                              WRef& wl) {
  const int C = d.c, cin = d.c0 + d.c1 + d.c2;
  w1 = WRef{d.w1, p.resident ? wsm + p.off_w1 : wsm, C, cin, p.sw1, 0, p.resident};
  wr = WRef{d.wr, p.resident ? wsm + p.off_wr : wsm, C, C, p.swc, 0, p.resident};
  wl = WRef{d.wl, p.resident ? wsm + p.off_wl : wsm, C, C, p.swc, 0, p.resident};
  if (p.resident) {
    stage_weights<DIM, false>(w1.s, p.sw1, d.w1, C, cin, Alg<DIM>::G, 0, cin);
    stage_weights<DIM, false>(wr.s, p.swc, d.wr, C, C, Alg<DIM>::G, 0, C);
    stage_weights<DIM, false>(wl.s, p.swc, d.wl, C, C, Alg<DIM>::G, 0, C);
  }
}

// dst[r][o] (+)= sum_k src[r][k] W(k, o) for all C output channels of the block; shared-memory to shared-memory.
template <int DIM, bool TRANS, bool ACCUM>
__device__ __forceinline__ void gemm_tile(const Grp& g, float* __restrict__ dst, int dstride, const float* __restrict__ src,
                                          int sstride, const WRef& w, const FusedPlan& p, int C, bool active, int c, int rg,
                                          bool lead_sync = true) {
  constexpr int B = Alg<DIM>::B, RB = FCfg<DIM>::RB, NCH = FCfg<DIM>::NCH;
  float acc[RB][NCH][B];
#pragma unroll
  for (int j = 0; j < RB; ++j)
#pragma unroll
    for (int a = 0; a < NCH; ++a)
#pragma unroll
      for (int i = 0; i < B; ++i) acc[j][a][i] = 0.f;
  gemm_run<DIM, TRANS, NCH>(g, acc, src + rg * RB * sstride, sstride, w, active, c, p.nc, 0, C, lead_sync);
  if (active) {
#pragma unroll
    for (int a = 0; a < NCH; ++a) {
      const int o = c + a * p.nc;
      if (o >= C) continue;
#pragma unroll
      for (int j = 0; j < RB; ++j) {
        float* q = dst + (rg * RB + j) * dstride + o * B;
        if (ACCUM) {
          float old[B];
          load_vec<B>(old, q);
#pragma unroll
          for (int i = 0; i < B; ++i) acc[j][a][i] += old[i];
        }
        store_vec<B>(q, acc[j][a]);
      }
    }
  }
}

// per-thread parameters of the channel a thread owns in the elementwise stages
template <int DIM>
struct ChanParams {
  float sa[Alg<DIM>::G], sb[Alg<DIM>::G], sn[Alg<DIM>::G], wv[Alg<DIM>::P], b1, bl, la;
  __device__ __forceinline__ void load(const csmpn_block_desc& d, int n, bool ok) {
    constexpr int G = Alg<DIM>::G, P = Alg<DIM>::P;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      sa[g] = ok ? d.sa[n * G + g] : 0.f;
      sb[g] = ok ? d.sb[n * G + g] : 0.f;
      sn[g] = ok ? sigmoidf_(d.na[n * G + g]) : 0.f;
    }
#pragma unroll
    for (int q = 0; q < P; ++q) wv[q] = ok ? d.wp[n * P + q] : 0.f;
    b1 = (ok && d.has_b1) ? d.b1[n] : 0.f;
    bl = ok ? d.bl[n] : 0.f;
    la = ok ? d.la[n] : 0.f;
  }
};

// ===================================================================================================
// forward
template <int DIM, bool MET>
__global__ void __launch_bounds__(256, 1) block_fwd_kernel(csmpn_block_desc d, FusedPlan p, MetricArg<MET> mp) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G;
  extern __shared__ __align__(128) float smem[];
  Grp g;
  g.id = threadIdx.x / p.threads;
  g.tid = threadIdx.x - g.id * p.threads;
  g.nthr = p.threads;
  float* wsm = smem;                                  // weights (shared by the groups)
  float* tA = smem + p.wbuf + g.id * p.tile_words;    // input row (wide) -> xr
  float* tB = tA + p.tr * p.s3;                       // sender rows (gather) -> y1 -> y2
  float* tC = tB + p.tr * p.s1;                       // xl -> o
  float* nu_s = tC + p.tr * p.s2;                     // [tr][C]
  float* mu_s = nu_s + 2 * p.tr * d.c;                // [tr]
  uint64_t* bar = reinterpret_cast<uint64_t*>(mu_s + 2 * p.tr);
  const int C = d.c;
  const int c = g.tid % p.nc, rg = g.tid / p.nc;
  const bool active = rg < p.rg;
  const int n_e = g.tid % C, rl = g.tid / C;  // elementwise mapping: channel n_e, rows rl, rl + ew_rows, ...
  const bool ew = rl < p.ew_rows;
  const int64_t tiles = (d.rows + p.tr - 1) / p.tr;
  WRef w1, wr, wl;
  setup_weights<DIM>(d, p, wsm, w1, wr, wl);
  if (!p.resident) { w1.kchunk = p.kc1; wr.kchunk = p.kcc; wl.kchunk = p.kcc; }
  if (g.tid == 0) mbar_init(bar, 1);
  ChanParams<DIM> cp;
  cp.load(d, n_e, ew);
  uint32_t phase = 0;
  __syncthreads();  // resident weights staged, barriers initialised

  for (int64_t tile = (int64_t)blockIdx.x * p.ng + g.id; tile < tiles; tile += (int64_t)gridDim.x * p.ng) {
    const int64_t row0 = tile * p.tr;
    const int valid = (d.rows - row0) < p.tr ? (int)(d.rows - row0) : p.tr;
    fence_proxy_async();
    g.sync();  // previous tile's generic accesses are done
    {
      RowPiece pc[5];
      const int np = input_pieces<DIM>(pc, tA, p.s3, tB, p.s1, d);
      tma_issue_pieces<DIM, 5>(g, pc, np, row0, valid, bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    finish_input_rows<DIM>(g, tA, p.s3, tB, p.s1, d, p.tr, valid);
    // ---- GEMM1: y1 (without bias) -> tB
    gemm_tile<DIM, false, false>(g, tB, p.s1, tA, p.s3, w1, p, C, active, c, rg);
    g.sync();
    // ---- bias + MVSiLU (in place): tB = y2
    if (ew) {
      for (int r = rl; r < p.tr; r += p.ew_rows) {
        float y1[B], sg[G], inv[G];
        float* q = tB + r * p.s1 + n_e * B;
        load_vec<B>(y1, q);
        y1[0] += cp.b1;
        if (d.save_y1 && r < valid) store_vec<B>(d.save_y1 + ((row0 + r) * C + n_e) * B, y1);
        silu_gates<DIM, MET>(y1, cp.sa, cp.sb, sg, inv, mp.qs);
#pragma unroll
        for (int i = 0; i < B; ++i) y1[i] *= sg[A::grade_of(i)];
        store_vec<B>(q, y1);
      }
    }
    // ---- GEMM-R: xr -> tA ; GEMM-L: xl -> tC   (the leading barrier of the first publishes y2)
    gemm_tile<DIM, false, false>(g, tA, p.s3, tB, p.s1, wr, p, C, active, c, rg);
    gemm_tile<DIM, false, false>(g, tC, p.s2, tB, p.s1, wl, p, C, active, c, rg, !p.resident);
    g.sync();
    // ---- normalisation, weighted geometric product, 1/sqrt2: tC = o ; norms for the layer norm
    if (ew) {
      for (int r = rl; r < p.tr; r += p.ew_rows) {
        float xr[B], y2[B], o[B], q[G], nrm[G], rinv[G];
        load_vec<B>(xr, tA + r * p.s3 + n_e * B);
        load_vec<B>(y2, tB + r * p.s1 + n_e * B);
        load_vec<B>(o, tC + r * p.s2 + n_e * B);
        if (d.save_xr && r < valid) store_vec<B>(d.save_xr + ((row0 + r) * C + n_e) * B, xr);
        norm_factors<DIM, MET>(xr, cp.sn, q, nrm, rinv, mp.qs);
#pragma unroll
        for (int i = 0; i < B; ++i) xr[i] *= rinv[A::grade_of(i)];
        o[0] += cp.bl;
        A::template wgp<MET>(y2, xr, cp.wv, mp.mf, o);
#pragma unroll
        for (int i = 0; i < B; ++i) o[i] *= kInvSqrt2;
        if (d.save_o && r < valid) store_vec<B>(d.save_o + ((row0 + r) * C + n_e) * B, o);
        store_vec<B>(tC + r * p.s2 + n_e * B, o);
        nu_s[r * C + n_e] = smooth_abs_sqrt(mv_q<DIM, MET>(o, mp.qs));
      }
    }
    g.sync();
    for (int r = g.tid >> 5; r < p.tr; r += (g.nthr >> 5)) {  // one warp per row, fixed-order tree
      float s = 0.f;
      for (int n = g.tid & 31; n < C; n += 32) s += nu_s[r * C + n];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if ((g.tid & 31) == 0) mu_s[r] = 1.f / (s / (float)C + kEps);
    }
    g.sync();
    // ---- MVLayerNorm scale (+ residual) -> global
    if (ew) {
      for (int r = rl; r < valid; r += p.ew_rows) {
        float o[B];
        load_vec<B>(o, tC + r * p.s2 + n_e * B);
        const float sc = cp.la * mu_s[r];
#pragma unroll
        for (int i = 0; i < B; ++i) o[i] *= sc;
        const int64_t off = ((row0 + r) * C + n_e) * B;
        if (d.res) {
          float rv[B];
          load_vec<B>(rv, d.res + off);
#pragma unroll
          for (int i = 0; i < B; ++i) o[i] += rv[i];
        }
        store_vec<B>(d.y + off, o);
      }
    }
  }
}

// ===================================================================================================
// backward helpers

// Tile-local weight-gradient GEMM over one column block of the m operand:
//   gacc[split][n][m_off + m][g] += sum_{r in split} sum_{i in g} nbuf[r][n][i] * mbuf[r][m][i],  m < cm_block
template <int DIM>
__device__ __forceinline__ void dw_tile(const Grp& g, const float* __restrict__ nbuf, int nstride, int cn_total,
                                        const float* __restrict__ mbuf, int mstride, int cm_block, int m_off, int m_ld,
                                        int tr, int ks_max, float* __restrict__ gacc) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G;
  constexpr int NA = (G <= 4) ? 4 : 2, MA = 4;
  const int ncn = (cn_total + NA - 1) / NA, ncm = (cm_block + MA - 1) / MA;
  const int tiles = ncn * ncm;
  int ks = g.nthr / tiles;
  if (ks < 1) ks = 1;
  if (ks > ks_max) ks = ks_max;
  while (ks > 1 && tr % ks) --ks;
  const int rows_per = tr / ks;
  for (int item = g.tid; item < tiles * ks; item += g.nthr) {
    const int split = item / tiles, tt = item - split * tiles;
    const int cm = tt % ncm, cn = tt / ncm;
    int nl[NA], ml[MA];
    bool nv[NA], mv[MA];
#pragma unroll
    for (int a = 0; a < NA; ++a) { int n = cn + a * ncn; nv[a] = n < cn_total; nl[a] = nv[a] ? n : 0; }
#pragma unroll
    for (int b = 0; b < MA; ++b) { int m = cm + b * ncm; mv[b] = m < cm_block; ml[b] = mv[b] ? m : 0; }
    float acc[NA][MA][G];
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
      for (int b = 0; b < MA; ++b)
#pragma unroll
        for (int g = 0; g < G; ++g) acc[a][b][g] = 0.f;
    const int rbeg = split * rows_per;
#pragma unroll 2
    for (int r = rbeg; r < rbeg + rows_per; ++r) {
      float dv[NA][B], xv[MA][B];
#pragma unroll
      for (int a = 0; a < NA; ++a) load_vec<B>(dv[a], nbuf + r * nstride + nl[a] * B);
#pragma unroll
      for (int b = 0; b < MA; ++b) load_vec<B>(xv[b], mbuf + r * mstride + ml[b] * B);
#pragma unroll
      for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int b = 0; b < MA; ++b)
#pragma unroll
          for (int i = 0; i < B; ++i) acc[a][b][A::grade_of(i)] = fmaf(dv[a][i], xv[b][i], acc[a][b][A::grade_of(i)]);
    }
    float* out = gacc + (size_t)split * cn_total * m_ld * G;
    if constexpr (G == 4) {
      // issue every load of the read-modify-write before the first dependent add (one L2 round trip, not 16)
      float4 old[NA][MA];
#pragma unroll
      for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int b = 0; b < MA; ++b)
          old[a][b] = (nv[a] && mv[b]) ? __ldcg(reinterpret_cast<const float4*>(out + ((size_t)nl[a] * m_ld + m_off + ml[b]) * G))
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int b = 0; b < MA; ++b) {
          if (!(nv[a] && mv[b])) continue;
          float4 t = old[a][b];
          t.x += acc[a][b][0]; t.y += acc[a][b][1]; t.z += acc[a][b][2]; t.w += acc[a][b][3];
          __stcg(reinterpret_cast<float4*>(out + ((size_t)nl[a] * m_ld + m_off + ml[b]) * G), t);
        }
    } else {
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        if (!nv[a]) continue;
#pragma unroll
        for (int b = 0; b < MA; ++b) {
          if (!mv[b]) continue;
          float* o = out + ((size_t)nl[a] * m_ld + m_off + ml[b]) * G;
#pragma unroll
          for (int g = 0; g < G; ++g) o[g] += acc[a][b][g];
        }
      }
    }
  }
}

struct BwdWorkspace {
  float* dw1;    // [grid][ks][c][cin][G]
  float* dwr;    // [grid][ks][c][c][G]
  float* dwl;    // [grid][ks][c][c][G]
  float* small;  // [grid][c * (P + 3G + 3)]:  dw[c][P] | dna[c][G] | dsa[c][G] | dsb[c][G] | dla[c] | db1[c] | dbl[c]
};

// one pass of the transposed W1 GEMM over output channels [ob, ob + width) with NCHT channels per thread -> global
template <int DIM, int NCHT>
__device__ __forceinline__ void dx_pass(const Grp& g, const float* __restrict__ tD, int sD, const FusedPlan& p, const WRef& w1,
                                        float* grad_x, int64_t row0, int valid, int cin, int ob, int width, int c, int rg,
                                        bool active) {
  constexpr int B = Alg<DIM>::B, RB = FCfg<DIM>::RB;
  float acc[RB][NCHT][B];
#pragma unroll
  for (int j = 0; j < RB; ++j)
#pragma unroll
    for (int a = 0; a < NCHT; ++a)
#pragma unroll
      for (int i = 0; i < B; ++i) acc[j][a][i] = 0.f;
  const bool act = active && c < width;
  gemm_run<DIM, true, NCHT>(g, acc, tD + rg * RB * sD, sD, w1, act, c, p.nc, ob, width);
  if (act && grad_x) {
#pragma unroll
    for (int j = 0; j < RB; ++j) {
      const int r = rg * RB + j;
      if (r >= valid) continue;
#pragma unroll
      for (int a = 0; a < NCHT; ++a) {
        const int ol = c + a * p.nc;
        if (ol < width) store_vec<B>(grad_x + ((row0 + r) * cin + ob + ol) * B, acc[j][a]);
      }
    }
  }
}

// ===================================================================================================
// backward
template <int DIM, bool MET>
__global__ void __launch_bounds__(256, 1) block_bwd_kernel(csmpn_block_desc d, csmpn_block_grads gr, FusedPlan p,
                                                           BwdWorkspace ws, MetricArg<MET> mp) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, P = A::P, NCH = FCfg<DIM>::NCH;
  extern __shared__ __align__(128) float smem[];
  Grp g;
  g.id = threadIdx.x / p.threads;
  g.tid = threadIdx.x - g.id * p.threads;
  g.nthr = p.threads;
  float* wsm = smem;                                  // weights (shared by the groups)
  float* t1 = smem + p.wbuf + g.id * p.tile_words;    // o -> y2 ; later sender rows of the gather
  float* t2 = t1 + p.tr * p.s1;           // dy -> d ; later y1 again
  float* t3 = t2 + p.tr * p.s2;           // xr -> dxr ; later the input row x0 (wide)
  float* t4 = t3 + p.tr * p.s3;           // y1 -> dy2 -> dy1
  float* nu_s = t4 + p.tr * p.s2;         // [tr][C]
  float* dt_s = nu_s + p.tr * d.c;        // [tr][C]
  float* mu_s = dt_s + p.tr * d.c;        // [tr] 1/mu
  float* dmu_s = mu_s + p.tr;             // [tr] d loss / d mu / C
  uint64_t* bar = reinterpret_cast<uint64_t*>(dmu_s + p.tr);  // bar[0]: tile inputs, bar[1]: y1 + x0 reload
  const int C = d.c, cin = d.c0 + d.c1 + d.c2;
  const int c = g.tid % p.nc, rg = g.tid / p.nc;
  const bool active = rg < p.rg;
  const int n_e = g.tid % C, rl = g.tid / C;
  const bool ew = rl < p.ew_rows;
  const int64_t tiles = (d.rows + p.tr - 1) / p.tr;
  const size_t slot = (size_t)blockIdx.x * p.ng + g.id;  // private weight-gradient accumulators of this group
  float* my_dw1 = ws.dw1 + slot * p.ks * C * cin * G;
  float* my_dwr = ws.dwr + slot * p.ks * C * C * G;
  float* my_dwl = ws.dwl + slot * p.ks * C * C * G;
  WRef w1, wr, wl;
  setup_weights<DIM>(d, p, wsm, w1, wr, wl);
  if (!p.resident) { w1.kchunk = p.kt1; wr.kchunk = p.ktc; wl.kchunk = p.ktc; }
  if (g.tid == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); }
  ChanParams<DIM> cp;
  cp.load(d, n_e, ew);
  // parameter-gradient accumulators of the channel this thread owns (registers, whole kernel)
  float g_w[P], g_na[G], g_sa[G], g_sb[G], g_la = 0.f, g_b1 = 0.f, g_bl = 0.f;
#pragma unroll
  for (int q = 0; q < P; ++q) g_w[q] = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) { g_na[g] = 0.f; g_sa[g] = 0.f; g_sb[g] = 0.f; }
  uint32_t phase = 0;
  const size_t rowsz = (size_t)C * B;
  __syncthreads();  // resident weights staged, barriers initialised

  for (int64_t tile = (int64_t)blockIdx.x * p.ng + g.id; tile < tiles; tile += (int64_t)gridDim.x * p.ng) {
    const int64_t row0 = tile * p.tr;
    const int valid = (d.rows - row0) < p.tr ? (int)(d.rows - row0) : p.tr;
    fence_proxy_async();
    g.sync();
    // ---- TMA: o -> t1, dy -> t2, xr -> t3, y1 -> t4
    {
      RowPiece pc[4] = {RowPiece{t1, p.s1, 0, d.save_o, C, nullptr}, RowPiece{t2, p.s2, 0, gr.grad_y, C, nullptr},
                        RowPiece{t3, p.s3, 0, d.save_xr, C, nullptr}, RowPiece{t4, p.s2, 0, d.save_y1, C, nullptr}};
      tma_issue_pieces<DIM, 4>(g, pc, 4, row0, valid, bar);
    }
    mbar_wait(bar, phase);
    if (valid < p.tr) {
      zero_tail_rows(g, t1, p.s1, (int)rowsz, p.tr, valid);
      zero_tail_rows(g, t2, p.s2, (int)rowsz, p.tr, valid);
      zero_tail_rows(g, t3, p.s3, (int)rowsz, p.tr, valid);
      zero_tail_rows(g, t4, p.s2, (int)rowsz, p.tr, valid);
      g.sync();
    }
    // ---- layer-norm statistics
    if (ew) {
      for (int r = rl; r < p.tr; r += p.ew_rows) {
        float o[B], dy[B];
        load_vec<B>(o, t1 + r * p.s1 + n_e * B);
        load_vec<B>(dy, t2 + r * p.s2 + n_e * B);
        float dot = 0.f;
#pragma unroll
        for (int i = 0; i < B; ++i) dot = fmaf(dy[i], o[i], dot);
        nu_s[r * C + n_e] = smooth_abs_sqrt(mv_q<DIM, MET>(o, mp.qs));
        dt_s[r * C + n_e] = cp.la * dot;
      }
    }
    g.sync();
    for (int r = g.tid >> 5; r < p.tr; r += (g.nthr >> 5)) {
      float s1 = 0.f, s2 = 0.f;
      for (int n = g.tid & 31; n < C; n += 32) { s1 += nu_s[r * C + n]; s2 += dt_s[r * C + n]; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
      if ((g.tid & 31) == 0) {
        const float inv_mu = 1.f / (s1 / (float)C + kEps);
        mu_s[r] = inv_mu;
        dmu_s[r] = -s2 * inv_mu * inv_mu / (float)C;
      }
    }
    g.sync();
    // ---- layer-norm backward -> d (t2); y2 (t1); product + normalisation backward -> dxr (t3), dy2 partial (t4)
    if (ew) {
      for (int r = rl; r < p.tr; r += p.ew_rows) {
        float o[B], dd[B];
        load_vec<B>(o, t1 + r * p.s1 + n_e * B);
        load_vec<B>(dd, t2 + r * p.s2 + n_e * B);
        {
          const float inv_mu = mu_s[r];
          float dot = 0.f;
#pragma unroll
          for (int i = 0; i < B; ++i) dot = fmaf(dd[i], o[i], dot);
          g_la = fmaf(dot, inv_mu, g_la);
          const float Q = mv_q<DIM, MET>(o, mp.qs);
          const float nu = smooth_abs_sqrt(Q);
          const float k1 = cp.la * inv_mu * kInvSqrt2;
          const float k2 = dmu_s[r] * Q / (nu * nu * nu) * kInvSqrt2;
#pragma unroll
          for (int i = 0; i < B; ++i) dd[i] = fmaf(k1, dd[i], k2 * qs_x<MET>(mp.qs, i, o[i]));  // d = do / sqrt2
        }
        store_vec<B>(t2 + r * p.s2 + n_e * B, dd);
        g_bl += dd[0];
        float y2[B], xr[B];
        {
          float sg[G], inv[G];
          load_vec<B>(y2, t4 + r * p.s2 + n_e * B);  // y1
          silu_gates<DIM, MET>(y2, cp.sa, cp.sb, sg, inv, mp.qs);
#pragma unroll
          for (int i = 0; i < B; ++i) y2[i] *= sg[A::grade_of(i)];
        }
        store_vec<B>(t1 + r * p.s1 + n_e * B, y2);
        load_vec<B>(xr, t3 + r * p.s3 + n_e * B);
        float q[G], nrm[G], rinv[G], xn[B], dxn[B], dy2[B];
        norm_factors<DIM, MET>(xr, cp.sn, q, nrm, rinv, mp.qs);
#pragma unroll
        for (int i = 0; i < B; ++i) { xn[i] = xr[i] * rinv[A::grade_of(i)]; dy2[i] = 0.f; dxn[i] = 0.f; }
        A::template wgp_bwd<MET>(y2, xn, cp.wv, dd, mp.mf, dy2, dxn, g_w);
        store_vec<B>(t4 + r * p.s2 + n_e * B, dy2);
        float t[G];
#pragma unroll
        for (int g = 0; g < G; ++g) t[g] = 0.f;
#pragma unroll
        for (int i = 0; i < B; ++i) t[A::grade_of(i)] = fmaf(dxn[i], xr[i], t[A::grade_of(i)]);
        float coef[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float ddn = -t[g] * rinv[g] * rinv[g];  // d loss / d denominator
          g_na[g] = fmaf(ddn * (nrm[g] - 1.f), cp.sn[g] * (1.f - cp.sn[g]), g_na[g]);
          coef[g] = ddn * cp.sn[g] * q[g] / (nrm[g] * nrm[g] * nrm[g]);
        }
#pragma unroll
        for (int i = 0; i < B; ++i) dxn[i] = fmaf(dxn[i], rinv[A::grade_of(i)], coef[A::grade_of(i)] * qs_x<MET>(mp.qs, i, xr[i]));
        store_vec<B>(t3 + r * p.s3 + n_e * B, dxn);  // dxr
      }
    }
    // ---- dy2 (t4) += D * WL + DXR * WR ;  dWL += D^T Y2 ; dWR += DXR^T Y2
    {
      constexpr int RB = FCfg<DIM>::RB;
      float acc[RB][NCH][B];
#pragma unroll
      for (int j = 0; j < RB; ++j)
#pragma unroll
        for (int a = 0; a < NCH; ++a)
#pragma unroll
          for (int i = 0; i < B; ++i) acc[j][a][i] = 0.f;
      gemm_run<DIM, true, NCH>(g, acc, t2 + rg * RB * p.s2, p.s2, wl, active, c, p.nc, 0, C);
      gemm_run<DIM, true, NCH>(g, acc, t3 + rg * RB * p.s3, p.s3, wr, active, c, p.nc, 0, C, !p.resident);
      if (active) {
#pragma unroll
        for (int a = 0; a < NCH; ++a) {
          const int o = c + a * p.nc;
          if (o >= C) continue;
#pragma unroll
          for (int j = 0; j < RB; ++j) {
            float* q = t4 + (rg * RB + j) * p.s2 + o * B;
            float old[B];
            load_vec<B>(old, q);
#pragma unroll
            for (int i = 0; i < B; ++i) old[i] += acc[j][a][i];
            store_vec<B>(q, old);
          }
        }
      }
    }
    dw_tile<DIM>(g, t2, p.s2, C, t1, p.s1, C, 0, C, p.tr, p.ks, my_dwl);
    dw_tile<DIM>(g, t3, p.s3, C, t1, p.s1, C, 0, C, p.tr, p.ks, my_dwr);
    // ---- TMA: y1 -> t2 again, the input row x0 -> t3 (sender rows through t1)
    fence_proxy_async();
    g.sync();  // generic accesses to t1, t2, t3 are done
    {
      RowPiece pc[5];
      pc[0] = RowPiece{t2, p.s2, 0, d.save_y1, C, nullptr};
      const int np = 1 + input_pieces<DIM>(pc + 1, t3, p.s3, t1, p.s1, d);
      tma_issue_pieces<DIM, 5>(g, pc, np, row0, valid, bar + 1);
    }
    mbar_wait(bar + 1, phase);
    phase ^= 1;
    finish_input_rows<DIM>(g, t3, p.s3, t1, p.s1, d, p.tr, valid);
    if (valid < p.tr) zero_tail_rows(g, t2, p.s2, (int)rowsz, p.tr, valid);
    g.sync();
    // ---- MVSiLU backward: dy1 -> t4
    if (ew) {
      for (int r = rl; r < p.tr; r += p.ew_rows) {
        float y1[B], dy[B], sg[G], inv[G], t[G];
        load_vec<B>(y1, t2 + r * p.s2 + n_e * B);
        load_vec<B>(dy, t4 + r * p.s2 + n_e * B);
        silu_gates<DIM, MET>(y1, cp.sa, cp.sb, sg, inv, mp.qs);
#pragma unroll
        for (int g = 0; g < G; ++g) t[g] = 0.f;
#pragma unroll
        for (int i = 0; i < B; ++i) t[A::grade_of(i)] = fmaf(dy[i], y1[i], t[A::grade_of(i)]);
        float ds[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
          ds[g] = t[g] * sg[g] * (1.f - sg[g]);
          g_sa[g] = fmaf(ds[g], inv[g], g_sa[g]);
          g_sb[g] += ds[g];
        }
#pragma unroll
        for (int i = 0; i < B; ++i) {
          const int g = A::grade_of(i);
          const float dinv = (g == 0) ? 1.f : 2.f * qs_x<MET>(mp.qs, i, y1[i]);
          dy[i] = fmaf(sg[g], dy[i], ds[g] * cp.sa[g] * dinv);
        }
        g_b1 += dy[0];
        store_vec<B>(t4 + r * p.s2 + n_e * B, dy);
      }
    }
    // ---- dx0 = DY1 * W1 in column blocks of C channels (straight to global);  dW1 += DY1^T X0
    for (int ob = 0; ob < cin; ob += C) {
      const int width = (cin - ob) < C ? (cin - ob) : C;
      if (width > (NCH - 1) * p.nc) {
        dx_pass<DIM, NCH>(g, t4, p.s2, p, w1, gr.grad_x, row0, valid, cin, ob, width, c, rg, active);
      } else {
        for (int o2 = 0; o2 < width; o2 += p.nc)
          dx_pass<DIM, 1>(g, t4, p.s2, p, w1, gr.grad_x, row0, valid, cin, ob + o2, (width - o2) < p.nc ? (width - o2) : p.nc, c,
                          rg, active);
      }
      dw_tile<DIM>(g, t4, p.s2, C, t3 + ob * B, p.s3, width, ob, cin, p.tr, p.ks, my_dw1);
    }
  }
  // ---- fixed-order reduction of the per-thread parameter gradients over the row lanes of the CTA
  {
    __syncthreads();
    float* red = smem;  // [threads]
    float* out = ws.small + (size_t)blockIdx.x * C * (P + 3 * G + 3);
    auto reduce_one = [&](float v, int offset, int Q, int q) {
      red[threadIdx.x] = ew ? v : 0.f;
      __syncthreads();
      if (threadIdx.x < C) {  // thread n sums the row lanes of every group in a fixed order
        float s = 0.f;
        for (int gi = 0; gi < p.ng; ++gi)
          for (int k = 0; k < p.ew_rows; ++k) s += red[gi * p.threads + k * C + threadIdx.x];
        out[offset + threadIdx.x * Q + q] = s;
      }
      __syncthreads();
    };
    int off = 0;
#pragma unroll
    for (int q = 0; q < P; ++q) reduce_one(g_w[q], off, P, q);
    off += C * P;
#pragma unroll
    for (int g = 0; g < G; ++g) reduce_one(g_na[g], off, G, g);
    off += C * G;
#pragma unroll
    for (int g = 0; g < G; ++g) reduce_one(g_sa[g], off, G, g);
    off += C * G;
#pragma unroll
    for (int g = 0; g < G; ++g) reduce_one(g_sb[g], off, G, g);
    off += C * G;
    reduce_one(g_la, off, 1, 0);
    off += C;
    reduce_one(g_b1, off, 1, 0);
    off += C;
    reduce_one(g_bl, off, 1, 0);
  }
}

template <int DIM, bool MET>
int run_block_fwd(const csmpn_block_desc& d, const FusedPlan& p, MetricArg<MET> mp, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    CSMPN_CUDA_TRY(cudaFuncSetAttribute(block_fwd_kernel<DIM, MET>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem + 1024));
    attr_set = true;
  }
  block_fwd_kernel<DIM, MET><<<p.grid, p.threads * p.ng, p.smem, s>>>(d, p, mp);
  CSMPN_LAUNCH_CHECK("block_fwd");
  return CSMPN_OK;
}

template <int DIM>
int launch_block_fwd(const csmpn_block_desc& d, cudaStream_t s) {
  FusedPlan p;
  int st = make_fused_plan<DIM>(d, false, &p);
  if (st) return st;
  MetricParams mp;
  if (block_metric(DIM, d, &mp)) return run_block_fwd<DIM, true>(d, p, mp, s);
  return run_block_fwd<DIM, false>(d, p, NoMetric{}, s);
}

template <int DIM>
int64_t block_bwd_ws_bytes(const csmpn_block_desc& d, FusedPlan* pp) {
  FusedPlan p;
  if (make_fused_plan<DIM>(d, true, &p)) return -1;
  if (pp) *pp = p;
  constexpr int G = Alg<DIM>::G, P = Alg<DIM>::P;
  const int64_t c = d.c, cin = d.c0 + d.c1 + d.c2;
  int64_t words = (int64_t)p.grid * ((int64_t)p.ng * p.ks * (c * cin * G + 2 * c * c * G) + c * (P + 3 * G + 3));
  return words * 4;
}

template <int DIM, bool MET>
int run_block_bwd(const csmpn_block_desc& d, const csmpn_block_grads& g, const FusedPlan& p, const BwdWorkspace& ws,
                  MetricArg<MET> mp, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    CSMPN_CUDA_TRY(cudaFuncSetAttribute(block_bwd_kernel<DIM, MET>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem + 1024));
    attr_set = true;
  }
  block_bwd_kernel<DIM, MET><<<p.grid, p.threads * p.ng, p.smem, s>>>(d, g, p, ws, mp);
  CSMPN_LAUNCH_CHECK("block_bwd");
  return CSMPN_OK;
}

template <int DIM>
int launch_block_bwd(const csmpn_block_desc& d, const csmpn_block_grads& g, void* workspace, int64_t bytes, cudaStream_t s) {
  FusedPlan p;
  int st;
  const int64_t need = block_bwd_ws_bytes<DIM>(d, &p);
  if (need < 0) return CSMPN_ERR_UNSUPPORTED;
  if (!workspace || bytes < need) return CSMPN_ERR_WORKSPACE;
  constexpr int G = Alg<DIM>::G, P = Alg<DIM>::P;
  const int c = d.c, cin = d.c0 + d.c1 + d.c2;
  BwdWorkspace ws;
  ws.dw1 = (float*)workspace;
  const size_t slots = (size_t)p.grid * p.ng * p.ks;
  ws.dwr = ws.dw1 + slots * c * cin * G;
  ws.dwl = ws.dwr + slots * c * c * G;
  ws.small = ws.dwl + slots * c * c * G;
  const size_t dw_bytes = (size_t)((char*)ws.small - (char*)workspace);
  CSMPN_CUDA_TRY(cudaMemsetAsync(workspace, 0, dw_bytes, s));  // the small partials are written, not accumulated
  MetricParams mp;
  st = block_metric(DIM, d, &mp) ? run_block_bwd<DIM, true>(d, g, p, ws, mp, s) : run_block_bwd<DIM, false>(d, g, p, ws, NoMetric{}, s);
  if (st) return st;
  // fixed-order sum of the per-CTA partials into the parameter gradients (one launch: 10 jobs)
  const int small_words = c * (P + 3 * G + 3);
  FinalJob jobs[10];
  memset(jobs, 0, sizeof(jobs));
  int k = 0;
  auto add = [&](const float* in, float* out, int n, int parts, int64_t stride) {
    jobs[k].in = in; jobs[k].out = out; jobs[k].n = n; jobs[k].parts = parts; jobs[k].stride = stride; ++k;  // kind 0
  };
  add(ws.dw1, g.g_w1, c * cin * G, (int)slots, (int64_t)c * cin * G);
  add(ws.dwr, g.g_wr, c * c * G, (int)slots, (int64_t)c * c * G);
  add(ws.dwl, g.g_wl, c * c * G, (int)slots, (int64_t)c * c * G);
  const float* sm = ws.small;
  add(sm, g.g_wp, c * P, p.grid, small_words); sm += c * P;
  add(sm, g.g_na, c * G, p.grid, small_words); sm += c * G;
  add(sm, g.g_sa, c * G, p.grid, small_words); sm += c * G;
  add(sm, g.g_sb, c * G, p.grid, small_words); sm += c * G;
  add(sm, g.g_la, c, p.grid, small_words); sm += c;
  add(sm, d.has_b1 ? g.g_b1 : nullptr, c, p.grid, small_words); sm += c;
  add(sm, g.g_bl, c, p.grid, small_words);
  return launch_final_reduce(jobs, k, s);
}

inline int check_desc(int dim, const csmpn_block_desc* d) {
  if (!d) return CSMPN_ERR_BAD_ARG;
  if (dim != 2 && dim != 3 && dim != 5) return CSMPN_ERR_UNSUPPORTED;
  if (d->rows < 0 || d->c <= 0 || d->c0 <= 0 || d->c1 < 0 || d->c2 < 0) return CSMPN_ERR_BAD_ARG;
  if (d->mode == 2 && d->engine != 1) return CSMPN_ERR_UNSUPPORTED;  // the vertex-table gather lives in the tensor-core engine
  if (d->mode != 0 && d->mode != 1 && d->mode != 2) return CSMPN_ERR_BAD_ARG;
  if (!d->p0 || (d->c1 > 0 && !d->p1) || (d->c2 > 0 && !d->p2)) return CSMPN_ERR_BAD_ARG;
  if (d->mode == 1 && (!d->src || !d->dst || (d->c1 > 0 && !d->eid && !d->pair_attr) || d->c2 != 0)) return CSMPN_ERR_BAD_ARG;
  if (d->pair_attr && (d->mode != 1 || (d->c1 & 1))) return CSMPN_ERR_BAD_ARG;
  if (!d->w1 || !d->sa || !d->sb || !d->wr || !d->na || !d->wl || !d->bl || !d->wp || !d->la) return CSMPN_ERR_BAD_ARG;
  if (d->has_b1 && !d->b1) return CSMPN_ERR_BAD_ARG;
  if (d->tf32 != 0 && d->tf32 != 1) return CSMPN_ERR_BAD_ARG;
  if (d->metric)  // degenerate metrics (a zero entry) change the grade-path set of the product: unit kernels only
    for (int i = 0; i < dim; ++i)
      if (d->metric[i] == 0.f) return CSMPN_ERR_UNSUPPORTED;
  return CSMPN_OK;
}

}  // namespace csmpn

namespace csmpn {
// tensor-core engine (tc_block_fwd.cu / tc_block_bwd.cu)
int tc_block_fwd(int dim, const csmpn_block_desc* d, cudaStream_t stream);
int tc_block_bwd(int dim, const csmpn_block_desc* d, const csmpn_block_grads* g, void* ws, int64_t bytes, cudaStream_t stream);
int64_t tc_block_bwd_workspace(int dim, const csmpn_block_desc* d);
int64_t tc_block_fwd_workspace(int dim, const csmpn_block_desc* d);
int tc_block_plan(int dim, int c_in, int c);
int tc_block_passes(int dim, int c_in, int c);
bool tc_block_supported(int dim, int c_in, int c);
}  // namespace csmpn

using namespace csmpn;

extern "C" {

int csmpn_block_tc_supported(int dim, int c_in, int c) { return tc_block_supported(dim, c_in, c) ? 1 : 0; }
int csmpn_block_tc_plan(int dim, int c_in, int c) { return tc_block_plan(dim, c_in, c); }
int csmpn_block_tc_passes(int dim, int c_in, int c) { return tc_block_passes(dim, c_in, c); }

// > 0 (= rows per shared-memory tile) if the FP32 SIMT engine keeps the three weight matrices of such a block resident in shared memory for both the forward
// and the backward kernel; 0 if it would fall back to staging them per GEMM (slower than the unit kernels: callers
// then compose the block from csmpn_mvlinear_* / csmpn_mvsilu_* / ... instead)
int csmpn_block_simt_resident(int dim, int c_in, int c) {
  csmpn_block_desc d;
  memset(&d, 0, sizeof(d));
  d.c0 = c_in; d.c = c; d.rows = 1;
  FusedPlan pf, pb;
  int sf, sb;
  switch (dim) {
    case 2: sf = make_fused_plan<2>(d, false, &pf); sb = make_fused_plan<2>(d, true, &pb); break;
    case 3: sf = make_fused_plan<3>(d, false, &pf); sb = make_fused_plan<3>(d, true, &pb); break;
    case 5: sf = make_fused_plan<5>(d, false, &pf); sb = make_fused_plan<5>(d, true, &pb); break;
    default: return 0;
  }
  if (!(sf == CSMPN_OK && sb == CSMPN_OK && pf.resident && pb.resident)) return 0;
  return pf.tr < pb.tr ? pf.tr : pb.tr;  // rows per tile that still fit next to the resident weights
}

int64_t csmpn_bpt_floats(int dim, int64_t rows, int channels) {
  if (dim < 1 || dim > 5 || rows < 0 || channels < 1) return -1;
  const int64_t cp = (channels + 15) / 16 * 16;
  return ((rows + 127) / 128) * (int64_t)(1 << dim) * cp * 128;
}

int csmpn_block_fwd(int dim, const csmpn_block_desc* desc, csmpn_stream_t stream) {
  int st = check_desc(dim, desc);
  if (st) return st;
  if (!desc->y) return CSMPN_ERR_BAD_ARG;
  if (desc->rows == 0) return CSMPN_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (desc->engine == 1) return tc_block_fwd(dim, desc, s);
  switch (dim) {
    case 2: return launch_block_fwd<2>(*desc, s);
    case 3: return launch_block_fwd<3>(*desc, s);
    case 5: return launch_block_fwd<5>(*desc, s);
  }
  return CSMPN_ERR_UNSUPPORTED;
}

int64_t csmpn_block_fwd_workspace(int dim, const csmpn_block_desc* desc) {
  if (check_desc(dim, desc)) return -1;
  return desc->engine == 1 ? tc_block_fwd_workspace(dim, desc) : 0;
}

int64_t csmpn_block_bwd_workspace(int dim, const csmpn_block_desc* desc) {
  if (check_desc(dim, desc)) return -1;
  if (desc->engine == 1) return tc_block_bwd_workspace(dim, desc);
  switch (dim) {
    case 2: return block_bwd_ws_bytes<2>(*desc, nullptr);
    case 3: return block_bwd_ws_bytes<3>(*desc, nullptr);
    case 5: return block_bwd_ws_bytes<5>(*desc, nullptr);
  }
  return -1;
}

int csmpn_block_bwd(int dim, const csmpn_block_desc* desc, const csmpn_block_grads* grads, void* workspace,
                    int64_t workspace_bytes, csmpn_stream_t stream) {
  int st = check_desc(dim, desc);
  if (st) return st;
  if (!grads || !grads->grad_y || !desc->save_y1 || !desc->save_xr || !desc->save_o) return CSMPN_ERR_BAD_ARG;
  if (!grads->g_w1 || !grads->g_sa || !grads->g_sb || !grads->g_wr || !grads->g_na || !grads->g_wl || !grads->g_bl ||
      !grads->g_wp || !grads->g_la)
    return CSMPN_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (desc->engine == 1) return tc_block_bwd(dim, desc, grads, workspace, workspace_bytes, s);
  switch (dim) {
    case 2: return launch_block_bwd<2>(*desc, *grads, workspace, workspace_bytes, s);
    case 3: return launch_block_bwd<3>(*desc, *grads, workspace, workspace_bytes, s);
    case 5: return launch_block_bwd<5>(*desc, *grads, workspace, workspace_bytes, s);
  }
  return CSMPN_ERR_UNSUPPORTED;
}

}  // extern "C"
