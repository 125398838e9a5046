// Shared definitions of the tensor-core CEMLP-block kernels (tc_block_fwd.cu, tc_block_bwd.cu).
//
// BPT ("blade-plane tile") tensor layout, used for every intermediate of the tensor-core path:
//     [tile = row / 128][blade][channel / 4][row % 128][channel % 4]      fp32, channels padded to Cp (multiple of 16)
// * one (tile, blade, 8-channel chunk) is 4 KB contiguous and already in the UMMA no-swizzle K-major operand layout,
//   so a GEMM kernel brings it in with two bulk copies and no transposition;
// * a thread that owns one row reads/writes 4 channels of a blade as one float4, and consecutive lanes (rows) touch
//   consecutive 16-byte units: every epilogue access is perfectly coalesced.
// Padded rows and padded channels always hold zeros.
#pragma once
#include "tc_common.cuh"

namespace csmpn {
namespace tcb {
using namespace tc;

constexpr int kTile = 128;     // rows per tile = UMMA M
constexpr int kThreads = 512;  // 16 warps: warp w owns TMEM lanes 32*(w%4).., channel groups (w/4), (w/4)+4, ...
constexpr float kInvSqrt2 = 0.70710678118654752440f;

// chunk buffer (one K step of 8 channels, all blades): hi planes then lo planes.  A plane is [2][128][4] fp32, 4 KB
// contiguous exactly as in a BPT tensor, so ONE bulk copy brings a blade of a chunk in (cp.async.bulk is issued from
// the uniform datapath: per-lane addresses serialise at ~70 cycles per copy, so fewer and larger copies matter).
// Planes are PS apart; the 16-byte pad makes the scalar stores of the transposing producer (lanes = 4 channels x 4
// rows x 2 blade quads) hit all 32 banks.
constexpr uint32_t kKH = 2048;
constexpr uint32_t kPS = 2 * kKH + 16;

__host__ __device__ constexpr int round_up(int x, int m) { return (x + m - 1) / m * m; }
__host__ __device__ constexpr int64_t bpt_floats(int B, int64_t rows, int cp) {
  return ((rows + kTile - 1) / kTile) * (int64_t)B * cp * kTile;
}
// float offset of (tile, blade, channel group c4, row r) -> 4 consecutive channels
__device__ __forceinline__ size_t bpt_off(int B, int cp, int64_t tile, int b, int c4, int r) {
  return ((((size_t)tile * B + b) * (cp >> 2) + c4) * kTile + r) * 4;
}

// Approximate SFU forms (rcp / sqrt / ex2 .approx: <= 2 ulp) instead of the IEEE-rounded sequences of sqrtf, expf and
// '/': each of those costs 8-20 instructions and the elementwise stages evaluate ~15 of them per multivector.  Their
// error (2^-22) is an order of magnitude below the fp32 parity budget (1e-5 forward, 1e-4 gradients).
__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sqrt(float x) { float y; asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_ex2(float x) { float y; asm("ex2.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sigmoid(float v) { return fast_rcp(1.f + fast_ex2(-1.4426950408889634f * v)); }
// (q^2 + 1e-16)^(1/4)
__device__ __forceinline__ float fast_sas(float q) { return fast_sqrt(fast_sqrt(fmaf(q, q, kSmoothEps))); }

template <int DIM>
__device__ __forceinline__ void silu_gates(const float* y1, const float* a, const float* b, float* sg, float* inv) {
  using A = Alg<DIM>;
#pragma unroll
  for (int g = 0; g < A::G; ++g) inv[g] = 0.f;
#pragma unroll
  for (int i = 0; i < A::B; ++i) inv[A::grade_of(i)] = fmaf(y1[i], y1[i], inv[A::grade_of(i)]);
  inv[0] = y1[0];
#pragma unroll
  for (int g = 0; g < A::G; ++g) sg[g] = fast_sigmoid(fmaf(a[g], inv[g], b[g]));
}

// normalisation: xn_i = xr_i * rinv[g];  den_g = s_g (nrm_g - 1) + 1 + eps
template <int DIM>
__device__ __forceinline__ void norm_factors(const float* xr, const float* s, float* q, float* nrm, float* rinv) {
  using A = Alg<DIM>;
#pragma unroll
  for (int g = 0; g < A::G; ++g) q[g] = 0.f;
#pragma unroll
  for (int i = 0; i < A::B; ++i) q[A::grade_of(i)] = fmaf(xr[i], xr[i], q[A::grade_of(i)]);
#pragma unroll
  for (int g = 0; g < A::G; ++g) {
    nrm[g] = fast_sas(q[g]);
    rinv[g] = fast_rcp(fmaf(s[g], nrm[g] - 1.f, 1.f) + kEps);
  }
}

template <int DIM>
__device__ __forceinline__ float mv_sumsq(const float* x) {
  float Q = 0.f;
#pragma unroll
  for (int i = 0; i < Alg<DIM>::B; ++i) Q = fmaf(x[i], x[i], Q);
  return Q;
}

// Numeric mode of the GEMM kernels: TERMS = 3 is the error-compensated split (hi*hi + hi*lo + lo*hi, fp32 accuracy, the
// default); TERMS = 1 is single-pass TF32 (csmpn_block_desc.tf32): every operand rounded to nearest TF32 once, one MMA
// per product, no `lo` operands.  Weight images per grade: hi and lo, or the rounded weight alone.
__host__ __device__ constexpr int n_images(int terms) { return terms == 1 ? 1 : 2; }

// Stage [c_out, c_in, G] weights (global, reference layout) as NI*G operand images each in shared memory (NI =
// n_images(TERMS)):
//   image (g, hl) = plane with R = rows_p rows;  TRANS == false: row = output channel, column = input channel
//                                                TRANS == true : row = input channel,  column = output channel
// TERMS = 3: hl = 0: TF32-exact high part, hl = 1: remainder.  TERMS = 1: the weight rounded to nearest TF32.
// Rows/columns beyond the real sizes are zero.
// A job = one weight: its image set (img0), its first plane row (two weights can share one image set: rows [0, n) and
// [n, 2n)).  [zero_base, zero_base + zero_bytes) -- all image sets of the call, contiguous -- is cleared first.
// The prologue of every GEMM kernel runs this once per CTA, and a one-tile-per-CTA launch (every per-simplex block) pays
// for it in full: the global loads are therefore issued in batches of 8 per thread, the first batch BEFORE the zero
// fill and the barrier, so that one L2/HBM latency is exposed per batch instead of one per element (the element-wise loop
// took 8-9 us of a 22 us single-tile kernel, profiles/r02_f2_timeline_prologue.log).
struct WJob {
  uint8_t* img0;
  const float* w;
  int c_out, c_in, row0;
};
// Work unit = one 8-row x 4-column block of a weight's image plane, one warp per unit: lane = (row % 8) * 4 + column % 4,
// so the 32 stores of one (grade, hi/lo) image are 128 contiguous bytes (conflict-free) and a lane's G grades of one
// (output, input) pair are one 16-byte load when G == 4.  Units of up to two weights are walked in one flat index space,
// four units per warp in flight.
template <int DIM, bool TRANS, int NJ, int TERMS = 3>
__device__ __forceinline__ void stage_weight_jobs(const WJob (&j)[NJ], int njobs, uint32_t img_bytes, int rows_p, int cols_p,
                                                  uint8_t* zero_base, uint32_t zero_bytes) {
  static_assert(NJ == 1 || NJ == 2, "one or two weights per call");
  static_assert(TERMS == 1 || TERMS == 3, "split or single-pass products");
  constexpr int G = Alg<DIM>::G, U = 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int rl = lane >> 2, cl = lane & 3;
  // job fields are selected with ?: (dynamic indexing of the job array would put it in local memory)
  const WJob& j0 = j[0];
  const WJob& j1 = j[NJ - 1];
  const bool two = NJ == 2 && njobs > 1;
  const int R0 = TRANS ? j0.c_in : j0.c_out, C0 = TRANS ? j0.c_out : j0.c_in;
  const int R1 = TRANS ? j1.c_in : j1.c_out, C1 = TRANS ? j1.c_out : j1.c_in;
  const int ncb0 = (C0 + 3) >> 2, ncb1 = (C1 + 3) >> 2;
  const int nb0 = ((R0 + 7) >> 3) * ncb0, nb1 = two ? ((R1 + 7) >> 3) * ncb1 : 0;
  const int total = nb0 + nb1;
  // unit -> (second job?, row, column, valid)
  auto decode = [&](int wb, bool& sj, int& row, int& col) -> bool {
    if (wb >= total) return false;
    sj = wb >= nb0;
    if (sj) wb -= nb0;
    const int ncb = sj ? ncb1 : ncb0;
    const int rb = wb / ncb, cb = wb - rb * ncb;
    row = rb * 8 + rl;
    col = cb * 4 + cl;
    return row < (sj ? R1 : R0) && col < (sj ? C1 : C0);
  };
  auto fetch = [&](int wb, float* v) {
#pragma unroll
    for (int g = 0; g < G; ++g) v[g] = 0.f;
    bool sj;
    int row, col;
    if (!decode(wb, sj, row, col)) return;
    const int o = TRANS ? col : row, i = TRANS ? row : col;
    const float* src = (sj ? j1.w : j0.w) + ((size_t)o * (sj ? j1.c_in : j0.c_in) + i) * G;
    if (G == 4 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(src));
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[G - 1] = x.w;
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g) v[g] = __ldg(src + g);
    }
  };
  auto put = [&](int wb, const float* v) {
    bool sj;
    int row, col;
    if (!decode(wb, sj, row, col)) return;
    const int r = (sj ? j1.row0 : j0.row0) + row;
    if (r >= rows_p || col >= cols_p) return;
    uint8_t* dst = (sj ? j1.img0 : j0.img0) + plane_off(rows_p, r, col);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if constexpr (TERMS == 1) {
        *reinterpret_cast<float*>(dst + (size_t)g * img_bytes) = tf32_rna(v[g]);
      } else {
        const float hi = tf32_hi(v[g]);
        *reinterpret_cast<float*>(dst + (size_t)(g * 2 + 0) * img_bytes) = hi;
        *reinterpret_cast<float*>(dst + (size_t)(g * 2 + 1) * img_bytes) = v[g] - hi;
      }
    }
  };
  float x[U][G];
#pragma unroll
  for (int u = 0; u < U; ++u) fetch(warp + u * nwarps, x[u]);  // in flight across the zero fill and the barrier
  for (uint32_t i = threadIdx.x; i < (zero_bytes >> 4); i += blockDim.x)
    reinterpret_cast<float4*>(zero_base)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  for (int base = 0; base < total; base += U * nwarps) {
    float nx[U][G];
    const int nbase = base + U * nwarps;
    if (nbase < total) {
#pragma unroll
      for (int u = 0; u < U; ++u) fetch(nbase + warp + u * nwarps, nx[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) put(base + warp + u * nwarps, x[u]);
    if (nbase < total) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int g = 0; g < G; ++g) x[u][g] = nx[u][g];
      }
    }
  }
}
// one weight into its own image set (cleared first)
template <int DIM, bool TRANS, int TERMS = 3>
__device__ __forceinline__ void stage_weight_images(uint8_t* img0, uint32_t img_bytes, const float* __restrict__ w, int c_out,
                                                    int c_in, int rows_p, int cols_p) {
  const WJob j[1] = {{img0, w, c_out, c_in, 0}};
  stage_weight_jobs<DIM, TRANS, 1, TERMS>(j, 1, img_bytes, rows_p, cols_p, img0,
                                          (uint32_t)Alg<DIM>::G * (uint32_t)n_images(TERMS) * img_bytes);
}

// A-operand descriptors of blade b in a chunk buffer half
__device__ __forceinline__ uint64_t chunk_desc(uint32_t half_saddr, int b) {
  return smem_desc(half_saddr + (uint32_t)b * kPS, kKH, 128u);
}

// ---- persistent CTAs, TMEM, prologue and teardown (every tcgen05 kernel) -----------------------------------------------
// One CTA per SM; this CTA runs tiles blockIdx.x, blockIdx.x + gridDim.x, ...
__device__ __forceinline__ int cta_tiles(int tiles) { return (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x; }
__device__ __forceinline__ int64_t cta_tile(int t) { return (int64_t)blockIdx.x + (int64_t)t * gridDim.x; }
// tcgen05.alloc takes a power of two >= 32 columns
__host__ __device__ constexpr uint32_t tmem_cols(uint32_t need) {
  return need <= 32 ? 32 : need <= 64 ? 64 : need <= 128 ? 128 : need <= 256 ? 256 : 512;
}
// End of the prologue: the barrier inits, the TMEM address written by tcgen05.alloc and the generic-proxy stores of the
// staged weights are visible to every thread and to the tensor cores.
__device__ __forceinline__ void prologue_sync() {
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
}
// End of the kernel: every warp's TMEM accesses are complete before the allocating warp 0 frees the columns.
__device__ __forceinline__ void tmem_teardown(int warp, uint32_t tbase, uint32_t tcols) {
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, tcols);
}

constexpr size_t kSmemMax = 227 * 1024;  // dynamic shared memory of one CTA
// The ring-fed kernels are persistent with one CTA per SM (grid = min(tiles, SMs)) and size their TMEM allocation for an SM
// of their own.  Several single-pass TF32 instantiations use <= 64 registers, so registers alone would let two 512-thread
// CTAs share an SM (and wait on each other's TMEM) while other SMs idle: their smaller shared-memory requests are raised
// to more than half of the SM's 228 KB (1 KB reserved per CTA), which keeps a second CTA off the SM.
constexpr size_t kOneCtaPerSm = 116 * 1024;
__host__ inline size_t one_cta_per_sm(size_t smem) { return smem < kOneCtaPerSm ? kOneCtaPerSm : smem; }

// ---- K-chunk pipeline of the ring-fed kernels (tc_f1, tc_f1db, tc_f2, tc_bgemm, tc_bgemmdb) ----------------------------
// A chunk = 8 channels of all blades of a 128-row tile.  Chunk q lands (bulk copies) in raw slot q % kRing; the split
// pass turns the slot into the TF32-exact high parts in place and writes the remainders to the single `lo` buffer;
// the MMAs of the chunk read both.  Loads run kRing-1 chunks ahead of the MMAs (two chunks = 64 KB per SM in flight).
// Single-pass TF32 (TERMS = 1): the conversion pass rounds the slot to nearest TF32 in place and the MMAs read the slot
// alone; `lo` and lo_bar are left unused.
//
// Roles during the K loop: warp 0 is the ISSUER (bulk copies + MMAs, nothing else); warps 1..15 are CONVERTERS (split
// pass / gathering producer).  They are decoupled by mbarriers only -- no CTA-wide barrier inside the K loop -- so the
// conversion of chunk q+1 overlaps the issue and execution of the MMAs of chunk q.  Every warp takes part in the tile
// epilogue.
// tcgen05.mma kind::tf32 reads fp32 operands and ignores the low 13 mantissa bits (truncation, verified on B200 by the
// 1e-5 parity tests, which a round-to-nearest read would fail by 2^-11): the raw chunk already IS the high operand, so the
// split pass only has to produce the remainders.  For the same reason single-pass TF32 rounds (cvt.rna) explicitly: raw
// fp32 operands would bias every product toward zero.
//
// Reuse rules (nothing but these mbarriers orders the K loop):
// * Raw slot q % kRing is overwritten by chunk q + kRing only once slot_bar has seen the MMAs of chunk q complete:
//   ChunkFeed::refill / refill_all for bulk copies, Pipe::wait_free(q - kRing) for the gathering producer's stores.
// * `lo` is rewritten for chunk q once lo_bar has seen the MMAs of chunk q-1 complete (split_chunk, store_chunk_api).
//   TERMS = 1 has no `lo`: the rounding pass writes only the raw slot, which the first rule already protects.
// * An accumulator is read (tcgen05.ld) only after wait_mmas of the last chunk that wrote it.  It is overwritten by the
//   first MMA of a later pass or tile, which the issuer issues only after wait_full of that chunk; every converter warp
//   arrives on full_bar (conv_done) after its own epilogue loads (tcgen05.wait::ld), and the issuer warp runs its part
//   of a plain epilogue itself, so the mbarrier orders the reuse.  The overlapped kernels alternate two accumulator
//   buffers by tile (PendingEpilogue).
constexpr bool kTf32Truncates = true;
constexpr int kRing = 3;
constexpr int kPipeBars = 3 * kRing + 1;
constexpr int kConvWarps = kThreads / 32 - 1;
constexpr int kConv = kConvWarps * 32;
struct Pipe {
  uint8_t* raw;        // kRing slots of `half` bytes
  uint8_t* lo;         // one slot
  uint64_t* load_bar;  // [kRing] the bulk copies of the chunk have landed
  uint64_t* slot_bar;  // [kRing] every MMA reading the slot has completed
  uint64_t* full_bar;  // [kRing] every converter warp has finished the chunk in this slot (count kConvWarps)
  uint64_t* lo_bar;    // [1]     the MMAs reading `lo` have completed
  uint32_t half;
  __device__ __forceinline__ uint8_t* slot(int q) const { return raw + (size_t)(q % kRing) * half; }
  __device__ __forceinline__ void init(uint8_t* base, uint64_t* bars, uint32_t half_bytes) {
    raw = base; lo = base + (size_t)kRing * half_bytes; half = half_bytes;
    load_bar = bars; slot_bar = bars + kRing; full_bar = bars + 2 * kRing; lo_bar = bars + 3 * kRing;
    if (threadIdx.x == 0) {
      for (int i = 0; i < kPipeBars; ++i) mbar_init(&bars[i], (i >= 2 * kRing && i < 3 * kRing) ? kConvWarps : 1);
      mbar_fence_init();
    }
  }
  // converter warps: this warp's part of chunk q is in shared memory (generic-proxy writes made visible to the MMAs)
  __device__ __forceinline__ void conv_done(int q) const {
    fence_async_smem();
    fence_before_sync();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&full_bar[q % kRing]);
  }
  // issuer warp: wait until chunk q is complete in shared memory
  __device__ __forceinline__ void wait_full(int q) const {
    mbar_wait(&full_bar[q % kRing], (q / kRing) & 1);
    fence_after_sync();
  }
  // the bulk copies of chunk q (activation planes and / or weight unit) have landed in its slot
  __device__ __forceinline__ void wait_landed(int q) const { mbar_wait(&load_bar[q % kRing], (q / kRing) & 1); }
  // the MMAs of chunk q have completed: its slot may be overwritten
  __device__ __forceinline__ void wait_free(int q) const { mbar_wait(&slot_bar[q % kRing], (q / kRing) & 1); }
  // ... and, with those of every earlier chunk, written their accumulators: tcgen05.ld may read them
  __device__ __forceinline__ void wait_mmas(int q) const {
    wait_free(q);
    fence_after_sync();
  }
};

// Copy-ahead of the issuer warp (all lanes of warp 0): chunk loads run kRing - 1 chunks ahead of the MMAs.  `load(q)`
// issues the bulk copies of the CTA's chunk q; `total` = chunks of this CTA.  ON == false (no bulk copies: gathered
// input with resident weights) compiles every call away.  The loader is an argument of each call rather than a member:
// a struct holding the lambda (or a reference to it) made nvcc widen shared-memory address arithmetic to 64 bits and
// cost the streamed-weight kernels 3 to 7 registers.
template <bool ON = true>
struct ChunkFeed {
  const Pipe& p;
  int total;
  int loaded = 0;  // chunks whose copies have been issued
  // The first kRing - 1 chunks, requested BEFORE the weights are staged: with one to three tiles per CTA the prologue is
  // a visible part of the kernel and these latencies overlap it.
  template <class Load>
  __device__ __forceinline__ void prime(Load&& load) {
    if (ON) for (; loaded < kRing - 1 && loaded < total; ++loaded) load(loaded);
  }
  // After wait_full(q): slot (q-1) % kRing was read by the MMAs of chunk q-1, issued a whole chunk period ago; reload it
  // before issuing the MMAs of chunk q, so that the copy has their issue time as extra lead.
  template <class Load>
  __device__ __forceinline__ void refill(int q, Load&& load) {
    if (ON && loaded == q + kRing - 1 && loaded < total) {
      if (q >= 1) p.wait_free(q - 1);
      load(loaded);
      ++loaded;
    }
  }
  // After wait_mmas(q - 1) at the end of a pass: every slot is free; prefetch the next chunks under the epilogue.
  template <class Load>
  __device__ __forceinline__ void refill_all(int q, Load&& load) {
    if (ON) for (; loaded < q + kRing && loaded < total; ++loaded) load(loaded);
  }
};

// ---- overlapped epilogue (tc_f1db_kernel, tc_bgemmdb_kernel) ---------------------------------------------------------
// Accumulators alternate between two TMEM buffers by tile.  The epilogue of tile t-1 stays pending on each epilogue warp
// (warps 4-15: lane quadrant warp & 3, channel groups (warp >> 2) - 1, + 3, ...) while the K loop of tile t runs; the
// warp runs one channel-group unit of it, unit(tile, c4, tb), between two of its chunks.
struct PendingEpilogue {
  int64_t tile = -1;  // nothing pending
  int c4 = 0;         // next channel group
  int q = 0;          // last chunk of the pending tile
  uint32_t tb = 0;    // its accumulator buffer
  bool ready = false;
  // after the K loop of `t` (last chunk last_q, accumulators at buf); warps 0-3 never run the epilogue
  __device__ __forceinline__ void start(int warp, int64_t t, int last_q, uint32_t buf) {
    if (warp >= 4) { tile = t; c4 = (warp >> 2) - 1; q = last_q; tb = buf; ready = false; }
  }
  // at most one unit
  template <class Unit>
  __device__ __forceinline__ void step(const Pipe& p, int n_c4, Unit&& unit) {
    if (tile < 0) return;
    if (!ready) {  // the MMAs of the pending tile have completed (its last chunk released its slot)
      p.wait_mmas(q);
      ready = true;
    }
    if (c4 < n_c4) {
      unit(tile, c4, tb);
      c4 += 3;
    }
    if (c4 >= n_c4) { tile = -1; fence_before_sync(); }
  }
  // Called at the end of each K loop: the previous tile's epilogue must be finished before this warp signals the next
  // tile's first chunk (conv_done).  The issuer waits for that full_bar before the first MMA of the next tile, which
  // overwrites the buffer this epilogue reads.
  template <class Unit>
  __device__ __forceinline__ void drain(const Pipe& p, int n_c4, Unit&& unit) {
    while (tile >= 0) step(p, n_c4, unit);
  }
};

// ---- streamed weights (wide blocks) --------------------------------------------------------------------------------
// When the weight images of a GEMM do not fit shared memory next to the chunk ring (Cl(3,0) with C >= 64), the weights
// are streamed WITH the activations: a raw slot holds the activation chunk followed by the "weight unit" of the same K
// chunk -- for every grade the hi and lo images of [R output rows x 8 input channels] (plane layout with R rows) --
// brought in by ONE more bulk copy from a pre-split image buffer in global memory (tc_weight_images_kernel), laid out
// unit after unit in the order the kernel walks them: [pass][K chunk][grade][hi | lo][2][R][4] floats.  Single-pass
// TF32: [pass][K chunk][grade][2][R][4], the rounded weight alone (nimg = 1), half the bytes.
template <int DIM>
__host__ __device__ constexpr uint32_t wunit_bytes(int rows, int nimg = 2) {
  return (uint32_t)Alg<DIM>::G * (uint32_t)nimg * (uint32_t)rows * 32u;
}

// bulk copies of chunk q: the activation planes (bpt != nullptr) and the weight unit; called by ALL lanes of one warp
template <int B>
__device__ __forceinline__ void issue_chunk_load_w(const Pipe& p, int q, const float* bpt, int cp, int64_t tile, int kc,
                                                   const uint8_t* wsrc, uint32_t wbytes) {
  const int lane = threadIdx.x & 31;
  uint64_t* bar = &p.load_bar[q % kRing];
  if (lane == 0) mbar_arrive_expect_tx(bar, (bpt ? B * 4096u : 0u) + wbytes);
  __syncwarp();
  if (bpt && lane < B) bulk_g2s(p.slot(q) + lane * kPS, bpt + bpt_off(B, cp, tile, lane, 2 * kc, 0), 4096u, bar);
  if (lane == B) bulk_g2s(p.slot(q) + B * kPS, wsrc, wbytes, bar);
}

// Pre-split weight images in global memory for the streamed mode.  One element per thread.
//   stack = 1: two weights share every unit along the rows ([0, np): w0 rows of the pass, [np, 2 np): w1 rows), one K range
//   stack = 0: w1 (if any) is a second K range after w0's chunks (the two-source GEMM of the backward)
//   trans = 0: w is [n_real][k_real][G] (image row = output channel n, column = input channel k)
//   trans = 1: w is [k_real][n_real][G]
struct WPrepArgs {
  const float *w0, *w1;
  int stack, trans, n_real, k_real0, k_real1, np, npass, nk0, nk1;
  float* out;
};
template <int DIM, int TERMS = 3>
__global__ void tc_weight_images_kernel(WPrepArgs a) {
  constexpr int G = Alg<DIM>::G, NI = n_images(TERMS);
  const int R = a.stack ? 2 * a.np : a.np;
  const int nk = a.nk0 + (a.stack ? 0 : a.nk1);
  const int64_t total = (int64_t)a.npass * nk * G * NI * R * 8;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e & 3), r = (int)((e >> 2) % R), cu = (int)((e / (4 * R)) & 1), hl = NI == 2 ? (int)((e / (8 * R)) & 1) : 0;
    const int g = (int)((e / (8 * NI * R)) % G);
    const int u = (int)(e / ((int64_t)8 * NI * R * G)), ps = u / nk, kc = u % nk;
    const int second_k = (!a.stack && kc >= a.nk0) ? 1 : 0;
    const int k = (second_k ? kc - a.nk0 : kc) * 8 + cu * 4 + c;
    const int k_real = second_k ? a.k_real1 : a.k_real0;
    const float* w = a.stack ? (r < a.np ? a.w0 : a.w1) : (second_k ? a.w1 : a.w0);
    const int n = ps * a.np + (a.stack ? r % a.np : r);
    float x = 0.f;
    if (w && n < a.n_real && k < k_real) x = a.trans ? w[((size_t)k * a.n_real + n) * G + g] : w[((size_t)n * k_real + k) * G + g];
    if constexpr (TERMS == 1) {
      a.out[e] = tf32_rna(x);
    } else {
      const float hi = tf32_hi(x);
      a.out[e] = hl ? x - hi : hi;
    }
  }
}
template <int DIM>
__host__ inline int64_t weight_image_floats(int stack, int np, int npass, int nk_total, int nimg = 2) {
  return (int64_t)npass * nk_total * Alg<DIM>::G * nimg * (stack ? 2 * np : np) * 8;
}
template <int DIM, int TERMS = 3>
__host__ int launch_weight_images(const WPrepArgs& w, int64_t floats, cudaStream_t stream) {
  int64_t blocks = (floats + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  tc_weight_images_kernel<DIM, TERMS><<<(unsigned)blocks, 256, 0, stream>>>(w);
  CSMPN_LAUNCH_CHECK("tc_weight_images_kernel");
  return CSMPN_OK;
}

// The overlapped-epilogue kernels (tc_f1db, tc_bgemmdb) need two accumulator buffers of B * ncols columns in TMEM.
// CSMPN_TC_OVERLAP=0 selects the plain kernels (epilogue after the K loop); read per call so a test can compare both.
__host__ inline bool use_overlapped_epilogue(int B, int ncols) {
  if (2 * B * ncols > 512) return false;
  const char* e = getenv("CSMPN_TC_OVERLAP");
  return !(e && e[0] == '0');
}

// bulk copies of chunk q (8 channels kc of a BPT tensor) into its raw slot: called by ALL lanes of one warp
template <int B>
__device__ __forceinline__ void issue_chunk_load(const Pipe& p, int q, const float* bpt, int cp, int64_t tile, int kc) {
  const int lane = threadIdx.x & 31;
  uint64_t* bar = &p.load_bar[q % kRing];
  if (lane == 0) mbar_arrive_expect_tx(bar, B * 4096u);
  __syncwarp();
  if (lane < B) bulk_g2s(p.slot(q) + lane * kPS, bpt + bpt_off(B, cp, tile, lane, 2 * kc, 0), 4096u, bar);
}
// split pass over the landed chunk q (CONVERTER warps only): high parts in place, remainders to `lo`.  The remainders
// wait in registers until the MMAs of chunk q-1 (the previous readers of `lo`) have completed, so reading the chunk,
// splitting it and storing the high parts overlap those MMAs.  Ends with conv_done(q).
// TERMS = 1: rounds the chunk to nearest TF32 in place; no `lo`, no lo_bar wait.
template <int B, int TERMS = 3>
__device__ __forceinline__ void split_chunk(const Pipe& p, int q) {
  uint8_t* hi = p.slot(q);
  constexpr int TOT = B * 2 * kTile;
  constexpr int N = (TOT + kConv - 1) / kConv;
  const int ct = (int)threadIdx.x - 32;
  if constexpr (TERMS == 1) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const int it = ct + i * kConv;
      if (it < TOT) {
        const int r = it & (kTile - 1), kh = (it >> 7) & 1, b = it >> 8;
        float4* x = reinterpret_cast<float4*>(hi + b * kPS + kh * kKH + r * 16);
        *x = tf32_rna4(*x);
      }
    }
    p.conv_done(q);
    return;
  }
  float4 l[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    if (it < TOT) {
      const int r = it & (kTile - 1), kh = (it >> 7) & 1, b = it >> 8;
      const uint32_t off = b * kPS + kh * kKH + r * 16;
      const float4 x = *reinterpret_cast<const float4*>(hi + off);
      float4 h;
      split4(x, h, l[i]);
      if (!kTf32Truncates) *reinterpret_cast<float4*>(hi + off) = h;
    }
  }
  if (q >= 1) mbar_wait(p.lo_bar, (q - 1) & 1);
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    if (it < TOT) {
      const int r = it & (kTile - 1), kh = (it >> 7) & 1, b = it >> 8;
      *reinterpret_cast<float4*>(p.lo + b * kPS + kh * kKH + r * 16) = l[i];
    }
  }
  p.conv_done(q);
}
// the MMAs of chunk q (called by every lane of one converged warp; an elected lane issues).  Weight set s: images at wimg0 + s*set_bytes, image (g, hi/lo) = 2g / 2g+1, plane
// rows = w_rows, K step ks, first output row n0; accumulator of (set s, blade b) at column (s*B + b)*ncols.
// TERMS = 1: image g = the rounded weight of grade g; one MMA per (set, blade) on the rounded chunk, one commit.
// The issuing thread's instruction stream is serial, so descriptors are formed by adding small 16-byte-unit offsets to
// bases computed once per chunk, and the loops are fully unrolled.
template <int DIM, int TERMS = 3>
__device__ __forceinline__ void issue_chunk_mma(const Pipe& p, int q, uint32_t tbase, uint32_t ncols, bool accumulate,
                                                const uint8_t* wimg0, uint32_t img_bytes, int s0, int nsets, uint32_t set_bytes,
                                                uint32_t w_rows, int ks, int n0, uint32_t idesc) {
  using A = Alg<DIM>;
  constexpr int B = A::B;
  const uint64_t a_hi = chunk_desc(smem_addr(p.slot(q)), 0), a_lo = chunk_desc(smem_addr(p.lo), 0);
  const uint64_t w0 = smem_desc(smem_addr(wimg0) + (uint32_t)s0 * set_bytes + 2u * ks * w_rows * 16u + (uint32_t)n0 * 16u,
                                w_rows * 16u, 128u);
  const uint64_t img16 = img_bytes >> 4, set16 = set_bytes >> 4;
  constexpr uint64_t ps16 = kPS >> 4;
  if constexpr (TERMS == 1) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      if (s < nsets) {
#pragma unroll
        for (int b = 0; b < B; ++b)
          mma_tf32_w(tbase + (uint32_t)(s * B + b) * ncols, a_hi + b * ps16, w0 + s * set16 + A::grade_of(b) * img16, idesc,
                     accumulate);
      }
    }
    mma_commit_w(&p.slot_bar[q % kRing]);
    return;
  }
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    if (s < nsets) {
#pragma unroll
      for (int b = 0; b < B; ++b)
        mma_tf32_w(tbase + (uint32_t)(s * B + b) * ncols, a_lo + b * ps16, w0 + s * set16 + (2 * A::grade_of(b)) * img16, idesc,
                 accumulate);
    }
  }
  mma_commit_w(p.lo_bar);
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    if (s < nsets) {
#pragma unroll
      for (int b = 0; b < B; ++b) {
        const uint64_t wd = w0 + s * set16 + (2 * A::grade_of(b)) * img16;
        const uint32_t d = tbase + (uint32_t)(s * B + b) * ncols;
        mma_tf32_w(d, a_hi + b * ps16, wd, idesc, 1);
        mma_tf32_w(d, a_hi + b * ps16, wd + img16, idesc, 1);
      }
    }
  }
  mma_commit_w(&p.slot_bar[q % kRing]);
}

}  // namespace tcb
}  // namespace csmpn
