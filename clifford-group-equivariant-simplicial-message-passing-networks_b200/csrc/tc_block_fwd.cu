// Tensor-core forward of one CEMLP block (cegnn_utils.py:180-207) for non-degenerate diagonal metrics of dimension 2 and 3:
//
//   tc_f1_kernel:  x0 (gathered / concatenated API-layout rows, or a BPT tensor) --MVLinear W1--> y1 (+bias, saved)
//                  --MVSiLU--> y2 (BPT)
//   tc_f2_kernel:  y2 --linear_right / linear_left--> xr, xl --normalisation, weighted geometric product, 1/sqrt2-->
//                  o --MVLayerNorm (+ residual)--> y        (xr and o saved for the backward)
//
// The three per-grade channel GEMMs run on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in
// TMEM) with the error-compensated split x = hi + lo (three MMAs per product) that keeps fp32 accuracy.  One CTA per
// SM, persistent over 128-row tiles.  Per tile the K dimension is streamed in 8-channel chunks through two
// shared-memory chunk buffers: chunk q+1 is produced (bulk copies + split pass, or the gathering/transposing
// producer) while the MMAs of chunk q run.  Blade b of a tile accumulates into TMEM columns [b*Cp, (b+1)*Cp) with the
// weight image of grade(b), so the [Cout, Cin, B] repeat_interleave'd weight of the reference never exists.
// The epilogues map one thread to one row (TMEM lane) and four channels at a time.
#include "tc_block.cuh"

namespace csmpn {
namespace tcb {

struct FwdArgs {
  int64_t rows;
  int tiles;
  int C, Cp;      // block width, padded to a multiple of 16
  int cin, kin8;  // input channels of the first linear, padded to a multiple of 8
  int in_bpt, in_cp;
  int mode, c0, c1, c2, pair_attr;
  int vt_k, vt_fp;  // mode 2 (vertex-table gather): vertices per row, channels per (feature type, vertex)
  const float *p0, *p1, *p2;
  const int32_t *src, *dst, *eid;
  const float *w1, *b1, *sa, *sb, *wr, *na, *wl, *bl, *wp, *la;
  float *save_y1, *y2, *save_xr, *save_o, *save_x0;
  float* y;
  const float* res;
  int out_bpt, has_b1;
  // streamed-weights mode (wide blocks): pre-split weight images in global memory and the channels per pass
  const float *wimg1, *wimg2;
  int ns1, ns2;
};

// ---- producer 2: gather / concatenate API-layout rows (all threads) ------------------------------------------------
// Item = (row r, channel cl of the chunk, blade quad h): one float4.  gather_chunk_api only LOADS (the values stay in
// registers, so the loads of chunk q+1 are in flight while chunk q is split, stored and multiplied);
// store_chunk_api transposes to planes, splits and stores.
template <int DIM>
struct ApiItems {
  static constexpr int H = Alg<DIM>::B / 4, PPR = 8 * H, TOT = kTile * PPR, N = (TOT + kConv - 1) / kConv;
  // item -> (row r, chunk channel cl, blade quad h).  A warp covers 4 channels x (8 / H) rows x H blade quads, so that
  // its transposing scalar stores (bank = 16 h + 4 (r % 4) + cl % 4 for Cl(3,0)) are conflict-free and its global
  // reads / x0 writes are 128 / 64 contiguous bytes per row.
  __device__ static __forceinline__ void decode(int it, int& r, int& cl, int& h) {
    const int l = it & 31, g = it >> 5;
    h = l % H;
    const int clo = (l / H) & 3, rlo = l / (4 * H);  // rlo < 8 / H
    cl = (g & 1) * 4 + clo;
    r = (g >> 1) * (8 / H) + rlo;
  }
};

// A thread's items keep their rows from chunk to chunk of a tile, so the gather indices of those rows (receiver, sender,
// position of the pair in the caller's order) are fetched ONCE per tile: the per-chunk gathers then start with the data
// loads instead of a dependent index load (the K loop of the gathering kernel is latency-bound on exactly that chain).
template <int DIM>
struct GatherIdx {
  int32_t d[ApiItems<DIM>::N], s[ApiItems<DIM>::N], e[ApiItems<DIM>::N];
};
template <int DIM>
__device__ __forceinline__ void load_gather_idx(const FwdArgs& a, int64_t row0, GatherIdx<DIM>& gi) {
  constexpr int N = ApiItems<DIM>::N, TOT = ApiItems<DIM>::TOT;
  if (a.mode == 0) return;
  const int ct = (int)threadIdx.x - 32;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    int r, cl, h;
    ApiItems<DIM>::decode(it, r, cl, h);
    const int64_t R = row0 + r;
    const bool ok = it < TOT && R < a.rows;
    if (a.mode == 2) {  // the (up to three) table rows of this row's vertices, in the row's vertex order
      gi.d[i] = ok ? a.src[R * a.vt_k] : 0;
      gi.s[i] = (ok && a.vt_k > 1) ? a.src[R * a.vt_k + 1] : 0;
      gi.e[i] = (ok && a.vt_k > 2) ? a.src[R * a.vt_k + 2] : 0;
    } else {
      gi.d[i] = ok ? a.dst[R] : 0;
      gi.s[i] = ok ? a.src[R] : 0;
      gi.e[i] = (ok && a.c1 > 0 && !a.pair_attr) ? a.eid[R] : 0;
    }
  }
}

template <int DIM>
__device__ __forceinline__ void gather_chunk_api(const FwdArgs& a, int64_t row0, int kc, float4* v, const GatherIdx<DIM>& gi) {
  constexpr int B = Alg<DIM>::B, H = ApiItems<DIM>::H, PPR = ApiItems<DIM>::PPR, N = ApiItems<DIM>::N, TOT = ApiItems<DIM>::TOT;
  const int ct = (int)threadIdx.x - 32;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    int r, cl, h;
    ApiItems<DIM>::decode(it, r, cl, h);
    const int c = kc * 8 + cl;
    const int64_t R = row0 + r;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (it < TOT && R < a.rows && c < a.cin) {
      if (a.mode == 2) {
        // channel c = (type t, vertex slot j, feature f): c = (t * k + j) * fp + f  ->  table[vertex_j][t * fp + f]
        const int kf = a.vt_k * a.vt_fp, t = c / kf, j = (c - t * kf) / a.vt_fp, f = c - t * kf - j * a.vt_fp;
        const int64_t vrow = j == 0 ? gi.d[i] : j == 1 ? gi.s[i] : gi.e[i];
        v[i] = __ldg(reinterpret_cast<const float4*>(a.p0 + (vrow * (a.c0 / a.vt_k) + t * a.vt_fp + f) * B + 4 * h));
      } else if (a.mode == 1) {
        if (c < a.c0) {
          const int64_t d = gi.d[i], s = gi.s[i];
          const float4 x = __ldg(reinterpret_cast<const float4*>(a.p0 + (d * a.c0 + c) * B + 4 * h));
          const float4 z = __ldg(reinterpret_cast<const float4*>(a.p0 + (s * a.c0 + c) * B + 4 * h));
          v[i] = make_float4(x.x - z.x, x.y - z.y, x.z - z.z, x.w - z.w);
        } else if (a.pair_attr) {  // (table[src] | table[dst]), table = p1 [n_nodes, c1/2, B]
          const int k = c - a.c0, half = a.c1 >> 1;
          const int64_t n = k < half ? gi.s[i] : gi.d[i];
          v[i] = __ldg(reinterpret_cast<const float4*>(a.p1 + (n * half + (k < half ? k : k - half)) * B + 4 * h));
        } else {
          const int64_t e = gi.e[i];
          v[i] = __ldg(reinterpret_cast<const float4*>(a.p1 + (e * a.c1 + (c - a.c0)) * B + 4 * h));
        }
      } else {
        if (c < a.c0) v[i] = __ldg(reinterpret_cast<const float4*>(a.p0 + (R * a.c0 + c) * B + 4 * h));
        else if (c < a.c0 + a.c1) v[i] = __ldg(reinterpret_cast<const float4*>(a.p1 + (R * a.c1 + (c - a.c0)) * B + 4 * h));
        else v[i] = __ldg(reinterpret_cast<const float4*>(a.p2 + (R * a.c2 + (c - a.c0 - a.c1)) * B + 4 * h));
      }
    }
  }
}
// high parts first (the raw slot of chunk q is free), then -- once the MMAs of chunk q-1 have released `lo` -- the remainders
// x0 != nullptr: the assembled input rows are also written to the BPT tensor x0 (kept for the weight-gradient GEMM of
// the backward) straight from the registers, between the two shared-memory phases: a warp covers two rows x 8 channels
// x all blades, i.e. full 32-byte sectors of every blade plane.
// TERMS = 1 (single-pass TF32): the values rounded to nearest TF32 go to the raw slot, x0 keeps the unrounded rows, and
// there is no `lo` phase.
template <int DIM, int TERMS = 3>
__device__ __forceinline__ void store_chunk_api(const Pipe& p, int q, const float4* v, float* x0, int x0_cp, int64_t tile, int kc) {
  constexpr int B = Alg<DIM>::B;
  constexpr int H = ApiItems<DIM>::H, PPR = ApiItems<DIM>::PPR, N = ApiItems<DIM>::N, TOT = ApiItems<DIM>::TOT;
  const int ct = (int)threadIdx.x - 32;
  uint8_t* hi = p.slot(q);
  uint8_t* lo = p.lo;
  float4 lv[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    if (it < TOT) {
      int r, cl, h;
      ApiItems<DIM>::decode(it, r, cl, h);
      float4 hv;
      if constexpr (TERMS == 1) hv = tf32_rna4(v[i]);
      else split4(v[i], hv, lv[i]);
      const uint32_t off = (4 * h) * kPS + (cl >> 2) * kKH + r * 16 + (cl & 3) * 4;
      *reinterpret_cast<float*>(hi + off) = hv.x;
      *reinterpret_cast<float*>(hi + off + kPS) = hv.y;
      *reinterpret_cast<float*>(hi + off + 2 * kPS) = hv.z;
      *reinterpret_cast<float*>(hi + off + 3 * kPS) = hv.w;
    }
  }
  if (x0) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const int it = ct + i * kConv;
      if (it < TOT) {
        int r, cl, h;
        ApiItems<DIM>::decode(it, r, cl, h);
        float* dst = x0 + bpt_off(B, x0_cp, tile, 4 * h, 2 * kc + (cl >> 2), r) + (cl & 3);
        const size_t bs = (size_t)(x0_cp >> 2) * kTile * 4;  // floats between blade planes
        dst[0] = v[i].x;
        dst[bs] = v[i].y;
        dst[2 * bs] = v[i].z;
        dst[3 * bs] = v[i].w;
      }
    }
  }
  if constexpr (TERMS == 1) return;
  if (q >= 1) mbar_wait(p.lo_bar, (q - 1) & 1);
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const int it = ct + i * kConv;
    if (it < TOT) {
      int r, cl, h;
      ApiItems<DIM>::decode(it, r, cl, h);
      const uint32_t off = (4 * h) * kPS + (cl >> 2) * kKH + r * 16 + (cl & 3) * 4;
      *reinterpret_cast<float*>(lo + off) = lv[i].x;
      *reinterpret_cast<float*>(lo + off + kPS) = lv[i].y;
      *reinterpret_cast<float*>(lo + off + 2 * kPS) = lv[i].z;
      *reinterpret_cast<float*>(lo + off + 3 * kPS) = lv[i].w;
    }
  }
}
// barrier among the converter warps only (named barrier 1; warp 0 never joins)
__device__ __forceinline__ void conv_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(kConv) : "memory"); }
// zero the 8 padding channels of chunk kc of a BPT tensor (c_in padded to 16 but staged in chunks of 8)
template <int B>
__device__ __forceinline__ void zero_chunk_bpt(float* dst, int cp, int64_t tile, int kc) {
  for (int it = (int)threadIdx.x - 32; it < B * 2 * kTile; it += kConv) {
    const int r = it & (kTile - 1), kh = (it >> 7) & 1, b = it >> 8;
    *reinterpret_cast<float4*>(dst + bpt_off(B, cp, tile, b, 2 * kc + kh, r)) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// F1 epilogue of channel group gc4 of row r of `tile`, from the accumulators already loaded from TMEM (v): bias -> y1
// (saved when requested), MVSiLU -> y2.  b1_s / sa_s / sb_s: the bias and gate parameters staged in shared memory.
template <int DIM, bool MET>
__device__ __forceinline__ void f1_epilogue_group(const FwdArgs& a, float (&v)[Alg<DIM>::B][4], int64_t tile, int gc4, int r,
                                                  const float* b1_s, const float* sa_s, const float* sb_s, const float* qs) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G;
  const bool row_ok = tile * kTile + r < a.rows;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ch = gc4 * 4 + j;
    float y1[B];
    const bool ok = row_ok && ch < a.C;
#pragma unroll
    for (int b = 0; b < B; ++b) y1[b] = ok ? v[b][j] : 0.f;
    if (ok) y1[0] += b1_s[ch];
#pragma unroll
    for (int b = 0; b < B; ++b) v[b][j] = y1[b];
  }
  if (a.save_y1) {
#pragma unroll
    for (int b = 0; b < B; ++b)
      *reinterpret_cast<float4*>(a.save_y1 + bpt_off(B, a.Cp, tile, b, gc4, r)) = make_float4(v[b][0], v[b][1], v[b][2], v[b][3]);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ch = gc4 * 4 + j;
    float y1[B], sg[G], inv[G];
#pragma unroll
    for (int b = 0; b < B; ++b) y1[b] = v[b][j];
    silu_gates<DIM, MET>(y1, sa_s + ch * G, sb_s + ch * G, sg, inv, qs);
#pragma unroll
    for (int b = 0; b < B; ++b) v[b][j] = y1[b] * sg[A::grade_of(b)];
  }
#pragma unroll
  for (int b = 0; b < B; ++b)
    *reinterpret_cast<float4*>(a.y2 + bpt_off(B, a.Cp, tile, b, gc4, r)) = make_float4(v[b][0], v[b][1], v[b][2], v[b][3]);
}

// The bias and gate parameters of f1 into shared memory: b1_s [Cp], sa_s / sb_s [Cp][G], zero beyond the real channels.
// Each thread's first elements are requested before stage_weights() runs (one exposed latency for the whole prologue
// instead of one per loop), the rest after it.
template <int DIM, class StageWeights>
__device__ __forceinline__ void stage_f1_params(const FwdArgs& a, float* b1_s, float* sa_s, float* sb_s, StageWeights&& stage_weights) {
  constexpr int G = Alg<DIM>::G;
  const int tid = threadIdx.x, C = a.C, Cp = a.Cp;
  const float pf_b1 = (tid < C && a.has_b1) ? __ldg(a.b1 + tid) : 0.f;
  const float pf_sa = tid < C * G ? __ldg(a.sa + tid) : 0.f;
  const float pf_sb = tid < C * G ? __ldg(a.sb + tid) : 0.f;
  stage_weights();
  if (tid < Cp) b1_s[tid] = pf_b1;
  for (int i = tid + kThreads; i < Cp; i += kThreads) b1_s[i] = (i < C && a.has_b1) ? a.b1[i] : 0.f;
  if (tid < Cp * G) { sa_s[tid] = pf_sa; sb_s[tid] = pf_sb; }
  for (int i = tid + kThreads; i < Cp * G; i += kThreads) {
    sa_s[i] = (i < C * G) ? a.sa[i] : 0.f;
    sb_s[i] = (i < C * G) ? a.sb[i] : 0.f;
  }
}

// =====================================================================================================================
// F1: MVLinear (W1) + bias + MVSiLU.  ST (streamed weights, wide blocks): the output channels are produced in passes of
// a.ns1 channels (accumulators = B * ns1 TMEM columns), the K chunks of the input are walked once per pass and every chunk
// arrives with its weight unit (tc_block.cuh); the resident weight images do not exist.  TERMS: numeric mode
// (tc_block.cuh, n_images).  MET: non-Euclidean metric (mp, common.cuh MetricArg) in the MVSiLU invariants.
template <int DIM, bool BPT_IN, bool ST, int TERMS, bool MET>
__global__ void __launch_bounds__(kThreads, 1) tc_f1_kernel(FwdArgs a, MetricArg<MET> mp) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, NI = n_images(TERMS);
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int C = a.C, Cp = a.Cp, nk = a.kin8 / 8;
  const int NS = ST ? a.ns1 : Cp;                     // output channels per pass
  const int npass = ST ? Cp / NS : 1;
  const uint32_t wunit = ST ? wunit_bytes<DIM>(NS, NI) : 0u;
  const uint32_t half = B * kPS + wunit;
  const uint32_t img = ST ? (uint32_t)NS * 32u : (uint32_t)a.kin8 * Cp * 4;
  uint8_t* wimg = smem + (size_t)kRing * half + B * kPS;
  float* b1_s = reinterpret_cast<float*>(wimg + (ST ? 0 : (size_t)G * NI * img));
  float* sa_s = b1_s + Cp;
  float* sb_s = sa_s + Cp * G;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb_s + Cp * G);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
  Pipe p;
  p.init(smem, bars, half);
  const int my_tiles = cta_tiles(a.tiles);
  const int per_tile = npass * nk;
  const int total_chunks = my_tiles * per_tile;
  auto tile_of = [&](int q) { return cta_tile(q / per_tile); };
  // the issuer's bulk copies: activation planes (BPT input) and / or weight units (ST)
  auto load = [&](int qq) {
    if constexpr (ST) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.wimg1) + (size_t)(qq % per_tile) * wunit;
      issue_chunk_load_w<B>(p, qq, BPT_IN ? a.p0 : nullptr, a.in_cp, tile_of(qq), qq % nk, wsrc, wunit);
    } else {
      issue_chunk_load<B>(p, qq, a.p0, a.in_cp, tile_of(qq), qq % nk);
    }
  };
  ChunkFeed<BPT_IN || ST> feed{p, total_chunks};
  // the gathering converters request their first chunk before the prologue as well (see ChunkFeed::prime)
  int q = 0;  // chunk sequence number of this CTA; chunk q lives in raw slot q % kRing
  float4 gv[BPT_IN ? 1 : ApiItems<DIM>::N];  // gathered items of the NEXT chunk to stage (API-layout input)
  GatherIdx<DIM> gi;
  if (!BPT_IN && warp != 0 && total_chunks > 0) {
    load_gather_idx<DIM>(a, tile_of(0) * kTile, gi);
    gather_chunk_api<DIM>(a, tile_of(0) * kTile, 0, gv, gi);
  }
  if (warp == 0) feed.prime(load);

  const uint32_t tcols = tmem_cols((uint32_t)B * NS);
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  stage_f1_params<DIM>(a, b1_s, sa_s, sb_s, [&] {
    if (!ST) stage_weight_images<DIM, false, TERMS>(wimg, img, a.w1, C, a.cin, Cp, a.kin8);
  });
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t idesc = idesc_tf32(kTile, NS, false, false);
  for (int t = 0; t < my_tiles; ++t) {
    const int64_t tile = cta_tile(t);
    for (int ps = 0; ps < npass; ++ps) {
      const int n0 = ps * NS;
      for (int kc = 0; kc < nk; ++kc, ++q) {
        if (warp == 0) {  // issuer
          p.wait_full(q);
          feed.refill(q, load);
          if constexpr (ST) {
            p.wait_landed(q);  // the weight unit of this chunk
            issue_chunk_mma<DIM, TERMS>(p, q, tbase, NS, kc > 0, p.slot(q) + B * kPS, img, 0, 1, 0, NS, 0, 0, idesc);
          } else {
            issue_chunk_mma<DIM, TERMS>(p, q, tbase, Cp, kc > 0, wimg, img, 0, 1, 0, Cp, kc, 0, idesc);
          }
        } else if (BPT_IN) {  // converters: split the landed chunk
          p.wait_landed(q);
          split_chunk<B, TERMS>(p, q);
        } else {              // converters: gathering producer (wide blocks gather the input rows once per pass)
          if (q >= kRing) p.wait_free(q - kRing);
          float* x0 = ps == 0 ? a.save_x0 : nullptr;
          store_chunk_api<DIM, TERMS>(p, q, gv, x0, round_up(a.kin8, 16), tile, kc);
          p.conv_done(q);
          if (q + 1 < total_chunks) {
            if ((q + 1) % per_tile == 0) load_gather_idx<DIM>(a, tile_of(q + 1) * kTile, gi);  // first chunk of the next tile
            gather_chunk_api<DIM>(a, tile_of(q + 1) * kTile, (q + 1) % nk, gv, gi);
          }
          if (x0 && kc == nk - 1 && (a.kin8 & 8)) zero_chunk_bpt<B>(x0, round_up(a.kin8, 16), tile, nk);
        }
      }
      // ---- epilogue of this pass
      p.wait_mmas(q - 1);
      if (warp == 0) feed.refill_all(q, load);
      const int r = (warp & 3) * 32 + lane;
      for (int c4 = warp >> 2; c4 < (NS >> 2); c4 += 4) {
        float v[B][4];
#pragma unroll
        for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tbase, (warp & 3) * 32, b * NS + c4 * 4), v[b]);
        tmem_wait_ld();
        f1_epilogue_group<DIM, MET>(a, v, tile, (n0 >> 2) + c4, r, b1_s, sa_s, sb_s, mp.qs);
      }
      fence_before_sync();  // the next pass's first MMA overwrites these accumulators (tc_block.cuh: reuse rules)
    }
  }
  tmem_teardown(warp, tbase, tcols);
}

// =====================================================================================================================
// F1 with OVERLAPPED epilogue (resident weights, B * Cp <= 256 TMEM columns): two accumulator buffers alternate by tile,
// and the epilogue of tile t-1 (TMEM -> bias -> y1 store -> MVSiLU -> y2 store) is cut into channel-group units that the
// converter warps run BETWEEN the chunks of tile t's K loop.  Loads, MMAs, the elementwise pass and the store drain of
// neighbouring tiles then overlap instead of running back to back (the plain kernel above spends two thirds of a tile in
// the epilogue and its drain with the tensor pipe and the copy engine idle).
// Roles: warp 0 issues copies and MMAs only; warps 1-15 convert / gather; warps 4-15 also own the epilogue: lane quadrant
// warp & 3, channel groups (warp >> 2) - 1, + 3, ... (PendingEpilogue).  Same epilogue body as tc_f1_kernel
// (f1_epilogue_group): results are bit-identical.
template <int DIM, bool BPT_IN, int TERMS, bool MET>
__global__ void __launch_bounds__(kThreads, 1) tc_f1db_kernel(FwdArgs a, MetricArg<MET> mp) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, NI = n_images(TERMS);
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int C = a.C, Cp = a.Cp, nk = a.kin8 / 8;
  const uint32_t img = (uint32_t)a.kin8 * Cp * 4;
  uint8_t* wimg = smem + (kRing + 1) * B * kPS;
  float* b1_s = reinterpret_cast<float*>(wimg + (size_t)G * NI * img);
  float* sa_s = b1_s + Cp;
  float* sb_s = sa_s + Cp * G;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb_s + Cp * G);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
  Pipe p;
  p.init(smem, bars, B * kPS);
  const int my_tiles = cta_tiles(a.tiles);
  const int total_chunks = my_tiles * nk;
  auto tile_of = [&](int q) { return cta_tile(q / nk); };
  auto load = [&](int qq) { issue_chunk_load<B>(p, qq, a.p0, a.in_cp, tile_of(qq), qq % nk); };
  ChunkFeed<BPT_IN> feed{p, total_chunks};
  // first chunks requested before the weights are staged (see tc_f1_kernel)
  int q = 0;
  float4 gv[BPT_IN ? 1 : ApiItems<DIM>::N];
  GatherIdx<DIM> gi;
  if (!BPT_IN && warp != 0 && total_chunks > 0) {
    load_gather_idx<DIM>(a, tile_of(0) * kTile, gi);
    gather_chunk_api<DIM>(a, tile_of(0) * kTile, 0, gv, gi);
  }
  if (warp == 0) feed.prime(load);

  const uint32_t bufcols = (uint32_t)B * Cp;  // <= 256 (host)
  const uint32_t tcols = tmem_cols(2 * bufcols);
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  stage_f1_params<DIM>(a, b1_s, sa_s, sb_s, [&] { stage_weight_images<DIM, false, TERMS>(wimg, img, a.w1, C, a.cin, Cp, a.kin8); });
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t idesc = idesc_tf32(kTile, Cp, false, false);
  const int r = (warp & 3) * 32 + lane;
  const int n_c4 = Cp >> 2;

  // one epilogue unit: channel group c4 of `tile`, accumulators at tb
  auto epilogue_unit = [&](int64_t tile, int c4, uint32_t tb) {
    float v[B][4];
#pragma unroll
    for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tb, (warp & 3) * 32, b * Cp + c4 * 4), v[b]);
    tmem_wait_ld();
    f1_epilogue_group<DIM, MET>(a, v, tile, c4, r, b1_s, sa_s, sb_s, mp.qs);
  };
  PendingEpilogue pend;

  for (int t = 0; t < my_tiles; ++t) {
    const int64_t tile = cta_tile(t);
    const uint32_t tb = tbase + (uint32_t)(t & 1) * bufcols;
    for (int kc = 0; kc < nk; ++kc, ++q) {
      if (warp == 0) {  // issuer
        p.wait_full(q);
        feed.refill(q, load);
        // buffer t & 1 was read by the epilogue of tile t-2: every epilogue warp finished it before its conv_done of
        // this tile's first chunk (full_bar observed above), so the first MMA may overwrite it
        issue_chunk_mma<DIM, TERMS>(p, q, tb, Cp, kc > 0, wimg, img, 0, 1, 0, Cp, kc, 0, idesc);
      } else {
        if (BPT_IN) {
          p.wait_landed(q);
          split_chunk<B, TERMS>(p, q);
        } else {
          if (q >= kRing) p.wait_free(q - kRing);
          store_chunk_api<DIM, TERMS>(p, q, gv, a.save_x0, round_up(a.kin8, 16), tile, kc);
          p.conv_done(q);
          if (q + 1 < total_chunks) {
            if ((q + 1) % nk == 0) load_gather_idx<DIM>(a, tile_of(q + 1) * kTile, gi);  // first chunk of the next tile
            gather_chunk_api<DIM>(a, tile_of(q + 1) * kTile, (q + 1) % nk, gv, gi);
          }
          if (a.save_x0 && kc == nk - 1 && (a.kin8 & 8)) zero_chunk_bpt<B>(a.save_x0, round_up(a.kin8, 16), tile, nk);
        }
        pend.step(p, n_c4, epilogue_unit);  // one unit of the previous tile between two chunks of this one
      }
    }
    pend.drain(p, n_c4, epilogue_unit);
    pend.start(warp, tile, q - 1, tb);
  }
  pend.drain(p, n_c4, epilogue_unit);
  tmem_teardown(warp, tbase, tcols);
}

// =====================================================================================================================
// F2: linear_right / linear_left + normalisation + weighted geometric product + MVLayerNorm (+ residual)
// The two linears share ONE MMA per (blade, split term): the weight images hold linear_right in plane rows [0, NS) and
// linear_left in rows [NS, 2 NS), so the instruction shape is 128 x 2 NS x 8 and the A operand (the activations, the
// expensive shared-memory read) is fetched once for both.  Blade b accumulates into columns [2 b NS, 2 (b+1) NS):
// xr first, xl second.
// ST (streamed weights, wide blocks): NS = a.ns2 < Cp output channels per pass, weight units streamed with the chunks; the
// row statistics of the MVLayerNorm accumulate over the passes and the final scaling pass re-reads the product sum `o`
// from the saved tensor (written by the same thread one pass earlier) instead of keeping it in TMEM.
template <int DIM, bool ST, int TERMS, bool MET>
__global__ void __launch_bounds__(kThreads, 1) tc_f2_kernel(FwdArgs a, MetricArg<MET> mp) {
  using A = Alg<DIM>;
  constexpr int B = A::B, G = A::G, P = A::P, NI = n_images(TERMS);
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int C = a.C, Cp = a.Cp, nk = Cp / 8;
  const int NS = ST ? a.ns2 : Cp;                      // output channels per pass
  const int npass = ST ? Cp / NS : 1;
  const uint32_t wunit = ST ? wunit_bytes<DIM>(2 * NS, NI) : 0u;
  const uint32_t half = B * kPS + wunit;
  const uint32_t img = ST ? (uint32_t)2 * NS * 32u : (uint32_t)2 * Cp * Cp * 4;  // one image: [2 NS rows (right | left)] x [K]
  const uint32_t set_bytes = ST ? 0u : G * NI * img;
  uint8_t* wimg = smem + (size_t)kRing * half + B * kPS;
  float* sn_s = reinterpret_cast<float*>(wimg + (size_t)set_bytes);  // sigmoid(normalization.a) [Cp][G]
  float* wv_s = sn_s + Cp * G;                                           // path weights [Cp][P]
  float* bl_s = wv_s + Cp * P;
  float* la_s = bl_s + Cp;
  float* rowsum_s = la_s + Cp;                                           // [2 tile parities][4][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(rowsum_s + 8 * kTile);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
  Pipe p;
  p.init(smem, bars, half);
  const int my_tiles = cta_tiles(a.tiles);
  const int per_tile = npass * nk;
  auto load = [&](int qq) {
    const int64_t tile = cta_tile(qq / per_tile);
    if constexpr (ST) {
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.wimg2) + (size_t)(qq % per_tile) * wunit;
      issue_chunk_load_w<B>(p, qq, a.y2, Cp, tile, qq % nk, wsrc, wunit);
    } else {
      issue_chunk_load<B>(p, qq, a.y2, Cp, tile, qq % nk);
    }
  };
  ChunkFeed<> feed{p, my_tiles * per_tile};
  int q = 0;
  if (warp == 0) feed.prime(load);

  const uint32_t tcols = tmem_cols(2 * B * NS);
  if (warp == 0) tmem_alloc(tmem_slot, tcols);
  // the first elements of the small per-channel parameters are requested before the weights are staged (one exposed
  // latency for the whole prologue instead of one per loop)
  const float pf_na = tid < C * G ? __ldg(a.na + tid) : 0.f;
  const float pf_wp0 = tid < C * P ? __ldg(a.wp + tid) : 0.f;
  const float pf_wp1 = tid + kThreads < C * P ? __ldg(a.wp + tid + kThreads) : 0.f;
  const float pf_bl = tid < C ? __ldg(a.bl + tid) : 0.f;
  const float pf_la = tid < C ? __ldg(a.la + tid) : 0.f;
  if (!ST) {
    const WJob wj[2] = {{wimg, a.wr, C, C, 0}, {wimg, a.wl, C, C, Cp}};  // right | left stacked along the image rows
    stage_weight_jobs<DIM, false, 2, TERMS>(wj, 2, img, 2 * Cp, Cp, wimg, (uint32_t)G * (uint32_t)NI * img);
  }
  if (tid < Cp * G) sn_s[tid] = tid < C * G ? sigmoidf_(pf_na) : 0.f;
  for (int i = tid + kThreads; i < Cp * G; i += kThreads) sn_s[i] = (i < C * G) ? sigmoidf_(a.na[i]) : 0.f;
  if (tid < Cp * P) wv_s[tid] = pf_wp0;
  if (tid + kThreads < Cp * P) wv_s[tid + kThreads] = pf_wp1;
  for (int i = tid + 2 * kThreads; i < Cp * P; i += kThreads) wv_s[i] = (i < C * P) ? a.wp[i] : 0.f;
  if (tid < Cp) { bl_s[tid] = pf_bl; la_s[tid] = pf_la; }
  for (int i = tid + kThreads; i < Cp; i += kThreads) {
    bl_s[i] = (i < C) ? a.bl[i] : 0.f;
    la_s[i] = (i < C) ? a.la[i] : 0.f;
  }
  prologue_sync();
  const uint32_t tbase = *tmem_slot;
  const uint32_t idesc = idesc_tf32(kTile, 2 * NS, false, false);
  const uint32_t col_r = 0, col_l = NS, bcols = 2 * NS;  // column of (blade b, channel c of the pass): b * bcols + col_{r,l} + c
  const bool wide_ok = aligned32(a.y) && (!a.res || aligned32(a.res));
  const uint32_t lane_base = (warp & 3) * 32;

  for (int t = 0; t < my_tiles; ++t) {
    const int64_t tile = cta_tile(t);
    const int64_t row0 = tile * kTile;
    const int r = lane_base + lane;
    const bool row_ok = row0 + r < a.rows;
    float rs = 0.f;  // this thread's part of the row sum of norms (MVLayerNorm), over all passes
    for (int ps = 0; ps < npass; ++ps) {
      const int n0 = ps * NS;
      for (int kc = 0; kc < nk; ++kc, ++q) {
        if (warp == 0) {  // issuer
          p.wait_full(q);
          feed.refill(q, load);
          if constexpr (ST) issue_chunk_mma<DIM, TERMS>(p, q, tbase, bcols, kc > 0, p.slot(q) + B * kPS, img, 0, 1, 0, bcols, 0, 0, idesc);
          else issue_chunk_mma<DIM, TERMS>(p, q, tbase, bcols, kc > 0, wimg, img, 0, 1, 0, bcols, kc, 0, idesc);
        } else {          // converters
          p.wait_landed(q);
          split_chunk<B, TERMS>(p, q);
        }
      }
      // y2 of this thread's first channel group is requested before waiting for the MMAs (left operand of the product)
      float4 y2v[B];
      if ((warp >> 2) < (NS >> 2)) {
#pragma unroll
        for (int b = 0; b < B; ++b) y2v[b] = *reinterpret_cast<const float4*>(a.y2 + bpt_off(B, Cp, tile, b, (n0 >> 2) + (warp >> 2), r));
      }
      p.wait_mmas(q - 1);
      if (warp == 0) feed.refill_all(q, load);
      // ---- pass 1: per channel normalisation + weighted geometric product; o -> TMEM over xl (ST: -> save_o only)
      for (int c4 = warp >> 2; c4 < (NS >> 2); c4 += 4) {
        const int gc4 = (n0 >> 2) + c4;
        float xr[B][4], o[B][4];
        if (c4 != (warp >> 2)) {
#pragma unroll
          for (int b = 0; b < B; ++b) y2v[b] = *reinterpret_cast<const float4*>(a.y2 + bpt_off(B, Cp, tile, b, gc4, r));
        }
#pragma unroll
        for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tbase, lane_base, b * bcols + col_r + c4 * 4), xr[b]);
#pragma unroll
        for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tbase, lane_base, b * bcols + col_l + c4 * 4), o[b]);
        tmem_wait_ld();
        // the saved tensors are stored from this (compute-bound) pass, so that their drain overlaps the arithmetic; the
        // second pass then only writes the block output
        if (a.save_xr) {
#pragma unroll
          for (int b = 0; b < B; ++b) {
            float4 x = make_float4(xr[b][0], xr[b][1], xr[b][2], xr[b][3]);
            if (!row_ok) x = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(a.save_xr + bpt_off(B, Cp, tile, b, gc4, r)) = x;
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = gc4 * 4 + j;
          float xn[B], oj[B], y2[B], qv[G], nrm[G], rinv[G];
#pragma unroll
          for (int b = 0; b < B; ++b) { xn[b] = xr[b][j]; oj[b] = o[b][j]; }
#pragma unroll
          for (int b = 0; b < B; ++b) y2[b] = j == 0 ? y2v[b].x : j == 1 ? y2v[b].y : j == 2 ? y2v[b].z : y2v[b].w;
          norm_factors<DIM, MET>(xn, sn_s + ch * G, qv, nrm, rinv, mp.qs);
#pragma unroll
          for (int b = 0; b < B; ++b) xn[b] *= rinv[A::grade_of(b)];
          oj[0] += bl_s[ch];
          A::template wgp<MET>(y2, xn, wv_s + ch * P, mp.mf, oj);
          const bool ok = row_ok && ch < C;
#pragma unroll
          for (int b = 0; b < B; ++b) oj[b] = ok ? oj[b] * kInvSqrt2 : 0.f;
          if (ok) rs += fast_sas(mv_q<DIM, MET>(oj, mp.qs));
#pragma unroll
          for (int b = 0; b < B; ++b) o[b][j] = oj[b];
        }
        if constexpr (!ST) {
#pragma unroll
          for (int b = 0; b < B; ++b) tmem_st4(tmem_at(tbase, lane_base, b * bcols + col_l + c4 * 4), o[b]);
        }
        if (ST || a.save_o) {
#pragma unroll
          for (int b = 0; b < B; ++b)
            *reinterpret_cast<float4*>(a.save_o + bpt_off(B, Cp, tile, b, gc4, r)) = make_float4(o[b][0], o[b][1], o[b][2], o[b][3]);
        }
      }
      if constexpr (!ST) tmem_wait_st();
      fence_before_sync();  // ST: the next pass's first MMA overwrites the accumulators (ordered by the full_bar chain)
    }
    // two copies, alternating by tile: a warp's reads of tile t and another warp's writes of tile t+1 are ordered by the
    // mbarrier chain of the next K loop anyway, but never touch the same words this way
    float* rowsum_t = rowsum_s + (t & 1) * 4 * kTile;
    rowsum_t[(warp >> 2) * kTile + r] = rs;
    __syncthreads();
    const float inv_mu = fast_rcp((rowsum_t[r] + rowsum_t[kTile + r] + rowsum_t[2 * kTile + r] + rowsum_t[3 * kTile + r]) / (float)C + kEps);
    // ---- pass 2: MVLayerNorm scale, residual, output (every channel group this thread handled in pass 1)
    for (int gc4 = warp >> 2; gc4 < (Cp >> 2); gc4 += 4) {
      float o[B][4];
      if constexpr (ST) {
#pragma unroll
        for (int b = 0; b < B; ++b) {
          const float4 x = *reinterpret_cast<const float4*>(a.save_o + bpt_off(B, Cp, tile, b, gc4, r));
          o[b][0] = x.x; o[b][1] = x.y; o[b][2] = x.z; o[b][3] = x.w;
        }
      } else {
#pragma unroll
        for (int b = 0; b < B; ++b) tmem_ld4(tmem_at(tbase, lane_base, b * bcols + col_l + gc4 * 4), o[b]);
        tmem_wait_ld();
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float sc = la_s[gc4 * 4 + j] * inv_mu;
#pragma unroll
        for (int b = 0; b < B; ++b) o[b][j] *= sc;
      }
      if (a.out_bpt) {
#pragma unroll
        for (int b = 0; b < B; ++b)
          *reinterpret_cast<float4*>(a.y + bpt_off(B, Cp, tile, b, gc4, r)) = make_float4(o[b][0], o[b][1], o[b][2], o[b][3]);
      } else if (row_ok) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = gc4 * 4 + j;
          if (ch >= C) continue;
          const size_t off = ((size_t)(row0 + r) * C + ch) * B;
          if constexpr (B == 8) {
            if (wide_ok) {  // one 32-byte sector per (row, channel)
              float v[8];
#pragma unroll
              for (int b = 0; b < 8; ++b) v[b] = o[b][j];
              if (a.res) {
                float rv[8];
                ld_global_v8(rv, a.res + off);
#pragma unroll
                for (int b = 0; b < 8; ++b) v[b] += rv[b];
              }
              st_global_v8(a.y + off, v);
              continue;
            }
          }
#pragma unroll
          for (int h = 0; h < B / 4; ++h) {
            float4 x = make_float4(o[4 * h][j], o[4 * h + 1][j], o[4 * h + 2][j], o[4 * h + 3][j]);
            if (a.res) {
              const float4 rv = *reinterpret_cast<const float4*>(a.res + off + 4 * h);
              x.x += rv.x; x.y += rv.y; x.z += rv.z; x.w += rv.w;
            }
            *reinterpret_cast<float4*>(a.y + off + 4 * h) = x;
          }
        }
      }
    }
    fence_before_sync();
  }
  tmem_teardown(warp, tbase, tcols);
}

// ---------------------------------------------------------------------------------------------------------------
// How the two forward kernels of a block of this shape run: weights resident in shared memory, or -- wide blocks --
// streamed with the K chunks in passes of ns1 / ns2 output channels (tc_block.cuh).  The choice is made for the default
// (split) weight images, so both numeric modes run a shape with the same plan; nimg = 1 (single-pass TF32) only shrinks
// the shared memory and the streamed image buffers.
struct FwdPlan {
  bool ok;
  bool st1, st2;
  int Cp, kin8, ns1, ns2;
  size_t s1, s2;            // dynamic shared memory of f1 / f2
  int64_t w1_floats, w2_floats;  // pre-split weight image buffers (streamed mode), floats
};

template <int DIM>
FwdPlan fwd_plan(int cin, int c, int nimg = 2) {
  constexpr int B = Alg<DIM>::B, G = Alg<DIM>::G, P = Alg<DIM>::P;
  FwdPlan p;
  memset(&p, 0, sizeof(p));
  if (c < 1 || cin < 1) return p;
  const int Cp = round_up(c, 16), kin8 = round_up(cin, 8);
  p.Cp = Cp; p.kin8 = kin8;
  const size_t ring = (size_t)(kRing + 1) * B * kPS;
  const size_t par1 = (size_t)Cp * (1 + 2 * G) * 4 + 96, par2 = (size_t)Cp * (G + P + 2) * 4 + 8 * kTile * 4 + 96;
  // ---- f1
  p.s1 = ring + (size_t)G * 2 * kin8 * Cp * 4 + par1;
  p.ns1 = Cp;
  if (B * Cp > 512 || p.s1 > kSmemMax) {
    p.st1 = true;
    int ns = (512 / B) / 16 * 16;
    while (ns >= 16 && (Cp % ns || (size_t)kRing * wunit_bytes<DIM>(ns) + ring + par1 > kSmemMax)) ns -= 16;
    if (ns < 16) return p;
    p.ns1 = ns;
    p.s1 = (size_t)kRing * wunit_bytes<DIM>(ns) + ring + par1;
    p.w1_floats = weight_image_floats<DIM>(0, ns, Cp / ns, kin8 / 8);
  }
  // ---- f2
  p.s2 = ring + (size_t)2 * G * 2 * Cp * Cp * 4 + par2;
  p.ns2 = Cp;
  if (2 * B * Cp > 512 || p.s2 > kSmemMax) {
    p.st2 = true;
    int ns = (512 / (2 * B)) / 16 * 16;
    while (ns >= 16 && (Cp % ns || (size_t)kRing * wunit_bytes<DIM>(2 * ns) + ring + par2 > kSmemMax)) ns -= 16;
    if (ns < 16) return p;
    p.ns2 = ns;
    p.s2 = (size_t)kRing * wunit_bytes<DIM>(2 * ns) + ring + par2;
    p.w2_floats = weight_image_floats<DIM>(1, ns, Cp / ns, Cp / 8);
  }
  if (nimg != 2) {
    p.s1 = one_cta_per_sm(p.st1 ? (size_t)kRing * wunit_bytes<DIM>(p.ns1, nimg) + ring + par1
                                : ring + (size_t)G * nimg * kin8 * Cp * 4 + par1);
    p.s2 = one_cta_per_sm(p.st2 ? (size_t)kRing * wunit_bytes<DIM>(2 * p.ns2, nimg) + ring + par2
                                : ring + (size_t)2 * G * nimg * Cp * Cp * 4 + par2);
    if (p.st1) p.w1_floats = weight_image_floats<DIM>(0, p.ns1, Cp / p.ns1, kin8 / 8, nimg);
    if (p.st2) p.w2_floats = weight_image_floats<DIM>(1, p.ns2, Cp / p.ns2, Cp / 8, nimg);
  }
  p.ok = true;
  return p;
}

template <int DIM>
bool fwd_supported(int cin, int c) { return fwd_plan<DIM>(cin, c).ok; }

inline int64_t align32f(int64_t floats) { return (floats + 31) / 32 * 32; }

template <int DIM>
int64_t fwd_ws_bytes(const csmpn_block_desc& d) {
  const FwdPlan p = fwd_plan<DIM>(d.c0 + d.c1 + d.c2, d.c, d.tf32 ? 1 : 2);
  if (!p.ok) return -1;
  return (align32f(p.w1_floats) + align32f(p.w2_floats)) * 4;
}

// TERMS: numeric mode (csmpn_block_desc.tf32 = 1 -> 1, else 3); MET: non-Euclidean metric mp
template <int DIM, int TERMS, bool MET>
int launch_fwd(const csmpn_block_desc& d, MetricArg<MET> mp, cudaStream_t stream) {
  constexpr int B = Alg<DIM>::B;
  FwdArgs a;
  memset(&a, 0, sizeof(a));
  a.rows = d.rows;
  a.tiles = (int)((d.rows + kTile - 1) / kTile);
  a.C = d.c;
  a.Cp = round_up(d.c, 16);
  a.cin = d.c0 + d.c1 + d.c2;
  a.kin8 = round_up(a.cin, 8);
  a.in_bpt = d.in_bpt;
  a.in_cp = round_up(a.cin, 16);
  a.mode = d.mode; a.c0 = d.c0; a.c1 = d.c1; a.c2 = d.c2; a.pair_attr = d.pair_attr;
  a.vt_k = d.vt_k; a.vt_fp = d.vt_fp;
  a.p0 = d.p0; a.p1 = d.p1; a.p2 = d.p2;
  a.src = d.src; a.dst = d.dst; a.eid = d.eid;
  a.w1 = d.w1; a.b1 = d.b1; a.sa = d.sa; a.sb = d.sb; a.wr = d.wr; a.na = d.na; a.wl = d.wl; a.bl = d.bl; a.wp = d.wp; a.la = d.la;
  a.save_y1 = d.save_y1; a.y2 = d.save_y2; a.save_xr = d.save_xr; a.save_o = d.save_o; a.save_x0 = d.save_x0;
  a.y = d.y; a.res = d.res; a.out_bpt = d.out_bpt; a.has_b1 = d.has_b1;
  if (!a.y2 || !a.y) return CSMPN_ERR_BAD_ARG;
  if (a.in_bpt && (d.mode != 0 || d.c1 || d.c2)) return CSMPN_ERR_BAD_ARG;
  if (d.mode == 2 && (d.vt_k < 1 || d.vt_k > 3 || d.vt_fp < 1 || d.c0 % (d.vt_k * d.vt_fp) || d.c1 || d.c2 || !d.src)) return CSMPN_ERR_BAD_ARG;
  if (a.out_bpt && d.res) return CSMPN_ERR_BAD_ARG;
  const FwdPlan p = fwd_plan<DIM>(a.cin, a.C, n_images(TERMS));
  if (!p.ok) return CSMPN_ERR_UNSUPPORTED;
  if (a.tiles == 0) return CSMPN_OK;
  a.ns1 = p.ns1; a.ns2 = p.ns2;
  const int mask = d.stage_mask ? d.stage_mask : ~0;
  if (p.st1 || p.st2) {
    // streamed weights: the pre-split images live in the caller's forward workspace (csmpn_block_fwd_workspace)
    if (!d.fwd_ws || d.fwd_ws_bytes < (align32f(p.w1_floats) + align32f(p.w2_floats)) * 4) return CSMPN_ERR_WORKSPACE;
    if (p.st2 && !d.save_o) return CSMPN_ERR_BAD_ARG;  // the scaling pass of f2 re-reads the product sum from it
    float* w1img = (float*)d.fwd_ws;
    float* w2img = w1img + align32f(p.w1_floats);
    a.wimg1 = w1img; a.wimg2 = w2img;
    if (p.st1 && (mask & 1)) {
      WPrepArgs w{d.w1, nullptr, 0, 0, a.C, a.cin, 0, p.ns1, a.Cp / p.ns1, a.kin8 / 8, 0, w1img};
      int st = launch_weight_images<DIM, TERMS>(w, p.w1_floats, stream);
      if (st) return st;
    }
    if (p.st2 && (mask & 2)) {
      WPrepArgs w{d.wr, d.wl, 1, 0, a.C, a.C, 0, p.ns2, a.Cp / p.ns2, a.Cp / 8, 0, w2img};
      int st = launch_weight_images<DIM, TERMS>(w, p.w2_floats, stream);
      if (st) return st;
    }
  }
  const int grid = a.tiles < sm_count_cached() ? a.tiles : sm_count_cached();
  auto run = [&](auto kern, size_t smem_bytes) -> int {
    CSMPN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    kern<<<grid, kThreads, smem_bytes, stream>>>(a, mp);
    return CSMPN_OK;
  };
  if (mask & 1) {
    const bool overlap = !p.st1 && use_overlapped_epilogue(B, a.Cp);
    int rc = overlap ? (a.in_bpt ? run(tc_f1db_kernel<DIM, true, TERMS, MET>, p.s1) : run(tc_f1db_kernel<DIM, false, TERMS, MET>, p.s1))
             : a.in_bpt ? (p.st1 ? run(tc_f1_kernel<DIM, true, true, TERMS, MET>, p.s1) : run(tc_f1_kernel<DIM, true, false, TERMS, MET>, p.s1))
                        : (p.st1 ? run(tc_f1_kernel<DIM, false, true, TERMS, MET>, p.s1) : run(tc_f1_kernel<DIM, false, false, TERMS, MET>, p.s1));
    if (rc) return rc;
    CSMPN_LAUNCH_CHECK("tc_f1_kernel");
  }
  if (mask & 2) {
    int rc = p.st2 ? run(tc_f2_kernel<DIM, true, TERMS, MET>, p.s2) : run(tc_f2_kernel<DIM, false, TERMS, MET>, p.s2);
    if (rc) return rc;
    CSMPN_LAUNCH_CHECK("tc_f2_kernel");
  }
  return CSMPN_OK;
}

template <int DIM, int TERMS>
int launch_fwd_metric(const csmpn_block_desc& d, cudaStream_t stream) {
  MetricParams mp;
  if (block_metric(DIM, d, &mp)) return launch_fwd<DIM, TERMS, true>(d, mp, stream);
  return launch_fwd<DIM, TERMS, false>(d, NoMetric{}, stream);
}

}  // namespace tcb

int tc_block_fwd(int dim, const csmpn_block_desc* d, cudaStream_t stream) {
  if (dim == 2) return d->tf32 ? tcb::launch_fwd_metric<2, 1>(*d, stream) : tcb::launch_fwd_metric<2, 3>(*d, stream);
  if (dim == 3) return d->tf32 ? tcb::launch_fwd_metric<3, 1>(*d, stream) : tcb::launch_fwd_metric<3, 3>(*d, stream);
  return CSMPN_ERR_UNSUPPORTED;
}
int64_t tc_block_fwd_workspace(int dim, const csmpn_block_desc* d) {
  if (dim == 2) return tcb::fwd_ws_bytes<2>(*d);
  if (dim == 3) return tcb::fwd_ws_bytes<3>(*d);
  return -1;
}
bool tc_block_bwd_supported(int dim, int c_in, int c);  // tc_block_bwd.cu
int tc_block_bwd_wide(int dim, int c_in, int c);         // tc_block_bwd.cu: np of the wide plan, 0 if resident
bool tc_block_supported(int dim, int c_in, int c);
// bit 0: supported, bit 1 / 2: f1 / f2 stream their weights, bit 3: the backward runs the wide plan
int tc_block_plan(int dim, int c_in, int c) {
  if (!tc_block_supported(dim, c_in, c)) return 0;
  tcb::FwdPlan p = dim == 2 ? tcb::fwd_plan<2>(c_in, c) : tcb::fwd_plan<3>(c_in, c);
  return 1 | (p.st1 ? 2 : 0) | (p.st2 ? 4 : 0) | (tc_block_bwd_wide(dim, c_in, c) ? 8 : 0);
}
// output channels per pass: bits 0-9 f1 (ns1), bits 10-19 f2 (ns2; both = Cp with resident weights), bits 20-29 the
// streamed backward GEMMs (np; 0 for the resident backward); 0 if the engine does not take the shape
int tc_block_passes(int dim, int c_in, int c) {
  if (!tc_block_supported(dim, c_in, c)) return 0;
  tcb::FwdPlan p = dim == 2 ? tcb::fwd_plan<2>(c_in, c) : tcb::fwd_plan<3>(c_in, c);
  return p.ns1 | (p.ns2 << 10) | (tc_block_bwd_wide(dim, c_in, c) << 20);
}
bool tc_block_supported(int dim, int c_in, int c) {
  if (dim == 2) return tcb::fwd_supported<2>(c_in, c) && tc_block_bwd_supported(2, c_in, c);
  if (dim == 3) return tcb::fwd_supported<3>(c_in, c) && tc_block_bwd_supported(3, c_in, c);
  return false;
}

}  // namespace csmpn
