// pgmuvi_b200 - the staged engine's big products on Blackwell tensor cores (tcgen05 / TMEM), for
// float32 models.  Two users of one 128x128-tile 3xTF32 product engine (tc_*):
//
// (G phase)
//   K~^-1 = X^T X   (X = L^-1, the "lauum" third of the n^3 flops)   as 3xTF32 products with FP32
//   accumulators in tensor memory, each 128x128 tile contracted at once - in the epilogue, straight
//   out of TMEM - with W = alpha alpha^T - K~^-1 and the regenerated dK/dtheta in FP64: the north
//   star's kernel (3) "0.5 tr((alpha alpha^T - K^-1) dK/dtheta) without ever materialising it",
//   for float32 models (the reference's default dtype, pgmuvi/lightcurve.py:2434-2446; loss.backward()
//   of pgmuvi/trainers.py:181).  The MLL itself (Cholesky, solves, log-det) stays on the FP64 path.
//
//   lg_pack_tf32   X^T tiles (fp64 64x64 images of the T phase) -> packed TF32 hi / lo operand images
//                  U[c, k] = X[k, c], one 16 KB SWIZZLE_128B image per (128 rows, 32 k) - byte for byte
//                  what tcgen05.mma reads from shared memory, so a pipeline stage is four bulk copies
//   lg_grad_tc     one CTA per 128x128 tile (I >= J) of K~^-1:  warp 0 = bulk-copy producer,
//                  warp 1 = MMA issuer (one thread; owns the TMEM allocation), warps 2-9 = epilogue
//                  (tcgen05.ld -> W -> dK/dtheta contraction in FP64 -> per-tile partial sums)
//
// (P phase, panel schedule)  the right-looking TRAILING UPDATE  C_ij -= sum_{k in panel} L_ik L_jk^T
//   - the north star's kernel (2), "trailing SYRK/GEMM updates on tensor cores, TF32-refined":
//   lg_pack_panel_tf32   the panel's L tiles (rows below the panel) -> packed TF32 hi / lo images
//   lg_update_tc         one CTA per 128x128 tile of the trailing triangle; epilogue = read-modify-write
//                        of the four 64x64 FP64 tile images (first panel: K~_ij generated in the epilogue
//                        instead, as lg_update does).  The 64x64 diagonal factorisations, the
//                        triangular solves and the in-panel updates stay FP64.
//
// Tensor memory (all 512 columns, one CTA per SM).  tcgen05.mma truncates on every accumulating
// instruction (tc_tf32.cuh), so the sum over k is split into PIECES of 16 k (half a 32-k chunk):
//   [256,512) two piece buffers, ping-pong between the MMA warp and the epilogue warps (mbarriers
//             pfull[2] / pempty[2]).  Per piece: the 4 cross-term MMAs (hi lo + lo hi) first - the
//             accumulator is still 2^-11 small, their truncation is harmless - then the 2 hi hi MMAs,
//             i.e. two truncating additions per piece instead of K / 8 * 3 per tile;
//   [  0,256) master accumulator as an unevaluated float pair (hi [0,128), lo [128,256)): the epilogue
//             warps drain every piece and add it with Fast2Sum on the CUDA cores (round to nearest,
//             the rounding error of each addition kept in lo).
#pragma once
#include "gp_large.cuh"
#include "tc_tf32.cuh"

namespace pgm {

constexpr int TC_THREADS = 320;        // producer warp + MMA warp + 8 epilogue warps
constexpr int TC_EPI_THREADS = 256;

// packed operand images of one light curve: piece (0 = hi, 1 = lo), 128-row block I, k-chunk kc
__host__ __device__ inline size_t tc_pack_floats(int n_max) {   // per light curve, both pieces
  const size_t N = (n_max + TS - 1) / TS, NT = (N + 1) / 2, KCH = 2 * N;
  return 2 * NT * KCH * (size_t)tc::IMG_FLOATS;
}
__host__ __device__ inline size_t large_ws_bytes_tc(int n_max, int B) {
  return ((large_ws_bytes(n_max, B) + 1023) & ~(size_t)1023) + tc_pack_floats(n_max) * 4 * (size_t)B;
}
__host__ __device__ inline float* tc_pack_base(double* ws, int n_max, int B, int b) {
  char* p = reinterpret_cast<char*>(ws) + ((large_ws_bytes(n_max, B) + 1023) & ~(size_t)1023);
  return reinterpret_cast<float*>(p) + tc_pack_floats(n_max) * (size_t)b;
}

// grid (Nmax, 2 * NTmax, B): block (a, b64) converts the 64 rows of tile column b64 of X (rows of U)
// against the 64 k of tile row a.  a > b64: the stored X_ab^T image; a == b64: X_bb^T (tilesT);
// a < b64 inside the same 128-row block or b64 >= N: zeros.
static __global__ void __launch_bounds__(NTHREADS) lg_pack_tf32(LargeArgs A) {
  const LcView v = lc_view(A, (int)blockIdx.z);
  if (v.st.state[v.b] != LG_FACTORED) return;
  const int a = blockIdx.x, b64 = blockIdx.y, I = b64 >> 1;
  if (a >= v.N || a < 2 * I || I >= (v.N + 1) / 2) return;
  const int Nmax = (A.n_max + TS - 1) / TS, NTmax = (Nmax + 1) / 2, KCH = 2 * Nmax;
  float* hi = tc_pack_base(A.ws, A.n_max, A.B, v.b);
  float* lo = hi + (size_t)NTmax * KCH * tc::IMG_FLOATS;
  const double* src = nullptr;
  if (b64 < v.N) {
    if (a > b64) src = lg_tile(v.w.tilesX, a, b64);
    else if (a == b64) src = v.w.tilesT + (size_t)b64 * TT;
  }
  const int row0 = (b64 & 1) * TS;
  for (int idx = threadIdx.x; idx < TT / 2; idx += NTHREADS) {
    const int c = idx >> 5, k = (idx & 31) * 2;     // row c of the image (column of X), k pair
    float2 h = make_float2(0.f, 0.f), l = make_float2(0.f, 0.f);
    if (src) {
      const double2 x = *reinterpret_cast<const double2*>(src + img(c, k));
      tc::split_tf32(x.x, h.x, l.x);
      tc::split_tf32(x.y, h.y, l.y);
    }
    const size_t o = ((size_t)I * KCH + 2 * a + (k >> 5)) * tc::IMG_FLOATS + tc::sw128_idx(row0 + c, k & 31);
    *reinterpret_cast<float2*>(hi + o) = h;
    *reinterpret_cast<float2*>(lo + o) = l;
  }
}


// ------------------------------------------------------------------------------------
// the 128x128-tile product engine:  D = sum_{kc0 <= kc < kc1} A(kc) B(kc)^T  over packed images
// ------------------------------------------------------------------------------------
constexpr unsigned T_MASTER = 0, T_MLO = 128, T_PIECE = 256;

// Pieces of 16 k, two per 32-k chunk (two truncating hi hi additions each): accuracy first.  32-k
// pieces halve the drain work - C4's G phase 170 -> 112 ms - at 1.8x the error (DESIGN.md 4.2b).
constexpr int TC_PPC = 2;              // pieces per 32-k chunk
constexpr int TC_KPP = 4 / TC_PPC;     // 8-k MMA steps per piece
constexpr int TC_FOLD = 4;             // pieces per register fold of tc_drain

struct TcCtx {
  unsigned base;        // shared address of stage 0 (1024-byte aligned)
  unsigned bar_full, bar_empty, bar_pfull, bar_pempty, tslot;
  unsigned tmem;
};

// all threads; `bars` = shared address of 14 doubles.  Ends with a block barrier.
template <int NST>
__device__ __forceinline__ void tc_setup(TcCtx& cx, unsigned stage_base, unsigned bars) {
  static_assert(NST >= 1 && NST <= 3, "the barrier region holds the full / empty pairs of 3 stages");
  cx.base = stage_base;
  cx.bar_full = bars; cx.bar_empty = bars + 24; cx.bar_pfull = bars + 48; cx.bar_pempty = bars + 64;
  cx.tslot = bars + 96;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NST; ++s) { mbar_init(cx.bar_full + 8 * s, 1); mbar_init(cx.bar_empty + 8 * s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(cx.bar_pfull + 8 * s, 1); mbar_init(cx.bar_pempty + 8 * s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    fence_proxy_async();
  }
  if ((threadIdx.x >> 5) == 1) tc::tmem_alloc(cx.tslot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(cx.tmem) : "r"(cx.tslot));
}
__device__ __forceinline__ void tc_teardown(const TcCtx& cx) {
  __syncthreads();
  if ((threadIdx.x >> 5) == 1) tc::tmem_dealloc(cx.tmem, 512);
}

// warp 0, one lane: stream the four operand images of every chunk (hi / lo at ahi / alo + kc * IMG)
template <int NST>
__device__ __forceinline__ void tc_producer(const TcCtx& cx, const float* ahi, const float* alo,
                                            const float* bhi, const float* blo, int nchunks) {
  for (int c = 0; c < nchunks; ++c) {
    const int s = c % NST, use = c / NST;
    if (use > 0) mbar_wait(cx.bar_empty + 8 * s, (use - 1) & 1);
    const unsigned bar = cx.bar_full + 8 * s, dst = cx.base + (unsigned)s * 4 * tc::IMG_BYTES;
    const size_t o = (size_t)c * tc::IMG_FLOATS;
    mbar_expect_tx(bar, 4 * tc::IMG_BYTES);
    bulk_g2s(dst, ahi + o, tc::IMG_BYTES, bar);
    bulk_g2s(dst + tc::IMG_BYTES, alo + o, tc::IMG_BYTES, bar);
    bulk_g2s(dst + 2 * tc::IMG_BYTES, bhi + o, tc::IMG_BYTES, bar);
    bulk_g2s(dst + 3 * tc::IMG_BYTES, blo + o, tc::IMG_BYTES, bar);
  }
}

// warp 1, one lane: per piece the cross terms (hi lo + lo hi) first, then hi hi
template <int NST>
__device__ __forceinline__ void tc_mma_issuer(const TcCtx& cx, int nchunks) {
  constexpr uint32_t idesc = tc::idesc_tf32(128, 128);
  for (int c = 0; c < nchunks; ++c) {
    const int s = c % NST, use = c / NST;
    mbar_wait(cx.bar_full + 8 * s, use & 1);
    tc::fence_after_sync();
    const unsigned st = cx.base + (unsigned)s * 4 * tc::IMG_BYTES;
    for (int hp = 0; hp < TC_PPC; ++hp) {
      const int piece = c * TC_PPC + hp, buf = piece & 1;
      if (piece >= 2) {                  // the epilogue has drained this piece buffer
        mbar_wait(cx.bar_pempty + 8 * buf, ((piece >> 1) - 1) & 1);
        tc::fence_after_sync();
      }
      const unsigned tp = cx.tmem + T_PIECE + 128u * (unsigned)buf;
      const int ks0 = hp * TC_KPP;
      for (int ks = ks0; ks < ks0 + TC_KPP; ++ks) {
        const uint64_t ahi = tc::smem_desc_sw128(st + ks * 32);
        const uint64_t alo = tc::smem_desc_sw128(st + tc::IMG_BYTES + ks * 32);
        const uint64_t bhi = tc::smem_desc_sw128(st + 2 * tc::IMG_BYTES + ks * 32);
        const uint64_t blo = tc::smem_desc_sw128(st + 3 * tc::IMG_BYTES + ks * 32);
        tc::mma_tf32(tp, alo, bhi, idesc, ks > ks0 ? 1u : 0u);
        tc::mma_tf32(tp, ahi, blo, idesc, 1u);
      }
      for (int ks = ks0; ks < ks0 + TC_KPP; ++ks) {
        const uint64_t ahi = tc::smem_desc_sw128(st + ks * 32);
        const uint64_t bhi = tc::smem_desc_sw128(st + 2 * tc::IMG_BYTES + ks * 32);
        tc::mma_tf32(tp, ahi, bhi, idesc, 1u);
      }
      tc::mma_commit(cx.bar_pfull + 8 * buf);   // piece complete
    }
    tc::mma_commit(cx.bar_empty + 8 * s);       // the stage is free once these MMAs have read it
  }
}

// The 8 epilogue warps drain every piece: two levels.  Level 1: a running sum of TC_FOLD consecutive
// pieces in REGISTERS (64 floats per thread, plain round-to-nearest adds: a fold of 4 keeps their error
// at the level of one piece's own truncation) - 4 LDTM + 64 FADD per piece.  Level 2: every TC_FOLD
// pieces the running sum goes into the float-pair master accumulator in TMEM by Fast2Sum (|hi| >= |sum|
// but for the first folds, where the missed rounding error is of no consequence).  Draining every piece
// straight into the TMEM master (r02k: ~400 instructions per thread and piece, tensor pipe 18 % active)
// made the drain, not the tensor pipe, the bound.  tlane = TMEM address of this thread's lane at its
// first column.
__device__ __forceinline__ void tc_drain(const TcCtx& cx, unsigned tlane, int nchunks) {
  const int lane = threadIdx.x & 31;
  const int npieces = nchunks * TC_PPC;
  float m1[64];
  int in_fold = 0, nfold = 0;
  for (int piece = 0; piece < npieces; ++piece) {
    const int buf = piece & 1;
    mbar_wait(cx.bar_pfull + 8 * buf, (piece >> 1) & 1);
    tc::fence_after_sync();
    const bool first = in_fold == 0;
    {
      // all four loads in flight, one wait, and the piece buffer goes back to the MMA warp before
      // the adds: the round trip pfull -> pempty, not the instruction count, paces the pipeline
      float p0[16], p1[16], p2[16], p3[16];
      const unsigned tpc = tlane + T_PIECE + 128u * (unsigned)buf;
      tc::tmem_ld16_async(tpc, p0);
      tc::tmem_ld16_async(tpc + 16, p1);
      tc::tmem_ld16_async(tpc + 32, p2);
      tc::tmem_ld16_async(tpc + 48, p3);
      tc::tmem_wait_ld();
      tc::tmem_tie(p0);
      tc::tmem_tie(p1);
      tc::tmem_tie(p2);
      tc::tmem_tie(p3);
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(cx.bar_pempty + 8 * buf);
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        m1[e] = first ? p0[e] : __fadd_rn(m1[e], p0[e]);
        m1[16 + e] = first ? p1[e] : __fadd_rn(m1[16 + e], p1[e]);
        m1[32 + e] = first ? p2[e] : __fadd_rn(m1[32 + e], p2[e]);
        m1[48 + e] = first ? p3[e] : __fadd_rn(m1[48 + e], p3[e]);
      }
    }
    if (++in_fold == TC_FOLD || piece == npieces - 1) {
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 16) {
        float hi[16], lo[16];
        if (nfold > 0) {
          tc::tmem_ld16(tlane + T_MASTER + (unsigned)c0, hi);
          tc::tmem_ld16(tlane + T_MLO + (unsigned)c0, lo);
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float s2 = __fadd_rn(hi[e], m1[c0 + e]);
            lo[e] = __fadd_rn(lo[e], __fsub_rn(m1[c0 + e], __fsub_rn(s2, hi[e])));
            hi[e] = s2;
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) { hi[e] = m1[c0 + e]; lo[e] = 0.f; }
        }
        tc::tmem_st16(tlane + T_MASTER + (unsigned)c0, hi);
        tc::tmem_st16(tlane + T_MLO + (unsigned)c0, lo);
      }
      tc::tmem_wait_st();
      in_fold = 0;
      ++nfold;
    }
  }
}

// Block -> tile of a lower-triangular set of Mt x Mt 128-tiles, in SUPER-BLOCKS of S x S tiles: the
// CTAs resident at the same time (one per SM) then cover a roughly square patch and share their A / B
// operand panels through L2 (row-major order: one A panel + ~148 B panels = 300 MB per wave, super-
// blocks of 12: 24 panels = 48 MB).  grid = nSB (nSB + 1) / 2 * S * S; blocks above the diagonal or
// past the edge return false.
__host__ __device__ inline int tc_super(int Mt) { return Mt < 12 ? Mt : 12; }
__host__ __device__ inline unsigned tc_grid(int Mt) {
  const int S = tc_super(Mt), nSB = (Mt + S - 1) / S;
  return (unsigned)(nSB * (nSB + 1) / 2) * (unsigned)(S * S);
}
__device__ __forceinline__ bool tc_tile_of_block(unsigned bid, int Mt, int& a, int& b) {
  const int S = tc_super(Mt);
  const unsigned sb = bid / (unsigned)(S * S), within = bid - sb * (unsigned)(S * S);
  int sI, sJ;
  tri_unrank((int)sb, sI, sJ);
  a = sI * S + (int)(within / (unsigned)S);
  b = sJ * S + (int)(within % (unsigned)S);
  return a < Mt && b <= a;
}

// per-point fields of the two 64-point sub-tiles of a side (128-block T128) -> vec, by the 256
// epilogue threads (et = 0..255); layout per sub-tile as lg_prefetch_side
template <int KIND, int QT, int D>
__device__ __forceinline__ void tc_load_side(double* vec, const LargeWs& w, int npad, int N, int T128,
                                             int et, bool with_alpha) {
  using C = Cfg<KIND, QT, D>;
  const int T0 = 2 * T128;
  for (int idx = et; idx < 2 * C::NF * TS; idx += TC_EPI_THREADS) {
    const int sub = idx / (C::NF * TS), o = idx - sub * C::NF * TS;
    const int f = o >> 6, p = o & 63;
    const int gp = (T0 + sub) * TS;
    double val = 0.0;
    if (T0 + sub < N) {
      if (o < D * TS) {
        val = w.fx[(size_t)f * npad + gp + p];
      } else if (o < C::NFB * TS) {
        const int o2 = o - D * TS, fc = o2 >> 7, pp = o2 & 127;   // (cos, sin) pairs: 128 doubles per field
        val = w.fcs[((size_t)fc * npad + gp) * 2 + pp];
      } else if (with_alpha) {
        val = w.alpha[gp + p];
      }
    } else if (o >= D * TS && o < C::NFB * TS) {
      val = ((o - D * TS) & 1) ? 0.0 : 1.0;                       // padded points: cos = 1, sin = 0
    }
    vec[sub * C::NF * TS + o] = val;
  }
}

template <int KIND, int QT, int D>
struct TcGradSmem {
  using C = Cfg<KIND, QT, D>;
  static constexpr int SIDE = 2 * C::NF * TS;                 // doubles per side (two 64-point sub-tiles)
  static constexpr int PAR_TAB = 0;                           // exp tables [96]
  static constexpr int PAR_RED = PAR_TAB + EXP_TAB;           // [8][NV] warp partials
  static constexpr int PAR_BAR = PAR_RED + 8 * C::NV;         // mbarriers (10) + TMEM slot
  static constexpr int PAR_END = PAR_BAR + 14;
  // 1024 bytes of alignment slack, NST pipeline stages of four operand images, the doubles above
  static constexpr size_t STAGE = 4 * tc::IMG_BYTES;
  static constexpr size_t FIXED = 1024 + (size_t)(2 * SIDE + PAR_END) * sizeof(double);
  // pipeline stages: the most, up to 3, that fit in a block's 227 KB of shared memory
  static constexpr int NST = FIXED + 3 * STAGE <= 227 * 1024 ? 3 : FIXED + 2 * STAGE <= 227 * 1024 ? 2 : 1;
  static constexpr size_t BYTES = FIXED + NST * STAGE;
  static_assert(BYTES <= 227 * 1024, "lg_grad_tc / lg_update_tc do not fit in shared memory");
};

template <int KIND, int QT, int D>
__global__ void __launch_bounds__(TC_THREADS, 1) lg_grad_tc(LargeArgs A) {
  using C = Cfg<KIND, QT, D>;
  using SM = TcGradSmem<KIND, QT, D>;
  constexpr int DS = C::DS;
  static_assert(C::NV <= LG_GP, "gradient partial slot too small");
  extern __shared__ __align__(1024) unsigned char smraw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  const LargeWs& w = v.w;
  const int n = v.n, N = v.N, npad = v.npad;
  const int Nmax = (A.n_max + TS - 1) / TS, NTmax = (Nmax + 1) / 2, KCH = 2 * Nmax;
  int I, J;
  if (!tc_tile_of_block(blockIdx.x, NTmax, I, J) || I >= (N + 1) / 2) return;
  const float* phi = tc_pack_base(A.ws, A.n_max, A.B, v.b);
  const float* plo = phi + (size_t)NTmax * KCH * tc::IMG_FLOATS;
  const int kc0 = 4 * I, nchunks = 2 * N - kc0;      // U[128 I .., k] = 0 for k < 128 I

  const unsigned base = (smem_u32(smraw) + 1023u) & ~1023u;
  unsigned char* gen = smraw + (base - smem_u32(smraw));
  double* sd = reinterpret_cast<double*>(gen + SM::NST * SM::STAGE);
  double* rowv = sd;
  double* colv = sd + SM::SIDE;
  double* par = sd + 2 * SM::SIDE;
  double* tab = par + SM::PAR_TAB;
  double* red = par + SM::PAR_RED;
  TcCtx cx;
  tc_setup<SM::NST>(cx, base, smem_u32(par + SM::PAR_BAR));

  if (warp == 0) {
    if (lane == 0) {
      const size_t oa = ((size_t)I * KCH + kc0) * tc::IMG_FLOATS, ob = ((size_t)J * KCH + kc0) * tc::IMG_FLOATS;
      tc_producer<SM::NST>(cx, phi + oa, plo + oa, phi + ob, plo + ob, nchunks);
    }
  } else if (warp == 1) {
    if (lane == 0) tc_mma_issuer<SM::NST>(cx, nchunks);
  } else {
    // ---------------- epilogue warps: per-point fields while the products run ----------------
    const int et = tid - 64;                              // 0..255
    const int q4 = warp & 3, half = (warp - 2) >> 2;      // TMEM lane quarter, column half
    const int r = 32 * q4 + lane;                         // accumulator row of this thread
    if (et < EXP_TAB) tab[et] = c_exp2_tab[et];
    tc_load_side<KIND, QT, D>(rowv, w, npad, N, I, et, true);
    tc_load_side<KIND, QT, D>(colv, w, npad, N, J, et, true);
    // Not LgConst: with nvcc 12.9 it raises <0,8,1> / <2,4,2> from 176 to 200 B of stack and their
    // spill stores / loads from 180 / 232 to 216 / 272 and 204 / 260 B.
    double wreg[QT], areg[QT * DS], lam[4];
#pragma unroll
    for (int q = 0; q < QT; ++q) wreg[q] = w.par[LG_PAR_WQ + q];
#pragma unroll
    for (int q = 0; q < QT * DS; ++q) areg[q] = w.par[LG_PAR_AQ + q];
#pragma unroll
    for (int q = 0; q < 4; ++q) lam[q] = w.par[LG_PAR_LM + q];
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
    double ga[C::NG];
#pragma unroll
    for (int t = 0; t < C::NG; ++t) ga[t] = 0.0;
    double trW = 0.0;
    const double* rv = rowv + (r >> 6) * C::NF * TS;
    const double* cv = colv + half * C::NF * TS;
    const int rr = r & 63;
    const int gi = I * 128 + r;
    const double al_i = rv[C::NFB * TS + rr];
    const unsigned tlane = cx.tmem + ((unsigned)(32 * q4) << 16) + (unsigned)(half * 64);
    tc_drain(cx, tlane, nchunks);
    // tcgen05.ld is warp-collective: the chunk loop is uniform over the warp (rows 32 q4 .. + 31),
    // the lower-triangle / n masks act per entry
    const int gi_hi = I * 128 + 32 * q4 + 31;
#pragma unroll 1
    for (int c0 = 0; c0 < 64; c0 += 16) {
      const int gj0 = J * 128 + half * 64 + c0;
      if (gj0 > gi_hi || I * 128 + 32 * q4 >= n) break;
      float kv[16], xv[16];
      tc::tmem_ld16(tlane + T_MASTER + (unsigned)c0, kv);
      tc::tmem_ld16(tlane + T_MLO + (unsigned)c0, xv);
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const int gj = gj0 + e;
        if (gi < n && gj <= gi) {
          const double W = al_i * cv[C::NFB * TS + c0 + e] - ((double)kv[e] + (double)xv[e]);
          if (gi == gj) trW += W;
          const double wgt = (gi == gj) ? W : 2.0 * W;
          k_grad_entry<KIND, QT, D>(rv, cv, rr, c0 + e, wreg, areg, lam, tab, wgt, ga);
        }
      }
    }
    tc::fence_before_sync();
    // reduction over the 256 epilogue threads (fixed order)
    double vv[C::NV];
#pragma unroll
    for (int t = 0; t < C::NG; ++t) vv[t] = ga[t];
    vv[C::NG] = trW;
#pragma unroll
    for (int t = 0; t < C::NV; ++t) {
      double s = vv[t];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += shfl_xor_d(s, o);
      if (lane == 0) red[(warp - 2) * C::NV + t] = s;
    }
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
    if (et < C::NV) {
      double s = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) s += red[w8 * C::NV + et];
      w.gpart[((size_t)I * (I + 1) / 2 + J) * LG_GP + et] = s;
    }
  }
  tc_teardown(cx);
}

// ------------------------------------------------------------------------------------
// P phase, panel schedule: the trailing update on tcgen05
// ------------------------------------------------------------------------------------
// grid (J1 - J0, 2 * NTmax - J1, B): block (kk, ii) packs tile L(i = J1 + ii, k = J0 + kk) - image rows
// = rows of L, image k = panel column - into image (I = i / 2, kc = 2 kk + {0, 1}); i >= N: zeros
static __global__ void __launch_bounds__(NTHREADS) lg_pack_panel_tf32(LargeArgs A, int J0, int J1) {
  const LcView v = lc_view(A, (int)blockIdx.z);
  if (v.st.state[v.b] != LG_ACTIVE || v.st.fail[v.b]) return;
  const int kk = blockIdx.x, i = J1 + blockIdx.y, I = i >> 1;
  if (I >= (v.N + 1) / 2) return;
  const int Nmax = (A.n_max + TS - 1) / TS, NTmax = (Nmax + 1) / 2, KCH = 2 * Nmax;
  float* hi = tc_pack_base(A.ws, A.n_max, A.B, v.b);
  float* lo = hi + (size_t)NTmax * KCH * tc::IMG_FLOATS;
  const double* src = (i < v.N) ? lg_tile(v.w.tilesL, i, J0 + kk) : nullptr;
  const int row0 = (i & 1) * TS;
  for (int idx = threadIdx.x; idx < TT / 2; idx += NTHREADS) {
    const int c = idx >> 5, k = (idx & 31) * 2;
    float2 h = make_float2(0.f, 0.f), l = make_float2(0.f, 0.f);
    if (src) {
      const double2 x = *reinterpret_cast<const double2*>(src + img(c, k));
      tc::split_tf32(x.x, h.x, l.x);
      tc::split_tf32(x.y, h.y, l.y);
    }
    const size_t o = ((size_t)I * KCH + 2 * kk + (k >> 5)) * tc::IMG_FLOATS + tc::sw128_idx(row0 + c, k & 31);
    *reinterpret_cast<float2*>(hi + o) = h;
    *reinterpret_cast<float2*>(lo + o) = l;
  }
}

// C_ij -= sum_{k in [J0, J1)} L_ik L_jk^T over the trailing triangle i >= j >= J1 (J1 even), one CTA
// per 128x128 tile; build: C_ij = K~_ij - sum (first panel), exactly as lg_update mode 1
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(TC_THREADS, 1)
    lg_update_tc(LargeArgs A, int J0, int J1, int build) {
  using C = Cfg<KIND, QT, D>;
  using SM = TcGradSmem<KIND, QT, D>;
  constexpr int DS = C::DS;
  extern __shared__ __align__(1024) unsigned char smraw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_ACTIVE || v.st.fail[v.b]) return;
  const LargeWs& w = v.w;
  const int n = v.n, N = v.N, npad = v.npad;
  const int Nmax = (A.n_max + TS - 1) / TS, NTmax = (Nmax + 1) / 2, KCH = 2 * Nmax;
  int a, b;
  if (!tc_tile_of_block(blockIdx.x, NTmax - (J1 >> 1), a, b)) return;
  const int I = (J1 >> 1) + a, J = (J1 >> 1) + b;
  if (I >= (N + 1) / 2) return;
  const float* phi = tc_pack_base(A.ws, A.n_max, A.B, v.b);
  const float* plo = phi + (size_t)NTmax * KCH * tc::IMG_FLOATS;
  const int nchunks = 2 * (J1 - J0);
  const double jitter = chol_jitter(v.st.attempt[v.b], A.flags);

  const unsigned base = (smem_u32(smraw) + 1023u) & ~1023u;
  unsigned char* gen = smraw + (base - smem_u32(smraw));
  double* sd = reinterpret_cast<double*>(gen + SM::NST * SM::STAGE);
  double* rowv = sd;
  double* colv = sd + SM::SIDE;
  double* par = sd + 2 * SM::SIDE;
  double* tab = par + SM::PAR_TAB;
  TcCtx cx;
  tc_setup<SM::NST>(cx, base, smem_u32(par + SM::PAR_BAR));

  if (warp == 0) {
    if (lane == 0) {
      const size_t oa = (size_t)I * KCH * tc::IMG_FLOATS, ob = (size_t)J * KCH * tc::IMG_FLOATS;
      tc_producer<SM::NST>(cx, phi + oa, plo + oa, phi + ob, plo + ob, nchunks);
    }
  } else if (warp == 1) {
    if (lane == 0) tc_mma_issuer<SM::NST>(cx, nchunks);
  } else {
    const int et = tid - 64;
    const int q4 = warp & 3, half = (warp - 2) >> 2;
    const int r = 32 * q4 + lane;
    // Not LgConst: with nvcc 12.9 it adds 12 to 16 B of spill loads to <0,4,1>, <1,4,2>, <2,4,2>.
    double wreg[QT], areg[QT * DS], lam[4];
    if (build) {
      if (et < EXP_TAB) tab[et] = c_exp2_tab[et];
      tc_load_side<KIND, QT, D>(rowv, w, npad, N, I, et, false);
      tc_load_side<KIND, QT, D>(colv, w, npad, N, J, et, false);
#pragma unroll
      for (int q = 0; q < QT; ++q) wreg[q] = w.par[LG_PAR_WQ + q];
#pragma unroll
      for (int q = 0; q < QT * DS; ++q) areg[q] = w.par[LG_PAR_AQ + q];
#pragma unroll
      for (int q = 0; q < 4; ++q) lam[q] = w.par[LG_PAR_LM + q];
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
    }
    const double* rv = rowv + (r >> 6) * C::NF * TS;
    const double* cv = colv + half * C::NF * TS;
    const int rr = r & 63;
    const int ti = 2 * I + (r >> 6), tj = 2 * J + half;       // the 64x64 tile of this thread's entries
    const int gi = I * 128 + r;
    const unsigned tlane = cx.tmem + ((unsigned)(32 * q4) << 16) + (unsigned)(half * 64);
    tc_drain(cx, tlane, nchunks);
    // every lane of the warp shares ti, tj (32 rows of one 64-row sub-tile)
    if (ti < N && tj <= ti) {
      double* out = lg_tile(w.tilesL, ti, tj);
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 16) {
        float kv[16], xv[16];
        tc::tmem_ld16(tlane + T_MASTER + (unsigned)c0, kv);
        tc::tmem_ld16(tlane + T_MLO + (unsigned)c0, xv);
#pragma unroll
        for (int e = 0; e < 16; e += 2) {
          double2* p = reinterpret_cast<double2*>(out + img(rr, c0 + e));
          const double s0 = (double)kv[e] + (double)xv[e], s1 = (double)kv[e + 1] + (double)xv[e + 1];
          double2 o2;
          if (build) {
            double k2[2];
#pragma unroll
            for (int u = 0; u < 2; ++u)
              k2[u] = lg_k_masked<KIND, QT, D>(rv, cv, rr, c0 + e + u, gi, tj * TS + c0 + e + u, n, w.dn,
                                               jitter, wreg, areg, lam, tab);
            o2 = make_double2(k2[0] - s0, k2[1] - s1);
          } else {
            o2 = *p;
            o2.x -= s0;
            o2.y -= s1;
          }
          *p = o2;
        }
      }
    }
    tc::fence_before_sync();
  }
  tc_teardown(cx);
}

}  // namespace pgm
