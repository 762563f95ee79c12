// pgmuvi_b200 - fused exact-GP evaluation for sm_100a (B200).
//
// One thread block owns one light curve at a time and runs the whole path for it:
//
//   (1) spectral-mixture K(x,x') tiles generated on the fly (never written to HBM)
//   (2) left-looking blocked Cholesky (64x64 tiles, trailing updates on FP64 tensor cores
//       through mma.sync.m8n8k4.f64 -> SASS DMMA), forward solve, log-det
//   (3) tiled triangular inverse + K^-1 = X^T X regenerated tile by tile and contracted at
//       once with dK/dtheta (regenerated per tile) -> gradient; K^-1 never materialised
//   (4) constraint chain rule, optional optimiser step (fit kernel)
//
// Reference semantics: gpytorch SpectralMixtureKernel / ExactMarginalLogLikelihood as driven
// by pgmuvi/trainers.py:177-182 and pgmuvi/gps.py:205-220, 302-318 (SURVEY.md Appendix A).
//
// Per-block scratch lives in a global workspace indexed by blockIdx.x (reused for every
// light curve the block processes); only L / L^-1 tiles go there, stored as the exact
// shared-memory operand image (two 32-deep k-chunks, XOR-swizzled), so that a pipeline stage
// is filled by ONE elected thread with two 16 KB bulk copies (cp.async.bulk -> SASS UBLKCP)
// that complete on an mbarrier: no per-chunk block barrier, and the stream of chunks runs
// ahead across tile boundaries.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/pgmuvi_b200.h"   // PGM_KIND_* / PGM_CON_* / PGM_FLAG_*

namespace pgm {

constexpr int TS = 64;          // tile edge
constexpr int TT = TS * TS;     // elements per tile
constexpr int KC = 32;          // k-chunk per pipeline stage
constexpr int NTHREADS = 256;   // 8 warps: 2 (M) x 4 (N), warp tile 32 x 16
constexpr int NSTAGES = 2;
constexpr int OPBUF = TS * KC;  // elements per operand per stage (XOR-swizzled, no padding)
constexpr int LD_S = 68;        // smem ld of the 64x64 work tile (diagonal blocks)
constexpr int STAGE_ELEMS = NSTAGES * 2 * OPBUF;   // 8192 doubles = 64 KB
constexpr int S_ELEMS = TS * LD_S;                 // 4352

// ------------------------------------------------------------------------------------
// small PTX wrappers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_f64(double (&d)[2], double a, double b) {
  asm volatile(
      "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(d[0]), "+d"(d[1])
      : "d"(a), "d"(b));
}
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
// mbarrier + bulk-copy (TMA, non-tensor form) primitives: one elected thread streams whole
// 16 KB operand chunks global -> shared, completion is counted in bytes on an mbarrier.
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes,
                                         unsigned bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::
          "r"(dst), "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, unsigned src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst),
               "r"(src), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() {
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
// source shared memory of all committed bulk stores has been read
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
}
// all committed bulk stores are complete (visible to later bulk loads of this thread)
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
}
// generic-proxy writes (st.global / st.shared) -> visible to later async-proxy (bulk) reads.
// The full fence drains the thread's global stores (slow): only the 64x64 diagonal blocks use
// it; off-diagonal tiles leave through shared memory + bulk store (shared-only fence).
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ double shfl_d(double v, int src) {
  return __shfl_sync(0xffffffffu, v, src);
}
__device__ __forceinline__ double shfl_xor_d(double v, int m) {
  return __shfl_xor_sync(0xffffffffu, v, m);
}

__host__ __device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }

// exp(x) for x <= 0 (small positive x also fine), branch free:
//   x = (2048 e + 32 j1 + j2) ln2/2048 + r, |r| <= ln2/4096,
//   exp(x) = 2^e * T1[j1] * T2[j2] * (1 + r + r^2/2 + r^3/6)   (truncation 3.4e-17 relative).
// T1 = correctly rounded 2^(j/64), T2 = 2^(j/2048), 96 doubles held in shared memory.
// One-constant argument reduction: |error| <= |x| * 8e-17 relative, <= 3e-17 absolute.
constexpr int EXP_TAB = 96;
__constant__ double c_exp2_tab[EXP_TAB] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0,
    // 2^(j/2048), j = 0..31
    0x1.0000000000000p+0, 0x1.00162f3904052p+0, 0x1.002c605e2e8cfp+0, 0x1.0042936faa3d8p+0,
    0x1.0058c86da1c0ap+0, 0x1.006eff583fc3dp+0, 0x1.0085382faef83p+0, 0x1.009b72f41a12bp+0,
    0x1.00b1afa5abcbfp+0, 0x1.00c7ee448ee02p+0, 0x1.00de2ed0ee0f5p+0, 0x1.00f4714af41d3p+0,
    0x1.010ab5b2cbd11p+0, 0x1.0120fc089ff63p+0, 0x1.0137444c9b5b5p+0, 0x1.014d8e7ee8d2fp+0,
    0x1.0163da9fb3335p+0, 0x1.017a28af25567p+0, 0x1.019078ad6a19fp+0, 0x1.01a6ca9aac5f3p+0,
    0x1.01bd1e77170b4p+0, 0x1.01d37442d5070p+0, 0x1.01e9cbfe113efp+0, 0x1.020025a8f6a35p+0,
    0x1.02168143b0281p+0, 0x1.022cdece68c4fp+0, 0x1.02433e494b755p+0, 0x1.02599fb483385p+0,
    0x1.027003103b10ep+0, 0x1.0286685c9e059p+0, 0x1.029ccf99d720ap+0, 0x1.02b338c811703p+0};
// cooperative copy of the table into shared memory (any block of >= 96 threads)
__device__ __forceinline__ void load_exp_tab(double* tab) {
  if (threadIdx.x < EXP_TAB) tab[threadIdx.x] = c_exp2_tab[threadIdx.x];
}

__device__ __forceinline__ double exp_neg(double x, const double* __restrict__ tab) {
  // clamp x >= -700 on the integer pipe (sign-magnitude: larger high word = more negative)
  const unsigned hx = min((unsigned)__double2hiint(x), 0xC085E000u);
  x = __hiloint2double((int)hx, __double2loint(x));
  double t = fma(x, 0x1.71547652b82fep+11, 6755399441055744.0);  // round(x * 2048/ln2)
  const int k = __double2loint(t);
  t -= 6755399441055744.0;
  const double r = fma(t, -0x1.62e42fefa39efp-12, x);            // ln2/2048
  const double tt = tab[(k >> 5) & 63] * tab[64 + (k & 31)];
  double p = fma(r, 1.66666666666666667e-01, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const double v = tt * p;
  return __hiloint2double(__double2hiint(v) + ((k >> 11) << 20), __double2loint(v));
}

// ------------------------------------------------------------------------------------
// static configuration per (kernel kind, padded mixture count, input dims)
// ------------------------------------------------------------------------------------
// the separable-kind code whose lam_factor implements an atom of the stationary kinds
#define PGM_ATOM_QP 100      // ScaleKernel(PeriodicKernel * RBFKernel), gps.py:915-935
#define PGM_ATOM_QP_RBF 101  // AdditiveKernel(QP, ScaleKernel(RBFKernel)), gps.py:1187-1236 (1-D)
#define PGM_ATOM_M12 102     // MaternKernel(nu=0.5): exp(-r), r = |tau| / l        (MaternGPModel nu)
#define PGM_ATOM_M25 103     // MaternKernel(nu=2.5): (1 + u + u^2/3) e^-u, u = sqrt5 |tau| / l
__host__ __device__ constexpr int stat_time_atom(int kind) {
  return ((kind - PGM_KIND_STAT_BASE) / 5 == 0) ? PGM_KIND_SEP_RBF
         : ((kind - PGM_KIND_STAT_BASE) / 5 == 1) ? PGM_KIND_SEP_MATERN15
         : ((kind - PGM_KIND_STAT_BASE) / 5 == 2) ? PGM_ATOM_QP
         : ((kind - PGM_KIND_STAT_BASE) / 5 == 3) ? PGM_ATOM_QP_RBF
         : ((kind - PGM_KIND_STAT_BASE) / 5 == 4) ? PGM_ATOM_M12 : PGM_ATOM_M25;
}
__host__ __device__ constexpr int stat_num_time(int kind) {   // time-kernel parameters
  return stat_time_atom(kind) == PGM_ATOM_QP ? 4 : stat_time_atom(kind) == PGM_ATOM_QP_RBF ? 6 : 2;
}
__host__ __device__ constexpr int stat_wave_atom(int kind) {   // 0 = no wavelength factor
  return ((kind - PGM_KIND_STAT_BASE) % 5 == 0) ? 0
         : (PGM_KIND_SEP_RBF + (kind - PGM_KIND_STAT_BASE) % 5 - 1);
}
__host__ __device__ constexpr int sep_num_lam(int sep_kind) {
  return (sep_kind == PGM_KIND_SEP_RBF || sep_kind == PGM_KIND_SEP_MATERN15) ? 2
         : (sep_kind == PGM_KIND_SEP_RQ) ? 3 : (sep_kind == PGM_KIND_SEP_CONST) ? 1 : 0;
}
// dims the spectral mixture acts on: d for the plain spectral-mixture kinds, else time only
__host__ __device__ constexpr int mix_dims(int kind, int d) {
  return kind >= PGM_KIND_SEP_RBF ? 1 : d;
}
// kernel parameters behind the mixture: wavelength kernel (outputscale, lengthscale[, alpha])
// or (constant); stationary kinds: time kernel (outputscale, lengthscale) + wavelength kernel
__host__ __device__ constexpr int num_lam(int kind) {
  return kind >= PGM_KIND_STAT_BASE ? stat_num_time(kind) + sep_num_lam(stat_wave_atom(kind))
                                    : sep_num_lam(kind);
}

template <int KIND, int QT, int D>
struct Cfg {
  static constexpr bool STAT = KIND >= PGM_KIND_STAT_BASE;
  static constexpr bool SEP = KIND >= PGM_KIND_SEP_RBF && !STAT;
  static constexpr int DS = mix_dims(KIND, D);
  static constexpr int NLT = STAT ? stat_num_time(KIND) : 0;   // time-kernel parameters of NL
  static constexpr int NL = num_lam(KIND);
  static_assert(!STAT || QT == 4, "stationary kinds carry the time-kernel constants in w[4]");
  static constexpr int NCS = DS * QT;         // (cos, sin) pairs per point
  static constexpr int NFB = D + 2 * NCS;     // per-point doubles: x[D], (cos,sin)[DS][QT]
  static constexpr int NF = NFB + 1;          // + alpha
  static constexpr int NG = QT + 2 * QT * DS + NL;  // kernel-gradient accumulators
  static constexpr int NV = NG + 1;           // + tr W
  static constexpr int PMAX = 2 + QT + 2 * QT * DS + NL;
  // shared memory (doubles)
  static constexpr int SM_STAGES = 0;
  static constexpr int SM_S = STAGE_ELEMS;
  static constexpr int SM_ROW = SM_S + S_ELEMS;
  static constexpr int SM_COL = SM_ROW + NF * TS;
  static constexpr int SM_PAR = SM_COL + NF * TS;
  static constexpr int PAR_THETA = 0;
  static constexpr int PAR_JAC = PAR_THETA + PMAX;
  static constexpr int PAR_W = PAR_JAC + PMAX;
  static constexpr int PAR_A = PAR_W + QT;
  static constexpr int PAR_LAM = PAR_A + QT * DS;   // wavelength-kernel constants [4]
  // the warp partials of block_reduce ([8][NV + 2]) live in the column-side field vector: every
  // reduction runs after a block barrier behind the last epilogue that read the fields.  (Kept out
  // of the parameter area so that the separable 2-D kinds fit two blocks per SM.)
  static constexpr int RED_ELEMS = 8 * (NV + 2);
  static_assert(RED_ELEMS <= NF * TS, "block_reduce scratch must fit the column field vector");
  static constexpr int PAR_FIN = PAR_LAM + 4;
  static constexpr int PAR_ZJ = (PAR_FIN + NV + 4 + 1) & ~1;   // z_j of the current block column [64], 16-B aligned
  static constexpr int PAR_ZI = PAR_ZJ + TS;          // z_i of the current tile row / scratch [64]
  static constexpr int PAR_DINV = PAR_ZI + TS;        // 1 / L_kk of the current diagonal block [64]
  static constexpr int PAR_TAB = PAR_DINV + TS;       // exp tables [EXP_TAB]
  static constexpr int PAR_RAW = PAR_TAB + EXP_TAB;        // raw / adam state / gradient (fit kernel)
  static constexpr int PAR_BAR = PAR_RAW + 4 * PMAX;  // 11 mbarriers (8 B each)
  static constexpr int PAR_END = PAR_BAR + 12;
  static constexpr int SM_TOTAL = SM_PAR + PAR_END + 8;
  static constexpr size_t SMEM_BYTES = (size_t)SM_TOTAL * sizeof(double);
  // Layout of the FUSED kernels (sm_mll_grad_kernel / sm_fit_kernel).  Kinds whose full layout does
  // not fit two blocks per SM (ARD 2-D SM-4, SM-8, ...) run LEAN when their fields fit one ring stage:
  // the per-point fields live in stage 0, fetched behind the k-loop (as lg_chol_all does), at the
  // price of the look-ahead across job boundaries in the P and G phases - two resident blocks
  // overlap more than the look-ahead did (r02z: C5 share 113.1 -> see DESIGN.md 4.1).
  static constexpr bool LEAN = (SMEM_BYTES > 113 * 1024) && (2 * NF * TS <= 2 * OPBUF);
  static constexpr int F_ROW = LEAN ? SM_STAGES : SM_ROW;
  static constexpr int F_COL = F_ROW + NF * TS;
  static constexpr int F_PAR = LEAN ? SM_ROW : SM_PAR;     // SM_ROW = first offset behind the S tile
  static constexpr size_t F_BYTES = (size_t)(F_PAR + PAR_END + 8) * sizeof(double);
};

// per-block global scratch layout (doubles)
struct Scratch {
  double* tiles;  // ntri * TT : L_ij (i>j), later X_ij^T; diagonal slots hold X_jj = L_jj^-1
  double* tilesT; // N * TT    : X_jj^T
  double* fx;     // D * npad      : centred inputs, [dd][i]
  double* fcs;    // NCS * npad * 2: (cos, sin)(2 pi mu_qd x_id), [(dd*QT+q)][i][2]
  double* alpha;  // npad
  double* rhs;    // npad  (y - mean)
  double* z;      // npad  (L^-1 rhs)
  double* dn;     // npad  (diagonal noise)
  double* fpart;  // ntri * 4 * 64 : partial products L_ij z_j per warp column (forward solve)
  double* apart;  // ntri * 4 * 64 : partial products X_ij^T z_i per warp column (alpha)
};
__host__ __device__ inline size_t scratch_elems(int n_max, int NF) {
  int N = (n_max + TS - 1) / TS;
  size_t npad = (size_t)N * TS;
  size_t ntri = (size_t)tri(N, 0);
  return ntri * TT + (size_t)N * TT + (size_t)(NF + 4) * npad + ntri * 8 * TS + 64;
}

// ------------------------------------------------------------------------------------
// the tensor-core tile engine:  acc += sum_kt  A(kt) * B(kt)^T   on 64x64 tiles
//   A(kt)[m][k], B(kt)[n][k] with k contiguous ("NT").  Every product of the algorithm is
//   brought to this form by storing the off-diagonal inverse tiles transposed.
//
// Tile image (global scratch == shared memory): two k-chunks of [64 rows][32 k] doubles,
// 16-byte groups XOR-swizzled by the row parity so that every fragment load is a
// conflict-free LDS.128:   img(r, k) below.
//
// Pipeline: a ring of NST stages (A chunk + B chunk = 32 KB each).  Thread 0 is the
// producer: before computing chunk c it waits for empty[stage of chunk c+NST-1] (all 8 warps
// released it) and issues that chunk's two bulk copies on full[stage]; every warp waits on
// full[stage], computes, and releases with one arrive per warp.  The producer runs ahead into
// the NEXT job's first chunks ("pre" of the following call) where the caller says the tiles
// are final.  Off-diagonal result tiles leave through shared memory and ONE bulk store
// (async proxy on both sides, no generic->async fence on global memory); the producer waits
// for that store before it issues anything beyond k-tile 0 of the following job.
//
// k <-> lane mapping of one 8-deep k-group: MMA step h in {0,1}, lane tq holds
// k = 8*k8 + 2*tq + h  (both operands).
// Accumulator layout acc[mi][ni][e] (lane = 4*g + tq), 8x8 MMA tiles interleaved over the
// warps so that triangular operands / outputs give every warp the same amount of work:
//   row = 8*mt + g,  mt = MT[wm][mi],  MT = {0,3,4,7} | {1,2,5,6}
//   col = 8*nt + 2*tq + e,  nt = wn (ni = 0) | 7 - wn (ni = 1)
//
// MODE0 describes the zero structure of k-tile 0 (the others are dense):
//   M_B_LE: B[n][k] = 0 for k > n   M_B_GE: B[n][k] = 0 for k < n
//   M_A_LE: A[m][k] = 0 for k > m   M_A_GE: A[m][k] = 0 for k < m
// LOWER: only MMA tiles with mt >= nt are computed (symmetric outputs).
// ------------------------------------------------------------------------------------
enum { M_FULL = 0, M_B_LE = 1, M_B_GE = 2, M_A_LE = 3, M_A_GE = 4 };

__host__ __device__ __forceinline__ int img(int r, int k) {
  return (k >> 5) * OPBUF + r * KC + ((((k & 31) >> 1) ^ ((r & 1) << 2)) << 1) + (k & 1);
}

__device__ __forceinline__ int frag_mt(int wm, int mi) {
  return 2 * mi + ((mi ^ wm) & 1);   // {0,3,4,7} | {1,2,5,6}, branch-free (rolled epilogue loops)
}
__device__ __forceinline__ int frag_nt(int wn, int ni) { return ni ? 7 - wn : wn; }
__device__ __forceinline__ int frag_row(int wm, int mi, int g) { return 8 * frag_mt(wm, mi) + g; }
__device__ __forceinline__ int frag_col(int wn, int ni, int tq, int e) {
  return 8 * frag_nt(wn, ni) + 2 * tq + e;
}

// Fragment loads of k-group k8l+1 are issued (and pinned in program order by an empty
// volatile asm) before the MMAs of k-group k8l; the two MMA steps of one accumulator are
// separated by the 7 other accumulators so that no DMMA waits on the one issued just before.
__device__ __forceinline__ void load_frags(double2 (&fa)[4], double2 (&fb)[2],
                                           const double* __restrict__ sA,
                                           const double* __restrict__ sB, int k8l, int wm, int wn,
                                           int g, int tq) {
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int r = frag_row(wm, mi, g);
    fa[mi] = *reinterpret_cast<const double2*>(sA + r * KC + (((k8l * 4 + tq) ^ ((r & 1) << 2)) << 1));
  }
#pragma unroll
  for (int ni = 0; ni < 2; ++ni) {
    const int r = 8 * frag_nt(wn, ni) + g;
    fb[ni] = *reinterpret_cast<const double2*>(sB + r * KC + (((k8l * 4 + tq) ^ ((r & 1) << 2)) << 1));
  }
  asm volatile("" : "+d"(fa[0].x), "+d"(fa[0].y), "+d"(fa[1].x), "+d"(fa[1].y), "+d"(fa[2].x),
                    "+d"(fa[2].y), "+d"(fa[3].x), "+d"(fa[3].y), "+d"(fb[0].x), "+d"(fb[0].y),
                    "+d"(fb[1].x), "+d"(fb[1].y));
}

template <int MODE, bool LOWER>
__device__ __forceinline__ void compute_chunk(double (&acc)[4][2][2], const double* __restrict__ sA,
                                              const double* __restrict__ sB, int k8base, int wm,
                                              int wn, int g, int tq) {
  double2 fa[2][4], fb[2][2];
  load_frags(fa[0], fb[0], sA, sB, 0, wm, wn, g, tq);
#pragma unroll
  for (int k8l = 0; k8l < KC / 8; ++k8l) {
    const int k8g = k8base + k8l;
    const int cur = k8l & 1;
    if (k8l + 1 < KC / 8) load_frags(fa[cur ^ 1], fb[cur ^ 1], sA, sB, k8l + 1, wm, wn, g, tq);
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 2; ++ni) {
          const int mt = frag_mt(wm, mi), nt = frag_nt(wn, ni);
          bool on = true;
          if (LOWER) on = on && (mt >= nt);
          if (MODE == M_B_LE) on = on && (k8g <= nt);
          if (MODE == M_B_GE) on = on && (k8g >= nt);
          if (MODE == M_A_LE) on = on && (k8g <= mt);
          if (MODE == M_A_GE) on = on && (k8g >= mt);
          if (on)
            mma_f64(acc[mi][ni], h ? fa[cur][mi].y : fa[cur][mi].x,
                    h ? fb[cur][ni].y : fb[cur][ni].x);
        }
  }
}

// ring of NST stages; `gq` counts the chunks consumed on this ring since the barriers were
// initialised (uniform over the block), which fixes the stage and the mbarrier phase.
struct Ring {
  unsigned full, empty;  // shared addresses of full[NST] / empty[NST]
  double* stages;        // stage s at stages + s * 2 * OPBUF
  int gq;
};
constexpr unsigned CHUNK_BYTES = OPBUF * sizeof(double);

// acc += sum over this job's nk k-tiles.  `pre` chunks of the job are already in flight
// (issued by the previous call); the first chunks of the next job (next_nk k-tiles, 0 = no
// look-ahead) are issued from here.  Returns the number of next-job chunks issued.
// `ready(kt)` is called by the producer thread before it issues the loads of k-tile kt of THIS
// job (a hook for operands another block of the same launch is still producing).
template <int MODE0, bool LOWER, int NST, typename FA, typename FB, typename FNA, typename FNB,
          typename FX, typename FR>
__device__ __forceinline__ int gemm_stream_r(double (&acc)[4][2][2], Ring& rg, int nk, FA tileA,
                                             FB tileB, int pre, int next_nk, FNA nextA, FNB nextB,
                                             FX extra_prefetch, FR ready) {
  constexpr int LA = NST - 1;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3;
  const int wm = warp >> 2, wn = warp & 3;
  const int n = 2 * nk, nn = 2 * next_nk;

  auto issue = [&](int t) {  // chunk t counted from this job's first chunk; thread 0 only
    const double *ga, *gb;
    if (t < n) {
      if (!(t & 1)) ready(t >> 1);
      ga = tileA(t >> 1) + (t & 1) * OPBUF;
      gb = tileB(t >> 1) + (t & 1) * OPBUF;
    } else {
      const int u = t - n;
      if (u >= nn) return;
      ga = nextA(u >> 1) + (u & 1) * OPBUF;
      gb = nextB(u >> 1) + (u & 1) * OPBUF;
    }
    const int q = rg.gq + t, s = q % NST, use = q / NST;
    if (use > 0) mbar_wait(rg.empty + 8 * s, (use - 1) & 1);
    const unsigned bar = rg.full + 8 * s;
    const unsigned dst = smem_u32(rg.stages + s * 2 * OPBUF);
    mbar_expect_tx(bar, 2 * CHUNK_BYTES);
    bulk_g2s(dst, ga, CHUNK_BYTES, bar);
    bulk_g2s(dst + CHUNK_BYTES, gb, CHUNK_BYTES, bar);
  };

  __syncthreads();  // job boundary: users of the stages / rowv / colv are done
  extra_prefetch();
  cp_async_commit();
  if (tid == 0) {
    // the previous job's bulk store has left its staging buffer; a cold start (nothing in
    // flight) also waits for every earlier store to be complete
    if (pre == 0) bulk_wait_all(); else bulk_wait_read();
    for (int t = pre; t < LA; ++t) issue(t);
  }
  for (int c = 0; c < n; ++c) {
    if (tid == 0) {
      // chunks >= 2 (k-tile 1 onwards) may read the tile the previous job stored
      if (c + LA == 2 || (c == 0 && LA > 2)) bulk_wait_all();
      issue(c + LA);
    }
    const int q = rg.gq + c, s = q % NST;
    mbar_wait(rg.full + 8 * s, (q / NST) & 1);
    const double* sA = rg.stages + s * 2 * OPBUF;
    const double* sB = sA + OPBUF;
    if (MODE0 != M_FULL && c < 2)
      compute_chunk<MODE0, LOWER>(acc, sA, sB, c * (KC / 8), wm, wn, g, tq);
    else
      compute_chunk<M_FULL, LOWER>(acc, sA, sB, 0, wm, wn, g, tq);
    __syncwarp();
    if (lane == 0) mbar_arrive(rg.empty + 8 * s);
  }
  rg.gq += n;
  cp_async_wait<0>();
  return nn < LA ? nn : LA;
}

template <int MODE0, bool LOWER, int NST, typename FA, typename FB, typename FNA, typename FNB,
          typename FX>
__device__ __forceinline__ int gemm_stream(double (&acc)[4][2][2], Ring& rg, int nk, FA tileA,
                                           FB tileB, int pre, int next_nk, FNA nextA, FNB nextB,
                                           FX extra_prefetch) {
  return gemm_stream_r<MODE0, LOWER, NST>(acc, rg, nk, tileA, tileB, pre, next_nk, nextA, nextB,
                                          extra_prefetch, [](int) {});
}

// Late look-ahead (LEAN layout): thread 0 issues the FIRST chunk of the next job at the ring's current
// position - always stage 0, every job consumes an even number of chunks - once stage 0 is free again;
// the following gemm_stream call is told `pre = 1`.
__device__ __forceinline__ void ring_issue_first(const Ring& rg, const double* ga, const double* gb) {
  const int q = rg.gq, s = q % 2, use = q / 2;
  if (use > 0) mbar_wait(rg.empty + 8 * s, (use - 1) & 1);
  const unsigned bar = rg.full + 8 * s;
  const unsigned dst = smem_u32(rg.stages + s * 2 * OPBUF);
  fence_proxy_async_smem();   // stage 0 was last written by cp.async (the per-point fields)
  mbar_expect_tx(bar, 2 * CHUNK_BYTES);
  bulk_g2s(dst, ga, CHUNK_BYTES, bar);
  bulk_g2s(dst + CHUNK_BYTES, gb, CHUNK_BYTES, bar);
}

__device__ __forceinline__ void zero_acc(double (&acc)[4][2][2]) {
#pragma unroll
  for (int mi = 0; mi < 4; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
}

// accumulator -> 64x64 tile image (global scratch or a shared-memory stage)
__device__ __forceinline__ void store_acc_tile(const double (&acc)[4][2][2], double* tile,
                                               double sign) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int r = frag_row(wm, mi, g);
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) {
      const int c = frag_col(wn, ni, tq, 0);
      *reinterpret_cast<double2*>(tile + img(r, c)) =
          make_double2(sign * acc[mi][ni][0], sign * acc[mi][ni][1]);
    }
  }
}

// accumulator -> global tile through a shared staging buffer (every warp must be done reading
// `stage`): image written by all threads, one bulk store issued by thread 0.
__device__ __forceinline__ void store_tile_bulk(const double (&acc)[4][2][2], double* stage,
                                                double* gtile, double sign) {
  __syncthreads();
  store_acc_tile(acc, stage, sign);
  fence_proxy_async_smem();
  __syncthreads();
  if (threadIdx.x == 0) {
    bulk_s2g(gtile, smem_u32(stage), 2 * OPBUF * sizeof(double));
    bulk_commit();
  }
}

// ------------------------------------------------------------------------------------
// kernel entry K(x_i, x_j) and its hyper-parameter derivatives (SURVEY.md A.3).
// Per-point data of the 64 rows / cols of a tile in shared memory:
//   xs[dd*64 + r] centred inputs;  cs[((dd*QT+q)*64 + r)] = (cos, sin)(2 pi mu_qd x_rd).
// cos(2 pi mu tau) = c_i c_j + s_i s_j,  sin(2 pi mu tau) = s_i c_j - c_i s_j.
// ------------------------------------------------------------------------------------
// wavelength factor f(tau) of the separable kinds and the two derivative carriers
//   lam = { outputscale | constant, c1, alpha, lengthscale }
//   RBF:     c1 = 1/(2 l^2)        f = exp(-c1 tau^2)          df/dl = f tau^2 / l^3
//   Matern:  c1 = sqrt(3)/l        f = (1+u) e^-u, u = c1|tau|  df/dl = u^2 e^-u / l
//   RQ:      c1 = 1/(2 alpha l^2)  f = (1+u)^-alpha, u = c1 tau^2
//            df/dl = 2 alpha f u / ((1+u) l),  df/dalpha = f (u/(1+u) - log1p(u))
// gl / ga_ return df/dl and df/dalpha WITHOUT their constant factors (applied once per light
// curve in the final assembly).
template <int KIND>
__device__ __forceinline__ double lam_factor(double tl, const double (&lam)[4],
                                             const double* __restrict__ tab, double& gl,
                                             double& ga_) {
  gl = 0.0;
  ga_ = 0.0;
  if (KIND == PGM_KIND_SEP_RBF) {
    const double t2 = tl * tl;
    const double f = exp_neg(-lam[1] * t2, tab);
    gl = f * t2;
    return f;
  } else if (KIND == PGM_KIND_SEP_MATERN15) {
    const double u = lam[1] * fabs(tl);
    const double e = exp_neg(-u, tab);
    gl = u * u * e;
    return (1.0 + u) * e;
  } else if (KIND == PGM_KIND_SEP_RQ) {
    const double u = lam[1] * tl * tl;
    const double l1 = log1p(u);
    const double f = exp(-lam[2] * l1);
    const double uu = u / (1.0 + u);
    gl = f * uu;
    ga_ = f * (uu - l1);
    return f;
  } else if (KIND == PGM_ATOM_M12) {
    const double u = lam[1] * fabs(tl);
    const double e = exp_neg(-u, tab);
    gl = u * e;                       // df/dl = u e^-u / l
    return e;
  } else if (KIND == PGM_ATOM_M25) {
    const double u = lam[1] * fabs(tl);
    const double e = exp_neg(-u, tab);
    const double u23 = u * u * (1.0 / 3.0);
    gl = u23 * (1.0 + u) * e;         // df/dl = (u^2 / 3)(1 + u) e^-u / l
    return (1.0 + u + u23) * e;
  }
  return 1.0;
}

// quasi-periodic time factor (GPyTorch PeriodicKernel x RBFKernel):
//   f = exp(-2 sin^2(pi tau / p) / lambda) * exp(-tau^2 / (2 l_r^2))
// w = {outputscale, lambda, p, l_r}, a = {2 / lambda, 1 / p, 1 / (2 l_r^2)}; g[] returns the
// derivative carriers f s^2, f sin(2 theta) tau, f tau^2 (constants applied at the end).
__device__ __forceinline__ double qp_factor(double tau, const double (&a)[4],
                                            const double* __restrict__ tab, double (&g)[3]) {
  double sn, cs;
  sincospi(tau * a[1], &sn, &cs);
  const double s2 = sn * sn, t2 = tau * tau;
  const double f = exp_neg(-(a[0] * s2 + a[2] * t2), tab);
  g[0] = f * s2;
  g[1] = f * (2.0 * sn * cs) * tau;
  g[2] = f * t2;
  return f;
}

template <int KIND, int QT, int D>
__device__ __forceinline__ double k_entry(const double* __restrict__ rowv,
                                          const double* __restrict__ colv, int r, int c,
                                          const double (&w)[QT],
                                          const double (&a)[QT * Cfg<KIND, QT, D>::DS],
                                          const double (&lam)[4],
                                          const double* __restrict__ tab) {
  constexpr int DS = Cfg<KIND, QT, D>::DS;
  if constexpr (Cfg<KIND, QT, D>::STAT) {
    // K = os_t f_T(tau_t) [x os_w f_W(tau_lambda)]; time-kernel constants travel in w[4]
    double gl, ga_, k;
    if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP) {
      double g3[3];
      k = w[0] * qp_factor(rowv[r] - colv[c], a, tab, g3);
    } else if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP_RBF) {
      // additive: the stochastic ScaleKernel(RBF) term travels in lam[] (no wavelength kernel)
      double g3[3];
      const double tt = rowv[r] - colv[c];
      k = w[0] * qp_factor(tt, a, tab, g3)
          + lam[0] * lam_factor<PGM_KIND_SEP_RBF>(tt, lam, tab, gl, ga_);
    } else {
      k = w[0] * lam_factor<stat_time_atom(KIND)>(rowv[r] - colv[c], w, tab, gl, ga_);
    }
    if constexpr (stat_wave_atom(KIND) != 0)
      k *= lam[0] * lam_factor<stat_wave_atom(KIND)>(rowv[TS + r] - colv[TS + c], lam, tab, gl, ga_);
    return k;
  }
  const double2* rcs = reinterpret_cast<const double2*>(rowv + D * TS);
  const double2* ccs = reinterpret_cast<const double2*>(colv + D * TS);
  double tau2[DS];
#pragma unroll
  for (int dd = 0; dd < DS; ++dd) {
    const double tau = rowv[dd * TS + r] - colv[dd * TS + c];
    tau2[dd] = tau * tau;
  }
  if (KIND == PGM_KIND_SM_ARD_SUMPROD) {
    double k = 0.0;
#pragma unroll
    for (int q = 0; q < QT; ++q) {
      double pr = w[q];
#pragma unroll
      for (int dd = 0; dd < DS; ++dd) {
        const double2 ri = rcs[(dd * QT + q) * TS + r], cj = ccs[(dd * QT + q) * TS + c];
        pr *= exp_neg(-a[q * DS + dd] * tau2[dd], tab) * (ri.x * cj.x + ri.y * cj.y);
      }
      k += pr;
    }
    return k;
  } else {
    double k = 1.0;
#pragma unroll
    for (int dd = 0; dd < DS; ++dd) {
      double s = 0.0;
#pragma unroll
      for (int q = 0; q < QT; ++q) {
        const double2 ri = rcs[(dd * QT + q) * TS + r], cj = ccs[(dd * QT + q) * TS + c];
        s += (w[q] * exp_neg(-a[q * DS + dd] * tau2[dd], tab)) * (ri.x * cj.x + ri.y * cj.y);
      }
      k *= s;
    }
    if (Cfg<KIND, QT, D>::SEP) {
      double gl, ga_;
      k *= lam[0] * lam_factor<KIND>(rowv[TS + r] - colv[TS + c], lam, tab, gl, ga_);
    }
    return k;
  }
}

// accumulate  wgt * dK/dtheta  into ga[NG] = { gw[q], gmu[q*DS+dd], gsg[q*DS+dd], glam[NL] }
// (raw sums; the constant factors -2 pi w_q, -4 pi^2 sigma w_q and those of the wavelength
// kernel are applied once at the end).
template <int KIND, int QT, int D>
__device__ __forceinline__ void k_grad_entry(const double* __restrict__ rowv,
                                             const double* __restrict__ colv, int r, int c,
                                             const double (&w)[QT],
                                             const double (&a)[QT * Cfg<KIND, QT, D>::DS],
                                             const double (&lam)[4],
                                             const double* __restrict__ tab, double wgt,
                                             double (&ga)[Cfg<KIND, QT, D>::NG]) {
  using C = Cfg<KIND, QT, D>;
  constexpr int DS = C::DS;
  if constexpr (C::STAT) {
    // raw carriers in the slots behind the (unused) mixture accumulators; constant factors
    // (outputscales, d c1 / d lengthscale) are applied once per light curve at the end
    constexpr int G0 = QT + 2 * QT * DS;
    constexpr int GW = G0 + C::NLT;        // first wavelength-kernel slot
    constexpr bool QP = stat_time_atom(KIND) == PGM_ATOM_QP ||
                        stat_time_atom(KIND) == PGM_ATOM_QP_RBF;
    double glt = 0.0, gat = 0.0, glw = 0.0, gaw = 0.0, g3[3] = {0.0, 0.0, 0.0}, ft;
    if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP_RBF) {
      // K = os qp + os2 rbf: six independent slots, nothing else multiplies them
      const double tt = rowv[r] - colv[c];
      ft = qp_factor(tt, a, tab, g3);
      const double fr = lam_factor<PGM_KIND_SEP_RBF>(tt, lam, tab, glt, gat);
      ga[G0] += wgt * ft;
      ga[G0 + 1] += wgt * g3[0];
      ga[G0 + 2] += wgt * g3[1];
      ga[G0 + 3] += wgt * g3[2];
      ga[G0 + 4] += wgt * fr;       // d / d outputscale_2
      ga[G0 + 5] += wgt * glt;      // d / d lengthscale_2  (x os_2 / l^3)
      return;
    }
    if constexpr (QP) ft = qp_factor(rowv[r] - colv[c], a, tab, g3);
    else ft = lam_factor<stat_time_atom(KIND)>(rowv[r] - colv[c], w, tab, glt, gat);
    double fw = 1.0, kw = 1.0;
    if constexpr (stat_wave_atom(KIND) != 0) {
      fw = lam_factor<stat_wave_atom(KIND)>(rowv[TS + r] - colv[TS + c], lam, tab, glw, gaw);
      kw = lam[0] * fw;
    }
    const double wk = wgt * kw;
    ga[G0] += wk * ft;            // d / d outputscale_t
    if constexpr (QP) {
      ga[G0 + 1] += wk * g3[0];   // d / d lambda   (x os_t x const)
      ga[G0 + 2] += wk * g3[1];   // d / d period
      ga[G0 + 3] += wk * g3[2];   // d / d l_rbf
    } else {
      ga[G0 + 1] += wk * glt;     // d / d lengthscale_t   (x os_t x const)
    }
    if constexpr (stat_wave_atom(KIND) != 0) {
      const double wkt = wgt * (w[0] * ft);
      ga[GW] += wkt * fw;                                          // d / d outputscale_w | constant
      if constexpr (C::NL - C::NLT >= 2) ga[GW + 1] += wkt * glw;  // d / d lengthscale_w
      if constexpr (C::NL - C::NLT >= 3) ga[GW + 2] += wkt * gaw;  // d / d alpha_w
    }
    return;
  }
  const double2* rcs = reinterpret_cast<const double2*>(rowv + D * TS);
  const double2* ccs = reinterpret_cast<const double2*>(colv + D * TS);
  double tau[DS], EC[DS][QT], ES[DS][QT], Ssum[DS];
#pragma unroll
  for (int dd = 0; dd < DS; ++dd) {
    tau[dd] = rowv[dd * TS + r] - colv[dd * TS + c];
    const double t2 = tau[dd] * tau[dd];
    Ssum[dd] = 0.0;
#pragma unroll
    for (int q = 0; q < QT; ++q) {
      const double2 ri = rcs[(dd * QT + q) * TS + r], cj = ccs[(dd * QT + q) * TS + c];
      const double E = exp_neg(-a[q * DS + dd] * t2, tab);
      EC[dd][q] = E * (ri.x * cj.x + ri.y * cj.y);
      ES[dd][q] = E * (ri.y * cj.x - ri.x * cj.y);
      Ssum[dd] += w[q] * EC[dd][q];
    }
  }
  if (C::SEP) {
    // K = kt * kl,  kt = Ssum[0],  kl = lam0 * f
    double gl, ga_;
    const double f = lam_factor<KIND>(rowv[TS + r] - colv[TS + c], lam, tab, gl, ga_);
    const double wk = wgt * (lam[0] * f);         // weight seen by the time-kernel parameters
    const double wt = wk * tau[0], wt2 = wt * tau[0];
#pragma unroll
    for (int q = 0; q < QT; ++q) {
      ga[q] += wk * EC[0][q];
      ga[QT + q] += wt * ES[0][q];
      ga[2 * QT + q] += wt2 * EC[0][q];
    }
    const double wkt = wgt * Ssum[0];
    ga[3 * QT] += wkt * f;                          // d/d outputscale  (or d/d constant)
    if (C::NL >= 2) ga[3 * QT + 1] += wkt * gl;     // d/d lengthscale  (x const at the end)
    if (C::NL >= 3) ga[3 * QT + 2] += wkt * ga_;    // d/d alpha
    return;
  }
#pragma unroll
  for (int dd = 0; dd < DS; ++dd) {
    const double wt = wgt * tau[dd];
    const double wt2 = wt * tau[dd];
#pragma unroll
    for (int q = 0; q < QT; ++q) {
      double R = 1.0;  // product of the other dimensions' factor
      if (DS == 2) R = (KIND == PGM_KIND_SM_ARD_SUMPROD) ? EC[1 - dd][q] : Ssum[1 - dd];
      const double ecr = (DS == 2) ? EC[dd][q] * R : EC[dd][q];
      if (KIND == PGM_KIND_SM_ARD_SUMPROD) {
        if (dd == 0) ga[q] += wgt * ecr;
      } else {
        ga[q] += wgt * ecr;
      }
      ga[QT + q * DS + dd] += wt * ((DS == 2) ? ES[dd][q] * R : ES[dd][q]);
      ga[QT + QT * DS + q * DS + dd] += wt2 * ecr;
    }
  }
}

// ------------------------------------------------------------------------------------
// 64x64 diagonal block:  S (lower) -> L in place,  X = L^-1 into S2,  dinv[k] = 1/L_kk.
// Panel width 8.  Warp 0 factors a panel in registers (shuffles); the trailing update and the
// next 8 rows of L^-1 (block forward substitution) run on the tensor cores (DMMA 8x8x4).
// The serial chain is what bounds this routine, so
//  * inside a panel the columns stay UNSCALED (v_ik) and the updates use v_ik v_ck / d_k with a
//    short reciprocal (MUFU.RCP64H + 2 Newton steps); the 8 rsqrt that turn v into L are
//    independent of each other and happen after the chain;
//  * look-ahead: after panel p only tile column p+1 of the trailing matrix is updated before
//    warp 0 starts panel p+1; the other warps finish the trailing update and the inverse rows
//    of panel p meanwhile (2 block barriers per panel).
// ------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp_pos(double d) {   // 1/d for normal d > 0
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  double e = fma(-d, y, 1.0);
  y = fma(y, e, y);
  e = fma(-d, y, 1.0);
  return fma(y, e, y);
}

// 1/d for normal d > 0: MUFU.RCP64H seed (|e| < 2^-20) + one cubic step e -> e^3 (3 dependent FMAs
// instead of the 4 of two Newton steps; relative error < 2^-60 before the final rounding)
__device__ __forceinline__ double rcp_pos3(double d) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double e = fma(-d, y, 1.0);
  const double t = fma(e, e, e);
  return fma(y, t, y);
}

// 1/sqrt(d) for normal d > 0: MUFU.RSQ64H seed + one cubic step (y (1 + e/2 + 3 e^2/8), e = 1 - d y^2):
// 1 MUFU + 5 dependent-free-ish FMAs instead of the ~18 instructions of rsqrt() / sqrt()
__device__ __forceinline__ double rsqrt_pos3(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double t = d * y;
  const double e = fma(-t, y, 1.0);
  const double q = fma(0.375, e, 0.5) * e;
  return fma(y, q, y);
}

// warp 0: factor columns c0..c0+7 (rows c0..63; lane holds rows c0+lane and c0+lane+32).
// The serial chain (pivot -> reciprocal -> update of the next pivot) runs on the 8x8 pivot block,
// which EVERY lane eliminates redundantly in its own registers (broadcast loads, no shuffle on the
// chain); the lanes then eliminate their own two rows against the finished multipliers
// u_ck = v_ck / d_k - 28 FMAs per row whose only chain is one FMA per column.  Rows are loaded and
// stored as 16-byte vectors (LD_S = 68: 2-way instead of 8-way bank conflicts).
__device__ __forceinline__ void potrf_panel8(double* __restrict__ S, double* __restrict__ dinv,
                                             int c0, int lane, int* fail) {
  const int r0 = c0 + lane, r1 = c0 + lane + 32;
  double P[8][8];      // lower triangle of the pivot block: v_ck -> u_ck; diagonal: d_k
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j2 = 0; j2 <= i / 2; ++j2) {
      const double2 v = *reinterpret_cast<const double2*>(S + (c0 + i) * LD_S + c0 + 2 * j2);
      P[i][2 * j2] = v.x;
      P[i][2 * j2 + 1] = v.y;          // (i, i + 1) for even i: unused upper entry
    }
  double a0[8], a1[8];
#pragma unroll
  for (int k2 = 0; k2 < 4; ++k2) {
    const double2 v0 = (r0 < TS) ? *reinterpret_cast<const double2*>(S + r0 * LD_S + c0 + 2 * k2)
                                 : make_double2(0.0, 0.0);
    const double2 v1 = (r1 < TS) ? *reinterpret_cast<const double2*>(S + r1 * LD_S + c0 + 2 * k2)
                                 : make_double2(0.0, 0.0);
    a0[2 * k2] = v0.x; a0[2 * k2 + 1] = v0.y;
    a1[2 * k2] = v1.x; a1[2 * k2 + 1] = v1.y;
  }
  bool bad = false, isnan_ = false;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double dpiv = P[k][k];
    if (!(dpiv > 0.0)) { bad = true; if (dpiv != dpiv) isnan_ = true; }
    dpiv = bad ? 1.0 : dpiv;
    P[k][k] = dpiv;
    const double rd = rcp_pos3(dpiv);
#pragma unroll
    for (int c = k + 1; c < 8; ++c) {
      const double v = P[c][k];
      const double u = v * rd;                  // v_ck / d_k
#pragma unroll
      for (int c2 = k + 1; c2 < c; ++c2) P[c][c2] = fma(-P[c2][k], v, P[c][c2]);   // P[c2][k] is u_c2k
      P[c][c] = fma(-v, u, P[c][c]);
      P[c][k] = u;
    }
  }
  // own rows: v_rc = a_rc - sum_{k<c} v_rk u_ck  (rows of the pivot block reproduce its elimination)
#pragma unroll
  for (int c = 1; c < 8; ++c) {
    double s0 = a0[c], s1 = a1[c];
#pragma unroll
    for (int k = 0; k < c; ++k) {
      s0 = fma(-a0[k], P[c][k], s0);
      s1 = fma(-a1[k], P[c][k], s1);
    }
    a0[c] = s0;
    a1[c] = s1;
  }
  double myrs = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const double rs = rsqrt_pos3(P[k][k]);      // 1 / L_kk
    if (lane == k) myrs = rs;
    a0[k] *= rs;
    a1[k] *= rs;
  }
  __syncwarp();   // every lane has read the pivot block (top) before lanes 0..7 overwrite its rows
#pragma unroll
  for (int k2 = 0; k2 < 4; ++k2) {
    if (r0 < TS)
      *reinterpret_cast<double2*>(S + r0 * LD_S + c0 + 2 * k2) = make_double2(a0[2 * k2], a0[2 * k2 + 1]);
    if (r1 < TS)
      *reinterpret_cast<double2*>(S + r1 * LD_S + c0 + 2 * k2) = make_double2(a1[2 * k2], a1[2 * k2 + 1]);
  }
  if (lane < 8) dinv[c0 + lane] = myrs;
  if (lane == 0 && bad) atomicOr(fail, isnan_ ? 2 : 1);
}

// C(ti,tj) -= P_ti P_tj^T on one 8x8 MMA tile, P = S[:, c0:c0+8]
__device__ __forceinline__ void potrf_syrk_tile(double* __restrict__ S, int c0, int ti, int tj,
                                                int g, int tq) {
  double2* cp = reinterpret_cast<double2*>(S + (8 * ti + g) * LD_S + 8 * tj + 2 * tq);
  const double2 cv = *cp;
  double c2[2] = {cv.x, cv.y};
#pragma unroll
  for (int s = 0; s < 2; ++s)
    mma_f64(c2, -S[(8 * ti + g) * LD_S + c0 + 4 * s + tq], S[(8 * tj + g) * LD_S + c0 + 4 * s + tq]);
  *cp = make_double2(c2[0], c2[1]);
}

__device__ __forceinline__ void potrf_inv_64(double* __restrict__ S, double* __restrict__ S2,
                                             double* __restrict__ dinv, int* fail) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3;
  if (warp == 0) potrf_panel8(S, dinv, 0, lane, fail);
  for (int p = 0; p < 8; ++p) {
    const int c0 = p * 8;
    __syncthreads();   // panel p is factored
    // step 1: tile column p+1 of the trailing matrix (what the next panel needs)
    if (p < 7 && warp < 7 - p) potrf_syrk_tile(S, c0, p + 1 + warp, p + 1, g, tq);
    __syncthreads();
    if (p < 7 && warp == 0) {
      potrf_panel8(S, dinv, c0 + 8, lane, fail);
    } else {
      const int nw = (p < 7) ? 7 : 8, w = (p < 7) ? warp - 1 : warp;
      // step 2a: the rest of the trailing update, tiles (ti >= tj >= p+2)
      const int m8 = 6 - p;
      const int cnt = (m8 > 0) ? m8 * (m8 + 1) / 2 : 0;
      for (int t = w; t < cnt; t += nw) {
        int a_ = 0;
        while ((a_ + 1) * (a_ + 2) / 2 <= t) ++a_;
        const int b_ = t - a_ * (a_ + 1) / 2;
        potrf_syrk_tile(S, c0, p + 2 + a_, p + 2 + b_, g, tq);
      }
      // step 2b: rows c0..c0+7 of X.  T = I - L[c0.., :c0] X[:c0, :] per column tile nt <= p,
      // then the 8x8 triangular solve of its 8 columns (lanes 0..7 of the same warp)
      for (int nt = w; nt <= p; nt += nw) {
        double c2[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) c2[e] = (c0 + g == 8 * nt + 2 * tq + e) ? 1.0 : 0.0;
        for (int kt = nt; kt < p; ++kt) {
#pragma unroll
          for (int s = 0; s < 2; ++s)
            mma_f64(c2, -S[(c0 + g) * LD_S + 8 * kt + 4 * s + tq],
                    S2[(8 * kt + 4 * s + tq) * LD_S + 8 * nt + g]);
        }
        *reinterpret_cast<double2*>(S2 + (c0 + g) * LD_S + 8 * nt + 2 * tq) = make_double2(c2[0], c2[1]);
        __syncwarp();
        if (lane < 8) {
          const int c = 8 * nt + lane;
          double v[8];
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) v[rr] = S2[(c0 + rr) * LD_S + c];
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            double sacc = v[rr];
#pragma unroll
            for (int kk = 0; kk < rr; ++kk) sacc -= S[(c0 + rr) * LD_S + c0 + kk] * v[kk];
            v[rr] = sacc * dinv[c0 + rr];
          }
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) S2[(c0 + rr) * LD_S + c] = v[rr];
        }
        __syncwarp();
      }
    }
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------
// arguments
// ------------------------------------------------------------------------------------
struct EvalArgs {
  const double* x;
  const int32_t* n_valid;
  const double* y;
  const double* fixed_noise;
  const double* raw;
  const int32_t* con_kind;
  const double* con_lb;
  const double* con_ub;
  int B, n_max, Q, flags;
  double* mll;
  double* grad;
  int32_t* info;
  double* ws;
  size_t ws_per_block;  // elements
  double* alpha_out;    // [B, n_max] or null: alpha = K~^-1 (y - mean)  (d MLL / d y = -alpha / n)
  int* sched;           // [PGM_SCHED_INTS] zeroed before the launch, or null: light-curve tickets
  int sms;              // SMs of the device (last-wave rule of next_lightcurve)
};

// Light curves are handed out by a ticket counter instead of a fixed stride, with one rule for the
// LAST wave.  The hardware fills every SM with both of its resident blocks before moving on, so with
// a fixed stride the left-over light curves of the last wave land two to an SM on the first SMs
// while the others idle (B = 444 on 148 SMs took the time of 592).  Here every block learns which
// of its SM's two slots it holds (atomic counter per %smid), and once no more than `sms` light
// curves are left only the slot-0 blocks - one per SM - take them.  The tickets make the
// assignment correct whatever the residency; the rule only balances.
constexpr int PGM_SCHED_INTS = 1024;     // [0] next ticket, [8 + smid] blocks seen on that SM
struct LcSched {
  int slot;
};
__device__ __forceinline__ LcSched sched_init(const EvalArgs& A, int* s_bcast) {
  LcSched sc{0};
  if (!A.sched) return sc;
  if (threadIdx.x == 0) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    *s_bcast = atomicAdd(A.sched + 8 + (smid % (PGM_SCHED_INTS - 8)), 1) & 1;
  }
  __syncthreads();
  sc.slot = *s_bcast;
  __syncthreads();
  return sc;
}
// next light curve of this block (first = true: its first one), or -1
__device__ __forceinline__ int next_lightcurve(const EvalArgs& A, const LcSched& sc, int prev,
                                               int* s_bcast) {
  if (!A.sched) {
    const int b = prev < 0 ? (int)blockIdx.x : prev + (int)gridDim.x;
    return b < A.B ? b : -1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int b = -1;
    const bool defer = sc.slot == 1 && prev >= 0 &&
                       A.B - atomicAdd(A.sched, 0) <= A.sms;   // leave the last ones to slot 0
    if (!defer) {
      b = atomicAdd(A.sched, 1);
      if (b >= A.B) b = -1;
    }
    *s_bcast = b;
  }
  __syncthreads();
  return *s_bcast;
}

struct FitArgs {
  EvalArgs e;
  double* raw_io;
  int optim_kind;
  double lr, beta1, beta2, eps, weight_decay, stop;
  int maxiter, miniter, stopavg;
  double* loss_hist;
  double* raw_hist;
  int32_t* n_iter;
};

// torch.nn.functional.softplus (beta 1, threshold 20), the transform of GPyTorch's Positive /
// GreaterThan: x itself above the threshold, where its derivative is exactly 1
__device__ __forceinline__ double softplus_d(double x) {
  return x > 20.0 ? x : log1p(exp(x));
}
__device__ __forceinline__ double softplus_grad_d(double x) {
  return x > 20.0 ? 1.0 : 1.0 / (1.0 + exp(-x));
}
__device__ __forceinline__ double sigmoid_d(double x) { return 1.0 / (1.0 + exp(-x)); }

template <int NVAL>
__device__ __forceinline__ void block_reduce(double (&v)[NVAL], double* red, double* fin) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int i = 0; i < NVAL; ++i) {
    double s = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += shfl_xor_d(s, o);
    if (lane == 0) red[warp * NVAL + i] = s;
  }
  __syncthreads();
  if (tid < NVAL) {
    double s = 0.0;
#pragma unroll
    for (int w8 = 0; w8 < NTHREADS / 32; ++w8) s += red[w8 * NVAL + tid];
    fin[tid] = s;
  }
  __syncthreads();
}

// packed raw-parameter layout:  [ mean | w[Q] | mu[Q*DS] | sigma[Q*DS] | (noise) | lam[NL] ]
// (mean at slot 0, w at slot 1): the first slot of each later group and the slot count P
struct ParamLayout {
  int o_mu, o_sigma, o_noise, o_lam, P;
};
__host__ __device__ constexpr ParamLayout param_layout(int kind, int d, int Q, bool learn_noise) {
  const int ds = mix_dims(kind, d), o_noise = 1 + Q + 2 * Q * ds;
  const int o_lam = o_noise + (learn_noise ? 1 : 0);
  return ParamLayout{1 + Q, 1 + Q + Q * ds, o_noise, o_lam, o_lam + num_lam(kind)};
}

// constraint of one slot (gpytorch.constraints): *th = theta(raw) and, if jc is given,
// *jc = d theta / d raw
__device__ __forceinline__ void constrain(int kd, double raw, double lb, double ub, double* th,
                                          double* jc) {
  double t = raw, j = 1.0;
  if (kd == PGM_CON_SOFTPLUS) {
    t = softplus_d(raw) + lb;
    j = softplus_grad_d(raw);
  } else if (kd == PGM_CON_INTERVAL) {
    const double s = sigmoid_d(raw);
    t = lb + (ub - lb) * s;
    j = (ub - lb) * s * (1.0 - s);
  } else if (kd == PGM_CON_RSOFTPLUS) {
    const double v = softplus_d(raw) + lb;
    t = ub / v;
    j = -ub * softplus_grad_d(raw) / (v * v);
  }
  *th = t;
  if (jc) *jc = j;
}
// threads 0..P-1: slot tid of light curve b's raw parameters -> theta[tid] (and jac[tid] unless
// jac is null), with the bounds of the light curve under PGM_FLAG_BOUNDS_PER_LC
template <class Args>
__device__ __forceinline__ void load_theta(const Args& A, int b, int P, const double* raw,
                                           double* theta, double* jac) {
  const int tid = threadIdx.x;
  if (tid < P) {
    const size_t bo = (A.flags & PGM_FLAG_BOUNDS_PER_LC) ? (size_t)b * P : 0;
    double th, jc;   // locals: passing theta + tid, jac + tid costs the dense builder registers
    constrain(A.con_kind[tid], raw[tid], A.con_lb[bo + tid], A.con_ub[bo + tid], &th,
              jac ? &jc : nullptr);
    theta[tid] = th;
    if (jac) jac[tid] = jc;
  }
}

// constants of the wavelength kernel from its constrained parameters (lam_factor above)
template <int KIND>
__device__ __forceinline__ void lam_setup(const double* th /* NL constrained values */,
                                          double* lam /* [4] */) {
  lam[0] = 1.0; lam[1] = 0.0; lam[2] = 1.0; lam[3] = 1.0;
  if (KIND == PGM_KIND_SEP_RBF) {
    lam[0] = th[0]; lam[3] = th[1]; lam[1] = 0.5 / (th[1] * th[1]);
  } else if (KIND == PGM_KIND_SEP_MATERN15) {
    lam[0] = th[0]; lam[3] = th[1]; lam[1] = 1.7320508075688772935 / th[1];
  } else if (KIND == PGM_KIND_SEP_RQ) {
    lam[0] = th[0]; lam[3] = th[1]; lam[2] = th[2]; lam[1] = 0.5 / (th[2] * th[1] * th[1]);
  } else if (KIND == PGM_KIND_SEP_CONST) {
    lam[0] = th[0];
  } else if (KIND == PGM_ATOM_M12) {
    lam[0] = th[0]; lam[3] = th[1]; lam[1] = 1.0 / th[1];
  } else if (KIND == PGM_ATOM_M25) {
    lam[0] = th[0]; lam[3] = th[1]; lam[1] = 2.2360679774997896964 / th[1];
  }
}

// stationary kinds: time-kernel constants into wq[4] (same {scale, c1, alpha, lengthscale}
// layout), wavelength-kernel constants into lamq[4]
template <int KIND>
__device__ __forceinline__ void stat_setup(const double* th, double* wq, double* aq, double* lamq) {
  if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP || stat_time_atom(KIND) == PGM_ATOM_QP_RBF) {
    // th = {outputscale, lambda (periodic lengthscale), period, l_rbf}
    wq[0] = th[0]; wq[1] = th[1]; wq[2] = th[2]; wq[3] = th[3];
    aq[0] = 2.0 / th[1]; aq[1] = 1.0 / th[2]; aq[2] = 0.5 / (th[3] * th[3]); aq[3] = 0.0;
  } else {
    lam_setup<stat_time_atom(KIND)>(th, wq);
    aq[0] = aq[1] = aq[2] = aq[3] = 0.0;
  }
  lamq[0] = 1.0; lamq[1] = 0.0; lamq[2] = 1.0; lamq[3] = 1.0;
  if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP_RBF) lam_setup<PGM_KIND_SEP_RBF>(th + 4, lamq);
  if constexpr (stat_wave_atom(KIND) != 0)
    lam_setup<stat_wave_atom(KIND)>(th + stat_num_time(KIND), lamq);
}

// d K / d theta constant factor of slot t of the parameters behind the mixture (carriers of
// lam_factor): 1 for scales / constants, scale x d c1-term for lengthscales, scale for alpha
template <int KIND>
__device__ __forceinline__ double lam_grad_factor(int t, const double* wq, const double* lamq) {
  auto ell_factor = [](int atom, const double* lm) {
    return (atom == PGM_KIND_SEP_RBF) ? lm[0] / (lm[3] * lm[3] * lm[3])
           : (atom == PGM_KIND_SEP_MATERN15 || atom == PGM_ATOM_M12 || atom == PGM_ATOM_M25)
               ? lm[0] / lm[3] : lm[0] * 2.0 * lm[2] / lm[3];
  };
  if constexpr (KIND >= PGM_KIND_STAT_BASE) {
    constexpr int NT = stat_num_time(KIND);
    if (t == 0 || t == NT) return 1.0;
    if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP_RBF) {
      if (t == 4) return 1.0;
      if (t == 5) return ell_factor(PGM_KIND_SEP_RBF, lamq);
    }
    if constexpr (stat_time_atom(KIND) == PGM_ATOM_QP || stat_time_atom(KIND) == PGM_ATOM_QP_RBF) {
      // wq = {os, lambda, p, l_r}: d f / d lambda = f s^2 2 / lambda^2,
      // d f / d p = f sin(2 theta) tau (2 / lambda) pi / p^2,  d f / d l_r = f tau^2 / l_r^3
      if (t == 1) return wq[0] * 2.0 / (wq[1] * wq[1]);
      if (t == 2) return wq[0] * (2.0 / wq[1]) * M_PI / (wq[2] * wq[2]);
      if (t == 3) return wq[0] / (wq[3] * wq[3] * wq[3]);
    } else {
      if (t == 1) return ell_factor(stat_time_atom(KIND), wq);
    }
    if (t == NT + 1) return ell_factor(stat_wave_atom(KIND), lamq);
    return lamq[0];
  } else {
    if (t == 1) return ell_factor(KIND, lamq);
    if (t == 2) return lamq[0];
    return 1.0;
  }
}

// kernel constants from theta: mixture weights wq[QT] and aq = 2 pi^2 sigma^2 [QT*DS] (zero for
// the padded mixtures), constants behind the mixture lamq[4]; the stationary kinds fill all three
// in stat_setup.  Threads 0..QT*DS-1 and 32 of the block write.
template <int KIND, int QT, int D>
__device__ __forceinline__ void kernel_constants(const double* theta, int Q, const ParamLayout& L,
                                                 double* wq, double* aq, double* lamq) {
  using C = Cfg<KIND, QT, D>;
  constexpr int DS = C::DS;
  const int tid = threadIdx.x;
  if (!C::STAT && tid < QT) wq[tid] = (tid < Q) ? theta[1 + tid] : 0.0;
  if (!C::STAT && tid < QT * DS) {
    const int q = tid / DS, dd = tid - q * DS;
    const double sg = (q < Q) ? theta[L.o_sigma + q * DS + dd] : 0.0;
    aq[q * DS + dd] = 2.0 * M_PI * M_PI * sg * sg;
  }
  if (tid == 32) {
    if constexpr (C::STAT) stat_setup<KIND>(theta + L.o_lam, wq, aq, lamq);
    else lam_setup<KIND>(theta + L.o_lam, lamq);
  }
}

// per-point fields of point i of the light curve's inputs x[n][D], centred on its first input:
// x_i - x_0 into fx[dd * stride + i], (cos, sin)(2 pi mu_qd (x_id - x_0d)) into
// fcs[2 * ((dd * QT + q) * stride + i)] (0 and (1, 0) for an invalid point or a padded mixture).
// mu = theta + o_mu.
template <int KIND, int QT, int D>
__device__ __forceinline__ void point_fields(const double* x, int i, bool valid, const double* mu,
                                             int Q, double* fx, double* fcs, int stride) {
  constexpr int DS = Cfg<KIND, QT, D>::DS;
#pragma unroll
  for (int dd = 0; dd < D; ++dd) {
    const double xc = valid ? (x[(size_t)i * D + dd] - x[dd]) : 0.0;
    fx[(size_t)dd * stride + i] = xc;
    if (dd < DS) {
#pragma unroll
      for (int q = 0; q < QT; ++q) {
        double sn = 0.0, cs = 1.0;
        if (valid && q < Q) sincospi(2.0 * mu[q * DS + dd] * xc, &sn, &cs);
        *reinterpret_cast<double2*>(fcs + ((size_t)(dd * QT + q) * stride + i) * 2) =
            make_double2(cs, sn);
      }
    }
  }
}

// NaN among the D inputs of point i: K~ then has a NaN in row and column i.  The Cholesky only meets
// it at a pivot, possibly after an earlier pivot has already failed; GPyTorch reports any NaN in K~
// as a NaN failure (info -1) before it tries the ladder, so both engines record it up front.
template <int D>
__device__ __forceinline__ bool point_has_nan(const double* x, int i) {
  bool r = false;
#pragma unroll
  for (int dd = 0; dd < D; ++dd) r |= isnan(x[(size_t)i * D + dd]);
  return r;
}

// per-datum exact marginal log-likelihood -(y^T K~^-1 y + log |K~| + n log 2 pi) / (2 n)
__device__ __forceinline__ double mll_value(double inv_quad, double logdet, int n) {
  return -0.5 * (inv_quad + logdet + (double)n * 1.8378770664093454836) / n;
}

// d mll / d theta of slot tid from the block-reduced carriers: fin[0..NG) the kernel-gradient
// accumulators, fin[NG] tr W, fin[NV] sum alpha.  The caller applies d theta / d raw.
template <int KIND, int QT, int D>
__device__ __forceinline__ double grad_slot(int tid, int n, const ParamLayout& L, const double* fin,
                                            const double* theta, const double* wq,
                                            const double* lamq) {
  using C = Cfg<KIND, QT, D>;
  constexpr int DS = C::DS;
  const double half = 0.5 / (double)n;
  if (tid == 0) return fin[C::NV] / (double)n;
  if (tid < L.o_mu) return half * fin[tid - 1];
  if (tid < L.o_sigma) {
    const int t = tid - L.o_mu, q = t / DS, dd = t - q * DS;
    return half * (-2.0 * M_PI * wq[q]) * fin[QT + q * DS + dd];
  }
  if (tid < L.o_noise) {
    const int t = tid - L.o_sigma, q = t / DS, dd = t - q * DS;
    return half * (-4.0 * M_PI * M_PI * theta[tid] * wq[q]) * fin[QT + QT * DS + q * DS + dd];
  }
  if (tid < L.o_lam) return half * fin[C::NG];   // learned noise: tr W
  // parameters behind the mixture: constant factors of lam_factor's derivative carriers
  const int t = tid - L.o_lam;
  return half * lam_grad_factor<KIND>(t, wq, lamq) * fin[QT + 2 * QT * DS + t];
}

// diagonal jitter of Cholesky attempt 0..3: psd_safe_cholesky's ladder 0, 1e-8, 1e-7, 1e-6
// (1e-6, 1e-5, 1e-4 under PGM_FLAG_JITTER_F32, GPyTorch's float32 cholesky_jitter)
__device__ __forceinline__ double chol_jitter(int attempt, int flags) {
  if (attempt <= 0) return 0.0;
  double j = (flags & PGM_FLAG_JITTER_F32) ? 1e-6 : 1e-8;
  for (int t = 1; t < attempt; ++t) j *= 10.0;
  return j;
}

// ------------------------------------------------------------------------------------
// pipeline state carried by a block across light curves (mbarrier phases keep running)
// ------------------------------------------------------------------------------------
struct PipeState {
  int gq2;   // chunks consumed on the 2-stage ring (phases P, T)
  int gq3;   // chunks consumed on the 3-stage ring (phase G)
  int rcnt;  // bulk loads of the resident tile R completed so far
};

template <int KIND, int QT, int D>
__device__ __forceinline__ void pipe_init_at(double* par, PipeState& ps);
template <int KIND, int QT, int D>
__device__ __forceinline__ void pipe_init(double* sm, PipeState& ps) {
  pipe_init_at<KIND, QT, D>(sm + Cfg<KIND, QT, D>::SM_PAR, ps);
}
template <int KIND, int QT, int D>
__device__ __forceinline__ void pipe_init_at(double* par, PipeState& ps) {
  using C = Cfg<KIND, QT, D>;
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(bars + 8 * s, 1); mbar_init(bars + 8 * (2 + s), NTHREADS / 32); }
    for (int s = 0; s < 3; ++s) { mbar_init(bars + 8 * (4 + s), 1); mbar_init(bars + 8 * (7 + s), NTHREADS / 32); }
    mbar_init(bars + 8 * 10, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    fence_proxy_async();
  }
  ps.gq2 = ps.gq3 = ps.rcnt = 0;
  __syncthreads();
}

// ------------------------------------------------------------------------------------
// one full evaluation of light curve b with raw parameters `raw` (global or shared).
// Writes the per-datum MLL to *mll_out and (PGM_FLAG_GRAD) d MLL / d raw to grad_out[P];
// returns info.
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
__device__ int eval_lightcurve(const EvalArgs& A, int b, const double* raw, double* sm,
                               const Scratch& sc, PipeState& ps, double* mll_out,
                               double* grad_out) {
  using C = Cfg<KIND, QT, D>;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Q = A.Q;
  const bool learn_noise = (A.flags & PGM_FLAG_LEARN_NOISE) != 0;
  const bool want_grad = (A.flags & PGM_FLAG_GRAD) != 0;
  constexpr int DS = C::DS;
  const ParamLayout L = param_layout(KIND, D, Q, learn_noise);
  const int P = L.P;
  const int n = A.n_valid ? A.n_valid[b] : A.n_max;
  const int N = (n + TS - 1) / TS;
  const int npad = N * TS;

  double* stages = sm + C::SM_STAGES;
  double* S2 = stages;         // diagonal blocks: X = L^-1 (aliases the idle pipeline stages)
  double* S = sm + C::SM_S;    // diagonal blocks: C_jj -> L_jj
  double* R = S;               // afterwards: resident X_jj / X_ii operand image (= stage 2 in G)
  double* Cst = stages + 2 * OPBUF;   // stage 1: staging of the register-resident A operand
  double* scr = stages + S_ELEMS;     // 256 doubles behind S2
  double* rowv = sm + C::F_ROW;
  double* colv = sm + C::F_COL;
  double* par = sm + C::F_PAR;
  double* theta = par + C::PAR_THETA;
  double* jac = par + C::PAR_JAC;
  double* wq = par + C::PAR_W;
  double* aq = par + C::PAR_A;
  double* lamq = par + C::PAR_LAM;
  double* red = colv;          // block_reduce scratch (see Cfg::RED_ELEMS)
  double* fin = par + C::PAR_FIN;
  double* zj = par + C::PAR_ZJ;
  double* zi = par + C::PAR_ZI;
  double* dinv = par + C::PAR_DINV;
  double* tab = par + C::PAR_TAB;
  int* s_fail = reinterpret_cast<int*>(sm + C::F_PAR + C::PAR_END);
  int* s_nan = s_fail + 1;     // a NaN among the inputs of K~ (point_has_nan)
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  const unsigned rbar = bars + 8 * 10;
  constexpr bool LEAN = C::LEAN;

  __syncthreads();
  // ---- constraints: raw -> theta, d theta / d raw  (A.2) -----------------------------
  load_theta(A, b, P, raw, theta, jac);
  load_exp_tab(tab);
  if (tid == 0) *s_nan = 0;
  __syncthreads();
  if (tid >= 1 && tid < P && isnan(theta[tid])) *s_nan = 1;   // every slot but the mean is in K~
  kernel_constants<KIND, QT, D>(theta, Q, L, wq, aq, lamq);
  const double mean = theta[0];
  const double lnoise = learn_noise ? theta[L.o_noise] : 0.0;
  // ---- per-point fields into the block's scratch ------------------------------------
  const double* xb = A.x + (size_t)b * A.n_max * D;
  const double* yb = A.y + (size_t)b * A.n_max;
  const double* fnb = A.fixed_noise ? A.fixed_noise + (size_t)b * A.n_max : nullptr;
  for (int i = tid; i < npad; i += NTHREADS) {
    const bool valid = i < n;
    point_fields<KIND, QT, D>(xb, i, valid, theta + L.o_mu, Q, sc.fx, sc.fcs, npad);
    sc.rhs[i] = valid ? (yb[i] - mean) : 0.0;
    const double dn = valid ? ((fnb ? fnb[i] : 0.0) + lnoise) : 0.0;
    sc.dn[i] = dn;
    if (valid && (isnan(dn) || point_has_nan<D>(xb, i))) *s_nan = 1;
  }
  __syncthreads();

  // asynchronous prefetch of the per-point data of tile row/col I into rowv / colv
  auto prefetch_side = [&](double* vec, int I, bool with_alpha) {
    // x: D*64 doubles, cs: NCS*128 doubles, alpha: 64 doubles -> 16-byte chunks
    constexpr int CH_X = D * 32, CH_CS = C::NCS * 64;
    for (int ch = tid; ch < CH_X + CH_CS + 32; ch += NTHREADS) {
      if (ch < CH_X) {
        const int dd = ch >> 5, o = (ch & 31) * 2;
        cp_async16(vec + dd * TS + o, sc.fx + (size_t)dd * npad + I * TS + o);
      } else if (ch < CH_X + CH_CS) {
        const int c2 = ch - CH_X, f = c2 >> 6, o = (c2 & 63) * 2;
        cp_async16(vec + D * TS + f * 2 * TS + o, sc.fcs + ((size_t)f * npad + I * TS) * 2 + o);
      } else if (with_alpha) {
        const int o = (ch - CH_X - CH_CS) * 2;
        cp_async16(vec + C::NFB * TS + o, sc.alpha + I * TS + o);
      }
    }
  };
  auto tile = [&](int i, int j) { return sc.tiles + (size_t)tri(i, j) * TT; };
  auto tileT = [&](int j) { return sc.tilesT + (size_t)j * TT; };

  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  double wreg[QT], areg[QT * DS], lam[4];
#pragma unroll
  for (int q = 0; q < QT; ++q) wreg[q] = wq[q];
#pragma unroll
  for (int q = 0; q < QT * DS; ++q) areg[q] = aq[q];
#pragma unroll
  for (int q = 0; q < 4; ++q) lam[q] = lamq[q];
  double acc[4][2][2];
  double iq_part = 0.0;  // partial of z^T z
  double ld_part = 0.0;  // partial of sum log L_kk
  int info = 0;
  Ring r2{bars, bars + 16, stages, ps.gq2};

  // the register-resident 64x64 result times the resident triangular tile R:
  //   acc <- acc_as_A * R^T   (R[n][k] = 0 for k > n), A staged through stage 1
  auto times_resident = [&]() {
    store_acc_tile(acc, Cst, 1.0);
    __syncthreads();
    zero_acc(acc);
    compute_chunk<M_B_LE, false>(acc, Cst, R, 0, wm, wn, g, tq);
    compute_chunk<M_B_LE, false>(acc, Cst + OPBUF, R + OPBUF, KC / 8, wm, wn, g, tq);
  };

  // ================= phase P: Cholesky + forward solve, with the jitter ladder ========
  for (int attempt = 0; attempt <= 3; ++attempt) {
    const double jitter = chol_jitter(attempt, A.flags);
    if (tid == 0) *s_fail = 0;
    iq_part = 0.0;
    ld_part = 0.0;
    bool failed = false;
    int pre = 0;
    for (int j = 0; j < N && !failed; ++j) {
      for (int i = j; i < N; ++i) {
        zero_acc(acc);
        // next job in column-major order; its k-tile 0 is final as soon as column 0 is
        // done.  No look-ahead across diagonal jobs (S2 aliases the stages there).
        int ni = i + 1, nj = j;
        if (ni >= N) { ni = j + 1; nj = j + 1; }
        const int nnk = (!LEAN && j >= 1 && i != j && ni < N) ? nj : 0;
        auto tA = [&](int k) { return tile(i, k); };
        auto tB = [&](int k) { return tile(j, k); };
        auto nA = [&](int k) { return tile(ni, k); };
        auto nB = [&](int k) { return tile(nj, k); };
        auto pf = [&]() { if (!LEAN) { prefetch_side(rowv, i, false); prefetch_side(colv, j, false); } };
        if (i == j) pre = gemm_stream<M_FULL, true, 2>(acc, r2, j, tA, tB, pre, nnk, nA, nB, pf);
        else pre = gemm_stream<M_FULL, false, 2>(acc, r2, j, tA, tB, pre, nnk, nA, nB, pf);
        __syncthreads();
        if (LEAN) {   // the ring is idle (no look-ahead): the fields of this job go into stage 0
          prefetch_side(rowv, i, false);
          prefetch_side(colv, j, false);
          cp_async_commit();
          cp_async_wait<0>();
          __syncthreads();
        }
        // epilogue: C = Ktilde_ij - acc (diagonal tiles: lower triangle only).  The
        // accumulators are parked in stage 1 (the image the next product reads as its A
        // operand) so that the registers go to the exp / cos chains: one rolled loop over the
        // 8 MMA tiles of the warp, 2 entries x QT mixtures in flight, no per-entry branches
        // (padded points carry finite dummy fields); MMA tiles above the diagonal are skipped.
        store_acc_tile(acc, Cst, 1.0);
#pragma unroll 1
        for (int p8 = 0; p8 < 8; ++p8) {
          const int mi = p8 >> 1, ni2 = p8 & 1;
          if (i == j && frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
          const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
          const int gi = i * TS + r;
          double2* cp = reinterpret_cast<double2*>(Cst + img(r, c0));
          const double2 cv = *cp;
          double out[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int gj = j * TS + c0 + e;
            double kv = k_entry<KIND, QT, D>(rowv, colv, r, c0 + e, wreg, areg, lam, tab);
            kv = (gi < n && gj <= gi) ? kv : 0.0;
            if (gi == gj) kv = (gi < n) ? (kv + sc.dn[gi] + jitter) : 1.0;
            out[e] = kv - (e ? cv.y : cv.x);
          }
          if (i == j) {
            S[r * LD_S + c0] = out[0];
            S[r * LD_S + c0 + 1] = out[1];
          } else {
            *cp = make_double2(out[0], out[1]);
          }
        }
        if (i == j) {
          __syncthreads();
          potrf_inv_64(S, S2, dinv, s_fail);
          if (*s_fail) { failed = true; break; }
          // X_jj -> tile(j,j) and the resident R, X_jj^T -> tilesT[j]  (tile images with
          // explicit zeros in the other triangle); L_jj itself is not needed any more
          double* dt = tile(j, j);
          double* dtT = tileT(j);
          for (int idx = tid; idx < TT / 2; idx += NTHREADS) {
            const int r = idx >> 5, c2 = (idx & 31) * 2;
            double2 v, vt;
            v.x = (c2 <= r) ? S2[r * LD_S + c2] : 0.0;
            v.y = (c2 + 1 <= r) ? S2[r * LD_S + c2 + 1] : 0.0;
            vt.x = (r <= c2) ? S2[c2 * LD_S + r] : 0.0;
            vt.y = (r <= c2 + 1) ? S2[(c2 + 1) * LD_S + r] : 0.0;
            const int o = img(r, c2);
            *reinterpret_cast<double2*>(dt + o) = v;
            *reinterpret_cast<double2*>(R + o) = v;
            *reinterpret_cast<double2*>(dtT + o) = vt;
          }
          fence_proxy_async();  // dt / dtT are read by bulk copies later (barriers follow)
          // forward solve: z_j = X_jj (rhs_j - sum_{k<j} L_jk z_k); the products L_jk z_k
          // were left in fpart by the epilogues of row j's tiles (4 partials per row).
          {
            const int r = tid & 63, part = tid >> 6;
            double u = 0.0;
            for (int k = 0; k < j; ++k) u += sc.fpart[((size_t)tri(j, k) * 4 + part) * TS + r];
            scr[part * TS + r] = u;
          }
          if (tid < TS) ld_part -= log(dinv[tid]);
          __syncthreads();
          if (tid < TS)
            zi[tid] = sc.rhs[j * TS + tid] - ((scr[tid] + scr[TS + tid]) + (scr[2 * TS + tid] + scr[3 * TS + tid]));
          __syncthreads();
          {
            const int r = tid >> 2, l4 = tid & 3;
            double zz = 0.0;
            for (int c = l4; c <= r; c += 4) zz += S2[r * LD_S + c] * zi[c];
            zz += shfl_xor_d(zz, 1);
            zz += shfl_xor_d(zz, 2);
            if (l4 == 0) {
              sc.z[j * TS + r] = zz;
              zj[r] = zz;
              iq_part += zz * zz;
            }
          }
          __syncthreads();
        } else {
          // L_ij = C * X_jj^T  straight from shared memory (C in stage 1, X_jj resident)
          __syncthreads();
          if (LEAN && j >= 1 && ni < N) {
            // the epilogue is done with the fields in stage 0: the next job's first chunk (k-tile 0 of
            // rows ni / nj, final since column 0) travels under the triangular solve and the tile store
            if (tid == 0) ring_issue_first(r2, nA(0), nB(0));
            pre = 1;
          }
          zero_acc(acc);
          compute_chunk<M_B_LE, false>(acc, Cst, R, 0, wm, wn, g, tq);
          compute_chunk<M_B_LE, false>(acc, Cst + OPBUF, R + OPBUF, KC / 8, wm, wn, g, tq);
          // partial products L_ij z_j for the forward solve of row i (deterministic order);
          // their global stores are issued after the tile has left, so that the proxy fence
          // of the bulk store (MEMBAR.ALL.CTA) has no global store of this thread to drain
          double pp[4];
#pragma unroll
          for (int mi = 0; mi < 4; ++mi) {
            double s = 0.0;
#pragma unroll
            for (int ni2 = 0; ni2 < 2; ++ni2)
#pragma unroll
              for (int e = 0; e < 2; ++e) s += acc[mi][ni2][e] * zj[frag_col(wn, ni2, tq, e)];
            s += shfl_xor_d(s, 1);
            s += shfl_xor_d(s, 2);
            pp[mi] = s;
          }
          store_tile_bulk(acc, Cst, tile(i, j), 1.0);
          if (tq == 0) {
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
              sc.fpart[((size_t)tri(i, j) * 4 + wn) * TS + frag_row(wm, mi, g)] = pp[mi];
          }
        }
      }
    }
    __syncthreads();
    const int fl = *s_fail;
    if (!fl) { info = attempt; break; }
    if ((fl & 2) || *s_nan) { info = -1; break; }
    info = -2;
    __syncthreads();
  }

  // ---- MLL ---------------------------------------------------------------------------
  {
    double v2[2] = {iq_part, ld_part};
    block_reduce<2>(v2, red, fin);
  }
  const double mll = (info >= 0) ? mll_value(fin[0], 2.0 * fin[1], n) : nan("");
  __syncthreads();
  if (tid == 0) *mll_out = mll;
  if (!want_grad || info < 0) {
    if (want_grad && tid < P) grad_out[tid] = nan("");
    if (A.alpha_out)   // info < 0 (alpha_out needs PGM_FLAG_GRAD): NaN like mll and grad
      for (int i2 = tid; i2 < A.n_max; i2 += NTHREADS)
        A.alpha_out[(size_t)b * A.n_max + i2] = (i2 < n) ? nan("") : 0.0;
    ps.gq2 = r2.gq;
    return info;
  }

  // ================= phase T: X = L^-1 in place, row by row ============================
  // Tm^T = sum_{k=j}^{i-1} X_kj^T L_ik^T (k = j: X_jj^T from tilesT), X_ij^T = -Tm^T X_ii^T
  // with X_ii resident in R for the whole row; the off-diagonal tiles keep holding X^T.
  {
    int pre = 0;
    for (int i = 1; i < N; ++i) {
      __syncthreads();  // the previous row is done with R and zi
      if (tid == 0) {
        mbar_expect_tx(rbar, 2 * CHUNK_BYTES);
        bulk_g2s(smem_u32(R), tile(i, i), 2 * CHUNK_BYTES, rbar);
      }
      if (tid < TS) zi[tid] = sc.z[i * TS + tid];
      bool rwait = true;
      for (int j = 0; j < i; ++j) {
        zero_acc(acc);
        int ni = i, nj = j + 1;
        if (nj >= i) { ni = i + 1; nj = 0; }
        const int nnk = (ni < N) ? ni - nj : 0;
        auto tA = [&](int kk) { return kk == 0 ? tileT(j) : tile(j + kk, j); };
        auto tB = [&](int kk) { return tile(i, j + kk); };
        auto nA = [&](int kk) { return kk == 0 ? tileT(nj) : tile(nj + kk, nj); };
        auto nB = [&](int kk) { return tile(ni, nj + kk); };
        pre = gemm_stream<M_A_GE, false, 2>(acc, r2, i - j, tA, tB, pre, nnk, nA, nB, []() {});
        __syncthreads();
        if (rwait) {
          mbar_wait(rbar, ps.rcnt & 1);
          ++ps.rcnt;
          rwait = false;
        }
        times_resident();
        // partial products X_ij^T z_i for alpha_j  (X_ij^T = -acc); stored after the tile
        // has left (see phase P)
        double pp[4];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
          double s = 0.0;
#pragma unroll
          for (int ni2 = 0; ni2 < 2; ++ni2)
#pragma unroll
            for (int e = 0; e < 2; ++e) s -= acc[mi][ni2][e] * zi[frag_col(wn, ni2, tq, e)];
          s += shfl_xor_d(s, 1);
          s += shfl_xor_d(s, 2);
          pp[mi] = s;
        }
        store_tile_bulk(acc, Cst, tile(i, j), -1.0);
        if (tq == 0) {
#pragma unroll
          for (int mi = 0; mi < 4; ++mi)
            sc.apart[((size_t)tri(i, j) * 4 + wn) * TS + frag_row(wm, mi, g)] = pp[mi];
        }
      }
    }
  }
  __syncthreads();
  // ---- alpha_j = X_jj^T z_j + sum_{i>j} X_ij^T z_i -----------------------------------
  {
    const int c = tid & 63, rg = tid >> 6;
    for (int j = 0; j < N; ++j) {
      const double* Xt = tile(j, j);
      const double* zz = sc.z + j * TS;
      double s = 0.0;
#pragma unroll
      for (int r = 0; r < 16; ++r) s += Xt[img(rg * 16 + r, c)] * zz[rg * 16 + r];
      for (int i = j + 1; i < N; ++i) s += sc.apart[((size_t)tri(i, j) * 4 + rg) * TS + c];
      scr[rg * TS + c] = s;
      __syncthreads();
      if (tid < TS)
        sc.alpha[j * TS + tid] = (scr[tid] + scr[TS + tid]) + (scr[2 * TS + tid] + scr[3 * TS + tid]);
      __syncthreads();
    }
  }
  // ================= phase G: K^-1 tiles -> gradient contraction =======================
  double ga[C::NG];
#pragma unroll
  for (int t = 0; t < C::NG; ++t) ga[t] = 0.0;
  double trW = 0.0;
  // G phase of the LEAN layout: no tile is resident in this phase, so the fields take the S / R region
  // (prefetched under the k-loop as in the full layout) and the K^-1 tile is parked in stage 1, which
  // the one-chunk look-ahead (always stage 0) never touches - the look-ahead stays on
  static_assert(!LEAN || 2 * C::NF * TS <= S_ELEMS, "LEAN: the fields must fit the S region in the G phase");
  double* rowg = LEAN ? S : rowv;
  double* colg = LEAN ? S + C::NF * TS : colv;
  double* parkg = LEAN ? Cst : R;
  {
    int pre = 0;
    if (tid == 0) bulk_wait_all();
    for (int i = 0; i < N; ++i) {
      for (int j = 0; j <= i; ++j) {
        zero_acc(acc);
        int ni = i, nj = j + 1;
        if (nj > i) { ni = i + 1; nj = 0; }
        const int nnk = (ni < N) ? N - ni : 0;
        // Kinv_ij = sum_kk X_{i+kk,i}^T X_{i+kk,j}: both operands are the stored X^T tiles
        auto tA = [&](int kk) { return kk == 0 ? tileT(i) : tile(i + kk, i); };
        auto tB = [&](int kk) { return (kk == 0 && i == j) ? tileT(j) : tile(i + kk, j); };
        auto nA = [&](int kk) { return kk == 0 ? tileT(ni) : tile(ni + kk, ni); };
        auto nB = [&](int kk) { return (kk == 0 && ni == nj) ? tileT(nj) : tile(ni + kk, nj); };
        auto pf = [&]() { prefetch_side(rowg, i, true); prefetch_side(colg, j, true); };
        if (i == j) pre = gemm_stream<M_A_GE, true, 2>(acc, r2, N - i, tA, tB, pre, nnk, nA, nB, pf);
        else pre = gemm_stream<M_A_GE, false, 2>(acc, r2, N - i, tA, tB, pre, nnk, nA, nB, pf);
        __syncthreads();
        // K^-1 tile parked (R, free in this phase; LEAN: stage 1); rolled, branch-free contraction
        store_acc_tile(acc, parkg, 1.0);
        const double* al_r = rowg + C::NFB * TS;
        const double* al_c = colg + C::NFB * TS;
#pragma unroll 1
        for (int p8 = 0; p8 < 8; ++p8) {
          const int mi = p8 >> 1, ni2 = p8 & 1;
          if (i == j && frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
          const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
          const int gi = i * TS + r;
          const double2 kinv = *reinterpret_cast<const double2*>(parkg + img(r, c0));
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int gj = j * TS + c0 + e;
            double W = al_r[r] * al_c[c0 + e] - (e ? kinv.y : kinv.x);
            W = (gi < n && gj <= gi) ? W : 0.0;
            if (gi == gj) trW += W;
            const double wgt = (gi == gj) ? W : 2.0 * W;
            k_grad_entry<KIND, QT, D>(rowg, colg, r, c0 + e, wreg, areg, lam, tab, wgt, ga);
          }
        }
      }
    }
    ps.gq2 = r2.gq;
  }
  // ---- reduce, apply constants and the constraint Jacobian ----------------------------
  {
    double v[C::NV + 1];
#pragma unroll
    for (int t = 0; t < C::NG; ++t) v[t] = ga[t];
    v[C::NG] = trW;
    double sa = 0.0;
    for (int i2 = tid; i2 < n; i2 += NTHREADS) sa += sc.alpha[i2];
    v[C::NV] = sa;
    if (A.alpha_out)
      for (int i2 = tid; i2 < A.n_max; i2 += NTHREADS)
        A.alpha_out[(size_t)b * A.n_max + i2] = (i2 < n) ? sc.alpha[i2] : 0.0;
    __syncthreads();
    block_reduce<C::NV + 1>(v, red, fin);
  }
  if (tid < P) grad_out[tid] = grad_slot<KIND, QT, D>(tid, n, L, fin, theta, wq, lamq) * jac[tid];
  __syncthreads();
  return info;
}

template <int KIND, int QT, int D>
__device__ __forceinline__ Scratch make_scratch(double* base, int n_max) {
  using C = Cfg<KIND, QT, D>;
  const int N = (n_max + TS - 1) / TS;
  const size_t npad = (size_t)N * TS;
  const size_t ntri = (size_t)tri(N, 0);
  Scratch sc;
  sc.tiles = base;
  sc.tilesT = sc.tiles + ntri * TT;
  sc.fx = sc.tilesT + (size_t)N * TT;
  sc.fcs = sc.fx + (size_t)D * npad;
  sc.alpha = sc.fcs + (size_t)C::NCS * npad * 2;
  sc.rhs = sc.alpha + npad;
  sc.z = sc.rhs + npad;
  sc.dn = sc.z + npad;
  sc.fpart = sc.dn + npad;
  sc.apart = sc.fpart + ntri * 4 * TS;
  return sc;
}

// ------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, (Cfg<KIND, QT, D>::F_BYTES <= 113 * 1024) ? 2 : 1)
    sm_mll_grad_kernel(EvalArgs A) {
  extern __shared__ __align__(16) double sm[];
  Scratch sc = make_scratch<KIND, QT, D>(A.ws + (size_t)blockIdx.x * A.ws_per_block, A.n_max);
  const int P = param_layout(KIND, D, A.Q, (A.flags & PGM_FLAG_LEARN_NOISE) != 0).P;
  PipeState ps;
  pipe_init_at<KIND, QT, D>(sm + Cfg<KIND, QT, D>::F_PAR, ps);
  // broadcast slot of the scheduler: in the spare words behind s_fail (static shared memory would
  // push the block over the two-per-SM limit)
  int* s_next = reinterpret_cast<int*>(sm + Cfg<KIND, QT, D>::F_PAR + Cfg<KIND, QT, D>::PAR_END) + 4;
  const LcSched lsc = sched_init(A, s_next);
  for (int b = next_lightcurve(A, lsc, -1, s_next); b >= 0; b = next_lightcurve(A, lsc, b, s_next)) {
    double* gout = A.grad ? A.grad + (size_t)b * P : nullptr;
    const int info =
        eval_lightcurve<KIND, QT, D>(A, b, A.raw + (size_t)b * P, sm, sc, ps, A.mll + b, gout);
    if (threadIdx.x == 0) A.info[b] = info;
  }
  if (threadIdx.x == 0) bulk_wait_all();  // no bulk store may outlive the block's shared memory
}

// rank t of the lower triangle (row-major) -> (a, b), a >= b
__device__ __forceinline__ void tri_unrank(int t, int& a, int& b) {
  a = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while ((a + 1) * (a + 2) / 2 <= t) ++a;
  while (a * (a + 1) / 2 > t) --a;
  b = t - a * (a + 1) / 2;
}

// dense K + D (north-star kernel 1 as a launch of its own; the fused and staged engines call the
// same k_entry from their Cholesky epilogues and never write K).  One block per (light curve,
// 64x64 tile of the LOWER triangle): the per-point fields of the 128 points are built by all 256
// threads, every entry is evaluated once with the larger index as its row, written row-wise and -
// for off-diagonal tiles - mirrored through a padded shared-memory tile so that both stores are
// coalesced and K_ij, K_ji are the same bits.  FP64-pipe bound (n^2/2 Q exp / cos chains).
template <int KIND, int QT, int D>
struct DenseSmem {
  using C = Cfg<KIND, QT, D>;
  static constexpr int LDT = TS + 1;
  static constexpr int ELEMS = 2 * C::NFB * TS + TS * LDT;
  static constexpr size_t BYTES = (size_t)ELEMS * sizeof(double);
};
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS)
    sm_kernel_dense_kernel(EvalArgs A, double* __restrict__ Kout) {
  using C = Cfg<KIND, QT, D>;
  constexpr int DS = C::DS;
  constexpr int LDT = DenseSmem<KIND, QT, D>::LDT;
  extern __shared__ __align__(16) double dsm[];
  double* rowv = dsm;
  double* colv = rowv + C::NFB * TS;
  double* tl = colv + C::NFB * TS;
  __shared__ double theta[C::PMAX], wq[QT], aq[QT * DS], lamq[4], tab[EXP_TAB];
  const int tid = threadIdx.x;
  const int b = blockIdx.y;
  int ti, tj;
  tri_unrank(blockIdx.x, ti, tj);
  const int Q = A.Q;
  const bool learn_noise = (A.flags & PGM_FLAG_LEARN_NOISE) != 0;
  const ParamLayout L = param_layout(KIND, D, Q, learn_noise);
  const int P = L.P;
  const int n = A.n_valid ? A.n_valid[b] : A.n_max;
  if (ti * TS >= n) return;
  load_theta(A, b, P, A.raw + (size_t)b * P, theta, nullptr);
  load_exp_tab(tab);
  __syncthreads();
  kernel_constants<KIND, QT, D>(theta, Q, L, wq, aq, lamq);
  // fields: item 0 of a point = its centred inputs, items 1.. = (cos, sin)(2 pi mu_qd x_d)
  const double* xb = A.x + (size_t)b * A.n_max * D;
  constexpr int ITEMS = 1 + DS * QT;
  for (int idx = tid; idx < 2 * TS * ITEMS; idx += NTHREADS) {
    const int item = idx / (2 * TS), pt = idx - item * (2 * TS);
    const int side = pt >> 6, r = pt & 63;
    const int gi = (side ? tj : ti) * TS + r;
    double* vec = side ? colv : rowv;
    const bool valid = gi < n;
    if (item == 0) {
#pragma unroll
      for (int dd = 0; dd < D; ++dd) vec[dd * TS + r] = valid ? (xb[(size_t)gi * D + dd] - xb[dd]) : 0.0;
    } else {
      const int f = item - 1, dd = f / QT, q = f - dd * QT;
      double sn = 0.0, cs = 1.0;
      if (valid && q < Q)
        sincospi(2.0 * theta[L.o_mu + q * DS + dd] * (xb[(size_t)gi * D + dd] - xb[dd]), &sn, &cs);
      vec[D * TS + (f * TS + r) * 2] = cs;
      vec[D * TS + (f * TS + r) * 2 + 1] = sn;
    }
  }
  __syncthreads();
  const double lnoise = learn_noise ? theta[L.o_noise] : 0.0;
  const double* fnb = A.fixed_noise ? A.fixed_noise + (size_t)b * A.n_max : nullptr;
  double* Kb = Kout + (size_t)b * A.n_max * A.n_max;
  double wreg[QT], areg[QT * DS], lam[4];
  for (int q = 0; q < QT; ++q) wreg[q] = wq[q];
  for (int q = 0; q < QT * DS; ++q) areg[q] = aq[q];
  for (int q = 0; q < 4; ++q) lam[q] = lamq[q];
  for (int idx = tid; idx < TT; idx += NTHREADS) {
    const int r = idx >> 6, c = idx & 63;
    const int gi = ti * TS + r, gj = tj * TS + c;
    if (gi < n && gj < n) {
      // the larger index is the row (on a diagonal tile rowv and colv hold the same points)
      double kv = (gi >= gj) ? k_entry<KIND, QT, D>(rowv, colv, r, c, wreg, areg, lam, tab)
                             : k_entry<KIND, QT, D>(colv, rowv, c, r, wreg, areg, lam, tab);
      if (gi == gj) kv += (fnb ? fnb[gi] : 0.0) + lnoise;
      Kb[(size_t)gi * A.n_max + gj] = kv;
      tl[r * LDT + c] = kv;
    }
  }
  if (ti == tj) return;
  __syncthreads();
  for (int idx = tid; idx < TT; idx += NTHREADS) {   // K_ji = K_ij, rows of the mirrored tile
    const int c = idx >> 6, r = idx & 63;
    const int gi = ti * TS + r, gj = tj * TS + c;
    if (gi < n && gj < n) Kb[(size_t)gj * A.n_max + gi] = tl[r * LDT + c];
  }
}

// torch.optim.{SGD,Adam,AdamW} step on one parameter (trainers.py:141-147 defaults; A.7).
// g is d loss / d raw; bc1 = 1 - beta1^step and bc2s = sqrt(1 - beta2^step) are the bias
// corrections of the step (the same for every parameter: computed once per step by the caller).
__device__ __forceinline__ double optim_update_bc(double p, double g, double& m, double& v,
                                                  int kind, double lr, double b1, double b2,
                                                  double eps, double wd, double bc1, double bc2s) {
  if (kind == 0) return p - lr * g;
  if (kind == 2) p *= (1.0 - lr * wd);
  else if (wd != 0.0) g += wd * p;
  m = b1 * m + (1.0 - b1) * g;
  v = b2 * v + (1.0 - b2) * g * g;
  const double denom = sqrt(v) / bc2s + eps;
  return p - (lr / bc1) * (m / denom);
}
__device__ __forceinline__ double optim_update(double p, double g, double& m, double& v,
                                               int kind, double lr, double b1, double b2,
                                               double eps, double wd, int step) {
  const double bc1 = 1.0 - pow(b1, (double)step);
  const double bc2s = sqrt(1.0 - pow(b2, (double)step));
  return optim_update_bc(p, g, m, v, kind, lr, b1, b2, eps, wd, bc1, bc2s);
}

// whole training loop of trainers.py:177-207 per light curve, on device
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, (Cfg<KIND, QT, D>::F_BYTES <= 113 * 1024) ? 2 : 1)
    sm_fit_kernel(FitArgs F) {
  using C = Cfg<KIND, QT, D>;
  extern __shared__ __align__(16) double sm[];
  const EvalArgs& A = F.e;
  Scratch sc = make_scratch<KIND, QT, D>(A.ws + (size_t)blockIdx.x * A.ws_per_block, A.n_max);
  const int P = param_layout(KIND, D, A.Q, (A.flags & PGM_FLAG_LEARN_NOISE) != 0).P;
  double* par = sm + C::F_PAR;
  double* s_raw = par + C::PAR_RAW;
  double* s_m = s_raw + C::PMAX;
  double* s_v = s_m + C::PMAX;
  double* s_grad = s_v + C::PMAX;
  double* s_mll = par + C::PAR_FIN + C::NV + 2;
  const int tid = threadIdx.x;
  PipeState ps;
  pipe_init_at<KIND, QT, D>(sm + Cfg<KIND, QT, D>::F_PAR, ps);
  // broadcast slot of the scheduler: in the spare words behind s_fail (static shared memory would
  // push the block over the two-per-SM limit)
  int* s_next = reinterpret_cast<int*>(sm + Cfg<KIND, QT, D>::F_PAR + Cfg<KIND, QT, D>::PAR_END) + 4;
  const LcSched lsc = sched_init(A, s_next);
  for (int b = next_lightcurve(A, lsc, -1, s_next); b >= 0; b = next_lightcurve(A, lsc, b, s_next)) {
    __syncthreads();
    if (tid < P) {
      s_raw[tid] = F.raw_io[(size_t)b * P + tid];
      s_m[tid] = 0.0;
      s_v[tid] = 0.0;
      if (F.raw_hist) F.raw_hist[(size_t)b * P + tid] = s_raw[tid];
    }
    int it = 0, info = 0;
    for (; it < F.maxiter; ++it) {
      __syncthreads();
      info = eval_lightcurve<KIND, QT, D>(A, b, s_raw, sm, sc, ps, s_mll, s_grad);
      __syncthreads();
      const double loss = -(*s_mll);
      if (tid == 0) F.loss_hist[(size_t)it * A.B + b] = loss;
      if (info < 0) { ++it; break; }
      if (tid < P) {
        s_raw[tid] = optim_update(s_raw[tid], -s_grad[tid], s_m[tid], s_v[tid], F.optim_kind,
                                  F.lr, F.beta1, F.beta2, F.eps, F.weight_decay, it + 1);
        if (F.raw_hist) F.raw_hist[((size_t)(it + 1) * A.B + b) * P + tid] = s_raw[tid];
      }
      // early stop: stop and i > miniter and std(loss[-stopavg:]) < stop  (np.std, ddof 0)
      if (F.stop > 0.0 && it > F.miniter) {
        const int cnt = min(F.stopavg, it + 1);
        double s1 = 0.0, s2 = 0.0;
        for (int t = 0; t < cnt; ++t) s1 += (t == 0) ? loss : F.loss_hist[(size_t)(it - t) * A.B + b];
        const double mu = s1 / cnt;
        for (int t = 0; t < cnt; ++t) {
          const double lv = (t == 0) ? loss : F.loss_hist[(size_t)(it - t) * A.B + b];
          s2 += (lv - mu) * (lv - mu);
        }
        if (sqrt(s2 / cnt) < F.stop) { ++it; break; }
      }
    }
    __syncthreads();
    if (tid < P) F.raw_io[(size_t)b * P + tid] = s_raw[tid];
    if (tid == 0) { F.n_iter[b] = it; A.info[b] = info; }
    // mark the unused tail of the history
    for (int t = it + tid; t < F.maxiter; t += NTHREADS) F.loss_hist[(size_t)t * A.B + b] = nan("");
  }
  if (threadIdx.x == 0) bulk_wait_all();
}

}  // namespace pgm
