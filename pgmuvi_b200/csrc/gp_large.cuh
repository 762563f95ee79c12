// pgmuvi_b200 - single large exact GP (n in the thousands .. tens of thousands) on ONE B200.
//
// BASELINE configs C3 (n = 8000, 2-D) and C4 (n = 32768): the factor no longer fits one
// block's scratch, so the whole GPU works on one matrix.  K~ lives in HBM as the lower
// triangle of 64x64 tile images (the shared-memory operand image of gp_fused.cuh) and every
// product runs through the same bulk-copy + mbarrier DMMA tile engine, one output tile per
// thread block, one kernel launch per dependency stage:
//
//   P  right-looking blocked Cholesky, panels of NB tile columns:
//        lg_update (column of the panel, k inside the panel)  -> lg_diag (64x64 potrf +
//        inverse, z_j, log-det)  -> lg_trsm (L_ij = C_ij X_jj^T, rhs_i -= L_ij z_j)
//        ... then ONE lg_update over the whole trailing triangle (k = the panel).
//      The first touch of a tile generates K~ in the epilogue (never a separate build pass).
//   T  X = L^-1 row by row (lg_inv_row: one block per tile of the row), alpha = X^T z.
//   G  K^-1_ij = sum_k X_ki^T X_kj per tile, contracted at once with W = alpha alpha^T - K^-1
//      and the regenerated dK/dtheta; per-tile partial sums, deterministic final reduction.
//
// The same kernels take a batch index (blockIdx.y = light curve): a batch of B light curves
// advances stage by stage in lock step, every launch carrying B x (tiles of the stage)
// independent blocks for the hardware scheduler to balance ("staged" engine; the fused
// one-block-per-light-curve kernel of gp_fused.cuh is the other engine).  The jitter ladder of
// psd_safe_cholesky is per light curve: state[b] / attempt[b] / fail[b] live behind the
// per-light-curve workspaces and failed members alone repeat the P phase.
//
// Reference semantics as gp_fused.cuh (pgmuvi/trainers.py:177-182, SURVEY.md Appendix A);
// the exact-Cholesky branch for n > 800 is the north star's definition of the path (F6).
#pragma once
#include "gp_fused.cuh"

namespace pgm {

constexpr int LG_NFB_MAX = 2 + 2 * 16;   // per-point doubles upper bound: x[2], (cos,sin)[16]
constexpr int LG_PAR = 160;              // theta[64] jac[64] wq[8] aq[16] lam[4] (+pad)
constexpr int LG_GP = 48;                // doubles per job in the gradient partials
constexpr int LG_PAR_TH = 0, LG_PAR_JC = 64, LG_PAR_WQ = 128, LG_PAR_AQ = 136, LG_PAR_LM = 152;

struct LargeWs {
  double *tilesL, *tilesX, *tilesT;
  double *fx, *fcs, *alpha, *rhs, *z, *dn, *par, *ldz, *gpart;
  double *fpart;   // [ntri][64]: L_ij z_j per tile (forward solve of the one-launch P phase)
};
// batch state behind the B per-light-curve workspaces
struct BatchState {
  int *state;     // 0 = needs the P phase, 1 = factored, 2 = failed
  int *attempt;   // jitter rung 0..3
  int *fail;      // potrf failure bits of the current pass
  int *nan_in;    // 1: a NaN among the inputs of K~ (lg_setup), so a failure is reported as -1
  int *count;     // light curves that must repeat the P phase
  int *tflag;     // [B, ntri(n_max)] "X tile is final" flags of the one-launch T phase
};
enum { LG_ACTIVE = 0, LG_FACTORED = 1, LG_FAILED = 2 };

__host__ __device__ inline size_t large_ws_elems(int n) {
  const size_t N = (n + TS - 1) / TS, npad = N * TS, ntri = N * (N + 1) / 2;
  return 2 * ntri * TT + N * TT + (size_t)(LG_NFB_MAX + 4) * npad + LG_PAR + 2 * N +
         ntri * LG_GP + ntri * TS + 16;
}
__host__ __device__ inline size_t large_ntri(int n_max) {
  const size_t N = (n_max + TS - 1) / TS;
  return N * (N + 1) / 2;
}
__host__ __device__ inline size_t large_ws_bytes(int n_max, int B) {
  return large_ws_elems(n_max) * sizeof(double) * (size_t)B +
         ((size_t)(4 * B + 4) + (size_t)B * large_ntri(n_max)) * sizeof(int);
}
__host__ __device__ inline BatchState make_batch_state(double* base, int n_max, int B) {
  BatchState st;
  st.state = reinterpret_cast<int*>(base + large_ws_elems(n_max) * (size_t)B);
  st.attempt = st.state + B;
  st.fail = st.attempt + B;
  st.nan_in = st.fail + B;
  st.count = st.nan_in + B;
  st.tflag = st.count + 4;
  return st;
}
__host__ __device__ inline LargeWs make_large_ws(double* base, int n) {
  const size_t N = (n + TS - 1) / TS, npad = N * TS, ntri = N * (N + 1) / 2;
  LargeWs w;
  w.tilesL = base;
  w.tilesX = w.tilesL + ntri * TT;
  w.tilesT = w.tilesX + ntri * TT;
  w.fx = w.tilesT + N * TT;
  w.fcs = w.fx + 2 * npad;
  w.alpha = w.fcs + 32 * npad;
  w.rhs = w.alpha + npad;
  w.z = w.rhs + npad;
  w.dn = w.z + npad;
  w.par = w.dn + npad;
  w.ldz = w.par + LG_PAR;
  w.gpart = w.ldz + 2 * N;
  w.fpart = w.gpart + ntri * LG_GP;
  return w;
}

struct LargeArgs {
  const double* x;            // [B, n_max, D]
  const int32_t* n_valid;     // [B] or null
  const double* y;            // [B, n_max]
  const double* fixed_noise;  // [B, n_max] or null
  const double* raw;          // [B, P]
  const int32_t* con_kind;
  const double* con_lb;
  const double* con_ub;
  int B, n_max, Q, flags;
  double* mll;                // [B]
  double* grad;               // [B, P]
  int32_t* info;              // [B] (device)
  double* ws;
  double* alpha_out;          // [B, n_max] or null
};

// the light curve of this block: its size and workspace
struct LcView {
  int b, n, N, npad;
  LargeWs w;
  BatchState st;
};
__device__ __forceinline__ LcView lc_view(const LargeArgs& A, int b = -1) {
  LcView v;
  v.b = b >= 0 ? b : (int)blockIdx.y;
  v.n = A.n_valid ? A.n_valid[v.b] : A.n_max;
  v.N = (v.n + TS - 1) / TS;
  v.npad = v.N * TS;
  v.w = make_large_ws(A.ws + large_ws_elems(A.n_max) * (size_t)v.b, A.n_max);
  v.st = make_batch_state(A.ws, A.n_max, A.B);
  return v;
}

__device__ __forceinline__ double* lg_tile(double* base, int i, int j) {
  return base + ((size_t)i * (i + 1) / 2 + j) * TT;
}
// linear index t -> (a, b) with a >= b >= 0 (row-major lower triangle)
// tri_unrank: gp_fused.cuh

// ------------------------------------------------------------------------------------
// setup: constraints -> parameter block; per-point fields, rhs, noise diagonal
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS) lg_setup(LargeArgs A) {
  __shared__ double theta[64], jac[64];
  const int tid = threadIdx.x;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_ACTIVE) return;
  const LargeWs& w = v.w;
  const int Q = A.Q;
  const bool learn_noise = (A.flags & PGM_FLAG_LEARN_NOISE) != 0;
  const ParamLayout L = param_layout(KIND, D, Q, learn_noise);
  const int P = L.P;
  const int n = v.n, npad = v.npad;
  if (blockIdx.x * NTHREADS >= npad) return;
  load_theta(A, v.b, P, A.raw + (size_t)v.b * P, theta, jac);
  __syncthreads();
  if (blockIdx.x == 0) {
    if (tid < P) {
      w.par[LG_PAR_TH + tid] = theta[tid];
      w.par[LG_PAR_JC + tid] = jac[tid];
    }
    if (tid >= 1 && tid < P && isnan(theta[tid])) v.st.nan_in[v.b] = 1;   // every slot but the mean
    kernel_constants<KIND, QT, D>(theta, Q, L, w.par + LG_PAR_WQ, w.par + LG_PAR_AQ,
                                  w.par + LG_PAR_LM);
  }
  const double mean = theta[0];
  const double lnoise = learn_noise ? theta[L.o_noise] : 0.0;
  const int i = blockIdx.x * NTHREADS + tid;
  if (i >= npad) return;
  const bool valid = i < n;
  const double* xb = A.x + (size_t)v.b * A.n_max * D;
  const double* yb = A.y + (size_t)v.b * A.n_max;
  const double* fnb = A.fixed_noise ? A.fixed_noise + (size_t)v.b * A.n_max : nullptr;
  point_fields<KIND, QT, D>(xb, i, valid, theta + L.o_mu, Q, w.fx, w.fcs, npad);
  w.rhs[i] = valid ? (yb[i] - mean) : 0.0;
  const double dn = valid ? ((fnb ? fnb[i] : 0.0) + lnoise) : 0.0;
  w.dn[i] = dn;
  if (valid && (isnan(dn) || point_has_nan<D>(xb, i))) v.st.nan_in[v.b] = 1;
}

// per-point data of tile row / col I -> rowv / colv (cp.async, as in the fused kernel)
template <int KIND, int QT, int D>
__device__ __forceinline__ void lg_prefetch_side(double* vec, const LargeWs& w, int npad, int I,
                                                 bool with_alpha) {
  using C = Cfg<KIND, QT, D>;
  constexpr int CH_X = D * 32, CH_CS = C::NCS * 64;
  for (int ch = threadIdx.x; ch < CH_X + CH_CS + 32; ch += NTHREADS) {
    if (ch < CH_X) {
      const int dd = ch >> 5, o = (ch & 31) * 2;
      cp_async16(vec + dd * TS + o, w.fx + (size_t)dd * npad + I * TS + o);
    } else if (ch < CH_X + CH_CS) {
      const int c2 = ch - CH_X, f = c2 >> 6, o = (c2 & 63) * 2;
      cp_async16(vec + D * TS + f * 2 * TS + o, w.fcs + ((size_t)f * npad + I * TS) * 2 + o);
    } else if (with_alpha) {
      const int o = (ch - CH_X - CH_CS) * 2;
      cp_async16(vec + C::NFB * TS + o, w.alpha + I * TS + o);
    }
  }
}

// kernel constants of the light curve (written by lg_setup) in registers, for k_entry / k_grad_entry
template <int KIND, int QT, int D>
struct LgConst {
  double w[QT], a[QT * Cfg<KIND, QT, D>::DS], lam[4];
  __device__ __forceinline__ void load(const double* par) {
#pragma unroll
    for (int q = 0; q < QT; ++q) w[q] = par[LG_PAR_WQ + q];
#pragma unroll
    for (int q = 0; q < QT * Cfg<KIND, QT, D>::DS; ++q) a[q] = par[LG_PAR_AQ + q];
#pragma unroll
    for (int q = 0; q < 4; ++q) lam[q] = par[LG_PAR_LM + q];
  }
};

// entry (gi, gj) of the lower triangle of K~ = K + noise + jitter: zero above the diagonal and
// outside the n valid points, 1 on the diagonal of the padding (r, c: rows of rowv / colv)
template <int KIND, int QT, int D>
__device__ __forceinline__ double lg_k_masked(const double* rowv, const double* colv, int r, int c,
                                              int gi, int gj, int n, const double* dn, double jitter,
                                              const double (&w)[QT],
                                              const double (&a)[QT * Cfg<KIND, QT, D>::DS],
                                              const double (&lam)[4], const double* tab) {
  double kv = k_entry<KIND, QT, D>(rowv, colv, r, c, w, a, lam, tab);
  kv = (gi < n && gj <= gi) ? kv : 0.0;
  if (gi == gj) kv = (gi < n) ? (kv + dn[gi] + jitter) : 1.0;
  return kv;
}

// thread 0: mbarriers of gemm_stream's 2-stage Ring{bars, bars + 16} (full / empty) and, unless
// `extra` is 0, one single-arrival barrier for a resident tile.  A block barrier must follow.
__device__ __forceinline__ void lg_ring_init(unsigned bars, unsigned extra = 0) {
  if (threadIdx.x != 0) return;
  for (int s = 0; s < 2; ++s) { mbar_init(bars + 8 * s, 1); mbar_init(bars + 8 * (2 + s), NTHREADS / 32); }
  if (extra) mbar_init(extra, 1);
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  fence_proxy_async();
}

// Job index of a block of a one-launch dataflow phase: a ticket taken when the block STARTS, so that
// the job order is the order in which blocks actually begin to run.  Every job only waits for jobs of
// lower index, and a block holding ticket t started after the blocks holding 0 .. t-1 did, so waiting
// can never deadlock whatever the hardware's dispatch order (MPS, preemption, debuggers) - the
// decoupled look-back idiom.  `counter` is zeroed by the host before the launch.
// `bcast`: any word of the block's (still unused) dynamic shared memory.
__device__ __forceinline__ unsigned lg_ticket(int* counter, void* bcast) {
  volatile unsigned* s_ticket = reinterpret_cast<volatile unsigned*>(bcast);
  if (threadIdx.x == 0) *s_ticket = (unsigned)atomicAdd(counter, 1);
  __syncthreads();
  const unsigned t = *s_ticket;
  __syncthreads();
  return t;
}

// per-tile "final" flags of the one-launch phases (lg_chol_all, lg_inv_all)
__device__ __forceinline__ void lg_wait_flag(const int* f) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
  if (!v) {
    // Watchdog: jobs come from a ticket taken at block start (lg_ticket), so every awaited producer
    // is running or done.  Should that ever not hold, fail the launch after 20 s
    // of waiting instead of hanging the device.
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t0));
    do {
      __nanosleep(40);
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
      if (!v) {
        asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t1));
        if (t1 - t0 > 20000000000ull) __trap();
      }
    } while (!v);
  }
  fence_proxy_async();   // the tile was written, and will be read, through the async proxy
}
// Non-blocking look at a flag: the acquire load is issued here, its value is consumed one k-tile later
// (lg_wait_flag_pf), so that the L2 round trip of the poll hides under the products of the tile in
// between (r02y: the blocking poll per operand tile paced the k-loops of the one-launch phases).
__device__ __forceinline__ int lg_peek_flag(const int* f) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
  return v;
}
// wait for a flag whose value was peeked earlier (0 = not yet set then: poll); no proxy fence
__device__ __forceinline__ void lg_wait_flag_pf(const int* f, int peeked) {
  if (peeked) return;
  int v;
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t0));
  do {
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
    if (!v) {
      __nanosleep(40);
      asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t1));
      if (t1 - t0 > 20000000000ull) __trap();
    }
  } while (!v);
}
__device__ __forceinline__ void lg_set_flag(int* f) {
  fence_proxy_async();
  // st.release.gpu is a gpu-scope release fence + store: no separate __threadfence() in front of it
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(f), "r"(1) : "memory");
}

// ------------------------------------------------------------------------------------
// C_ij -= sum_{k0 <= k < k1} L_ik L_jk^T   (build: C_ij = K~_ij - sum, first touch)
//   mode 0: one tile column j = jj, i = jj + blockIdx.x
//   mode 1: the whole trailing triangle i >= j >= jj, blockIdx.x -> (i - jj, j - jj)
// ------------------------------------------------------------------------------------
// Shared memory of lg_update: ring + ONE 32 KB region that is the block's own C tile when the launch
// updates an existing tile (read-modify-write) and the per-point fields when it builds K~ (first
// touch; the result is then formed in stage 1) - never both.  102-105 KB for every kind, i.e. two
// blocks per SM also for SM-8 (C4's trailing updates) and the ARD 2-D kinds (r02z).
template <int KIND, int QT, int D>
struct UpdSmem {
  using C = Cfg<KIND, QT, D>;
  static constexpr int CT_OFF = STAGE_ELEMS;
  static constexpr int UNION = (2 * C::NF * TS > 2 * OPBUF) ? 2 * C::NF * TS : 2 * OPBUF;
  static constexpr int PAR_OFF = CT_OFF + UNION;
  static constexpr size_t BYTES = (size_t)(PAR_OFF + C::PAR_END + 8) * sizeof(double);
  static constexpr int MIN_BLOCKS = (BYTES <= 113 * 1024) ? 2 : 1;
};
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, UpdSmem<KIND, QT, D>::MIN_BLOCKS)
    lg_update(LargeArgs A, int mode, int jj, int k0, int k1, int build) {
  using C = Cfg<KIND, QT, D>;
  using L = UpdSmem<KIND, QT, D>;
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_ACTIVE) return;
  const LargeWs& w = v.w;
  const int n = v.n, N = v.N, npad = v.npad;
  int i, j;
  if (mode == 0) {
    j = jj;
    i = jj + blockIdx.x;
  } else {
    int a, b;
    tri_unrank(blockIdx.x, a, b);
    i = jj + a;
    j = jj + b;
  }
  if (i >= N || j >= N) return;
  if (v.st.fail[v.b]) return;
  const double jitter = chol_jitter(v.st.attempt[v.b], A.flags);
  double* stages = sm;
  double* Cst = stages + 2 * OPBUF;
  double* Ct = sm + L::CT_OFF;            // !build: the block's own C tile
  double* rowv = Ct;                      // build: per-point fields (same region)
  double* colv = rowv + C::NF * TS;
  double* par = sm + L::PAR_OFF;
  double* tab = par + C::PAR_TAB;
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  const unsigned cbar = bars + 8 * 10;
  load_exp_tab(tab);
  lg_ring_init(bars, cbar);
  __syncthreads();
  Ring r2{bars, bars + 16, stages, 0};
  double* out = lg_tile(w.tilesL, i, j);
  if (!build && tid == 0) {
    // read-modify-write of C_ij through shared memory: one bulk load now (lands under the k-loop),
    // one bulk store at the end, instead of 16 scattered 16-byte global accesses per thread
    mbar_expect_tx(cbar, 2 * CHUNK_BYTES);
    bulk_g2s(smem_u32(Ct), out, 2 * CHUNK_BYTES, cbar);
  }
  double acc[4][2][2];
  zero_acc(acc);
  auto tA = [&](int kk) { return lg_tile(w.tilesL, i, k0 + kk); };
  auto tB = [&](int kk) { return lg_tile(w.tilesL, j, k0 + kk); };
  auto none = [&](int) { return (double*)nullptr; };
  auto pf = [&]() {
    if (build) {
      lg_prefetch_side<KIND, QT, D>(rowv, w, npad, i, false);
      lg_prefetch_side<KIND, QT, D>(colv, w, npad, j, false);
    }
  };
  if (i == j) gemm_stream<M_FULL, true, 2>(acc, r2, k1 - k0, tA, tB, 0, 0, none, none, pf);
  else gemm_stream<M_FULL, false, 2>(acc, r2, k1 - k0, tA, tB, 0, 0, none, none, pf);
  __syncthreads();
  if (!build) {
    mbar_wait(cbar, 0);
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
      for (int ni = 0; ni < 2; ++ni) {
        const int r = frag_row(wm, mi, g), c = frag_col(wn, ni, tq, 0);
        double2* p = reinterpret_cast<double2*>(Ct + img(r, c));
        double2 vv = *p;
        vv.x -= acc[mi][ni][0];
        vv.y -= acc[mi][ni][1];
        *p = vv;
      }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      bulk_s2g(out, smem_u32(Ct), 2 * OPBUF * sizeof(double));
      bulk_commit();
      bulk_wait_all();
    }
    return;
  }
  LgConst<KIND, QT, D> kc;
  kc.load(w.par);
  store_acc_tile(acc, Cst, 1.0);
#pragma unroll 1
  for (int p8 = 0; p8 < 8; ++p8) {
    const int mi = p8 >> 1, ni2 = p8 & 1;
    if (i == j && frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
    const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
    const int gi = i * TS + r;
    double2* cp = reinterpret_cast<double2*>(Cst + img(r, c0));
    const double2 cv = *cp;
    double o2[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const double kv = lg_k_masked<KIND, QT, D>(rowv, colv, r, c0 + e, gi, j * TS + c0 + e, n, w.dn,
                                                 jitter, kc.w, kc.a, kc.lam, tab);
      o2[e] = kv - (e ? cv.y : cv.x);
    }
    *cp = make_double2(o2[0], o2[1]);
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (tid == 0) {
    bulk_s2g(out, smem_u32(Cst), 2 * OPBUF * sizeof(double));
    bulk_commit();
    bulk_wait_all();
  }
}

// ------------------------------------------------------------------------------------
// diagonal block j: C_jj -> X_jj = L_jj^-1 (tilesL / tilesX diagonal slots), X_jj^T (tilesT),
// z_j = X_jj rhs_j, log-det and z^T z partials
// ------------------------------------------------------------------------------------
// After potrf_inv_64 (S2 = X_jj, dinv = 1 / diag L_jj), in two steps.  (a) What the other tiles of
// column j wait for: X_jj in the L array's diagonal slot and z_j = X_jj zi; red[r] = z_r^2 and
// red[64 + r] = -log dinv[r] for step (b).
__device__ __forceinline__ void lg_diag_solve(const LargeWs& w, int j, const double* S2,
                                              const double* zi, const double* dinv, double* red) {
  const int tid = threadIdx.x;
  double* tl = lg_tile(w.tilesL, j, j);
  for (int idx = tid; idx < TT / 2; idx += NTHREADS) {
    const int r = idx >> 5, c2 = (idx & 31) * 2;
    double2 vv;
    vv.x = (c2 <= r) ? S2[r * LD_S + c2] : 0.0;
    vv.y = (c2 + 1 <= r) ? S2[r * LD_S + c2 + 1] : 0.0;
    *reinterpret_cast<double2*>(tl + img(r, c2)) = vv;
  }
  const int r = tid >> 2, l4 = tid & 3;
  double zz = 0.0;
  for (int c = l4; c <= r; c += 4) zz += S2[r * LD_S + c] * zi[c];
  zz += shfl_xor_d(zz, 1);
  zz += shfl_xor_d(zz, 2);
  if (l4 == 0) {
    w.z[j * TS + r] = zz;
    red[r] = zz * zz;
    red[TS + r] = -log(dinv[r]);
  }
}
// (b) What later phases read: X_jj (tilesX) and X_jj^T (tilesT), and the log-det / quadratic-form
// partials.  `red` of step (a) must be complete (a block barrier in between).
__device__ __forceinline__ void lg_diag_images(const LargeWs& w, int j, const double* S2,
                                               const double* red) {
  const int tid = threadIdx.x;
  double* tx = lg_tile(w.tilesX, j, j);
  double* tt = w.tilesT + (size_t)j * TT;
  for (int idx = tid; idx < TT / 2; idx += NTHREADS) {
    const int r = idx >> 5, c2 = (idx & 31) * 2;
    double2 vv, vt;
    vv.x = (c2 <= r) ? S2[r * LD_S + c2] : 0.0;
    vv.y = (c2 + 1 <= r) ? S2[r * LD_S + c2 + 1] : 0.0;
    vt.x = (r <= c2) ? S2[c2 * LD_S + r] : 0.0;
    vt.y = (r <= c2 + 1) ? S2[(c2 + 1) * LD_S + r] : 0.0;
    const int o = img(r, c2);
    *reinterpret_cast<double2*>(tx + o) = vv;
    *reinterpret_cast<double2*>(tt + o) = vt;
  }
  if (tid < 2) {
    double s = 0.0;
    for (int r = 0; r < TS; ++r) s += red[tid * TS + r];
    w.ldz[2 * j + (tid ? 0 : 1)] = s;   // ldz[2j] = sum log L_kk, ldz[2j+1] = z_j^T z_j
  }
}

constexpr size_t LG_DIAG_SMEM = (size_t)(2 * S_ELEMS + 4 * TS + 8) * sizeof(double);
static __global__ void __launch_bounds__(NTHREADS) lg_diag(LargeArgs A, int j) {
  extern __shared__ __align__(16) double sm[];
  double* S = sm;
  double* S2 = sm + S_ELEMS;
  double* dinv = S2 + S_ELEMS;
  double* zi = dinv + TS;
  double* red = zi + TS;   // [2 * 64]
  int* s_fail = reinterpret_cast<int*>(red + 2 * TS);
  const int tid = threadIdx.x;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_ACTIVE || j >= v.N) return;
  if (v.st.fail[v.b]) return;   // an earlier diagonal block failed: keep its failure bits
  const LargeWs& w = v.w;
  double* tl = lg_tile(w.tilesL, j, j);
  if (tid == 0) *s_fail = 0;
  for (int idx = tid; idx < TT / 2; idx += NTHREADS) {
    const int r = idx >> 5, c2 = (idx & 31) * 2;
    const double2 vv = *reinterpret_cast<const double2*>(tl + img(r, c2));
    S[r * LD_S + c2] = vv.x;
    S[r * LD_S + c2 + 1] = vv.y;
  }
  if (tid < TS) zi[tid] = w.rhs[j * TS + tid];
  __syncthreads();
  potrf_inv_64(S, S2, dinv, s_fail);
  if (*s_fail) {
    if (tid == 0) atomicOr(v.st.fail + v.b, *s_fail);
    return;
  }
  lg_diag_solve(w, j, S2, zi, dinv, red);
  __syncthreads();
  lg_diag_images(w, j, S2, red);
}

// ------------------------------------------------------------------------------------
// L_ij = C_ij X_jj^T for i > j;  rhs_i -= L_ij z_j
// ------------------------------------------------------------------------------------
// row t (< 64) of a [4][64] set of per-warp-column partials, summed in a fixed order
__device__ __forceinline__ double lg_sum4(const double* red, int t) {
  return (red[t] + red[TS + t]) + (red[2 * TS + t] + red[3 * TS + t]);
}

// L_ij = C X_jj^T (images of C in Cst, of X_jj in R), the row partials of L_ij z_j over the four
// warp columns into red[4][64], and the bulk store of L_ij to `dst`, left in flight.  The barriers of
// the store also publish `red`.
__device__ __forceinline__ void lg_offdiag_solve(double* Cst, const double* R, const double* zj,
                                                 double* red, double* dst) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  double acc[4][2][2];
  zero_acc(acc);
  compute_chunk<M_B_LE, false>(acc, Cst, R, 0, wm, wn, g, tq);
  compute_chunk<M_B_LE, false>(acc, Cst + OPBUF, R + OPBUF, KC / 8, wm, wn, g, tq);
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    double s = 0.0;
#pragma unroll
    for (int ni = 0; ni < 2; ++ni)
#pragma unroll
      for (int e = 0; e < 2; ++e) s += acc[mi][ni][e] * zj[frag_col(wn, ni, tq, e)];
    s += shfl_xor_d(s, 1);
    s += shfl_xor_d(s, 2);
    if (tq == 0) red[wn * TS + frag_row(wm, mi, g)] = s;
  }
  store_tile_bulk(acc, Cst, dst, 1.0);
}

constexpr size_t LG_TRSM_SMEM = (size_t)(4 * OPBUF + 5 * TS + 8) * sizeof(double);
static __global__ void __launch_bounds__(NTHREADS, 2) lg_trsm(LargeArgs A, int j) {
  extern __shared__ __align__(16) double sm[];
  double* Cst = sm;
  double* R = sm + 2 * OPBUF;
  double* zj = R + 2 * OPBUF;
  double* red = zj + TS;   // [4][64]
  const unsigned bar = smem_u32(red + 4 * TS);
  const int tid = threadIdx.x;
  const LcView v = lc_view(A);
  const int i = j + 1 + blockIdx.x;
  if (v.st.state[v.b] != LG_ACTIVE || i >= v.N) return;
  if (v.st.fail[v.b]) return;   // a diagonal block of this light curve already failed
  const LargeWs& w = v.w;
  double* tij = lg_tile(w.tilesL, i, j);
  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    fence_proxy_async();
  }
  if (tid < TS) zj[tid] = w.z[j * TS + tid];
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(bar, 4 * CHUNK_BYTES);
    bulk_g2s(smem_u32(Cst), tij, 2 * CHUNK_BYTES, bar);
    bulk_g2s(smem_u32(R), lg_tile(w.tilesL, j, j), 2 * CHUNK_BYTES, bar);
  }
  mbar_wait(bar, 0);
  lg_offdiag_solve(Cst, R, zj, red, tij);
  if (tid < TS) w.rhs[i * TS + tid] -= lg_sum4(red, tid);
  if (tid == 0) bulk_wait_all();
}

// ------------------------------------------------------------------------------------
// The whole P phase (blocked Cholesky + forward solve) of one pass in ONE launch: block t <->
// tile (i, j), i >= j, in COLUMN-major order (tile-major over a batch).  Left-looking: the
// block accumulates sum_{k<j} L_ik L_jk^T, waiting on the "final" flag of each operand tile
// right before its bulk copies are issued, generates K~_ij in the epilogue, then
//   i == j: 64x64 potrf + inverse, z_j = X_jj (rhs_j - sum_k L_jk z_k), log-det partials;
//   i >  j: waits for the diagonal tile, L_ij = C X_jj^T, partial product L_ij z_j -> fpart.
// Every dependency has a lower block index (earlier column, or the head of the same column),
// and blocks are dispatched in index order, so waiting cannot deadlock.  A failed diagonal
// block records its failure BEFORE it raises its flag; blocks that come later see it, skip
// their factorisation (so that garbage never turns a "not p.d." into a NaN report) and still
// raise their flags.
// ------------------------------------------------------------------------------------
// Block order: column-major with look-ahead on the critical path.  t = 0 is tile (0, 0); then,
// per column j: (j+1, j), the NEXT diagonal tile (j+1, j+1), and the rest of column j
// (j+2.., j).  The two tiles that gate the next column are dispatched first and run while the
// bulk of column j is still being processed; every dependency keeps a lower index.
__device__ __forceinline__ void col_unrank(int t, int N, int& i, int& j) {
  if (t == 0) { i = 0; j = 0; return; }
  t -= 1;
  // group j starts at offset(j) = j N - j (j - 1) / 2 and holds N - j tiles
  const double b = 2.0 * N + 1.0;
  j = (int)((b - sqrt(b * b - 8.0 * (double)t)) * 0.5);
  if (j < 0) j = 0;
  if (j > N - 2) j = N - 2;
  while (j > 0 && j * N - j * (j - 1) / 2 > t) --j;
  while (j < N - 2 && (j + 1) * N - (j + 1) * j / 2 <= t) ++j;
  const int r = t - (j * N - j * (j - 1) / 2);
  if (r == 0) { i = j + 1; }
  else if (r == 1) { i = j + 1; j = j + 1; }
  else { i = j + r; }
}

// shared memory: [stages 64 KB | S 34 KB | par]; the per-point fields of the epilogue are fetched
// AFTER the k-loop into idle buffers (rows: stage 0; columns: the S region, which an
// off-diagonal job needs only later for X_jj - a diagonal job's columns ARE its rows), so that
// two blocks fit on an SM for every kind
template <int KIND, int QT, int D>
struct CholAllSmem {
  using C = Cfg<KIND, QT, D>;
  static_assert(C::NFB * TS <= 2 * OPBUF, "row fields must fit in stage 0");
  static constexpr int S_OFF = STAGE_ELEMS;
  static constexpr int PAR_OFF = S_OFF + S_ELEMS;
  static constexpr size_t BYTES = (size_t)(PAR_OFF + C::PAR_END + 8) * sizeof(double);
};

template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, 2) lg_chol_all(LargeArgs A) {
  using C = Cfg<KIND, QT, D>;
  using L = CholAllSmem<KIND, QT, D>;
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  const unsigned job = lg_ticket(make_batch_state(A.ws, A.n_max, A.B).count + 1, sm);
  const unsigned tix = job / (unsigned)A.B;
  const LcView v = lc_view(A, (int)(job - tix * (unsigned)A.B));
  const int Nmax = (A.n_max + TS - 1) / TS;
  int i, j;
  col_unrank((int)tix, Nmax, i, j);
  if (v.st.state[v.b] != LG_ACTIVE || i >= v.N) return;
  const LargeWs& w = v.w;
  const int n = v.n, npad = v.npad;
  int* flags = v.st.tflag + (size_t)v.b * large_ntri(A.n_max);
  auto flag_of = [&](int a, int b2) { return flags + ((size_t)a * (a + 1) / 2 + b2); };
  volatile int* failp = v.st.fail + v.b;
  const double jitter = chol_jitter(v.st.attempt[v.b], A.flags);
  double* stages = sm;
  double* S2 = stages;                  // diagonal job: X = L^-1 (the stages are idle then)
  double* Cst = stages + 2 * OPBUF;
  double* red = stages;                 // off-diagonal job: [4][64] partial products
  double* S = sm + L::S_OFF;
  double* R = S;
  double* rowv = stages;                // epilogue only: stage 0 is idle after the k-loop
  double* colv = (i == j) ? rowv : S;   // S is idle until the off-diagonal job loads X_jj
  double* par = sm + L::PAR_OFF;
  double* tab = par + C::PAR_TAB;
  double* zj = par + C::PAR_ZJ;
  double* zi = par + C::PAR_ZI;
  double* dinv = par + C::PAR_DINV;
  double* red2 = stages + S_ELEMS;      // [2][64] small reductions of the diagonal job (behind S2)
  int* s_fail = reinterpret_cast<int*>(par + C::PAR_END);
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  const unsigned rbar = bars + 8 * 10;
  load_exp_tab(tab);
  lg_ring_init(bars, rbar);
  if (tid == 0) *s_fail = 0;
  __syncthreads();
  Ring r2{bars, bars + 16, stages, 0};
  LgConst<KIND, QT, D> kc;
  kc.load(w.par);
  if (i == j) {
    // Diagonal job = the critical path of the factorisation (column j + 1 cannot start before it):
    // K~_jj (+ noise, jitter) does not depend on the operands this block is about to wait for, so it
    // is generated into S BEFORE the k-loop (fields through stage 0, which the ring takes over
    // afterwards); behind the k-loop only C = K~ - acc is left (r02y).
    lg_prefetch_side<KIND, QT, D>(rowv, w, npad, i, false);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
#pragma unroll 1
    for (int p8 = 0; p8 < 8; ++p8) {
      const int mi = p8 >> 1, ni2 = p8 & 1;
      if (frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
      const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
      const int gi = i * TS + r;
#pragma unroll
      for (int e = 0; e < 2; ++e)
        S[r * LD_S + c0 + e] = lg_k_masked<KIND, QT, D>(rowv, rowv, r, c0 + e, gi, j * TS + c0 + e, n,
                                                        w.dn, jitter, kc.w, kc.a, kc.lam, tab);
    }
    __syncthreads();      // everyone is done with the fields in stage 0
  }
  double acc[4][2][2];
  zero_acc(acc);
  auto tA = [&](int kk) { return lg_tile(w.tilesL, i, kk); };
  auto tB = [&](int kk) { return lg_tile(w.tilesL, j, kk); };
  auto none = [&](int) { return (double*)nullptr; };
  // producer thread only: both operand tiles of k-tile kk must be final; the flags of k-tile kk + 1 are
  // peeked here and looked at one k-tile later
  int pk_k = -1, pk_j = 0, pk_i = 0;
  auto ready = [&](int kk) {
    const bool have = (pk_k == kk);
    lg_wait_flag_pf(flag_of(j, kk), have ? pk_j : 0);
    if (i != j) lg_wait_flag_pf(flag_of(i, kk), have ? pk_i : 0);
    fence_proxy_async();   // the tiles were written, and will be read, through the async proxy
    if (kk + 1 < j) {
      pk_j = lg_peek_flag(flag_of(j, kk + 1));
      pk_i = (i != j) ? lg_peek_flag(flag_of(i, kk + 1)) : 1;
      pk_k = kk + 1;
    }
  };
  if (i == j) gemm_stream_r<M_FULL, true, 2>(acc, r2, j, tA, tB, 0, 0, none, none, []() {}, ready);
  else gemm_stream_r<M_FULL, false, 2>(acc, r2, j, tA, tB, 0, 0, none, none, []() {}, ready);
  __syncthreads();
  if (i == j) {
    // C = K~ - acc on the lower MMA tiles; every thread revisits the entries it wrote itself
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
      for (int ni2 = 0; ni2 < 2; ++ni2) {
        if (frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
        double2* sp = reinterpret_cast<double2*>(S + frag_row(wm, mi, g) * LD_S + frag_col(wn, ni2, tq, 0));
        double2 kv = *sp;
        kv.x -= acc[mi][ni2][0];
        kv.y -= acc[mi][ni2][1];
        *sp = kv;
      }
  } else {
    // the stages are idle now: per-point fields of tile row i / column j into stage 0 / S
    lg_prefetch_side<KIND, QT, D>(rowv, w, npad, i, false);
    lg_prefetch_side<KIND, QT, D>(colv, w, npad, j, false);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    // epilogue: C = K~_ij - acc, image in stage 1.  The entry is masked here rather than by
    // lg_k_masked (i > j: no diagonal entry): with nvcc 12.9 its dead diagonal branch raises
    // lg_chol_all<1,4,2> and <4,8,2> from 126 to 128 registers.
    store_acc_tile(acc, Cst, 1.0);
#pragma unroll 1
    for (int p8 = 0; p8 < 8; ++p8) {
      const int mi = p8 >> 1, ni2 = p8 & 1;
      const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
      const int gi = i * TS + r;
      double2* cp = reinterpret_cast<double2*>(Cst + img(r, c0));
      const double2 cv = *cp;
      double o2[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int gj = j * TS + c0 + e;
        double kv = k_entry<KIND, QT, D>(rowv, colv, r, c0 + e, kc.w, kc.a, kc.lam, tab);
        kv = (gi < n && gj <= gi) ? kv : 0.0;
        o2[e] = kv - (e ? cv.y : cv.x);
      }
      *cp = make_double2(o2[0], o2[1]);
    }
  }
  if (i == j) {
    // ---- diagonal tile: all operands (j, k < j) were awaited in the k-loop
    if (tid < TS) {
      double u = 0.0;
      for (int k = 0; k < j; ++k) u += __ldcg(w.fpart + ((size_t)j * (j + 1) / 2 + k) * TS + tid);
      zi[tid] = w.rhs[j * TS + tid] - u;
    }
    __syncthreads();
    const bool earlier_failure = (*failp != 0);
    if (!earlier_failure) potrf_inv_64(S, S2, dinv, s_fail);
    const bool ok = !earlier_failure && (*s_fail == 0);
    if (!earlier_failure && *s_fail && tid == 0) atomicOr(v.st.fail + v.b, *s_fail);
    // What column j's other blocks wait for goes out FIRST (X_jj in the L array's diagonal slot and
    // z_j), then the flag; the copies later phases read (X_jj / X_jj^T for the inverse and the
    // gradient, the log-det / quadratic-form partials) follow behind the flag (r02y).
    if (ok) lg_diag_solve(w, j, S2, zi, dinv, red2);
    fence_proxy_async();   // the tile written above is read by bulk copies of other blocks
    __syncthreads();
    if (tid == 0) lg_set_flag(flag_of(j, j));
    if (ok) {
      lg_diag_images(w, j, S2, red2);
      fence_proxy_async();   // tilesX / tilesT are read by bulk copies of the following kernels
    }
    return;
  }
  // ---- off-diagonal tile: L_ij = C X_jj^T once the diagonal tile is final
  __syncthreads();         // C image complete in stage 1; stage 0 free for `red`
  if (tid == 0) {
    lg_wait_flag(flag_of(j, j));
    mbar_expect_tx(rbar, 2 * CHUNK_BYTES);
    bulk_g2s(smem_u32(R), lg_tile(w.tilesL, j, j), 2 * CHUNK_BYTES, rbar);
  }
  __syncthreads();         // the acquire of thread 0 is ordered before everyone's loads below
  if (tid < TS) zj[tid] = __ldcg(w.z + j * TS + tid);
  const bool failed = (*failp != 0);
  mbar_wait(rbar, 0);
  __syncthreads();
  lg_offdiag_solve(Cst, R, zj, red, lg_tile(w.tilesL, i, j));
  if (tid < TS && !failed) w.fpart[((size_t)i * (i + 1) / 2 + j) * TS + tid] = lg_sum4(red, tid);
  __syncthreads();
  if (tid == 0) {
    bulk_wait_all();
    lg_set_flag(flag_of(i, j));
  }
}

// per-light-curve jitter ladder (psd_safe_cholesky, A.5) after a P pass
static __global__ void lg_ladder(LargeArgs A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  BatchState st = make_batch_state(A.ws, A.n_max, A.B);
  if (st.state[b] != LG_ACTIVE) return;
  const int fl = st.fail[b];
  if (!fl) {
    st.state[b] = LG_FACTORED;
    A.info[b] = st.attempt[b];
  } else if ((fl & 2) || st.nan_in[b]) {   // a NaN in K~, possibly behind an earlier failed pivot
    st.state[b] = LG_FAILED;
    A.info[b] = -1;
  } else if (st.attempt[b] < 3) {
    st.attempt[b] += 1;
    st.fail[b] = 0;
    atomicAdd(st.count, 1);
  } else {
    st.state[b] = LG_FAILED;
    A.info[b] = -2;
  }
}

// ------------------------------------------------------------------------------------
// row i of X = L^-1:  X_ij^T = -(sum_{k=j}^{i-1} X_kj^T L_ik^T) X_ii^T,  j = blockIdx.x < i
// (reads L from tilesL, writes X^T tiles to tilesX: blocks of one launch never conflict)
// ------------------------------------------------------------------------------------
// alpha_j = X_jj^T z_j + sum_{i>j} X_ij^T z_i: the products X_ij^T z_i ride along with the T phase
// (the tile is in the accumulators as -X_ij^T; 4 partials per row over the warp columns, summed in
// a fixed order) and land in fpart - dead after the P phase -, so that lg_alpha only adds N of
// them per point instead of walking the tile column (r02y: 32 -> 6 us at n = 1000).
__device__ __forceinline__ void lg_inv_partial(const double (&acc)[4][2][2], const double* __restrict__ zi,
                                               double* red /* [4][64], stage 0 is idle */, int wm, int wn,
                                               int g, int tq) {
  double zc[2][2];
#pragma unroll
  for (int ni = 0; ni < 2; ++ni)
#pragma unroll
    for (int e = 0; e < 2; ++e) zc[ni][e] = __ldcg(zi + frag_col(wn, ni, tq, e));
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    double s = 0.0;
#pragma unroll
    for (int ni = 0; ni < 2; ++ni)
#pragma unroll
      for (int e = 0; e < 2; ++e) s -= acc[mi][ni][e] * zc[ni][e];
    s += shfl_xor_d(s, 1);
    s += shfl_xor_d(s, 2);
    if (tq == 0) red[wn * TS + frag_row(wm, mi, g)] = s;
  }
}
// Tile (i, j), i > j, of X = L^-1 and its alpha partial.  `ready(kk)`: producer-thread hook run
// before the operands of k-tile kk are loaded; `flags` (or null): the light curve's per-tile flags,
// the tile's own is raised once the tile is stored.  The alpha partial is stored behind the flag (no
// block of the launch reads it).
constexpr size_t LG_INV_SMEM = (size_t)(6 * OPBUF + 16) * sizeof(double);
template <typename FR>
__device__ __forceinline__ void lg_inv_tile(double* sm, const LargeWs& w, int i, int j, FR ready,
                                            int* flags) {
  double* stages = sm;
  double* Cst = stages + 2 * OPBUF;
  double* R = sm + 4 * OPBUF;
  const unsigned bars = smem_u32(sm + 6 * OPBUF);
  const unsigned rbar = bars + 8 * 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  lg_ring_init(bars, rbar);
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(rbar, 2 * CHUNK_BYTES);
    bulk_g2s(smem_u32(R), lg_tile(w.tilesX, i, i), 2 * CHUNK_BYTES, rbar);
  }
  Ring r2{bars, bars + 16, stages, 0};
  double acc[4][2][2];
  zero_acc(acc);
  auto tA = [&](int kk) { return kk == 0 ? w.tilesT + (size_t)j * TT : lg_tile(w.tilesX, j + kk, j); };
  auto tB = [&](int kk) { return lg_tile(w.tilesL, i, j + kk); };
  auto none = [&](int) { return (double*)nullptr; };
  gemm_stream_r<M_A_GE, false, 2>(acc, r2, i - j, tA, tB, 0, 0, none, none, []() {}, ready);
  __syncthreads();
  store_acc_tile(acc, Cst, 1.0);
  __syncthreads();
  mbar_wait(rbar, 0);
  zero_acc(acc);
  compute_chunk<M_B_LE, false>(acc, Cst, R, 0, wm, wn, g, tq);
  compute_chunk<M_B_LE, false>(acc, Cst + OPBUF, R + OPBUF, KC / 8, wm, wn, g, tq);
  lg_inv_partial(acc, w.z + i * TS, stages, wm, wn, g, tq);
  store_tile_bulk(acc, Cst, lg_tile(w.tilesX, i, j), -1.0);   // its barriers also publish the partials
  if (tid == 0) {
    bulk_wait_all();
    if (flags) lg_set_flag(flags + ((size_t)i * (i + 1) / 2 + j));
  }
  if (tid < TS) w.fpart[((size_t)i * (i + 1) / 2 + j) * TS + tid] = lg_sum4(stages, tid);
}

static __global__ void __launch_bounds__(NTHREADS, 2) lg_inv_row(LargeArgs A, int i) {
  extern __shared__ __align__(16) double sm[];
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED || i >= v.N) return;
  lg_inv_tile(sm, v.w, i, (int)blockIdx.x, [](int) {}, nullptr);
}

// ------------------------------------------------------------------------------------
// The whole T phase in ONE launch: block t <-> tile (i, j), i > j, in row-major order.  Tile
// (i, j) needs the X tiles (k, j), j < k < i - all of lower block index.  Blocks are
// dispatched in index order, so every producer a block waits for is running or done: the
// producer thread spins on the "tile is final" flag of an operand just before it issues that
// operand's bulk copies, and each block publishes its tile (bulk store complete -> proxy fence
// -> release store of the flag) at the end.  Rows overlap: the dependency depth drops from one
// launch per tile row (N^2 / 2 tile products along column 0) to about two products per row.
// ------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(NTHREADS, 2) lg_inv_all(LargeArgs A) {
  extern __shared__ __align__(16) double sm[];
  // tile-major block order (all light curves' tile t before any tile t + 1): in a batch the
  // blocks adjacent in dispatch order are independent, a single GP gets plain row-major order
  const unsigned job = lg_ticket(make_batch_state(A.ws, A.n_max, A.B).count + 2, sm);
  const unsigned tix = job / (unsigned)A.B;
  const LcView v = lc_view(A, (int)(job - tix * (unsigned)A.B));
  int i, j;
  tri_unrank((int)tix, i, j);   // (a, b), a >= b  ->  tile (a + 1, b)
  i += 1;
  if (v.st.state[v.b] != LG_FACTORED || i >= v.N) return;
  int* flags = v.st.tflag + (size_t)v.b * large_ntri(A.n_max);
  // producer thread only: X_{j+kk, j} must be final; the flag of k-tile kk + 1 is peeked one tile ahead
  int pk_k = -1, pk_v = 0;
  auto xflag = [&](int kk) { return flags + ((size_t)(j + kk) * (j + kk + 1) / 2 + j); };
  auto ready = [&](int kk) {
    if (kk > 0) {
      lg_wait_flag_pf(xflag(kk), (pk_k == kk) ? pk_v : 0);
      fence_proxy_async();
    }
    if (kk + 1 < i - j) {
      pk_v = lg_peek_flag(xflag(kk + 1));
      pk_k = kk + 1;
    }
  };
  lg_inv_tile(sm, v.w, i, j, ready, flags);
}

// alpha_j = X_jj^T z_j + sum_{i>j} X_ij^T z_i   (tilesX holds X_jj and the X_ij^T tiles)
static __global__ void __launch_bounds__(NTHREADS) lg_alpha(LargeArgs A) {
  __shared__ double scr[4 * TS];
  const int tid = threadIdx.x;
  const LcView v = lc_view(A);
  const int N = v.N, j = blockIdx.x;
  if (v.st.state[v.b] != LG_FACTORED || j >= N) return;
  const LargeWs& w = v.w;
  const int m = tid & 63, part = tid >> 6;
  double s = 0.0;
  {
    const double* Xd = lg_tile(w.tilesX, j, j);
    const double* zz = w.z + j * TS;
#pragma unroll 4
    for (int r = part * 16; r < part * 16 + 16; ++r) s += Xd[img(r, m)] * zz[r];
  }
  // the off-diagonal products were left in fpart by the T phase (lg_inv_partial)
  for (int i = j + 1 + part; i < N; i += 4) s += w.fpart[((size_t)i * (i + 1) / 2 + j) * TS + m];
  scr[part * TS + m] = s;
  __syncthreads();
  if (tid < TS)
    w.alpha[j * TS + tid] = (scr[tid] + scr[TS + tid]) + (scr[2 * TS + tid] + scr[3 * TS + tid]);
}

// ------------------------------------------------------------------------------------
// gradient partials of tile (i, j), i >= j:  K^-1_ij = sum_kk X_{i+kk,i}^T X_{i+kk,j}
// ------------------------------------------------------------------------------------
// Shared memory of lg_grad: one tile job per block and no look-ahead, so the ring is idle behind the
// k-loop and the K^-1 tile is parked in stage 1 - no separate 34 KB work tile.  That brings the ARD
// 2-D kinds (19 per-point fields per side) under the two-blocks-per-SM limit (r02z); two blocks are
// only asked for while the gradient accumulators leave room in 128 registers (NG <= 24).
template <int KIND, int QT, int D>
struct GradSmem {
  using C = Cfg<KIND, QT, D>;
  static constexpr int ROW_OFF = STAGE_ELEMS;
  static constexpr int COL_OFF = ROW_OFF + C::NF * TS;
  static constexpr int PAR_OFF = COL_OFF + C::NF * TS;
  static constexpr size_t BYTES = (size_t)(PAR_OFF + C::PAR_END + 8) * sizeof(double);
  static constexpr int MIN_BLOCKS = (BYTES <= 113 * 1024 && C::NG <= 24) ? 2 : 1;
};
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, GradSmem<KIND, QT, D>::MIN_BLOCKS)
    lg_grad(LargeArgs A) {
  using C = Cfg<KIND, QT, D>;
  using L = GradSmem<KIND, QT, D>;
  static_assert(C::NV <= LG_GP, "gradient partial slot too small");
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  const LargeWs& w = v.w;
  const int n = v.n, N = v.N, npad = v.npad;
  int i, j;
  tri_unrank(blockIdx.x, i, j);
  if (i >= N) return;
  double* stages = sm;
  double* R = stages + 2 * OPBUF;   // K^-1 tile parked in stage 1 (the ring is idle by then)
  double* rowv = sm + L::ROW_OFF;
  double* colv = sm + L::COL_OFF;
  double* par = sm + L::PAR_OFF;
  double* red = colv;          // block_reduce scratch: the fields are dead by then (Cfg::RED_ELEMS)
  double* fin = par + C::PAR_FIN;
  double* tab = par + C::PAR_TAB;
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  load_exp_tab(tab);
  lg_ring_init(bars);
  __syncthreads();
  Ring r2{bars, bars + 16, stages, 0};
  double acc[4][2][2];
  zero_acc(acc);
  auto tA = [&](int kk) { return kk == 0 ? w.tilesT + (size_t)i * TT : lg_tile(w.tilesX, i + kk, i); };
  auto tB = [&](int kk) {
    return (kk == 0 && i == j) ? w.tilesT + (size_t)j * TT : lg_tile(w.tilesX, i + kk, j);
  };
  auto none = [&](int) { return (double*)nullptr; };
  auto pf = [&]() {
    lg_prefetch_side<KIND, QT, D>(rowv, w, npad, i, true);
    lg_prefetch_side<KIND, QT, D>(colv, w, npad, j, true);
  };
  if (i == j) gemm_stream<M_A_GE, true, 2>(acc, r2, N - i, tA, tB, 0, 0, none, none, pf);
  else gemm_stream<M_A_GE, false, 2>(acc, r2, N - i, tA, tB, 0, 0, none, none, pf);
  __syncthreads();
  LgConst<KIND, QT, D> kc;
  kc.load(w.par);
  store_acc_tile(acc, R, 1.0);
  double ga[C::NG];
#pragma unroll
  for (int t = 0; t < C::NG; ++t) ga[t] = 0.0;
  double trW = 0.0;
  const double* al_r = rowv + C::NFB * TS;
  const double* al_c = colv + C::NFB * TS;
#pragma unroll 1
  for (int p8 = 0; p8 < 8; ++p8) {
    const int mi = p8 >> 1, ni2 = p8 & 1;
    if (i == j && frag_mt(wm, mi) < frag_nt(wn, ni2)) continue;
    const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
    const int gi = i * TS + r;
    const double2 kinv = *reinterpret_cast<const double2*>(R + img(r, c0));
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int gj = j * TS + c0 + e;
      double W = al_r[r] * al_c[c0 + e] - (e ? kinv.y : kinv.x);
      W = (gi < n && gj <= gi) ? W : 0.0;
      if (gi == gj) trW += W;
      const double wgt = (gi == gj) ? W : 2.0 * W;
      k_grad_entry<KIND, QT, D>(rowv, colv, r, c0 + e, kc.w, kc.a, kc.lam, tab, wgt, ga);
    }
  }
  double vv[C::NV];
#pragma unroll
  for (int t = 0; t < C::NG; ++t) vv[t] = ga[t];
  vv[C::NG] = trW;
  __syncthreads();
  block_reduce<C::NV>(vv, red, fin);
  if (tid < C::NV) w.gpart[(size_t)blockIdx.x * LG_GP + tid] = fin[tid];
}

// ------------------------------------------------------------------------------------
// final reduction (fixed order), MLL, gradient assembly: one block per light curve
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS) lg_finish(LargeArgs A, int want_grad) {
  using C = Cfg<KIND, QT, D>;
  __shared__ double red[8 * (C::NV + 4)], fin[C::NV + 4];
  const int tid = threadIdx.x;
  const LcView v = lc_view(A);
  const LargeWs& w = v.w;
  const int n = v.n, N = v.N;
  const ParamLayout L = param_layout(KIND, D, A.Q, (A.flags & PGM_FLAG_LEARN_NOISE) != 0);
  const int P = L.P;
  double* mll_out = A.mll + v.b;
  double* grad_out = A.grad ? A.grad + (size_t)v.b * P : nullptr;
  if (v.st.state[v.b] != LG_FACTORED) {
    if (tid == 0) *mll_out = nan("");
    if (want_grad && tid < P) grad_out[tid] = nan("");
    if (want_grad && A.alpha_out)
      for (int i2 = tid; i2 < A.n_max; i2 += NTHREADS)
        A.alpha_out[(size_t)v.b * A.n_max + i2] = (i2 < n) ? nan("") : 0.0;
    return;
  }
  double vv[C::NV + 3];
#pragma unroll
  for (int t = 0; t < C::NV + 3; ++t) vv[t] = 0.0;
  for (int jb = tid; jb < N; jb += NTHREADS) {
    vv[C::NV + 1] += w.ldz[2 * jb];
    vv[C::NV + 2] += w.ldz[2 * jb + 1];
  }
  if (want_grad) {
    // per-tile partials: 64x64 tiles (lg_grad) or 128x128 tiles (lg_grad_tc, PGM_FLAG_TF32X3)
    const int NTg = (A.flags & PGM_FLAG_TF32X3) ? (N + 1) / 2 : N;
    const int njobs = NTg * (NTg + 1) / 2;
    for (int t = tid; t < njobs; t += NTHREADS)
#pragma unroll
      for (int k = 0; k < C::NV; ++k) vv[k] += w.gpart[(size_t)t * LG_GP + k];
    for (int i2 = tid; i2 < n; i2 += NTHREADS) vv[C::NV] += w.alpha[i2];
    if (A.alpha_out)
      for (int i2 = tid; i2 < A.n_max; i2 += NTHREADS)
        A.alpha_out[(size_t)v.b * A.n_max + i2] = (i2 < n) ? w.alpha[i2] : 0.0;
  }
  block_reduce<C::NV + 3>(vv, red, fin);
  if (tid == 0) *mll_out = mll_value(fin[C::NV + 2], 2.0 * fin[C::NV + 1], n);
  if (!want_grad || tid >= P) return;
  grad_out[tid] = grad_slot<KIND, QT, D>(tid, n, L, fin, w.par + LG_PAR_TH, w.par + LG_PAR_WQ,
                                         w.par + LG_PAR_LM) *
                  w.par[LG_PAR_JC + tid];
}

// ------------------------------------------------------------------------------------
// N1: exact posterior prediction at m test inputs per light curve (the step after the fit:
// pgmuvi/lightcurve.py:9607-9640, 9862, 9937 evaluate likelihood(model(x_fine)) on a 10000-point
// grid; GPyTorch does it under fast_pred_var, i.e. with an approximate variance - this is the
// exact one it approximates).   mean* = c + K*^T alpha,   var* = k** - || L^-1 k* ||^2.
// Runs after the P and T phases (X = L^-1 and alpha in the workspace).
// ------------------------------------------------------------------------------------
// row-major X_ij (i > j) into tilesL: the stored X_ij^T image transposed (tilesL is dead after T)
static __global__ void __launch_bounds__(NTHREADS) lg_transpose(LargeArgs A) {
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  int i, j;
  tri_unrank(blockIdx.x, i, j);
  if (i >= v.N || i == j) return;
  const double* src = lg_tile(v.w.tilesX, i, j);
  double* dst = lg_tile(v.w.tilesL, i, j);
  for (int idx = threadIdx.x; idx < TT / 2; idx += NTHREADS) {
    const int r = idx >> 5, c2 = (idx & 31) * 2;   // dst[r][c2..c2+1] = src[c2..][r]
    *reinterpret_cast<double2*>(dst + img(r, c2)) = make_double2(src[img(c2, r)], src[img(c2 + 1, r)]);
  }
}

struct PredictArgs {
  LargeArgs a;
  const double* xstar;   // [B, m, D]
  int m;
  double* mean;          // [B, m]
  double* var;           // [B, m]   latent variance (no likelihood noise)
  double* kscratch;      // gridDim.x * N_max tiles: K*^T panels of the block's current job
};

template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS, (Cfg<KIND, QT, D>::SMEM_BYTES <= 113 * 1024) ? 2 : 1)
    lg_predict(PredictArgs PA) {
  using C = Cfg<KIND, QT, D>;
  constexpr int DS = C::DS;
  extern __shared__ __align__(16) double sm[];
  const LargeArgs& A = PA.a;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tq = lane & 3, wm = warp >> 2, wn = warp & 3;
  double* stages = sm + C::SM_STAGES;
  double* rowv = sm + C::SM_ROW;   // test tile fields
  double* colv = sm + C::SM_COL;   // train tile fields (+ alpha)
  double* par = sm + C::SM_PAR;
  double* scr = sm + C::SM_S;      // 34 KB free region: reductions
  double* tab = par + C::PAR_TAB;
  const unsigned bars = smem_u32(par + C::PAR_BAR);
  load_exp_tab(tab);
  PipeState ps;
  pipe_init<KIND, QT, D>(sm, ps);
  Ring r2{bars, bars + 16, stages, 0};
  const int Nmax = (A.n_max + TS - 1) / TS;
  const int Mt = (PA.m + TS - 1) / TS;
  double* ks = PA.kscratch + (size_t)blockIdx.x * Nmax * TT;
  const BatchState st = make_batch_state(A.ws, A.n_max, A.B);
  const int Q = A.Q;
  const bool learn_noise = (A.flags & PGM_FLAG_LEARN_NOISE) != 0;
  (void)learn_noise;
  for (int job = blockIdx.x; job < A.B * Mt; job += gridDim.x) {
    const int b = job / Mt, t = job - b * Mt;
    double* mean_out = PA.mean + (size_t)b * PA.m;
    double* var_out = PA.var + (size_t)b * PA.m;
    __syncthreads();
    if (st.state[b] != LG_FACTORED) {
      if (tid < TS && t * TS + tid < PA.m) {
        mean_out[t * TS + tid] = nan("");
        var_out[t * TS + tid] = nan("");
      }
      continue;
    }
    const int n = A.n_valid ? A.n_valid[b] : A.n_max;
    const int N = (n + TS - 1) / TS, npad = N * TS;
    const LargeWs w = make_large_ws(A.ws + large_ws_elems(A.n_max) * (size_t)b, A.n_max);
    LgConst<KIND, QT, D> kc;
    kc.load(w.par);
    const double* theta = w.par + LG_PAR_TH;
    // ---- test tile fields (centred on the light curve's first training input, as lg_setup).
    // Written out rather than through point_fields / param_layout: with nvcc 12.9 either form
    // raises the registers of lg_predict<1,1,2> from 104 to 107 and of <1,8,2> from 244 to 250.
    const double* xb = A.x + (size_t)b * A.n_max * D;
    const double* xs = PA.xstar + ((size_t)b * PA.m + (size_t)t * TS) * D;
    if (tid < TS) {
      const bool valid = t * TS + tid < PA.m;
#pragma unroll
      for (int dd = 0; dd < D; ++dd) {
        const double xc = valid ? (xs[(size_t)tid * D + dd] - xb[dd]) : 0.0;
        rowv[dd * TS + tid] = xc;
        if (dd < DS) {
#pragma unroll
          for (int q = 0; q < QT; ++q) {
            double sn = 0.0, cs = 1.0;
            if (valid && q < Q) sincospi(2.0 * theta[1 + Q + q * DS + dd] * xc, &sn, &cs);
            rowv[D * TS + ((dd * QT + q) * TS + tid) * 2] = cs;
            rowv[D * TS + ((dd * QT + q) * TS + tid) * 2 + 1] = sn;
          }
        }
      }
    }
    // ---- phase 1: K*^T_j tiles (rows = test points, k = training points of tile j) ----------
    double mu[4] = {0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < N; ++j) {
      __syncthreads();
      lg_prefetch_side<KIND, QT, D>(colv, w, npad, j, true);
      cp_async_commit();
      cp_async_wait<0>();
      __syncthreads();
      const double* al_c = colv + C::NFB * TS;
      double* kt = ks + (size_t)j * TT;
#pragma unroll 1
      for (int p8 = 0; p8 < 8; ++p8) {
        const int mi = p8 >> 1, ni2 = p8 & 1;
        const int r = frag_row(wm, mi, g), c0 = frag_col(wn, ni2, tq, 0);
        double kv[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int gc = j * TS + c0 + e;
          double k1 = k_entry<KIND, QT, D>(rowv, colv, r, c0 + e, kc.w, kc.a, kc.lam, tab);
          k1 = (gc < n && t * TS + r < PA.m) ? k1 : 0.0;
          kv[e] = k1;
          mu[mi] += k1 * al_c[c0 + e];
        }
        *reinterpret_cast<double2*>(kt + img(r, c0)) = make_double2(kv[0], kv[1]);
      }
    }
    fence_proxy_async();   // the K* tiles are read back by bulk copies
    // ---- phase 2: v_i^T = sum_{j<=i} K*^T_j X_ij^T,  vsq += row sums of v_i^T squared ---------
    double vs[4] = {0.0, 0.0, 0.0, 0.0};
    double acc[4][2][2];
    for (int i = 0; i < N; ++i) {
      zero_acc(acc);
      auto tA = [&](int kk) { return ks + (size_t)(i - kk) * TT; };
      auto tB = [&](int kk) { return lg_tile(w.tilesL, i, i - kk); };
      auto none = [&](int) { return (double*)nullptr; };
      gemm_stream<M_B_LE, false, 2>(acc, r2, i + 1, tA, tB, 0, 0, none, none, []() {});
#pragma unroll
      for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 2; ++ni) vs[mi] += acc[mi][ni][0] * acc[mi][ni][0] + acc[mi][ni][1] * acc[mi][ni][1];
    }
    // ---- reduce over the column lanes / warps; k** and outputs ------------------------------
    __syncthreads();
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      double a1 = mu[mi], a2 = vs[mi];
      a1 += shfl_xor_d(a1, 1); a1 += shfl_xor_d(a1, 2);
      a2 += shfl_xor_d(a2, 1); a2 += shfl_xor_d(a2, 2);
      if (tq == 0) {
        scr[wn * TS + frag_row(wm, mi, g)] = a1;
        scr[4 * TS + wn * TS + frag_row(wm, mi, g)] = a2;
      }
    }
    __syncthreads();
    if (tid < TS && t * TS + tid < PA.m) {
      const double m1 = (scr[tid] + scr[TS + tid]) + (scr[2 * TS + tid] + scr[3 * TS + tid]);
      const double v1 = (scr[4 * TS + tid] + scr[5 * TS + tid]) + (scr[6 * TS + tid] + scr[7 * TS + tid]);
      const double kss = k_entry<KIND, QT, D>(rowv, rowv, tid, tid, kc.w, kc.a, kc.lam, tab);
      mean_out[t * TS + tid] = theta[0] + m1;
      var_out[t * TS + tid] = kss - v1;
    }
  }
  if (tid == 0) bulk_wait_all();
}

}  // namespace pgm
