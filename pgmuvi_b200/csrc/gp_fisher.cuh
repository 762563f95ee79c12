// pgmuvi_b200 - expected (Fisher) information of the exact Gaussian log-likelihood on the staged
// engine: standard errors of fitted hyper-parameters.
//
//   l(theta) = log p(y | theta),  I_pq = 1/2 tr(K~^-1 dK~_p K~^-1 dK~_q),  I_cc = 1^T K~^-1 1
//   (constant mean c; the cross terms between c and the covariance slots are exactly 0).
//
// dK~_p = s_p C_c(p): C_k is derivative carrier k of k_grad_entry (weight 1), the learned noise's
// carrier is the identity, and c(p) / s_p are the carrier index and constant factor grad_slot
// applies.  With X = L^-1 (after the P and T phases of gp_large.cuh):
//
//   I_pq = 1/2 s_p s_q <B_p, B_q>_F,   B_s = X C_s X^T   (symmetric: lower tiles, off-diagonal x 2)
//
// One launch per stage, every launch carrying (light curve) x (tile) [x (carrier)] independent
// blocks on blockIdx.x / blockIdx.y = light curve; no block waits for another:
//   fs_carriers  C_s tile images of every used slot s = p - 1 (both (I, J) and (J, I): full square)
//   fs_xc        T_s(I, J) = sum_{K <= I} X_IK C_s(K, J)            lower tiles, DMMA tile engine
//   fs_xcx       B_s(I, J) = sum_{K <= J} T_s(I, K) X_JK^T          lower tiles, over the dead C_s
//   fs_gram      per tile: <B_p, B_q> of all pairs, fixed order
//   fs_ones      per tile row: || (X 1)_I ||^2                       (1^T K~^-1 1)
//   fs_finish    fixed-order sum over tiles, scales, [P, P] per light curve
// Slot 0 (mean) has no carrier; padded mixtures (q >= Q) have no slot and never enter.
#pragma once
#include "gp_large.cuh"

namespace pgm {

constexpr int FS_NC_MAX = 44;   // carriers per light curve (ARD 2-D SM-8 + learned noise: 41)
constexpr int FS_PAIRS_PER_THREAD = (FS_NC_MAX * (FS_NC_MAX + 1) / 2 + NTHREADS - 1) / NTHREADS;

// Workspace: the staged engine's (rounded up to 256 bytes), then per light curve
//   cb  [nc][N][N] tile images   C_s (full square), later B_s in the [nc][ntri] layout
//   t   [nc][ntri] tile images   T_s
//   gp  [ntri][nc (nc + 1) / 2]  per-tile Gram partials
//   up  [N]                      per-tile-row partials of 1^T K~^-1 1
// N = tile rows of n_max for every light curve of the batch (shorter ones use a prefix).
struct FisherWs {
  double *cb, *t, *gp, *up;
};
// rounded up to 32 doubles: every light curve's tile images start 256-byte aligned (bulk copies
// need 16-byte aligned global addresses)
__host__ __device__ inline size_t fisher_lc_elems(int n_max, int nc) {
  const size_t N = (n_max + TS - 1) / TS, ntri = N * (N + 1) / 2;
  const size_t e = (size_t)nc * (N * N + ntri) * TT + ntri * (size_t)(nc * (nc + 1) / 2) + N;
  return (e + 31) & ~(size_t)31;
}
__host__ __device__ inline size_t fisher_base_bytes(int n_max, int B) {
  return (large_ws_bytes(n_max, B) + 255) & ~(size_t)255;
}
__host__ __device__ inline size_t fisher_ws_bytes(int n_max, int B, int nc) {
  return fisher_base_bytes(n_max, B) + (size_t)B * fisher_lc_elems(n_max, nc) * sizeof(double);
}
__host__ __device__ inline FisherWs fisher_ws(double* ws, int n_max, int B, int nc, int b) {
  const size_t N = (n_max + TS - 1) / TS, ntri = N * (N + 1) / 2;
  FisherWs f;
  f.cb = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + fisher_base_bytes(n_max, B)) +
         (size_t)b * fisher_lc_elems(n_max, nc);
  f.t = f.cb + (size_t)nc * N * N * TT;
  f.gp = f.t + (size_t)nc * ntri * TT;
  f.up = f.gp + ntri * (size_t)(nc * (nc + 1) / 2);
  return f;
}

struct FisherArgs {
  int nc;           // carriers = P - 1
  double* fisher;   // [B, P, P]
};

// block -> (carrier s, lower tile (I, J)) of the product launches: tile-major, so that the blocks
// of one tile (same X operands) are adjacent in dispatch order
__device__ __forceinline__ void fs_job(int nc, int& s, int& I, int& J) {
  const int t = (int)(blockIdx.x / (unsigned)nc);
  s = (int)blockIdx.x - t * nc;
  tri_unrank(t, I, J);
}
__device__ __forceinline__ double* fs_sq(double* base, int N, int s, int I, int J) {
  return base + (((size_t)s * N + I) * N + J) * TT;
}
__device__ __forceinline__ double* fs_lo(double* base, int N, int s, int I, int J) {
  return base + ((size_t)s * (N * (N + 1) / 2) + ((size_t)I * (I + 1) / 2 + J)) * TT;
}

// slot of k_grad_entry carrier t (t == NG: the identity, learned noise), or -1 if it has none
template <int KIND, int QT, int D>
__device__ __forceinline__ int fs_slot_of(int t, int Q, const ParamLayout& L, bool learn_noise) {
  constexpr int DS = Cfg<KIND, QT, D>::DS, G0 = QT + 2 * QT * DS;
  if (t < QT) return (t < Q) ? 1 + t : -1;
  if (t < QT + QT * DS) return ((t - QT) / DS < Q) ? L.o_mu + (t - QT) : -1;
  if (t < G0) return ((t - QT - QT * DS) / DS < Q) ? L.o_sigma + (t - QT - QT * DS) : -1;
  if (t < Cfg<KIND, QT, D>::NG) return L.o_lam + (t - G0);
  return learn_noise ? L.o_noise : -1;
}

// constant factor s_p of slot p >= 1 (the factors grad_slot applies to the carriers)
template <int KIND, int QT, int D>
__device__ __forceinline__ double fs_scale(int p, const ParamLayout& L, const double* theta,
                                           const double* wq, const double* lamq) {
  constexpr int DS = Cfg<KIND, QT, D>::DS;
  if (p < L.o_mu) return 1.0;
  if (p < L.o_sigma) return -2.0 * M_PI * wq[(p - L.o_mu) / DS];
  if (p < L.o_noise) return -4.0 * M_PI * M_PI * theta[p] * wq[(p - L.o_sigma) / DS];
  if (p < L.o_lam) return 1.0;
  return lam_grad_factor<KIND>(p - L.o_lam, wq, lamq);
}

// ------------------------------------------------------------------------------------
// carrier tiles: block (tile (I, J), light curve); every entry of the 64x64 tile runs k_grad_entry
// once and writes the used carriers to C_s(I, J) and, off the diagonal, C_s(J, I)
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
struct FsCarrierSmem {
  using C = Cfg<KIND, QT, D>;
  static constexpr size_t BYTES = (size_t)(2 * C::NF * TS + EXP_TAB) * sizeof(double);
};
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS) fs_carriers(LargeArgs A, FisherArgs F) {
  using C = Cfg<KIND, QT, D>;
  extern __shared__ __align__(16) double sm[];
  double* rowv = sm;
  double* colv = sm + C::NF * TS;
  double* tab = colv + C::NF * TS;
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  int I, J;
  tri_unrank(blockIdx.x, I, J);
  if (I >= v.N) return;
  const LargeWs& w = v.w;
  const int n = v.n, Nm = (A.n_max + TS - 1) / TS;
  const bool learn_noise = (A.flags & PGM_FLAG_LEARN_NOISE) != 0;
  const ParamLayout L = param_layout(KIND, D, A.Q, learn_noise);
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, F.nc, v.b);
  load_exp_tab(tab);
  lg_prefetch_side<KIND, QT, D>(rowv, w, v.npad, I, false);
  lg_prefetch_side<KIND, QT, D>(colv, w, v.npad, J, false);
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  LgConst<KIND, QT, D> kc;
  kc.load(w.par);
  for (int idx = threadIdx.x; idx < TT; idx += NTHREADS) {
    const int r = idx >> 6, c = idx & 63;
    const int gi = I * TS + r, gj = J * TS + c;
    const bool valid = gi < n && gj < n;
    double ga[C::NG];
#pragma unroll
    for (int t = 0; t < C::NG; ++t) ga[t] = 0.0;
    k_grad_entry<KIND, QT, D>(rowv, colv, r, c, kc.w, kc.a, kc.lam, tab, 1.0, ga);
#pragma unroll
    for (int t = 0; t <= C::NG; ++t) {
      const int p = fs_slot_of<KIND, QT, D>(t, A.Q, L, learn_noise);
      if (p < 1) continue;
      double val = (t < C::NG) ? ga[t < C::NG ? t : 0] : (gi == gj ? 1.0 : 0.0);
      val = valid ? val : 0.0;
      fs_sq(f.cb, Nm, p - 1, I, J)[img(r, c)] = val;
      if (I != J) fs_sq(f.cb, Nm, p - 1, J, I)[img(c, r)] = val;
    }
  }
  fence_proxy_async();   // the tiles are read by bulk copies of the next launch
}

// ------------------------------------------------------------------------------------
// the two triangular tile products per carrier (tilesL holds the row-major X tiles after
// lg_transpose, X_jj in the diagonal slots)
// ------------------------------------------------------------------------------------
constexpr size_t FS_PROD_SMEM = (size_t)(STAGE_ELEMS + 8) * sizeof(double);

// acc of the product, then the tile out of stage 0 by one bulk store
template <int MODE0, typename FA, typename FB>
__device__ __forceinline__ void fs_product(double* sm, int nk, FA tA, FB tB, double* out) {
  const unsigned bars = smem_u32(sm + STAGE_ELEMS);
  lg_ring_init(bars);
  __syncthreads();
  Ring r2{bars, bars + 16, sm, 0};
  double acc[4][2][2];
  zero_acc(acc);
  auto none = [&](int) { return (double*)nullptr; };
  gemm_stream<MODE0, false, 2>(acc, r2, nk, tA, tB, 0, 0, none, none, []() {});
  store_tile_bulk(acc, sm, out, 1.0);
  if (threadIdx.x == 0) bulk_wait_all();
}

// T_s(I, J) = sum_{K <= I} X_IK C_s(K, J);  k-tile kk <-> K = I - kk (X_II lower: M_A_LE)
static __global__ void __launch_bounds__(NTHREADS, 2) fs_xc(LargeArgs A, FisherArgs F) {
  extern __shared__ __align__(16) double sm[];
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  int s, I, J;
  fs_job(F.nc, s, I, J);
  if (I >= v.N) return;
  const int Nm = (A.n_max + TS - 1) / TS;
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, F.nc, v.b);
  double* tilesL = v.w.tilesL;
  // C_s(K, J) as the B operand [n][k] is the row-major image of C_s(J, K) (C_s symmetric)
  fs_product<M_A_LE>(sm, I + 1, [&](int kk) { return lg_tile(tilesL, I, I - kk); },
                     [&](int kk) { return fs_sq(f.cb, Nm, s, J, I - kk); }, fs_lo(f.t, Nm, s, I, J));
}

// B_s(I, J) = sum_{K <= J} T_s(I, K) X_JK^T;  k-tile kk <-> K = J - kk (X_JJ lower: M_B_LE)
static __global__ void __launch_bounds__(NTHREADS, 2) fs_xcx(LargeArgs A, FisherArgs F) {
  extern __shared__ __align__(16) double sm[];
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  int s, I, J;
  fs_job(F.nc, s, I, J);
  if (I >= v.N) return;
  const int Nm = (A.n_max + TS - 1) / TS;
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, F.nc, v.b);
  double* tilesL = v.w.tilesL;
  fs_product<M_B_LE>(sm, J + 1, [&](int kk) { return fs_lo(f.t, Nm, s, I, J - kk); },
                     [&](int kk) { return lg_tile(tilesL, J, J - kk); }, fs_lo(f.cb, Nm, s, I, J));
}

// ------------------------------------------------------------------------------------
// Gram partials of tile (I, J): <B_p(I, J), B_q(I, J)> for every pair p >= q (pair index
// p (p + 1) / 2 + q), 64 entries of all carriers at a time through shared memory; each thread owns
// fixed pairs and sums its entries in a fixed order.  Off-diagonal tiles count twice.
// ------------------------------------------------------------------------------------
constexpr int FS_CHUNK = 64, FS_LDC = FS_CHUNK + 1;
static __global__ void __launch_bounds__(NTHREADS) fs_gram(LargeArgs A, FisherArgs F) {
  __shared__ double buf[FS_NC_MAX * FS_LDC];
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  int I, J;
  const int t = (int)blockIdx.x;
  tri_unrank(t, I, J);
  if (I >= v.N) return;
  const int nc = F.nc, npair = nc * (nc + 1) / 2, Nm = (A.n_max + TS - 1) / TS;
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, nc, v.b);
  const int tid = threadIdx.x;
  int pp[FS_PAIRS_PER_THREAD], pq[FS_PAIRS_PER_THREAD];
  double acc[FS_PAIRS_PER_THREAD];
#pragma unroll
  for (int k = 0; k < FS_PAIRS_PER_THREAD; ++k) {
    const int pi = tid + k * NTHREADS;
    int a = 0, b = 0;
    if (pi < npair) tri_unrank(pi, a, b);
    pp[k] = a * FS_LDC;
    pq[k] = b * FS_LDC;
    acc[k] = 0.0;
  }
  for (int e0 = 0; e0 < TT; e0 += FS_CHUNK) {
    __syncthreads();
    for (int i = tid; i < nc * FS_CHUNK; i += NTHREADS) {
      const int s = i / FS_CHUNK, e = i - s * FS_CHUNK;
      buf[s * FS_LDC + e] = fs_lo(f.cb, Nm, s, I, J)[e0 + e];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < FS_PAIRS_PER_THREAD; ++k) {
      if (tid + k * NTHREADS >= npair) break;
      double a = acc[k];
#pragma unroll 8
      for (int e = 0; e < FS_CHUNK; ++e) a = fma(buf[pp[k] + e], buf[pq[k] + e], a);
      acc[k] = a;
    }
  }
  const double wgt = (I == J) ? 1.0 : 2.0;
#pragma unroll
  for (int k = 0; k < FS_PAIRS_PER_THREAD; ++k) {
    const int pi = tid + k * NTHREADS;
    if (pi < npair) f.gp[(size_t)t * npair + pi] = wgt * acc[k];
  }
}

// ------------------------------------------------------------------------------------
// 1^T K~^-1 1 = || X 1 ||^2 (1 on the n valid points): block (tile row I, light curve) sums the
// squares of its 64 row sums in a fixed order into up[I]
// ------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(NTHREADS) fs_ones(LargeArgs A, FisherArgs F) {
  __shared__ double red[TS];
  const LcView v = lc_view(A);
  if (v.st.state[v.b] != LG_FACTORED) return;
  const int I = blockIdx.x;
  if (I >= v.N) return;
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, F.nc, v.b);
  const int tid = threadIdx.x, r = tid >> 2, part = tid & 3;
  double u = 0.0;
  for (int K = 0; K <= I; ++K) {
    const double* xt = lg_tile(v.w.tilesL, I, K);
    for (int c = part; c < TS; c += 4)
      if (K * TS + c < v.n) u += xt[img(r, c)];
  }
  u += shfl_xor_d(u, 1);
  u += shfl_xor_d(u, 2);
  if (part == 0) red[r] = u * u;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int k = 0; k < TS; ++k) s += red[k];
    f.up[I] = s;
  }
}

// ------------------------------------------------------------------------------------
// [P, P] of one light curve: fixed-order sums over its tiles, I_pq = 1/2 s_p s_q G_pq,
// I_00 = 1^T K~^-1 1, I_0p = 0; NaN rows for a light curve whose Cholesky failed
// ------------------------------------------------------------------------------------
template <int KIND, int QT, int D>
__global__ void __launch_bounds__(NTHREADS) fs_finish(LargeArgs A, FisherArgs F) {
  __shared__ double sc[64];
  const LcView v = lc_view(A);
  const ParamLayout L = param_layout(KIND, D, A.Q, (A.flags & PGM_FLAG_LEARN_NOISE) != 0);
  const int P = L.P, tid = threadIdx.x;
  double* out = F.fisher + (size_t)v.b * P * P;
  if (v.st.state[v.b] != LG_FACTORED) {
    for (int i = tid; i < P * P; i += NTHREADS) out[i] = nan("");
    return;
  }
  const double* par = v.w.par;
  if (tid >= 1 && tid < P)
    sc[tid] = fs_scale<KIND, QT, D>(tid, L, par + LG_PAR_TH, par + LG_PAR_WQ, par + LG_PAR_LM);
  __syncthreads();
  const int nc = F.nc, npair = nc * (nc + 1) / 2;
  const int ntri = v.N * (v.N + 1) / 2;
  const FisherWs f = fisher_ws(A.ws, A.n_max, A.B, nc, v.b);
  for (int pi = tid; pi < npair; pi += NTHREADS) {
    double g = 0.0;
    for (int t = 0; t < ntri; ++t) g += f.gp[(size_t)t * npair + pi];
    int a, b;
    tri_unrank(pi, a, b);
    const double val = 0.5 * sc[a + 1] * sc[b + 1] * g;
    out[(a + 1) * P + (b + 1)] = val;
    out[(b + 1) * P + (a + 1)] = val;
  }
  if (tid == 0) {
    double s = 0.0;
    for (int I = 0; I < v.N; ++I) s += f.up[I];
    out[0] = s;
  }
  if (tid >= 1 && tid < P) {
    out[tid] = 0.0;
    out[tid * P] = 0.0;
  }
}

}  // namespace pgm
