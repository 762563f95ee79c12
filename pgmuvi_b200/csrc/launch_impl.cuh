// Host launchers of the fused kernels; explicitly instantiated per (KIND, QT, D) in inst.cu so
// the heavy kernels compile in parallel translation units.
#pragma once
#include "gp_fused.cuh"
#include "gp_large.cuh"
#include "gp_large_tc.cuh"
#include "gp_fisher.cuh"
#include <algorithm>
#include <cstdlib>
#include <string>

namespace pgm {
int fail(const std::string& m);
int cuda_fail(const char* what, cudaError_t e);
int device_sms();
inline int predict_blocks() { return 2 * device_sms(); }   // persistent blocks of lg_predict

// the per-light-curve arguments inside a fused kernel's argument block
inline EvalArgs& eval_args(EvalArgs& A) { return A; }
inline EvalArgs& eval_args(FitArgs& F) { return F.e; }

// Persistent launch of a fused kernel: as many blocks as are resident at once, at most one per light
// curve.  The ticket scheduler (sched) runs only on the full grid of two blocks per SM it is built
// for; every other grid takes the light curves at a fixed stride.
template <typename Args>
int launch_persistent(void (*kern)(Args), Args args, size_t smem, const char* what, cudaStream_t st) {
  EvalArgs& A = eval_args(args);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute", e);
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NTHREADS, smem);
  if (e != cudaSuccess) return cuda_fail("occupancy", e);
  if (occ < 1) return fail("kernel does not fit on an SM");
  A.sms = device_sms();
  int grid = A.sms * occ;
  if (grid > A.B) grid = A.B;
  if (A.sched && (occ != 2 || grid != 2 * A.sms || getenv("PGM_STATIC_STRIDE"))) A.sched = nullptr;
  if (A.sched) cudaMemsetAsync(A.sched, 0, PGM_SCHED_INTS * sizeof(int), st);
  kern<<<grid, NTHREADS, smem, st>>>(args);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(what, e);
  return 0;
}

template <int KIND, int QT, int D>
int launch_eval(const EvalArgs& A, cudaStream_t st) {
  return launch_persistent(sm_mll_grad_kernel<KIND, QT, D>, A, Cfg<KIND, QT, D>::F_BYTES,
                           "sm_mll_grad_kernel launch", st);
}

template <int KIND, int QT, int D>
int launch_fit(const FitArgs& F, cudaStream_t st) {
  return launch_persistent(sm_fit_kernel<KIND, QT, D>, F, Cfg<KIND, QT, D>::F_BYTES,
                           "sm_fit_kernel launch", st);
}

template <int KIND, int QT, int D>
int launch_dense(const pgm::EvalArgs& A, double* K, cudaStream_t st) {
  const int N = (A.n_max + pgm::TS - 1) / pgm::TS;
  if (A.B > 65535) return fail("sm_kernel_dense: at most 65535 light curves per call");
  auto kern = pgm::sm_kernel_dense_kernel<KIND, QT, D>;
  const size_t smem = pgm::DenseSmem<KIND, QT, D>::BYTES;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(sm_kernel_dense_kernel)", e);
  dim3 grid(N * (N + 1) / 2, A.B);
  kern<<<grid, pgm::NTHREADS, smem, st>>>(A, K);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("sm_kernel_dense_kernel launch", e);
  return 0;
}


// Staged engine (gp_large.cuh): B light curves advance stage by stage, one launch per
// dependency stage with B x (tiles of the stage) blocks; B = 1 is the single large GP.
// Host-orchestrated on `st`; synchronises once per Cholesky pass to read how many light curves
// must repeat it with more jitter (psd_safe_cholesky's ladder) - the call is blocking.
template <int KIND, int QT, int D>
int launch_large(const pgm::LargeArgs& A, int want_grad, cudaStream_t st, int predict_only = 0) {
  using C = pgm::Cfg<KIND, QT, D>;
  using namespace pgm;
  const int n = A.n_max, N = (n + TS - 1) / TS, npad = N * TS, B = A.B;
  if (B > 65535) return fail("staged engine: B > 65535 (split the batch)");
  // tile columns per panel (one right-looking trailing update every NB columns): wider panels
  // amortise the C-tile round trip of the trailing update once there are enough tile rows to
  // keep the in-panel launches busy (B200, C4: NB 8 -> 32 takes the P phase from 497 to 416 ms)
  int NB = (N <= 64) ? 8 : (N <= 256) ? 16 : 32;
  if (const char* f = getenv("PGM_STAGED_NB")) NB = std::max(1, atoi(f));
  auto k_upd = lg_update<KIND, QT, D>;
  auto k_grad = lg_grad<KIND, QT, D>;
  auto k_chol = lg_chol_all<KIND, QT, D>;
  cudaError_t e;
  constexpr size_t UPD_SMEM = UpdSmem<KIND, QT, D>::BYTES;
  e = cudaFuncSetAttribute(k_upd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UPD_SMEM);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_update)", e);
  constexpr size_t CHOL_SMEM = CholAllSmem<KIND, QT, D>::BYTES;
  e = cudaFuncSetAttribute(k_chol, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CHOL_SMEM);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_chol_all)", e);
  constexpr size_t GRAD_SMEM = GradSmem<KIND, QT, D>::BYTES;
  e = cudaFuncSetAttribute(k_grad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GRAD_SMEM);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_grad)", e);
  e = cudaFuncSetAttribute(lg_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_DIAG_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(lg_trsm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_TRSM_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(lg_inv_row, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_INV_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(lg_inv_all, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG_INV_SMEM);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(staged engine kernels)", e);
  BatchState bs = make_batch_state(A.ws, n, B);
  cudaMemsetAsync(bs.state, 0, (size_t)(4 * B + 4) * sizeof(int), st);
  const dim3 blk(NTHREADS);
  for (int pass = 0; pass <= 3; ++pass) {
    cudaMemsetAsync(bs.count, 0, 4 * sizeof(int), st);   // [0] repeat count, [1] / [2] job tickets
    lg_setup<KIND, QT, D><<<dim3((npad + NTHREADS - 1) / NTHREADS, B), blk, 0, st>>>(A);
    const long long ncb = (long long)(N * (N + 1) / 2) * B;
    // up to PGM_STAGED_CHOL_ALL_N tile rows (default 200) the left-looking one-launch schedule
    // wins (no launch latencies, potrf overlapped: n=2048 1.62 -> 1.16 ms, C3 11.8 -> 8.6 ms); the
    // two meet at N = 256 (63.1 vs 64.4 ms) and beyond the panel scheme's operand reuse in L2
    // wins (C4: 425 vs 500 ms)
    int all_n = 200;
    if (const char* f = getenv("PGM_STAGED_CHOL_ALL_N")) all_n = atoi(f);
    // ... and only while a dependency stage cannot fill the device by itself: big batches have
    // all the parallelism they need in one launch per stage (C5: 52.8 vs 62.9 ms)
    const bool few = (long long)B * N < 1024;
    const bool one_launch = few && N <= all_n && ncb <= 2147483647LL;
    if (one_launch) {   // dataflow Cholesky: the whole pass in one flag-ordered launch
      cudaMemsetAsync(bs.tflag, 0, (size_t)B * large_ntri(n) * sizeof(int), st);
      k_chol<<<dim3((unsigned)ncb), blk, CHOL_SMEM, st>>>(A);
    }
    for (int J0 = 0; J0 < N && !one_launch; J0 += NB) {
      const int J1 = std::min(J0 + NB, N);
      const int build = (J0 == 0) ? 1 : 0;
      for (int j = J0; j < J1; ++j) {
        if (build || j > J0)
          k_upd<<<dim3(N - j, B), blk, UPD_SMEM, st>>>(A, 0, j, J0, j, build);
        lg_diag<<<dim3(1, B), blk, LG_DIAG_SMEM, st>>>(A, j);
        if (j + 1 < N) lg_trsm<<<dim3(N - j - 1, B), blk, LG_TRSM_SMEM, st>>>(A, j);
      }
      if (J1 < N && (A.flags & PGM_FLAG_TF32X3_CHOL) && !(J1 & 1)) {
        // trailing update on tcgen05 (3xTF32): pack the panel's L tiles, one CTA per 128x128 tile
        constexpr size_t TC_SMEM = TcGradSmem<KIND, QT, D>::BYTES;
        auto k_utc = lg_update_tc<KIND, QT, D>;
        e = cudaFuncSetAttribute(k_utc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM);
        if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_update_tc)", e);
        const int NT = (N + 1) / 2, Mt = NT - J1 / 2;
        lg_pack_panel_tf32<<<dim3(J1 - J0, 2 * NT - J1, B), blk, 0, st>>>(A, J0, J1);
        k_utc<<<dim3(tc_grid(Mt), B), TC_THREADS, TC_SMEM, st>>>(A, J0, J1, build);
      } else if (J1 < N) {
        const int M = N - J1;
        k_upd<<<dim3(M * (M + 1) / 2, B), blk, UPD_SMEM, st>>>(A, 1, J1, J0, J1, build);
      }
    }
    lg_ladder<<<(B + 255) / 256, 256, 0, st>>>(A);
    if (A.flags & PGM_FLAG_NOSYNC) {
      // no host round trip: all four ladder passes are enqueued; for a light curve that is already
      // factored (or failed) every kernel of a later pass returns at once
      if (!one_launch) return fail("PGM_FLAG_NOSYNC needs the one-launch schedule (B * N < 1024, N <= 200)");
      continue;
    }
    int again = 0;
    e = cudaMemcpyAsync(&again, bs.count, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail("staged engine, Cholesky phase", e);
    if (!again) break;
  }
  if (want_grad || predict_only) {
    if ((long long)B * N >= 1024) {            // one launch per tile row
      for (int i = 1; i < N; ++i) lg_inv_row<<<dim3(i, B), blk, LG_INV_SMEM, st>>>(A, i);
    } else if (N > 1) {                        // whole T phase in one launch, flag-ordered
      cudaMemsetAsync(bs.tflag, 0, (size_t)B * large_ntri(n) * sizeof(int), st);
      cudaMemsetAsync(bs.count + 2, 0, sizeof(int), st);
      const long long nblk = (long long)(N * (N - 1) / 2) * B;
      if (nblk > 2147483647LL) return fail("staged engine: too many tiles x light curves");
      lg_inv_all<<<dim3((unsigned)nblk), blk, LG_INV_SMEM, st>>>(A);
    }
    lg_alpha<<<dim3(N, B), blk, 0, st>>>(A);
    if (!predict_only && (A.flags & PGM_FLAG_TF32X3)) {
      // G phase on tcgen05: X^T -> packed TF32 hi / lo operand images, then one CTA per 128x128
      // tile of K~^-1 (3xTF32 products in tensor memory, FP64 contraction epilogue)
      const int NT = (N + 1) / 2;
      constexpr size_t TC_SMEM = TcGradSmem<KIND, QT, D>::BYTES;
      auto k_tc = lg_grad_tc<KIND, QT, D>;
      e = cudaFuncSetAttribute(k_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM);
      if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_grad_tc)", e);
      lg_pack_tf32<<<dim3(N, 2 * NT, B), blk, 0, st>>>(A);
      k_tc<<<dim3(tc_grid(NT), B), TC_THREADS, TC_SMEM, st>>>(A);
    } else if (!predict_only) {
      k_grad<<<dim3(N * (N + 1) / 2, B), blk, GRAD_SMEM, st>>>(A);
    }
  }
  if (predict_only) {
    lg_transpose<<<dim3(N * (N + 1) / 2, B), blk, 0, st>>>(A);
  } else {
    lg_finish<KIND, QT, D><<<dim3(1, B), blk, 0, st>>>(A, want_grad);
  }
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("staged engine launch", e);
  return 0;
}

// N1: posterior prediction = P + T phases of the staged engine, then lg_predict (persistent
// blocks over (light curve, test tile) jobs, each with its own K* panel scratch).
template <int KIND, int QT, int D>
int launch_predict(const pgm::PredictArgs& PA0, cudaStream_t st) {
  using C = pgm::Cfg<KIND, QT, D>;
  using namespace pgm;
  PredictArgs PA = PA0;
  if (int r = launch_large<KIND, QT, D>(PA.a, 0, st, 1)) return r;
  auto kern = lg_predict<KIND, QT, D>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)C::SMEM_BYTES);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(lg_predict)", e);
  const int Mt = (PA.m + TS - 1) / TS;
  int grid = predict_blocks();
  const long long jobs = (long long)PA.a.B * Mt;
  if (jobs < grid) grid = (int)jobs;
  if (grid < 1) return 0;
  kern<<<grid, NTHREADS, C::SMEM_BYTES, st>>>(PA);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("lg_predict launch", e);
  return 0;
}

// Fisher information = P + T phases of the staged engine (X = L^-1, row-major in tilesL), then one
// launch per stage of gp_fisher.cuh.  The caller has checked the grid sizes (pgm_sm_fisher_f64).
template <int KIND, int QT, int D>
int launch_fisher(const pgm::LargeArgs& A, const pgm::FisherArgs& F, cudaStream_t st) {
  using namespace pgm;
  if (int r = launch_large<KIND, QT, D>(A, 0, st, 1)) return r;
  const int N = (A.n_max + TS - 1) / TS, ntri = N * (N + 1) / 2, B = A.B;
  auto k_car = fs_carriers<KIND, QT, D>;
  constexpr size_t CAR_SMEM = FsCarrierSmem<KIND, QT, D>::BYTES;
  cudaError_t e = cudaFuncSetAttribute(k_car, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAR_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(fs_xc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_PROD_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(fs_xcx, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_PROD_SMEM);
  if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute(fisher kernels)", e);
  const dim3 blk(NTHREADS);
  k_car<<<dim3(ntri, B), blk, CAR_SMEM, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_carriers launch", e);
  fs_xc<<<dim3((unsigned)(ntri * F.nc), B), blk, FS_PROD_SMEM, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_xc launch", e);
  fs_xcx<<<dim3((unsigned)(ntri * F.nc), B), blk, FS_PROD_SMEM, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_xcx launch", e);
  fs_gram<<<dim3(ntri, B), blk, 0, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_gram launch", e);
  fs_ones<<<dim3(N, B), blk, 0, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_ones launch", e);
  fs_finish<KIND, QT, D><<<dim3(1, B), blk, 0, st>>>(A, F);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail("fs_finish launch", e);
  return 0;
}

}  // namespace pgm
