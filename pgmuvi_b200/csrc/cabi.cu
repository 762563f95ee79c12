// C ABI of pgmuvi_b200 (see include/pgmuvi_b200.h).  Host-side dispatch only; all device
// code is in gp_fused.cuh.
#include "gp_fused.cuh"
#include "gp_large.cuh"
#include "gp_large_tc.cuh"
#include "gp_fisher.cuh"
#include "lombscargle.cuh"
#include "../../include/pgmuvi_b200.h"

#include <algorithm>
#include <cstdio>
#include <cmath>
#include <initializer_list>
#include <string>

namespace pgm {
// launchers are explicitly instantiated in inst.cu (one translation unit per config)
template <int KIND, int QT, int D> int launch_eval(const EvalArgs& A0, cudaStream_t st);
template <int KIND, int QT, int D> int launch_fit(const FitArgs& F, cudaStream_t st);
template <int KIND, int QT, int D> int launch_dense(const EvalArgs& A, double* K, cudaStream_t st);
template <int KIND, int QT, int D>
int launch_large(const LargeArgs& A, int want_grad, cudaStream_t st, int predict_only);
template <int KIND, int QT, int D> int launch_predict(const PredictArgs& PA, cudaStream_t st);
template <int KIND, int QT, int D>
int launch_fisher(const LargeArgs& A, const FisherArgs& F, cudaStream_t st);

thread_local std::string g_err;
int fail(const std::string& m) {
  g_err = m;
  return -1;
}
int cuda_fail(const char* what, cudaError_t e) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return -2;
}
int device_sms() {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms > 0 ? sms : 148;
}
}  // namespace pgm

namespace pgm {
__global__ void optim_step_kernel(double* raw, const double* grad_mll, double* m, double* v,
                                  const int32_t* active, int B, int P, int kind, double lr,
                                  double b1, double b2, double eps, double wd, double bc1,
                                  double bc2s) {
  // HBM-bound: 4 reads + 3 writes of 8 bytes per parameter; the bias corrections (two pow per
  // step) come from the host so that no transcendental is left in the kernel
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * P) return;
  if (active && !active[idx / P]) return;
  double mm = m ? m[idx] : 0.0, vv = v ? v[idx] : 0.0;
  raw[idx] = optim_update_bc(raw[idx], -grad_mll[idx], mm, vv, kind, lr, b1, b2, eps, wd, bc1, bc2s);
  if (m) m[idx] = mm;
  if (v) v[idx] = vv;
}


// fp32 <-> fp64 staging of the _f32 entry points (fp32 storage, fp64 arithmetic)
__global__ void widen_kernel(const float* __restrict__ src, double* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    dst[i] = (double)src[i];
}
__global__ void narrow_kernel(const double* __restrict__ src, float* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    dst[i] = (float)src[i];
}
}  // namespace pgm

namespace {
using pgm::cuda_fail;
using pgm::fail;
using pgm::launch_dense;
using pgm::launch_eval;
using pgm::launch_fit;
using pgm::launch_large;
using pgm::launch_predict;
using pgm::launch_fisher;

// NF of the instantiated config serving (d, Q): sizes the workspace (upper bound over kinds)
int nf_for(int d, int Q) { return d + 2 * d * (Q <= 4 ? 4 : 8) + 1; }  // Q = 0 -> QT = 4

// one row per compiled instantiation (configs.h): its launchers and the resident fused blocks per SM
struct Config {
  int kind, qt, d;
  int (*eval)(const pgm::EvalArgs&, cudaStream_t);
  int (*fit)(const pgm::FitArgs&, cudaStream_t);
  int (*dense)(const pgm::EvalArgs&, double*, cudaStream_t);
  int (*large)(const pgm::LargeArgs&, int, cudaStream_t, int);
  int (*predict)(const pgm::PredictArgs&, cudaStream_t);
  int (*fisher)(const pgm::LargeArgs&, const pgm::FisherArgs&, cudaStream_t);
  int fused_blocks_per_sm;
};
#define PGM_CONFIG(KIND, QT, D)                                                              \
  {KIND, QT, D, launch_eval<KIND, QT, D>, launch_fit<KIND, QT, D>, launch_dense<KIND, QT, D>, \
   launch_large<KIND, QT, D>, launch_predict<KIND, QT, D>, launch_fisher<KIND, QT, D>,       \
   pgm::Cfg<KIND, QT, D>::F_BYTES <= 113 * 1024 ? 2 : 1},
const Config kConfigs[] = {
#include "configs.h"
};
#undef PGM_CONFIG

const Config* reject(const char* why) {
  fail(why);
  return nullptr;
}

// Validates a model and returns the compiled instantiation that serves it: the row of its kind with
// the smallest QT >= max(Q, 1).  Null (and pgm_last_error set) if the model is rejected.
const Config* check_common(int B, int n_max, int d, int Q, int kernel_kind) {
  if (B < 0 || n_max < 1) return reject("B must be >= 0 and n_max >= 1");
  if (kernel_kind >= PGM_KIND_STAT_BASE && kernel_kind <= PGM_KIND_STAT(5, 0)) {
    if (Q != 0) return reject("stationary kinds have no mixtures: pass Q == 0");
    const int wk = (kernel_kind - PGM_KIND_STAT_BASE) % 5;
    if ((kernel_kind - PGM_KIND_STAT_BASE) / 5 >= 3 && wk != 0)
      return reject("time kernels 3..5 exist for 1-D models only (wk = 0)");
    if (d != (wk == 0 ? 1 : 2))
      return reject("stationary kind / d mismatch (d = 1 without, 2 with a wavelength kernel)");
  } else {
    if (Q < 1 || Q > 8) return reject("Q (num_mixtures) must be in 1..8");
    if (kernel_kind == PGM_KIND_SM1D && d != 1) return reject("PGM_KIND_SM1D needs d == 1");
    if ((kernel_kind == PGM_KIND_SM_ARD_PRODSUM || kernel_kind == PGM_KIND_SM_ARD_SUMPROD) && d != 2)
      return reject("ARD spectral-mixture kinds need d == 2");
    if (kernel_kind >= PGM_KIND_SEP_RBF && kernel_kind <= PGM_KIND_SEP_CONST && d != 2)
      return reject("separable kinds need d == 2 (time, wavelength)");
  }
  const Config* best = nullptr;
  for (const Config& c : kConfigs)
    if (c.kind == kernel_kind && c.qt >= std::max(Q, 1) && (!best || c.qt < best->qt)) best = &c;
  return best ? best : reject("unknown kernel_kind");
}

int check_ptrs(std::initializer_list<const void*> ptrs) {
  for (const void* p : ptrs)
    if (!p) return fail("null pointer argument");
  return 0;
}

// the members EvalArgs and LargeArgs share: the model's inputs, its info output and the workspace
template <typename Args>
Args model_args(const double* x, const int32_t* n_valid, const double* y,
                const double* fixed_noise, const double* raw, const int32_t* con_kind,
                const double* con_lb, const double* con_ub, int B, int n_max, int Q, int flags,
                int32_t* info, void* workspace) {
  Args A{};
  A.x = x; A.n_valid = n_valid; A.y = y; A.fixed_noise = fixed_noise; A.raw = raw;
  A.con_kind = con_kind; A.con_lb = con_lb; A.con_ub = con_ub;
  A.B = B; A.n_max = n_max; A.Q = Q; A.flags = flags;
  A.info = info; A.ws = static_cast<double*>(workspace);
  return A;
}


// number of packed raw parameters of a model (layout in include/pgmuvi_b200.h)
int host_param_count(int d, int Q, int kernel_kind, int flags) {
  return pgm::param_layout(kernel_kind, d, Q, (flags & PGM_FLAG_LEARN_NOISE) != 0).P;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// the fused kernels' workspace (pgm_workspace_bytes): per-block scratch, then the light-curve
// ticket counters at its tail
int fused_ws(pgm::EvalArgs& A, int d, size_t workspace_bytes) {
  const size_t need = pgm_workspace_bytes(8, A.n_max, d, A.Q, -1);
  if (workspace_bytes < need) return fail("workspace too small (see pgm_workspace_bytes)");
  A.ws_per_block = pgm::scratch_elems(A.n_max, nf_for(d, A.Q));
  A.sched = reinterpret_cast<int*>(reinterpret_cast<char*>(A.ws) + need -
                                   pgm::PGM_SCHED_INTS * sizeof(int));
  return 0;
}

// fp64 staging area of the _f32 entry points, carved from the tail of the workspace
struct Stage32 {
  double *x, *y, *fn, *raw, *lb, *ub, *mll, *grad, *loss, *hist;
  size_t bytes;
};
Stage32 carve32(char* base, int B, int n_max, int d, int P, bool bounds_per_lc, int maxiter,
                bool want_hist) {
  Stage32 s;
  size_t off = 0;
  auto take = [&](size_t elems) {
    double* p = base ? reinterpret_cast<double*>(base + off) : nullptr;
    off += align256(elems * sizeof(double));
    return p;
  };
  const size_t Bn = (size_t)B * n_max, BP = (size_t)B * P;
  s.x = take(Bn * d); s.y = take(Bn); s.fn = take(Bn); s.raw = take(BP);
  s.lb = take(bounds_per_lc ? BP : (size_t)P); s.ub = take(bounds_per_lc ? BP : (size_t)P);
  s.mll = take((size_t)B); s.grad = take(BP);
  s.loss = take((size_t)maxiter * B);
  s.hist = take(want_hist ? (size_t)(maxiter + 1) * BP : 0);
  s.bytes = off;
  return s;
}
void widen(const float* src, double* dst, size_t n, cudaStream_t st) {
  if (!n || !src) return;
  const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 8);
  pgm::widen_kernel<<<blocks, 256, 0, st>>>(src, dst, n);
}
void narrow(const double* src, float* dst, size_t n, cudaStream_t st) {
  if (!n || !dst) return;
  const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 8);
  pgm::narrow_kernel<<<blocks, 256, 0, st>>>(src, dst, n);
}

// the arrays of an _f32 entry point: inputs, and the outputs it returns (null: none)
struct Io32 {
  const float *x, *y, *fixed_noise, *raw, *con_lb, *con_ub;
  float *mll, *grad, *raw_out, *loss, *hist;
};

// An _f32 entry point on an fp64 one (fp32 storage, fp64 arithmetic), for a call its caller has
// validated up to the workspace size.  The fp64 entry's workspace (f64_bytes, rounded up to 256)
// comes first, the staging area (pgm_f32_staging_bytes) behind it.  The inputs are widened into
// the staging area, f64(staged, rounded f64_bytes) runs the fp64 entry on them, and the outputs
// are narrowed back.
template <typename F64>
int stage_f32(const Io32& io, int B, int n_max, int d, int Q, int kernel_kind, int flags,
              int maxiter, size_t f64_bytes, const char* f64_ws, void* workspace,
              size_t workspace_bytes, void* stream, F64 f64) {
  const size_t base = align256(f64_bytes);
  if (workspace_bytes < base + pgm_f32_staging_bytes(B, n_max, d, Q, kernel_kind, flags, maxiter,
                                                     io.hist != nullptr))
    return fail(std::string("workspace too small (") + f64_ws +
                " rounded up to 256 + pgm_f32_staging_bytes)");
  const int P = host_param_count(d, Q, kernel_kind, flags);
  const bool per_lc = (flags & PGM_FLAG_BOUNDS_PER_LC) != 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Stage32 s = carve32(static_cast<char*>(workspace) + base, B, n_max, d, P, per_lc, maxiter,
                      io.hist != nullptr);
  const size_t Bn = (size_t)B * n_max, BP = (size_t)B * P, nb = per_lc ? BP : (size_t)P;
  widen(io.x, s.x, Bn * d, st); widen(io.y, s.y, Bn, st); widen(io.fixed_noise, s.fn, Bn, st);
  widen(io.raw, s.raw, BP, st); widen(io.con_lb, s.lb, nb, st); widen(io.con_ub, s.ub, nb, st);
  if (!io.fixed_noise) s.fn = nullptr;
  if (!io.grad) s.grad = nullptr;
  if (!io.hist) s.hist = nullptr;
  if (int r = f64(s, base)) return r;
  narrow(s.mll, io.mll, (size_t)B, st); narrow(s.grad, io.grad, BP, st);
  narrow(s.raw, io.raw_out, BP, st); narrow(s.loss, io.loss, (size_t)maxiter * B, st);
  narrow(s.hist, io.hist, (size_t)(maxiter + 1) * BP, st);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("f32 staging", e);
  return 0;
}

}  // namespace

extern "C" {

int pgm_version(void) { return 101; }
const char* pgm_last_error(void) { return pgm::g_err.c_str(); }

size_t pgm_workspace_bytes(int elem_size, int n_max, int d, int Q, int device) {
  (void)elem_size;
  int sms = 148;
  if (device >= 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  else { int dv = 0; if (cudaGetDevice(&dv) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dv); }
  if (sms <= 0) sms = 148;
  const size_t per_block = pgm::scratch_elems(n_max, nf_for(d, Q));
  // up to 2 resident blocks per SM, + the light-curve ticket counters of the fused kernels
  return per_block * sizeof(double) * (size_t)sms * 2 + pgm::PGM_SCHED_INTS * sizeof(int);
}

int pgm_sm_mll_grad_f64(const double* x, const int32_t* n_valid, const double* y,
                        const double* fixed_noise, const double* raw, const int32_t* con_kind,
                        const double* con_lb, const double* con_ub, int B, int n_max, int d,
                        int Q, int kernel_kind, int flags, double* mll, double* grad_raw,
                        int32_t* info, void* workspace, size_t workspace_bytes, void* stream) {
  return pgm_sm_mll_grad_alpha_f64(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub, B,
                                   n_max, d, Q, kernel_kind, flags, mll, grad_raw, nullptr, info,
                                   workspace, workspace_bytes, stream);
}

int pgm_sm_mll_grad_alpha_f64(const double* x, const int32_t* n_valid, const double* y,
                              const double* fixed_noise, const double* raw,
                              const int32_t* con_kind, const double* con_lb, const double* con_ub,
                              int B, int n_max, int d, int Q, int kernel_kind, int flags,
                              double* mll, double* grad_raw, double* alpha_out, int32_t* info,
                              void* workspace, size_t workspace_bytes, void* stream) {
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (alpha_out && !(flags & PGM_FLAG_GRAD)) return fail("alpha_out needs PGM_FLAG_GRAD");
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, mll, info, workspace})) return r;
  if ((flags & PGM_FLAG_GRAD) && !grad_raw) return fail("PGM_FLAG_GRAD needs grad_raw");
  auto A = model_args<pgm::EvalArgs>(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub,
                                     B, n_max, Q, flags, info, workspace);
  A.mll = mll; A.grad = grad_raw; A.alpha_out = alpha_out;
  if (int r = fused_ws(A, d, workspace_bytes)) return r;
  return cfg->eval(A, static_cast<cudaStream_t>(stream));
}

int pgm_fused_grid(int d, int Q, int kernel_kind) {
  const Config* cfg = check_common(1, 64, d, Q, kernel_kind);
  return cfg ? pgm::device_sms() * cfg->fused_blocks_per_sm : -1;
}

size_t pgm_staged_workspace_bytes(int n_max, int B) {
  return (n_max < 1 || B < 1) ? 0 : pgm::large_ws_bytes(n_max, B);
}

int pgm_sm_mll_grad_staged_f64(const double* x, const int32_t* n_valid, const double* y,
                               const double* fixed_noise, const double* raw,
                               const int32_t* con_kind, const double* con_lb,
                               const double* con_ub, int B, int n_max, int d, int Q,
                               int kernel_kind, int flags, double* mll, double* grad_raw,
                               int32_t* info, void* workspace, size_t workspace_bytes,
                               void* stream) {
  return pgm_sm_mll_grad_staged_alpha_f64(x, n_valid, y, fixed_noise, raw, con_kind, con_lb,
                                          con_ub, B, n_max, d, Q, kernel_kind, flags, mll,
                                          grad_raw, nullptr, info, workspace, workspace_bytes,
                                          stream);
}

int pgm_sm_mll_grad_staged_alpha_f64(const double* x, const int32_t* n_valid, const double* y,
                                     const double* fixed_noise, const double* raw,
                                     const int32_t* con_kind, const double* con_lb,
                                     const double* con_ub, int B, int n_max, int d, int Q,
                                     int kernel_kind, int flags, double* mll, double* grad_raw,
                                     double* alpha_out, int32_t* info, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (alpha_out && !(flags & PGM_FLAG_GRAD)) return fail("alpha_out needs PGM_FLAG_GRAD");
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, mll, info, workspace})) return r;
  if ((flags & PGM_FLAG_GRAD) && !grad_raw) return fail("PGM_FLAG_GRAD needs grad_raw");
  if (workspace_bytes < ((flags & PGM_FLAG_TF32X3) ? pgm_staged_tf32x3_workspace_bytes(n_max, B)
                                                   : pgm_staged_workspace_bytes(n_max, B)))
    return fail("workspace too small (see pgm_staged_workspace_bytes / pgm_staged_tf32x3_workspace_bytes)");
  auto A = model_args<pgm::LargeArgs>(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub,
                                      B, n_max, Q, flags, info, workspace);
  A.mll = mll; A.grad = grad_raw; A.alpha_out = alpha_out;
  return cfg->large(A, (flags & PGM_FLAG_GRAD) ? 1 : 0, static_cast<cudaStream_t>(stream), 0);
}

size_t pgm_staged_tf32x3_workspace_bytes(int n_max, int B) {
  return (n_max < 1 || B < 1) ? 0 : pgm::large_ws_bytes_tc(n_max, B);
}

int pgm_sm_mll_grad_staged_tf32x3_f64(const double* x, const int32_t* n_valid, const double* y,
                                      const double* fixed_noise, const double* raw,
                                      const int32_t* con_kind, const double* con_lb,
                                      const double* con_ub, int B, int n_max, int d, int Q,
                                      int kernel_kind, int flags, double* mll, double* grad_raw,
                                      int32_t* info, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  return pgm_sm_mll_grad_staged_alpha_f64(x, n_valid, y, fixed_noise, raw, con_kind, con_lb,
                                          con_ub, B, n_max, d, Q, kernel_kind,
                                          flags | PGM_FLAG_TF32X3, mll, grad_raw, nullptr, info,
                                          workspace, workspace_bytes, stream);
}

int pgm_sm_mll_grad_tf32x3_f32(const float* x, const int32_t* n_valid, const float* y,
                               const float* fixed_noise, const float* raw,
                               const int32_t* con_kind, const float* con_lb, const float* con_ub,
                               int B, int n_max, int d, int Q, int kernel_kind, int flags,
                               float* mll, float* grad_raw, int32_t* info, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!check_common(B, n_max, d, Q, kernel_kind)) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, mll, info, workspace})) return r;
  if ((flags & PGM_FLAG_GRAD) && !grad_raw) return fail("PGM_FLAG_GRAD needs grad_raw");
  const Io32 io{x, y, fixed_noise, raw, con_lb, con_ub, mll,
                (flags & PGM_FLAG_GRAD) ? grad_raw : nullptr, nullptr, nullptr, nullptr};
  return stage_f32(io, B, n_max, d, Q, kernel_kind, flags, 0,
                   pgm_staged_tf32x3_workspace_bytes(n_max, B), "pgm_staged_tf32x3_workspace_bytes",
                   workspace, workspace_bytes, stream, [&](const Stage32& s, size_t f64_bytes) {
    return pgm_sm_mll_grad_staged_alpha_f64(
        s.x, n_valid, s.y, s.fn, s.raw, con_kind, s.lb, s.ub, B, n_max, d, Q, kernel_kind,
        flags | PGM_FLAG_JITTER_F32 | PGM_FLAG_TF32X3 | PGM_FLAG_TF32X3_CHOL, s.mll, s.grad,
        nullptr, info, workspace, f64_bytes, stream);
  });
}

size_t pgm_predict_workspace_bytes(int n_max, int B, int device) {
  if (n_max < 1 || B < 1) return 0;
  int sms = 148;
  if (device >= 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  else sms = pgm::device_sms();
  if (sms <= 0) sms = 148;
  const size_t N = (n_max + pgm::TS - 1) / pgm::TS;
  size_t staged = (pgm::large_ws_bytes(n_max, B) + 255) & ~(size_t)255;
  return staged + (size_t)2 * sms * N * pgm::TT * sizeof(double);
}

int pgm_sm_predict_f64(const double* x, const int32_t* n_valid, const double* y,
                       const double* fixed_noise, const double* raw, const int32_t* con_kind,
                       const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                       int kernel_kind, int flags, const double* xstar, int m, double* mean,
                       double* var, int32_t* info, void* workspace, size_t workspace_bytes,
                       void* stream) {
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (B == 0 || m == 0) return 0;
  if (m < 0) return fail("m must be >= 0");
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, xstar, mean, var, info, workspace}))
    return r;
  if (workspace_bytes < pgm_predict_workspace_bytes(n_max, B, -1))
    return fail("workspace too small (see pgm_predict_workspace_bytes)");
  pgm::PredictArgs PA{};
  PA.a = model_args<pgm::LargeArgs>(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub, B,
                                    n_max, Q, flags & ~PGM_FLAG_GRAD, info, workspace);
  PA.xstar = xstar; PA.m = m; PA.mean = mean; PA.var = var;
  PA.kscratch = reinterpret_cast<double*>(static_cast<char*>(workspace) +
                                          align256(pgm::large_ws_bytes(n_max, B)));
  return cfg->predict(PA, static_cast<cudaStream_t>(stream));
}

size_t pgm_fisher_workspace_bytes(int n_max, int B, int d, int Q, int kernel_kind, int flags) {
  if (n_max < 1 || B < 1 || !check_common(B, n_max, d, Q, kernel_kind)) return 0;
  return pgm::fisher_ws_bytes(n_max, B, host_param_count(d, Q, kernel_kind, flags) - 1);
}

int pgm_sm_fisher_f64(const double* x, const int32_t* n_valid, const double* y,
                      const double* fixed_noise, const double* raw, const int32_t* con_kind,
                      const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                      int kernel_kind, int flags, double* fisher, int32_t* info, void* workspace,
                      size_t workspace_bytes, void* stream) {
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, fisher, info, workspace})) return r;
  if (B > 65535) return fail("pgm_sm_fisher_f64: B > 65535 (split the batch)");
  const int nc = host_param_count(d, Q, kernel_kind, flags) - 1;
  if (nc < 1 || nc > pgm::FS_NC_MAX) return fail("pgm_sm_fisher_f64: unsupported parameter count");
  const long long N = (n_max + pgm::TS - 1) / pgm::TS, ntri = N * (N + 1) / 2;
  if (ntri * nc > 2147483647LL) return fail("pgm_sm_fisher_f64: n_max too large (tiles x carriers)");
  if (workspace_bytes < pgm_fisher_workspace_bytes(n_max, B, d, Q, kernel_kind, flags))
    return fail("workspace too small (see pgm_fisher_workspace_bytes)");
  const int fs_flags = flags & (PGM_FLAG_LEARN_NOISE | PGM_FLAG_BOUNDS_PER_LC | PGM_FLAG_JITTER_F32);
  auto A = model_args<pgm::LargeArgs>(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub,
                                      B, n_max, Q, fs_flags, info, workspace);
  pgm::FisherArgs F;
  F.nc = nc;
  F.fisher = fisher;
  return cfg->fisher(A, F, static_cast<cudaStream_t>(stream));
}

int pgm_sm_kernel_dense_f64(const double* x, const int32_t* n_valid, const double* fixed_noise,
                            const double* raw, const int32_t* con_kind, const double* con_lb,
                            const double* con_ub, int B, int n_max, int d, int Q,
                            int kernel_kind, int flags, double* K_out, void* stream) {
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, raw, con_kind, con_lb, con_ub, K_out})) return r;
  if (B > 65535) return fail("B > 65535 not supported by the dense builder");
  const auto A = model_args<pgm::EvalArgs>(x, n_valid, nullptr, fixed_noise, raw, con_kind,
                                           con_lb, con_ub, B, n_max, Q, flags, nullptr, nullptr);
  return cfg->dense(A, K_out, static_cast<cudaStream_t>(stream));
}

int pgm_optim_step_f64(double* raw, const double* grad_mll, double* exp_avg, double* exp_avg_sq,
                       const int32_t* active, int B, int P, int optim_kind, double lr,
                       double beta1, double beta2, double eps, double weight_decay, int step,
                       void* stream) {
  if (B < 0 || P < 1) return fail("bad B / P");
  if (B == 0) return 0;
  if (int r = check_ptrs({raw, grad_mll})) return r;
  if (optim_kind != PGM_OPT_SGD && (!exp_avg || !exp_avg_sq))
    return fail("Adam / AdamW need exp_avg and exp_avg_sq");
  if (optim_kind < 0 || optim_kind > 2) return fail("unknown optim_kind");
  if (step < 1) return fail("step counts from 1");
  const size_t total = (size_t)B * P;
  const int threads = 256;
  const unsigned blocks = (unsigned)((total + threads - 1) / threads);
  // torch.optim computes the bias corrections in host double precision as well (1 - beta ** step)
  const double bc1 = 1.0 - std::pow(beta1, (double)step);
  const double bc2s = std::sqrt(1.0 - std::pow(beta2, (double)step));
  pgm::optim_step_kernel<<<blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      raw, grad_mll, exp_avg, exp_avg_sq, active, B, P, optim_kind, lr, beta1, beta2, eps,
      weight_decay, bc1, bc2s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("optim_step_kernel launch", e);
  return 0;
}

int pgm_sm_fit_f64(const double* x, const int32_t* n_valid, const double* y,
                   const double* fixed_noise, double* raw, const int32_t* con_kind,
                   const double* con_lb, const double* con_ub, int B, int n_max, int d, int Q,
                   int kernel_kind, int flags, int optim_kind, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int maxiter, int miniter,
                   double stop, int stopavg, double* loss_hist, double* raw_hist,
                   int32_t* n_iter, int32_t* info, double* opt_state, void* workspace,
                   size_t workspace_bytes, void* stream) {
  (void)opt_state;  // optimiser state lives in shared memory for the whole loop
  const Config* cfg = check_common(B, n_max, d, Q, kernel_kind);
  if (!cfg) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, loss_hist, n_iter, info, workspace}))
    return r;
  if (maxiter < 1) return fail("maxiter must be >= 1");
  if (optim_kind < 0 || optim_kind > 2) return fail("unknown optim_kind");
  if (stopavg < 1) stopavg = 1;
  pgm::FitArgs F{};
  F.e = model_args<pgm::EvalArgs>(x, n_valid, y, fixed_noise, raw, con_kind, con_lb, con_ub, B,
                                  n_max, Q, flags | PGM_FLAG_GRAD, info, workspace);
  if (int r = fused_ws(F.e, d, workspace_bytes)) return r;
  F.raw_io = raw; F.optim_kind = optim_kind; F.lr = lr; F.beta1 = beta1; F.beta2 = beta2;
  F.eps = eps; F.weight_decay = weight_decay; F.stop = stop; F.maxiter = maxiter;
  F.miniter = miniter; F.stopavg = stopavg; F.loss_hist = loss_hist; F.raw_hist = raw_hist;
  F.n_iter = n_iter;
  return cfg->fit(F, static_cast<cudaStream_t>(stream));
}

size_t pgm_f32_staging_bytes(int B, int n_max, int d, int Q, int kernel_kind, int flags,
                             int maxiter, int want_raw_hist) {
  if (B < 1 || n_max < 1) return 0;
  const int P = host_param_count(d, Q, kernel_kind, flags);
  return carve32(nullptr, B, n_max, d, P, (flags & PGM_FLAG_BOUNDS_PER_LC) != 0,
                 maxiter < 0 ? 0 : maxiter, want_raw_hist != 0).bytes;
}

int pgm_sm_mll_grad_f32(const float* x, const int32_t* n_valid, const float* y,
                        const float* fixed_noise, const float* raw, const int32_t* con_kind,
                        const float* con_lb, const float* con_ub, int B, int n_max, int d, int Q,
                        int kernel_kind, int flags, float* mll, float* grad_raw, int32_t* info,
                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!check_common(B, n_max, d, Q, kernel_kind)) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, mll, info, workspace})) return r;
  if ((flags & PGM_FLAG_GRAD) && !grad_raw) return fail("PGM_FLAG_GRAD needs grad_raw");
  const Io32 io{x, y, fixed_noise, raw, con_lb, con_ub, mll,
                (flags & PGM_FLAG_GRAD) ? grad_raw : nullptr, nullptr, nullptr, nullptr};
  return stage_f32(io, B, n_max, d, Q, kernel_kind, flags, 0,
                   pgm_workspace_bytes(8, n_max, d, Q, -1), "pgm_workspace_bytes", workspace,
                   workspace_bytes, stream, [&](const Stage32& s, size_t f64_bytes) {
    return pgm_sm_mll_grad_f64(s.x, n_valid, s.y, s.fn, s.raw, con_kind, s.lb, s.ub, B, n_max, d,
                               Q, kernel_kind, flags | PGM_FLAG_JITTER_F32, s.mll, s.grad, info,
                               workspace, f64_bytes, stream);
  });
}

int pgm_sm_fit_f32(const float* x, const int32_t* n_valid, const float* y,
                   const float* fixed_noise, float* raw, const int32_t* con_kind,
                   const float* con_lb, const float* con_ub, int B, int n_max, int d, int Q,
                   int kernel_kind, int flags, int optim_kind, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int maxiter, int miniter,
                   double stop, int stopavg, float* loss_hist, float* raw_hist, int32_t* n_iter,
                   int32_t* info, void* workspace, size_t workspace_bytes, void* stream) {
  if (!check_common(B, n_max, d, Q, kernel_kind)) return -1;
  if (B == 0) return 0;
  if (int r = check_ptrs({x, y, raw, con_kind, con_lb, con_ub, loss_hist, n_iter, info, workspace}))
    return r;
  if (maxiter < 1) return fail("maxiter must be >= 1");
  const Io32 io{x, y, fixed_noise, raw, con_lb, con_ub, nullptr, nullptr, raw, loss_hist,
                raw_hist};
  return stage_f32(io, B, n_max, d, Q, kernel_kind, flags, maxiter,
                   pgm_workspace_bytes(8, n_max, d, Q, -1), "pgm_workspace_bytes", workspace,
                   workspace_bytes, stream, [&](const Stage32& s, size_t f64_bytes) {
    return pgm_sm_fit_f64(s.x, n_valid, s.y, s.fn, s.raw, con_kind, s.lb, s.ub, B, n_max, d, Q,
                          kernel_kind, flags | PGM_FLAG_JITTER_F32, optim_kind, lr, beta1, beta2,
                          eps, weight_decay, maxiter, miniter, stop, stopavg, s.loss, s.hist,
                          n_iter, info, nullptr, workspace, f64_bytes, stream);
  });
}

int pgm_lombscargle_f64(const double* t, const int32_t* n_valid, const double* y, const double* dy,
                        int B, int n_max, const double* f0, const double* df, const int32_t* nf,
                        int nf_max, int flags, double* power, void* stream) {
  if (B < 0 || n_max < 1 || nf_max < 1) return fail("B >= 0, n_max >= 1, nf_max >= 1 required");
  if (B == 0) return 0;
  if (B > 65535) return fail("B > 65535 (split the batch)");
  if (int r = check_ptrs({t, y, f0, df, nf, power})) return r;
  pgm::LsArgs A;
  A.t = t; A.n_valid = n_valid; A.y = y; A.dy = dy; A.f0 = f0; A.df = df; A.nf = nf;
  A.B = B; A.n_max = n_max; A.nf_max = nf_max; A.flags = flags; A.power = power;
  dim3 grid((nf_max + pgm::LS_FPB - 1) / pgm::LS_FPB, B);
  pgm::ls_power_kernel<<<grid, pgm::LS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(A);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("ls_power_kernel launch", e);
  return 0;
}

int pgm_ls_peaks_f64(const double* power, const int32_t* nf, int B, int nf_max, int distance,
                     int num_peaks, int32_t* peak_idx, double* peak_power, void* scratch,
                     size_t scratch_bytes, void* stream) {
  if (B < 0 || nf_max < 1 || num_peaks < 1) return fail("bad B / nf_max / num_peaks");
  if (B == 0) return 0;
  if (distance < 1) return fail("distance must be >= 1 (scipy.signal.find_peaks)");
  if (int r = check_ptrs({power, nf, peak_idx, peak_power, scratch})) return r;
  if (scratch_bytes < (size_t)B * nf_max) return fail("scratch too small (B * nf_max bytes)");
  pgm::LsPeakArgs A;
  A.power = power; A.nf = nf; A.B = B; A.nf_max = nf_max; A.distance = distance;
  A.num_peaks = num_peaks; A.mask = static_cast<uint8_t*>(scratch); A.peak_idx = peak_idx;
  A.peak_power = peak_power;
  pgm::ls_peaks_kernel<<<B, pgm::LS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(A);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("ls_peaks_kernel launch", e);
  return 0;
}

int pgm_sm_psd_peak_f64(const double* freq, const double* fscale, const double* weight,
                        const double* fmin, const double* fmax, int B, int Q, int n_grid,
                        double* grid, double* psd, int32_t* dom_idx, double* dom_freq,
                        double* dom_height, int32_t* n_peaks, void* stream) {
  if (B < 0 || Q < 1 || Q > 8 || n_grid < 3) return fail("bad B / Q (1..8) / n_grid (>= 3)");
  if (B == 0) return 0;
  if (int r = check_ptrs({freq, fscale, weight, fmin, fmax, psd, dom_idx, dom_freq, dom_height,
                          n_peaks}))
    return r;
  pgm::PsdArgs A;
  A.freq = freq; A.fscale = fscale; A.weight = weight; A.fmin = fmin; A.fmax = fmax;
  A.B = B; A.Q = Q; A.n_grid = n_grid; A.grid = grid; A.psd = psd; A.dom_idx = dom_idx;
  A.dom_freq = dom_freq; A.dom_height = dom_height; A.n_peaks = n_peaks;
  pgm::sm_psd_peak_kernel<<<B, pgm::LS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(A);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("sm_psd_peak_kernel launch", e);
  return 0;
}

}  // extern "C"

// ---- FP64 yardsticks ---------------------------------------------------------------------
namespace pgm {
__global__ void __launch_bounds__(256) probe_dmma(int iters, double* out) {
  double acc[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i][0] = acc[i][1] = 0.0;
  double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) mma_f64(acc[i], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += acc[i][0] + acc[i][1];
  if (s == 123.456) out[0] = s;
}
__global__ void __launch_bounds__(256) probe_dfma(int iters, double* out) {
  double acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = threadIdx.x * 1e-9 + i;
  const double a = 1.0000001, b = 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = fma(acc[i], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  if (s == 123.456) out[0] = s;
}
// DMMA and DFMA interleaved (equal flops each): tells whether they share one FP64 pipe
__global__ void __launch_bounds__(256) probe_mixed(int iters, double* out) {
  double acc[4][2], f[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) f[i] = threadIdx.x * 1e-9 + i;
  double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
  const double fa = 1.0000001, fb = 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      mma_f64(acc[i], a, b);                        // 512 flops / warp
#pragma unroll
      for (int j = 0; j < 8; ++j) f[(i * 8 + j) & 15] = fma(f[(i * 8 + j) & 15], fa, fb);  // 8 x 64
    }
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) s += acc[i][0] + acc[i][1];
#pragma unroll
  for (int i = 0; i < 16; ++i) s += f[i];
  if (s == 123.456) out[0] = s;
}
__global__ void __launch_bounds__(256) probe_ffma(int iters, double* out) {
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = threadIdx.x * 1e-9f + i;
  const float a = 1.0000001f, b = 1e-9f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = fmaf(acc[i], a, b);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  if (s == 123.456f) out[0] = s;
}
// dense TF32 tcgen05.mma rate (M = N = 128, K = 8 per instruction): one CTA per SM, one thread issues
// `iters` rounds of 16 MMAs (4 k-steps x 2 accumulators x A/B image pairs) from a resident stage
__global__ void __launch_bounds__(64, 1) probe_tcgen05_tf32(int iters, double* out) {
  extern __shared__ __align__(1024) unsigned char smraw[];
  const unsigned base = (smem_u32(smraw) + 1023u) & ~1023u;
  const unsigned bar = base + 2 * tc::IMG_BYTES, tslot = bar + 16;
  float* img = reinterpret_cast<float*>(smraw + (base - smem_u32(smraw)));
  for (int i = threadIdx.x; i < 2 * tc::IMG_FLOATS; i += 64) img[i] = 1e-3f * (float)((i * 37) % 101);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    fence_proxy_async();
  }
  if ((threadIdx.x >> 5) == 1) tc::tmem_alloc(tslot, 256);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  unsigned tmem;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(tmem) : "r"(tslot));
  if (threadIdx.x == 0) {
    constexpr uint32_t idesc = tc::idesc_tf32(128, 128);
    for (int it = 0; it < iters; ++it)
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t a = tc::smem_desc_sw128(base + ks * 32);
        const uint64_t b = tc::smem_desc_sw128(base + tc::IMG_BYTES + ks * 32);
        tc::mma_tf32(tmem, a, b, idesc, (it | ks) ? 1u : 0u);
        tc::mma_tf32(tmem + 128, b, a, idesc, (it | ks) ? 1u : 0u);
        tc::mma_tf32(tmem, b, a, idesc, 1u);
        tc::mma_tf32(tmem + 128, a, b, idesc, 1u);
      }
    tc::mma_commit(bar);
    mbar_wait(bar, 0);
    tc::fence_after_sync();
  }
  __syncthreads();
  if ((threadIdx.x >> 5) == 1) {
    float v[16];
    tc::tmem_ld16(tmem + ((unsigned)(32 * 1) << 16), v);
    if (v[0] == 123.456f) out[0] = v[0];
    tc::fence_before_sync();
    tc::tmem_dealloc(tmem, 256);
  }
}
}  // namespace pgm

extern "C" int pgm_peak_probe(int kind, int iters, double* tflops_host, void* stream) {
  if (!tflops_host || iters < 1) return fail("bad arguments");
  const int sms = pgm::device_sms();
  double* dout = nullptr;
  cudaError_t e = cudaMalloc(&dout, 8);
  if (e != cudaSuccess) return cuda_fail("cudaMalloc", e);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  int blocks = sms * 8, threads = 256;
  double flops_per_thread_iter = 0.0;
  float best = 1e30f;
  const size_t tc_smem = 2 * pgm::tc::IMG_BYTES + 1024 + 64;
  if (kind == 4) {
    blocks = sms; threads = 64;
    cudaFuncSetAttribute(pgm::probe_tcgen05_tf32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem);
  }
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0, st);
    if (kind == 4) {
      pgm::probe_tcgen05_tf32<<<blocks, threads, tc_smem, st>>>(iters, dout);
      flops_per_thread_iter = 16.0 * (128.0 * 128 * 8 * 2) / 64.0;
    } else if (kind == 0) {
      pgm::probe_dmma<<<blocks, threads, 0, st>>>(iters, dout);
      flops_per_thread_iter = 8.0 * (8 * 8 * 4 * 2) / 32.0;
    } else if (kind == 1) {
      pgm::probe_dfma<<<blocks, threads, 0, st>>>(iters, dout);
      flops_per_thread_iter = 16.0 * 2;
    } else if (kind == 3) {
      pgm::probe_mixed<<<blocks, threads, 0, st>>>(iters, dout);
      flops_per_thread_iter = 4.0 * (8 * 8 * 4 * 2) / 32.0 + 32.0 * 2;
    } else {
      pgm::probe_ffma<<<blocks, threads, 0, st>>>(iters, dout);
      flops_per_thread_iter = 16.0 * 2;
    }
    cudaEventRecord(e1, st);
    e = cudaEventSynchronize(e1);
    if (e != cudaSuccess) { cudaFree(dout); return cuda_fail("probe", e); }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(dout);
  const double total = flops_per_thread_iter * (double)iters * (double)blocks * threads;
  *tflops_host = total / (best * 1e-3) / 1e12;
  return 0;
}
