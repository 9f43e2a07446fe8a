// Kernel launchers, one translation unit per kernel family (xt_k1.cu, xt_k2f.cu, ...) so that the
// engine builds in parallel; the host driver (xt_engine.cu) only sees these non-template entry points.
#pragma once
#include "xt_common.cuh"

struct K1Args;
struct K2Args;
struct K2Lin;
struct K2FArgs;
struct K2Tab;
struct K3Args;
struct K3SArgs;
struct KRArgs;
struct K4Args;
// what a state-annotation launch writes next to the posteriors (selects the k3_predict instantiation)
enum K3Out { K3_OUT_PREDS = 0, K3_OUT_PAIRS = 1, K3_OUT_RESID = 2, K3_OUT_PATH = 3 };

#define XT_DISPATCH(D_, KS_, CALL)                                   \
  do {                                                               \
    if (D_ == 1) { CALL(1, 1); }                                     \
    else if (D_ == 2 && KS_ == 1) { CALL(2, 1); }                    \
    else if (D_ == 2) { CALL(2, 2); }                                \
    else if (KS_ == 1) { CALL(3, 1); }                               \
    else { CALL(3, 3); }                                             \
  } while (0)

// Dynamic shared memory above 48 KB needs an opt-in per kernel.  The attribute belongs to the function (per device),
// not to a context, so several contexts of one process (xt_multi, one thread each) must never lower it between
// another thread's opt-in and its launch: it is set once per kernel and device to the most the device allows
// (opt-in maximum minus the kernel's static shared memory).  `done`: one bit per device ordinal, owned by the call site.
template <class Kern>
inline cudaError_t xt_allow_smem(Kern kern, size_t smem, unsigned long long* done) {
  if (smem <= 32 * 1024) return cudaSuccess;  // (static + dynamic stay below the 48 KB that need no opt-in)
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if ((__atomic_load_n(done, __ATOMIC_ACQUIRE) >> (dev & 63)) & 1ull) return cudaSuccess;
  cudaFuncAttributes at;
  e = cudaFuncGetAttributes(&at, kern);
  if (e != cudaSuccess) return e;
  int optin = 0;
  e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)at.sharedSizeBytes);
  if (e == cudaSuccess) __atomic_or_fetch(done, 1ull << (dev & 63), __ATOMIC_RELEASE);
  return e;
}

inline bool xt_is_var(const xt_params* p) { return (p->flags & (XT_FLAG_VAR_LOC | XT_FLAG_VAR_DT)) != 0; }

// plan kernel (xt_plan.cuh); nthreads = 256, 512 or 1024
cudaError_t xt_launch_k1(const K1Args& a, const xt_params& p, size_t smem, int n_chunks, cudaStream_t stream, int nthreads);
// ... in verification mode (k1_plan<.., VERIFY>): scalar models, scratch in shared memory, nthreads = 256 or 512
cudaError_t xt_launch_k1_verify(const K1Args& a, const xt_params& p, size_t smem, int n_chunks, cudaStream_t stream, int nthreads);
// fused replay kernel, FP64 (xt_replay_fused.cuh): shared-memory state, GST or VAR instantiation
cudaError_t xt_launch_k2_fused(int d, int ks, const K2FArgs& a, const K2Tab& tab, size_t smem, int wpc, int tpt,
                               cudaStream_t stream, bool var);
// optional single-precision replay (xt_replay_f32.cuh)
cudaError_t xt_launch_k2_f32(int d, int ks, const K2FArgs& a, const K2Tab& tab, size_t smem, cudaStream_t stream);
// first-generation linear-domain kernel / log-domain fallback (xt_replay_lin.cuh, xt_replay.cuh)
cudaError_t xt_launch_k2_old(const K2Args& a, const xt_params& p, const K2Lin& lin, size_t smem, bool use_smem, int grid,
                             int wpc, cudaStream_t stream);
// state annotation (xt_predict.cuh); `out`: the instantiation that also writes the two-slice posteriors (a.pairs), the
// residuals (a.resid) or the MAP paths (a.path)
cudaError_t xt_launch_k3(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream, K3Out out);
int xt_k3_regs(const xt_params& p, int hot_smem, K3Out out);  // registers per thread of the kernel xt_launch_k3 would launch
// ... with plans shared by the nb_max tracks of a chunk (xt_predict_shared.cuh): the plans, then the annotation along them
cudaError_t xt_launch_k3_shared_plan(const K3SArgs& a, const xt_params& p, int grid, cudaStream_t stream);
cudaError_t xt_launch_k3_follow(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream,
                                K3Out out);
// position refinement (xt_refine.cuh): recursion that stores every step, combination of its two passes
cudaError_t xt_launch_k3_refine(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream);
cudaError_t xt_launch_refine_combine(int d, int ks, const KRArgs& a, unsigned grid, cudaStream_t stream);
// segment-length histogram (xt_seglen.cuh)
cudaError_t xt_launch_k4(const K4Args& a, const xt_params& p, int grid, size_t smem, cudaStream_t stream);
// final fixed-order sums (xt_replay.cuh: k_reduce) and the FP64 FMA microbenchmark live in xt_engine.cu
