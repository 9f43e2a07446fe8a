// Translation unit of the state-annotation kernel (k3_predict).
#include "xt_launch.h"
#include "xt_predict.cuh"
#include "xt_predict_shared.cuh"
#include "xt_refine.cuh"

// The own-plan annotation kernel of a model: scalar models with 2 or 3 states and the hot scratch in shared memory get
// the instantiation with the number of states fixed at compile time (NSC), everything else the generic one.  `OUT`: the
// instantiation that also writes the two-slice posteriors (K3Args::pairs), the residuals (K3Args::resid) or the MAP
// paths (K3Args::path).
using K3Kern = void (*)(const K3Args, const xt_params);
struct K3Pick {
  K3Kern kern;
  unsigned long long* smem_ok;
};
template <int D, int KS, bool VAR, int NSC, K3Out OUT>
static K3Pick k3_one() {
  static unsigned long long smem_ok = 0;
  return K3Pick{k3_predict<D, KS, VAR, false, false, NSC, OUT == K3_OUT_PAIRS, OUT == K3_OUT_RESID, OUT == K3_OUT_PATH>,
                &smem_ok};
}
template <int D, int KS, K3Out OUT>
static K3Pick k3_pick_nsc(bool var, int nsc) {
  return var ? k3_one<D, KS, true, 0, OUT>()
             : (nsc == 2 ? k3_one<D, KS, false, 2, OUT>()
                         : (nsc == 3 ? k3_one<D, KS, false, 3, OUT>() : k3_one<D, KS, false, 0, OUT>()));
}
static K3Pick k3_pick(const xt_params& p, int hot_smem, K3Out out) {
  K3Pick k{nullptr, nullptr};
  const bool var = xt_is_var(&p);
  const int nsc = (!var && hot_smem && (p.nS == 2 || p.nS == 3)) ? p.nS : 0;
#define PICK_K3(D_, KS_)                                                         \
  k = out == K3_OUT_PAIRS   ? k3_pick_nsc<D_, KS_, K3_OUT_PAIRS>(var, nsc)       \
      : out == K3_OUT_RESID ? k3_pick_nsc<D_, KS_, K3_OUT_RESID>(var, nsc)       \
      : out == K3_OUT_PATH  ? k3_pick_nsc<D_, KS_, K3_OUT_PATH>(var, nsc)        \
                            : k3_pick_nsc<D_, KS_, K3_OUT_PREDS>(var, nsc)
  XT_DISPATCH(p.d, p.n_loc, PICK_K3);
#undef PICK_K3
  return k;
}

int xt_k3_regs(const xt_params& p, int hot_smem, K3Out out) {
  cudaFuncAttributes at;
  if (cudaFuncGetAttributes(&at, k3_pick(p, hot_smem, out).kern) != cudaSuccess) {
    cudaGetLastError();
    return 128;
  }
  return at.numRegs;
}

cudaError_t xt_launch_k3(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream, K3Out out) {
  const K3Pick k = k3_pick(p, a.hot_smem, out);
  cudaError_t e = xt_allow_smem(k.kern, smem, k.smem_ok);
  if (e != cudaSuccess) return e;
  k.kern<<<grid, 32 * nwarps, smem, stream>>>(a, p);
  return cudaGetLastError();
}

// predict_Bs with nb_max > 1: the plans shared by the tracks of a chunk, then the annotation that follows them
template <int D, int KS>
static cudaError_t launch_k3s(const K3SArgs& a, const xt_params& p, int grid, cudaStream_t stream) {
  k3_shared_plan<D, KS><<<grid, 256, 0, stream>>>(a, p);
  return cudaGetLastError();
}
cudaError_t xt_launch_k3_shared_plan(const K3SArgs& a, const xt_params& p, int grid, cudaStream_t stream) {
  cudaError_t e = cudaSuccess;
#define CALL_K3S(D_, KS_) e = launch_k3s<D_, KS_>(a, p, grid, stream)
  XT_DISPATCH(p.d, p.n_loc, CALL_K3S);
#undef CALL_K3S
  return e;
}
template <int D, int KS, K3Out OUT>
static cudaError_t launch_k3f(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream) {
  auto kern = k3_predict<D, KS, false, true, false, 0, OUT == K3_OUT_PAIRS, OUT == K3_OUT_RESID, OUT == K3_OUT_PATH>;
  static unsigned long long smem_ok = 0;
  cudaError_t e = xt_allow_smem(kern, smem, &smem_ok);
  if (e != cudaSuccess) return e;
  kern<<<grid, 32 * nwarps, smem, stream>>>(a, p);
  return cudaGetLastError();
}
cudaError_t xt_launch_k3_follow(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream,
                                K3Out out) {
  cudaError_t e = cudaSuccess;
#define CALL_K3F(D_, KS_)                                                                                  \
  e = out == K3_OUT_PAIRS   ? launch_k3f<D_, KS_, K3_OUT_PAIRS>(a, p, grid, nwarps, smem, stream)        \
      : out == K3_OUT_RESID ? launch_k3f<D_, KS_, K3_OUT_RESID>(a, p, grid, nwarps, smem, stream)        \
      : out == K3_OUT_PATH  ? launch_k3f<D_, KS_, K3_OUT_PATH>(a, p, grid, nwarps, smem, stream)         \
                            : launch_k3f<D_, KS_, K3_OUT_PREDS>(a, p, grid, nwarps, smem, stream)
  XT_DISPATCH(p.d, p.n_loc, CALL_K3F);
#undef CALL_K3F
  return e;
}

// position refinement: the recursion along the buckets' plans that stores every step, and the combination of its two passes
template <int D, int KS>
static cudaError_t launch_k3r(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream) {
  auto kern = k3_predict<D, KS, false, true, true>;
  static unsigned long long smem_ok = 0;
  cudaError_t e = xt_allow_smem(kern, smem, &smem_ok);
  if (e != cudaSuccess) return e;
  kern<<<grid, 32 * nwarps, smem, stream>>>(a, p);
  return cudaGetLastError();
}
cudaError_t xt_launch_k3_refine(const K3Args& a, const xt_params& p, int grid, int nwarps, size_t smem, cudaStream_t stream) {
  cudaError_t e = cudaSuccess;
#define CALL_K3R(D_, KS_) e = launch_k3r<D_, KS_>(a, p, grid, nwarps, smem, stream)
  XT_DISPATCH(p.d, p.n_loc, CALL_K3R);
#undef CALL_K3R
  return e;
}
cudaError_t xt_launch_refine_combine(int d, int ks, const KRArgs& a, unsigned grid, cudaStream_t stream) {
#define CALL_KR(D_, KS_) k_refine_combine<D_, KS_><<<grid, 256, 0, stream>>>(a)
  XT_DISPATCH(d, ks, CALL_KR);
#undef CALL_KR
  return cudaGetLastError();
}
