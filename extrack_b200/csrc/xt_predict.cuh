// K3 — state annotation kernel (predict_Bs, tracking.py:792-906 with the default nb_max = 1:
// every track is its own chunk, so the grouping plan is decided per track from that track alone).
//
// One warp per track, lanes stride over state sequences.  Forward pass = the recursion of
// P_Cs_inter_bound_stats_th(do_preds=1) in the reference's operation order (same faithful
// arithmetic as the plan kernel, because here every track's own numbers drive the discontinuous
// grouping decisions).  The reference carries, for every sequence, the posterior of *all* past
// states (cur_Bs_cat[nT, nB, L, nS], rewritten at every step: O(L^2) traffic).  Only the newest
// frame_len rows ever influence a decision (tracking.py:679-681), so the forward pass keeps that
// window, records the normalised merge weights of every fusion, and a backward sweep over the
// recorded lattice produces the same posteriors in O(L):
//     a_final[c]  = softmax_c(LP_c)                                   (:641-648)
//     pred[s][label_s(c)] += a_child[c];  a_parent[p] = sum_r a_child[pK + r]
//     a_child(step s-1)[c'] = a_parent(step s)[gid[c']] * w[c'] / sum_group w
// The history labels keep the reference's int8 wrap (:543).  nb_substeps is 1 (:839).
// With PAIRS the same sweep also yields the two-slice posteriors (the Baum-Welch "xi"): the newest history row of a
// group q of the fusion at step s-1 is the weighted mixture of its members' labels, so with v_q[j] = mass of q's
// children at step s that carry label j,
//     pair[s-1][label(c')][j] += w[c'] * v_q[j]   for every member c' of q (normalised weight w[c'])
// and the initial sequences give pair[0] directly.  This equals carrying a pair history through the reference's
// expansions and fusions (oracle/pair_oracle.py).
// With RESID the forward pass also yields the one-step-ahead predictive of every localisation c_k (k >= 1): at the step
// that consumes c_k, every live sequence j (a child of the expansion, or a final sequence at the end of the track) has
// the predictive Gaussian N(m_j, q_j) of c_k (its parent's mean, q_j = l2 + s2_j), the Gaussian term LC_j of c_k and
// the log-weight A_j = (log-weight after the step) - LC_j.  The mixture over j gives
//     logpred[k] = logsumexp_j(A_j + LC_j) - logsumexp_j(A_j)
//     pit[k][x]  = sum_j softmax(A)_j Phi((c_k,x - m_j,x) / sqrt(q_j,kappa(x)))
// m, q and LC are those of the parent, so they and Phi are evaluated once per parent (oracle/resid_oracle.py).
// With PATH the forward pass also yields the most probable state path (MAP / Viterbi path) of the lattice above: a route
// from an initial to a final sequence has the weight softmax(LP)_final * prod of the merge weights w along it, the
// routes' weights sum to 1 and the backward sweep sums them by label.  Every sequence carries a score V updated like its
// LP, except that a fusion sets its group's V to the *maximum* of the members' V (LP: their log-sum-exp); the argmax
// member (ties: the first in member order) is recorded per group and level (recArg).  The final choice is the argmax of
// V + the end-of-track term of LP (the bleaching end's Lsum included; ties: the lowest index), and one lane backtracks
// along recArg and the implicit parents c / K.  The labels are those of the posteriors (the int8 wrap included) and
//     path_logp = V* - logsumexp(final LP) = log(weight of the heaviest route)
// by telescoping.  Without fusion V = LP, so the path is the exact argmax over the state sequences
// (oracle/path_oracle.py).
#pragma once
#include <math_constants.h>
#include "xt_common.cuh"
#include "xt_plan.cuh"

#define XT_K3_WARPS 8
#ifndef XT_K3_MIN_CTAS
#define XT_K3_MIN_CTAS 2  // resident CTAs of 8 warps the register allocation leaves room for (2: 128 registers)
#endif

struct K3Args {
  const XtChunk* chunks;
  const XtWork* work;
  const double* soa;
  double* scratch;     // per resident warp
  double* pred;        // [sum over tracks of L][nS], forward time
  int32_t* err;        // [n_work]  0 ok, 1 grouping failure, 2 capacity overflow (need in err_need)
  int32_t* err_need;
  int32_t n_work;
  int32_t cap;         // children capacity
  int32_t maxL;
  int32_t bits;
  double Lsum[XT_MAX_STATES];
  size_t warp_scratch; // 8-byte units per warp in `scratch`: cold part (+ hot part unless hot_smem)
  int32_t hot_smem;    // 1: the hot part of every warp is in dynamic shared memory
  XtAux ax;            // VAR instantiation only; stay = [n_tracks][K] Lp_stay, leave = [n_tracks][nS] log-sums
  // FOLLOW instantiation (predict_Bs with nb_max > 1): the groups of every fusion step come from the chunk's shared
  // plan (k3_shared_plan, xt_predict_shared.cuh) instead of this track's own decisions
  const int32_t* splan;  // [n_chunks][splan_stride]: nC[maxL], nG[maxL], then per step goff[cap + 1], order[cap]
  size_t splan_stride;
  // REFINE instantiation (position refinement, refined_localization.py:48-204 get_LC_Km_Ks): the recursion without
  // field-of-view / bleaching terms, initial fractions added at the end; instead of posteriors it stores, for every
  // step, (mean[d], std[KS], log-weight, newest state) of every surviving sequence of every track
  int32_t rev;           // 1: consume the localisations from the last to the first (get_LC_Km_Ks' own order)
  union {
    double* dump;        // [n_tracks][L - 1 entries][capD][d + KS + 2] doubles, per chunk at dump_off[chunk]
    // PAIRS instantiation (predict_transitions, never REFINE): two-slice posteriors P(s_k = i, s_k+1 = j | track),
    // [sum over tracks of (L - 1)][nS][nS] in forward time; a track's rows start at loc_off - trk_off + t (L - 1)
    double* pairs;
    // RESID instantiation (predict_residuals, never REFINE nor PAIRS): {logpred, pit}, a device array of two pointers
    // to [sum over tracks of L] and [sum over tracks of L][d] doubles in forward time, a track's rows at loc_off + t L
    double* const* resid;
    // PATH instantiation (predict_path, never REFINE, PAIRS nor RESID): {labels, path_logp}, a device array of two
    // pointers to int8_t[sum over tracks of L] in forward time (a track's labels at loc_off + t L) and double[n_tracks]
    // (a track's entry at trk_off + t)
    void* const* path;
  };
  const int64_t* dump_off;
  int32_t* ent_n;        // [n_chunks][maxL]: sequences per entry (written by the chunk's first track)
  int32_t capD;
  double LF[XT_MAX_STATES];  // log initial fractions by state (REFINE: added at the end, refined_localization.py:190)
};

// per-warp scratch layout, in 8-byte units: the *hot* part (state of the forward pass, touched at
// every step) lives in shared memory when the launch could be sized for it (hot_smem), the *cold*
// part (records of the fusions for the backward sweep: written once, read once) in global memory
struct K3Layout {
  size_t bufP, bufC, histP, histN, codeP, codeC, aC, aP, gid, order, goff, curP, hot_total;
  size_t recW, recN, recGid, cold_total;
};
// PATH instantiation: its own regions after the hot and the cold part of the other modes' layout `l`, and the totals
// that include them
struct K3PathLayout {
  size_t vP, vC, hot_total;  // path scores of the parents / groups [cap / nS + 1] and of the children [cap]
  size_t recArg, cold_total; // uint16[maxL][cap / nS + 1]: argmax member of every group of every fused step
};
__host__ __device__ inline K3PathLayout k3_path_layout(const K3Layout& l, int cap, int nS, int maxL) {
  K3PathLayout q;
  size_t o = l.hot_total;
  q.vP = o;     o += cap / nS + 1;
  q.vC = o;     o += cap;
  q.hot_total = (o + 1) & ~(size_t)1;
  q.recArg = l.cold_total;
  q.cold_total = l.cold_total + ((size_t)maxL * (cap / nS + 1) + 3) / 4;
  return q;
}
// The PATH arrays of one warp (hot part at `base`, cold part at `cold`)
struct K3PathPtrs {
  double* vP;        // path scores V of the parents / groups [cap / nS + 1]
  double* vC;        // ... of the children [cap]
  uint16_t* recArg;  // [maxL][cap / nS + 1]: argmax member of every group of every fused step
};
template <bool PATH = false>
__host__ __device__ inline K3Layout k3_layout(int cap, int CO, int fl, int nS, int maxL) {
  K3Layout l;
  size_t o = 0;
  // parents / groups: at most cap / nS of them (see the history rows below)
  l.bufP = o;   o += (size_t)(cap / nS + 1) * CO;
  l.bufC = o;   o += (size_t)cap * CO;
  // history rows exist per parent / group only: at most cap / nS of them (a step with more groups
  // could not expand into cap children and reports the overflow, see the check after the grouping)
  l.histP = o;  o += (size_t)(cap / nS + 1) * fl * nS;
  l.histN = o;  o += (size_t)(cap / nS + 1) * fl * nS;
  l.codeP = o;  o += cap / nS + 1;
  l.codeC = o;  o += cap;
  l.aC = o;     o += cap;
  l.aP = o;     o += cap / nS + 1;
  l.gid = o;    o += (cap + 1) / 2;        // int32[cap]
  l.order = o;  o += (cap + 1) / 2;
  l.goff = o;   o += (cap + 2) / 2;        // int32[cap+1]
  l.curP = o;   o += (cap + 1) / 2;
  l.recN = o;   o += (maxL + 2) / 2;       // int32[maxL+1]: children per fused step (read again by the backward sweep)
  l.hot_total = (o + 1) & ~(size_t)1;
  o = 0;
  l.recW = o;   o += (size_t)maxL * cap;
  l.recGid = o; o += ((size_t)maxL * cap + 3) / 4;  // uint16[maxL][cap]
  l.cold_total = o + 4;
  if constexpr (PATH) {
    const K3PathLayout q = k3_path_layout(l, cap, nS, maxL);
    l.hot_total = q.hot_total;
    l.cold_total = q.cold_total;
  }
  return l;
}
static __device__ __forceinline__ K3PathPtrs k3_path_ptrs(double* base, double* cold, int cap, int CO, int fl, int nS, int maxL) {
  const K3PathLayout q = k3_path_layout(k3_layout(cap, CO, fl, nS, maxL), cap, nS, maxL);
  return K3PathPtrs{base + q.vP, base + q.vC, (uint16_t*)(cold + q.recArg)};
}

// The annotation kernel is sensitive to instruction fetch (ncu: 32 % of the stall samples were "no instruction" with
// 4 k SASS instructions and 16 warps per SM in different phases): its run-time loops are kept rolled (`#pragma unroll 1`:
// 4096 -> 3472 instructions, 116 -> 87.5 ms per 10^6 tracks).  Going further - log / exp / the rarely taken exact division
// of the grouping predicate as shared out-of-line subroutines, one predicate copy for both register halves - was measured
// and is slower (the macros below keep the experiment reproducible).
#ifndef XT_K3_NOINLINE
#define XT_K3_NOINLINE 0  // (measured: out-of-line log / exp / exact-division helpers cost more in calls than they save in fetch: 92 vs 87.5 ms)
#endif
#if XT_K3_NOINLINE
#define K3_NI __noinline__
#else
#define K3_NI __forceinline__
#endif
#ifndef XT_K3_HLOOP
#define XT_K3_HLOOP 0     // (measured: one predicate copy with operand selects 90.5 vs 87.5 ms with the two inline copies)
#endif
static __device__ K3_NI double k3_log(double x) { return log(x); }
static __device__ K3_NI double k3_exp(double x) { return exp(x); }
static __device__ K3_NI bool k3_div_lt(double a, double s, double th) { return __ddiv_rn(a, s) < th; }

// Pair row `row` (states at localisations row, row + 1) of one track into po[nS][nS], from the n sequences c' of level
// `row` and av = the posterior of the children of level row + 1 (child q*nS + r of sequence / group q).  rw / rg: the
// fusion records of level `row` (normalised weight, group); nullptr at level 1, whose sequences are the initial ones
// (newest state c' % nS, unfused: weight 1, parent of the children c' itself).
template <int NSC>
static __device__ __forceinline__ void k3_emit_pairs(double* po, const double* av, int n, const double* rw, const uint16_t* rg,
                                                     int nS, bool wrap, int lane) {
  if constexpr (NSC == 2 || NSC == 4) {
    // the label of c' is the residue of its lane (also c' % nS at level 1), and child q*NSC + j carries label j
    double acc[NSC];
#pragma unroll
    for (int j = 0; j < NSC; ++j) acc[j] = 0.0;
    #pragma unroll 1
    for (int c = lane; c < n; c += 32) {
      const double w = rw ? rw[c] : 1.0;
      const int q = rw ? (int)rg[c] : c;
#pragma unroll
      for (int j = 0; j < NSC; ++j) acc[j] += w * av[q * NSC + j];
    }
#pragma unroll
    for (int j = 0; j < NSC; ++j) {
#pragma unroll
      for (int o2 = 16; o2 >= NSC; o2 >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o2);
    }
    if (lane < NSC) {
#pragma unroll
      for (int j = 0; j < NSC; ++j) po[lane * NSC + j] = acc[j];
    }
  } else {
    for (int i = 0; i < nS; ++i) {
      for (int j = 0; j < nS; ++j) {
        double acc = 0.0;
        #pragma unroll 1
        for (int c = lane; c < n; c += 32) {
          if ((rw ? xt_label(c, nS, wrap) : c % nS) != i) continue;
          const int q = rw ? (int)rg[c] : c;
          double v = 0.0;
          #pragma unroll 1
          for (int r = 0; r < nS; ++r)
            if (xt_label(q * nS + r, nS, wrap) == j) v += av[q * nS + r];
          acc += (rw ? rw[c] : 1.0) * v;
        }
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
        if (lane == 0) po[i * nS + j] = acc;
      }
    }
  }
}

// Residuals of one localisation cl (RESID): the n sequences p of buf (slot pitch `pitch`: mean [D], s2 [KS], log-weight at
// component D + 2 KS) are the parents of nch sequences each, the r-th with A = log-weight + add(p, r).  Lane 0 writes
// logpred to lp[0] and the PIT values to pit[0..D).
template <int D, int KS, class AddF>
static __device__ __forceinline__ void k3_emit_resid(double* lp, double* pit, const double* buf, int pitch, int n, int nch,
                                                     const double* cl, const double* l2, AddF add, int lane) {
  auto lc_of = [&](int p) {  // the Gaussian term of cl under the predictive of parent p
    double lc = 0.0;
#pragma unroll
    for (int dim = 0; dim < D; ++dim) {
      const int k = (KS == 1) ? 0 : dim;
      const double q = buf[(D + k) * pitch + p] + l2[k];
      const double df = cl[dim] - buf[dim * pitch + p];
      lc += -0.5 * log(XT_TWO_PI * q) - df * df / (2.0 * q);
    }
    return lc;
  };
  double mA = -INFINITY, mB = -INFINITY;
  #pragma unroll 1
  for (int p = lane; p < n; p += 32) {
    const double lc = lc_of(p), a0 = buf[(D + 2 * KS) * pitch + p];
    #pragma unroll 1
    for (int r = 0; r < nch; ++r) {
      const double A = a0 + add(p, r);
      mA = fmax(mA, A);
      mB = fmax(mB, A + lc);
    }
  }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    mA = fmax(mA, __shfl_xor_sync(0xffffffffu, mA, o2));
    mB = fmax(mB, __shfl_xor_sync(0xffffffffu, mB, o2));
  }
  double s0 = 0.0, s1 = 0.0, sx[D];
#pragma unroll
  for (int dim = 0; dim < D; ++dim) sx[dim] = 0.0;
  #pragma unroll 1
  for (int p = lane; p < n; p += 32) {
    const double lc = lc_of(p), a0 = buf[(D + 2 * KS) * pitch + p];
    double w = 0.0;  // softmax numerators of p's children
    #pragma unroll 1
    for (int r = 0; r < nch; ++r) {
      const double A = a0 + add(p, r);
      w += exp(A - mA);
      s1 += exp(A + lc - mB);
    }
    s0 += w;
#pragma unroll
    for (int dim = 0; dim < D; ++dim) {
      const int k = (KS == 1) ? 0 : dim;
      const double q = buf[(D + k) * pitch + p] + l2[k];
      sx[dim] += w * normcdf((cl[dim] - buf[dim * pitch + p]) / sqrt(q));
    }
  }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o2);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o2);
#pragma unroll
    for (int dim = 0; dim < D; ++dim) sx[dim] += __shfl_xor_sync(0xffffffffu, sx[dim], o2);
  }
  if (lane == 0) {
    lp[0] = (log(s1) + mB) - (log(s0) + mA);
#pragma unroll
    for (int dim = 0; dim < D; ++dim) pit[dim] = sx[dim] / s0;
  }
}

template <int D, int KS, bool VAR = false, bool FOLLOW = false, bool REFINE = false, int NSC = 0, bool PAIRS = false,
          bool RESID = false, bool PATH = false>
__global__ void __launch_bounds__(32 * XT_K3_WARPS, XT_K3_MIN_CTAS) k3_predict(const K3Args a, const __grid_constant__ xt_params P) {
  static_assert(!(VAR && FOLLOW), "shared plans are built for scalar LocErr / dt models");
  static_assert(!REFINE || FOLLOW, "the refinement recursion follows the bucket's shared plan");
  static_assert(!(REFINE && PAIRS), "the refinement stores no posteriors");
  static_assert(!(REFINE && RESID) && !(PAIRS && RESID), "the residuals share the output pointer of the other modes");
  static_assert(!(PATH && (REFINE || PAIRS || RESID)), "the MAP paths share the output pointer of the other modes");
  // NSC > 0: the number of states is the compile-time constant NSC and the hot scratch is known to be in shared memory
  // (32-bit shared-memory addressing, shifts / multiply-shifts instead of integer divisions); NSC == 0: both at run time
  constexpr bool HOT = NSC > 0;
  extern __shared__ double k3_smem[];
  const int nwarps = blockDim.x >> 5;  // <= XT_K3_WARPS (fewer when the hot scratch of 8 warps exceeds shared memory)
  constexpr int CO = D + 2 * KS + 1;  // m[D], s2[KS], s[KS], LP
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nS = NSC ? NSC : P.nS, K = nS, cap = a.cap, fl = P.frame_len, bits = a.bits;
  const bool wrap = (P.flags & XT_FLAG_INT8_WRAP) != 0;
  const unsigned long long rowmask = (1ull << bits) - 1ull;
  const unsigned lt_mask = (1u << lane) - 1u;
  // history label of child c (tracking.py:543: the int8 wrap); 256 is a multiple of a power-of-two nS, so there the
  // wrap leaves the residue alone
  auto label = [&](int c) -> int {
    if constexpr (NSC == 2 || NSC == 4) return c & (NSC - 1);
    else return xt_label(c, nS, wrap);
  };

  // ---- per-warp scratch carve-up ----
  const K3Layout lay = k3_layout<PATH>(cap, CO, fl, nS, a.maxL);
  double* cold = a.scratch + (size_t)(blockIdx.x * nwarps + warp) * a.warp_scratch;
  double* base;
  if constexpr (HOT) base = k3_smem + warp * (int)lay.hot_total;
  else base = a.hot_smem ? k3_smem + (size_t)warp * lay.hot_total : cold + lay.cold_total;
  double* bufP = base + (int)lay.bufP;            // [CO][capP]
  double* bufC = base + (int)lay.bufC;            // [CO][cap]
  int hP = (int)lay.histP, hN = (int)lay.histN;   // history windows [fl][nS][capP] (offsets: the two swap every step)
  unsigned long long* codeP = (unsigned long long*)(base + (int)lay.codeP);
  unsigned long long* codeC = (unsigned long long*)(base + (int)lay.codeC);
  double* aC = base + (int)lay.aC;
  double* aP = base + (int)lay.aP;
  int* gid = (int*)(base + (int)lay.gid);
  int* order = (int*)(base + (int)lay.order);
  int* goff = (int*)(base + (int)lay.goff);       // [cap+1]
  int* curP = (int*)(base + (int)lay.curP);
  int* recN = (int*)(base + (int)lay.recN);       // children per fused step
  double* recW = cold + lay.recW;                 // [maxL][cap]
  uint16_t* recGid = (uint16_t*)(cold + lay.recGid);
  // PATH: its arrays (K3PathPtrs) are fetched inside the PATH-only blocks, so that the other instantiations compile to
  // exactly the code they had without this mode
#define K3_PATH_PTRS const K3PathPtrs pa = k3_path_ptrs(base, cold, cap, CO, fl, nS, a.maxL)

  const int capP = cap / nS + 1;  // parent / group slots
#define BP(slot, comp) bufP[(comp) * capP + (slot)]
#define BC(slot, comp) bufC[(comp) * cap + (slot)]
  // history window [row][state][slot]: consecutive lanes (slots) hit consecutive shared-memory banks
#define HIX(slot, row, st) (((row) * nS + (st)) * capP + (slot))
#define HISTP(slot, row, st) base[hP + HIX(slot, row, st)]
#define HISTN(slot, row, st) base[hN + HIX(slot, row, st)]

  double l2[KS];
#pragma unroll
  for (int k = 0; k < KS; ++k) l2[k] = P.l2[k];
  const bool var_loc = VAR && (P.flags & XT_FLAG_VAR_LOC), var_dt = VAR && (P.flags & XT_FLAG_VAR_DT);

  for (int wi = blockIdx.x; wi < a.n_work; wi += gridDim.x) {
    const XtWork wk = a.work[wi];
    const XtChunk ck = a.chunks[wk.chunk];
    const int L = ck.L;
    for (int tsub = warp; tsub < 32; tsub += nwarps) {
      const int t = wk.t0 + tsub;
      if (t >= ck.nT) break;  // warp-uniform
      const double* Cp = a.soa + ck.xyz_off + t;
      const size_t npad = (size_t)ck.nTpad;
      double* out = a.pred + ((size_t)ck.loc_off + (size_t)t * L) * nS;
      // RESID: this track's logpred [L] and pit [L][D] start at localisation loc_off + t L; the first localisation has no
      // predictive
      if constexpr (RESID) {
        const size_t row0 = (size_t)ck.loc_off + (size_t)t * L;
        if (lane == 0) {
          a.resid[0][row0] = CUDART_NAN;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) a.resid[1][row0 * D + dim] = CUDART_NAN;
        }
      }
      int errc = 0;
      const bool rev = REFINE && a.rev;
#define LROW(j) (rev ? (L - 1 - (j)) : (j))  // localisation consumed j-th
      // REFINE: this track's entries [L - 1][capD][d + KS + 2]
      constexpr int COD = D + KS + 2;
      double* dmp = REFINE ? a.dump + a.dump_off[wk.chunk] + (size_t)t * (L - 1) * a.capD * COD : nullptr;
      int32_t* entn = (REFINE && t == 0) ? a.ent_n + (size_t)wk.chunk * a.maxL : nullptr;
      // VAR: row j of the aux block = (sigma components, time-reversed dt) of localisation j
      const double* Ap = VAR ? a.ax.aux + (size_t)(ck.xyz_off / D) * a.ax.R + t : nullptr;
      const double* Lps = (VAR && a.ax.stay) ? a.ax.stay + (size_t)(ck.trk_off + t) * K : P.Lp_stay;
      const double* Lsm = (VAR && a.ax.leave) ? a.ax.leave + (size_t)(ck.trk_off + t) * nS : a.Lsum;
      double dtv = 0.0;
      auto var_row = [&](int j) {
        if (var_loc) {
#pragma unroll
          for (int k = 0; k < KS; ++k) l2[k] = xt_sigma2(P, Ap[(size_t)(j * a.ax.R + k) * npad]);
        }
        if (var_dt) dtv = Ap[(size_t)(j * a.ax.R + a.ax.ka) * npad];
      };
#define DDX(head) ((VAR && var_dt) ? xt_dd_exact(P, head, dtv) : P.dd[head])
      if (VAR) var_row(0);

      // ---- first localisation (tracking.py:478-529) ----
      int nP = nS * nS;
      #pragma unroll 1
      for (int c = lane; c < nP; c += 32) {
#pragma unroll
        for (int dim = 0; dim < D; ++dim) BP(c, dim) = Cp[(size_t)(LROW(0) * D + dim) * npad];
#pragma unroll
        for (int k = 0; k < KS; ++k) BP(c, D + k) = __dadd_rn(l2[k], DDX(c));
        BP(c, D + 2 * KS) = REFINE ? P.LT[c] : __dadd_rn(P.LT[c], P.LF[c]);
        if (REFINE && L > 2) {  // entry 0 (for L == 2 the only entry is written at the end, with the final weights)
          double* e0 = dmp + (size_t)c * COD;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) e0[dim] = BP(c, dim);
#pragma unroll
          for (int k = 0; k < KS; ++k) e0[D + k] = __dsqrt_rn(BP(c, D + k));
          e0[D + KS] = BP(c, D + 2 * KS);
          e0[D + KS + 1] = (double)(c % nS);
        }
        if constexpr (PATH) {
          K3_PATH_PTRS;
          pa.vP[c] = BP(c, D + 2 * KS);
        }
        curP[c] = c % nS;
        const int d0 = c % nS, d1 = c / nS;
        codeP[c] = (unsigned long long)d0 | ((unsigned long long)d1 << bits);
        for (int s = 0; s < nS; ++s) {
          HISTP(c, 0, s) = (d0 == s) ? 1.0 : 0.0;
          if (fl > 1) HISTP(c, 1, s) = (d1 == s) ? 1.0 : 0.0;
        }
      }
      int LhP = 2;       // full history length (never truncated in predict mode)
      double th = P.threshold;
      if (entn && lane == 0) entn[0] = nP;
      __syncwarp();

      for (int step = 2; step <= L - 1; ++step) {
        const int nC = nP * K;
        if (nC > cap) {
          errc = 2;
          if (lane == 0) atomicMax(&a.err_need[wi], nC);
          break;
        }
        const int LhC = LhP + 1;
        const int rows_cmp = LhC < fl ? LhC : fl;    // rows stored / compared for the children
        const bool use_window = LhC > fl;
        const unsigned long long cmask = (bits * rows_cmp >= 64) ? ~0ull : ((1ull << (bits * rows_cmp)) - 1ull);
        // the own-plan grouping keeps the candidates of up to 64 children in registers (two per lane)
        const bool reg_grouping = !FOLLOW && nC <= 64;
        double cl[D];
#pragma unroll
        for (int dim = 0; dim < D; ++dim) cl[dim] = Cp[(size_t)(LROW(step - 1) * D + dim) * npad];
        const bool stay = !REFINE && step >= P.min_len;
        if (VAR) var_row(step - 1);
        // ---- expansion + Gaussian update (tracking.py:540-570, :87-98), lane = child ----
        for (int c = lane; c < nC; c += 32) {
          const int p = c / K, r = c - p * K;
          const int head = r + K * curP[p];
          const double dd = DDX(head);
          double s2[KS], q[KS];
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            s2[k] = BP(p, D + k);
            q[k] = __dadd_rn(l2[k], s2[k]);
          }
          double quad = 0.0, logs = 0.0;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) {
            const int k = (KS == 1) ? 0 : dim;
            const double mm = BP(p, dim);
            const double df = __dsub_rn(cl[dim], mm);
            const double term = __ddiv_rn(__dmul_rn(df, df), __dmul_rn(2.0, q[k]));
            quad = (dim == 0) ? term : __dadd_rn(quad, term);
            BC(c, dim) = __ddiv_rn(__dadd_rn(__dmul_rn(mm, l2[k]), __dmul_rn(cl[dim], s2[k])), __dadd_rn(l2[k], s2[k]));
          }
          if (KS == 1) {
            logs = __dmul_rn((double)D * -0.5, k3_log(__dmul_rn(XT_TWO_PI, q[0])));
          } else {
#pragma unroll
            for (int k = 0; k < KS; ++k) {
              const double lg = __dmul_rn(-0.5, k3_log(__dmul_rn(XT_TWO_PI, q[k])));
              logs = (k == 0) ? lg : __dadd_rn(logs, lg);
            }
          }
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            const double ns2 = __ddiv_rn(
                __dadd_rn(__dadd_rn(__dmul_rn(dd, l2[k]), __dmul_rn(dd, s2[k])), __dmul_rn(l2[k], s2[k])), q[k]);
            BC(c, D + k) = ns2;
            BC(c, D + KS + k) = __dsqrt_rn(ns2);
          }
          double add = __dadd_rn(P.LT[head], __dsub_rn(logs, quad));
          if (stay) add = __dadd_rn(add, Lps[r]);
          BC(c, D + 2 * KS) = __dadd_rn(BP(p, D + 2 * KS), add);
          if constexpr (PATH) {
            K3_PATH_PTRS;
            pa.vC[c] = __dadd_rn(pa.vP[p], add);
          }
          codeC[c] = ((codeP[p] << bits) | (unsigned long long)label(c)) & cmask;
          if (!FOLLOW && !reg_grouping) gid[c] = -1;
        }
        if (nC > P.max_nb_states) th = __dmul_rn(th, 1.2);
        __syncwarp();
        if constexpr (RESID) {  // localisation step - 1 under the K children of every parent
          const size_t row = (size_t)ck.loc_off + (size_t)t * L + step - 1;
          k3_emit_resid<D, KS>(a.resid[0] + row, a.resid[1] + row * D, bufP, capP, nP, K, cl, l2,
                               [&](int p, int r) { return P.LT[r + K * curP[p]] + (stay ? Lps[r] : 0.0); }, lane);
        }
        if (step == L - 1) {  // last step: no fusion (tracking.py:591)
          nP = nC;
          LhP = LhC;
          break;
        }

        // ---- greedy grouping from this track alone (tracking.py:667-698 with one leader track) ----
        const double th_lo = __dmul_rn(th, 1.0 - 1e-14), th_hi = __dmul_rn(th, 1.0 + 1e-14);
        // does the leader (ci, mi, si) capture the candidate (cj, mj, sj)?
        auto captures = [&](unsigned long long ci, const double* mi, const double* si, unsigned long long cj, const double* mj,
                            const double* sj) -> bool {
          if (use_window && cj == ci) return true;
          if ((cj & rowmask) != (ci & rowmask)) return false;
          double am = 0.0, as = 0.0;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) {
            const double v = fabs(__dsub_rn(mj[dim], mi[dim]));
            am = (dim == 0) ? v : __dadd_rn(am, v);
          }
          am = (D == 2) ? __dmul_rn(am, 0.5) : ((D == 1) ? am : __ddiv_rn(am, (double)D));
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            const double v = fabs(__dsub_rn(sj[k], si[k]));
            as = (k == 0) ? v : __dadd_rn(as, v);
          }
          as = (KS == 2) ? __dmul_rn(as, 0.5) : ((KS == 1) ? as : __ddiv_rn(as, (double)KS));
          // one leader track: mean(bool over KS comps) > 0.8  <=>  every component passes
          // fl(x / s) < th decided without a division unless x is within 1e-14 (relative) of th*s
          bool ok = true;
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            const double lo = __dmul_rn(th_lo, sj[k]), hi = __dmul_rn(th_hi, sj[k]);
            bool pm = am < lo, ps = as < lo;
            if (!pm && !(am > hi)) pm = k3_div_lt(am, sj[k], th);
            if (!ps && !(as > hi)) ps = k3_div_lt(as, sj[k], th);
            ok = ok && pm && ps;
          }
          return ok;
        };
        int nG = 0, off = 0;
        if (FOLLOW) {  // the chunk's shared plan: member lists of this step
          const int32_t* plan = a.splan + (size_t)wk.chunk * a.splan_stride;
          const int32_t* pl = plan + 2 * a.maxL + (size_t)step * (2 * cap + 1);
          nG = plan[a.maxL + step];
          if (plan[step] != nC || nG < 1 || nG > nC) errc = 1;  // (cannot happen: same expansion, same groups)
          else {
            for (int g = lane; g <= nG; g += 32) goff[g] = pl[g];
            for (int c = lane; c < nC; c += 32) order[c] = pl[cap + 1 + c];
            off = nC;
          }
          __syncwarp();
        } else if (reg_grouping) {
          // lane holds the children lane and lane + 32; the next leader is the first child nobody captured yet
          double mj0[D], sj0[KS], mj1[D], sj1[KS];
          unsigned long long cj0 = 0, cj1 = 0;
          const bool has0 = lane < nC, has1 = lane + 32 < nC;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) {
            mj0[dim] = has0 ? BC(lane, dim) : 0.0;
            mj1[dim] = has1 ? BC(lane + 32, dim) : 0.0;
          }
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            sj0[k] = has0 ? BC(lane, D + KS + k) : 1.0;
            sj1[k] = has1 ? BC(lane + 32, D + KS + k) : 1.0;
          }
          if (has0) cj0 = codeC[lane];
          if (has1) cj1 = codeC[lane + 32];
          unsigned u0 = __ballot_sync(0xffffffffu, has0), u1 = __ballot_sync(0xffffffffu, has1);
          while (u0 | u1) {
            const int i = u0 ? (__ffs(u0) - 1) : (31 + __ffs(u1));
            double mi[D], si[KS];
#pragma unroll
            for (int dim = 0; dim < D; ++dim) mi[dim] = BC(i, dim);
#pragma unroll
            for (int k = 0; k < KS; ++k) si[k] = BC(i, D + KS + k);
            const unsigned long long ci = codeC[i];
            if (lane == 0) goff[nG] = off;
            const int off_in = off;
#if XT_K3_HLOOP
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {  // (one copy of the predicate: the two halves select their operands)
              const unsigned uh = h ? u1 : u0;
              if (!uh) continue;
              double mj[D], sj[KS];
#pragma unroll
              for (int dim = 0; dim < D; ++dim) mj[dim] = h ? mj1[dim] : mj0[dim];
#pragma unroll
              for (int k = 0; k < KS; ++k) sj[k] = h ? sj1[k] : sj0[k];
              const bool ok = ((uh >> lane) & 1u) && captures(ci, mi, si, h ? cj1 : cj0, mj, sj);
              const unsigned m = __ballot_sync(0xffffffffu, ok);
              if (ok) order[off + __popc(m & lt_mask)] = lane + 32 * h;
              off += __popc(m);
              if (h) u1 &= ~m; else u0 &= ~m;
            }
#else
            if (u0) {
              const bool ok = ((u0 >> lane) & 1u) && captures(ci, mi, si, cj0, mj0, sj0);
              const unsigned m = __ballot_sync(0xffffffffu, ok);
              if (ok) order[off + __popc(m & lt_mask)] = lane;
              off += __popc(m);
              u0 &= ~m;
            }
            if (u1) {
              const bool ok = ((u1 >> lane) & 1u) && captures(ci, mi, si, cj1, mj1, sj1);
              const unsigned m = __ballot_sync(0xffffffffu, ok);
              if (ok) order[off + __popc(m & lt_mask)] = lane + 32;
              off += __popc(m);
              u1 &= ~m;
            }
#endif
            if (off == off_in) {  // leader failed its own test and captured nobody (:725, :700-701)
              errc = 1;
              break;
            }
            ++nG;
          }
          if (lane == 0) goff[nG] = off;
        } else {
          for (int i = 0; i < nC; ++i) {
            if (gid[i] >= 0) continue;  // warp-uniform (memory made visible by __syncwarp)
            double mi[D], si[KS];
#pragma unroll
            for (int dim = 0; dim < D; ++dim) mi[dim] = BC(i, dim);
#pragma unroll
            for (int k = 0; k < KS; ++k) si[k] = BC(i, D + KS + k);
            const unsigned long long ci = codeC[i];
            goff[nG] = off;
            for (int j0 = 0; j0 < nC; j0 += 32) {
              const int j = j0 + lane;
              bool ok = false;
              if (j < nC && gid[j] < 0) {
                double mj[D], sj[KS];
#pragma unroll
                for (int dim = 0; dim < D; ++dim) mj[dim] = BC(j, dim);
#pragma unroll
                for (int k = 0; k < KS; ++k) sj[k] = BC(j, D + KS + k);
                ok = captures(ci, mi, si, codeC[j], mj, sj);
              }
              const unsigned m = __ballot_sync(0xffffffffu, ok);
              if (ok) {
                gid[j] = nG;
                order[off + __popc(m & lt_mask)] = j;
              }
              off += __popc(m);
            }
            if (off == goff[nG]) errc = 1;  // leader failed its own test and captured nobody (:725)
            ++nG;
            __syncwarp();
          }
          if (lane == 0) goff[nG] = off;
          for (int c = lane; c < nC; c += 32)
            if (gid[c] < 0) errc = 1;  // tracking.py:700-701
        }
        if (errc == 0 && nG * K > cap) {  // the next expansion would not fit (history rows are sized for it)
          errc = 2;
          if (lane == 0) atomicMax(&a.err_need[wi], nG * K);
        }
        errc = __reduce_max_sync(0xffffffffu, errc);
        __syncwarp();
        if (errc) break;

        // ---- merge, lane = group (tracking.py:723-741); record normalised weights ----
        if (lane == 0) recN[step] = nC;
        const int rows_out = rows_cmp;  // window rows kept (older rows never influence a decision)
        double* rw = recW + (size_t)step * cap;
        uint16_t* rg = recGid + (size_t)step * cap;
        int nM = 0;  // groups of several members, listed in gid[] (free after the grouping)
        for (int g0 = 0; g0 < nG; g0 += 32) {
          const int g = g0 + lane;
          bool multi = false;
          if (g < nG) {
            const int o = goff[g], n = goff[g + 1] - o;
            const int c0 = order[o];
            if (n == 1) {
#pragma unroll
              for (int q = 0; q < CO; ++q) BP(g, q) = BC(c0, q);
              rw[c0] = 1.0;
              rg[c0] = (uint16_t)g;
              if constexpr (PATH) {
                K3_PATH_PTRS;
                pa.vP[g] = pa.vC[c0];
                pa.recArg[(size_t)step * capP + g] = (uint16_t)c0;
              }
              if (!FOLLOW) {  // (history window and codes only serve this track's own decisions)
                const int lab = label(c0), p0 = c0 / K;
                for (int s = 0; s < nS; ++s) HISTN(g, 0, s) = (lab == s) ? 1.0 : 0.0;
                #pragma unroll 1
                for (int it = nS; it < rows_out * nS; ++it) base[hN + it * capP + g] = base[hP + (it - nS) * capP + p0];
                // the window code of an unmerged sequence is its own (codes are the per-row argmax of the window)
                codeP[g] = codeC[c0];
              }
            } else {
              multi = true;
              double mx = BC(c0, D + 2 * KS);
              #pragma unroll 1
              for (int k = 1; k < n; ++k) mx = fmax(mx, BC(order[o + k], D + 2 * KS));
              double sw = 0.0, am[D], as2[KS];
              #pragma unroll 1
              for (int k = 0; k < n; ++k) {
                const int c = order[o + k];
                const double w = k3_exp(__dsub_rn(BC(c, D + 2 * KS), mx));
                aC[c] = w;  // (aC is only used after the forward pass: free scratch here)
                rg[c] = (uint16_t)g;
                sw = (k == 0) ? w : __dadd_rn(sw, w);
#pragma unroll
                for (int dim = 0; dim < D; ++dim) {
                  const double v = __dmul_rn(w, BC(c, dim));
                  am[dim] = (k == 0) ? v : __dadd_rn(am[dim], v);
                }
#pragma unroll
                for (int k2 = 0; k2 < KS; ++k2) {
                  const double v = __dmul_rn(w, BC(c, D + k2));
                  as2[k2] = (k == 0) ? v : __dadd_rn(as2[k2], v);
                }
              }
#pragma unroll
              for (int dim = 0; dim < D; ++dim) BP(g, dim) = __ddiv_rn(am[dim], sw);
#pragma unroll
              for (int k2 = 0; k2 < KS; ++k2) BP(g, D + k2) = __ddiv_rn(as2[k2], sw);
              BP(g, D + 2 * KS) = __dadd_rn(k3_log(sw), mx);
              #pragma unroll 1
              for (int k = 0; k < n; ++k) {  // the recorded weights, normalised
                const int c = order[o + k];
                rw[c] = __ddiv_rn(aC[c], sw);
              }
              aP[g] = sw;  // (aP, like aC, is only used after the forward pass) for the history rows below
              if constexpr (PATH) {  // the group's path score: its best member's (ties: the first in member order)
                K3_PATH_PTRS;
                double bv = pa.vC[c0];
                int bc = c0;
                #pragma unroll 1
                for (int k = 1; k < n; ++k) {
                  const int c = order[o + k];
                  if (pa.vC[c] > bv) {
                    bv = pa.vC[c];
                    bc = c;
                  }
                }
                pa.vP[g] = bv;
                pa.recArg[(size_t)step * capP + g] = (uint16_t)bc;
              }
            }
            curP[g] = c0 % nS;  // newest true state (curP / codeP are only read by the expansion)
          }
          if (!FOLLOW) {
            const unsigned mm = __ballot_sync(0xffffffffu, multi);
            if (multi) gid[nM + __popc(mm & lt_mask)] = g;
            nM += __popc(mm);
          }
        }
        if (!FOLLOW && nM > 0) {
          // Groups of several members: weighted mean of the members' window rows (tracking.py:733, member order), one lane
          // per (group, row, state) over all of them at once, then their window codes (argmax per row, ties -> lowest
          // state), lane = group again.
          __syncwarp();
          const int items = rows_out * nS, tot = nM * items;
          const float inv_items = 1.0f / (float)items;
          for (int idx = lane; idx < tot; idx += 32) {
            const int gm = (int)(((float)idx + 0.5f) * inv_items), it = idx - gm * items;
            const int row = it / nS, st = it - row * nS;
            const int g = gid[gm];
            const int o = goff[g], n = goff[g + 1] - o;
            double acc = 0.0;
            #pragma unroll 1
            for (int k = 0; k < n; ++k) {
              const int c = order[o + k];
              const double hv = (row == 0) ? ((label(c) == st) ? 1.0 : 0.0) : base[hP + (it - nS) * capP + c / K];
              const double v = __dmul_rn(aC[c], hv);  // aC[c] = exp(LP_c - max) of this fusion
              acc = (k == 0) ? v : __dadd_rn(acc, v);
            }
            base[hN + it * capP + g] = __ddiv_rn(acc, aP[g]);
          }
          __syncwarp();
          for (int gm = lane; gm < nM; gm += 32) {
            const int g = gid[gm];
            unsigned long long code = 0;
            #pragma unroll 1
            for (int row = 0; row < rows_out; ++row) {
              int best = 0;
              double bv = HISTN(g, row, 0);
              for (int st = 1; st < nS; ++st) {
                const double v = HISTN(g, row, st);
                if (v > bv) { bv = v; best = st; }
              }
              code |= (unsigned long long)best << (bits * row);
            }
            codeP[g] = code;
          }
        }
        __syncwarp();
        if (REFINE) {  // entry step - 1: the merged sequences (refined_localization.py:183-186)
          for (int g = lane; g < nG; g += 32) {
            double* e1 = dmp + ((size_t)(step - 1) * a.capD + g) * COD;
#pragma unroll
            for (int dim = 0; dim < D; ++dim) e1[dim] = BP(g, dim);
#pragma unroll
            for (int k = 0; k < KS; ++k) e1[D + k] = __dsqrt_rn(BP(g, D + k));
            e1[D + KS] = BP(g, D + 2 * KS);
            e1[D + KS + 1] = (double)curP[g];
          }
        }
        if (entn && lane == 0) entn[step - 1] = nG;
        {
          const int tmp = hP;
          hP = hN;
          hN = tmp;
        }
        nP = nG;
        LhP = LhC;
        __syncwarp();
      }
      if (errc) {
        if (lane == 0) atomicMax(&a.err[wi], errc);
        continue;
      }

      // ---- end of track: last-localisation term, optional leave expansion (tracking.py:613-639) ----
      const bool have_children = L > 2;  // final sequences live in bufC (children of the last step) or bufP (L == 2)
      double* FB = have_children ? bufC : bufP;
      const int fbs = have_children ? cap : capP;  // slot pitch of that buffer
      double clast[D];
#pragma unroll
      for (int dim = 0; dim < D; ++dim) clast[dim] = Cp[(size_t)(LROW(L - 1) * D + dim) * npad];
      if (VAR) var_row(L - 1);
      if constexpr (RESID) {  // the last localisation under the final sequences (the bleaching end sums its heads in Lsm)
        const size_t row = (size_t)ck.loc_off + (size_t)t * L + L - 1;
        k3_emit_resid<D, KS>(a.resid[0] + row, a.resid[1] + row * D, FB, fbs, nP, 1, clast, l2,
                             [&](int c, int) { return ck.isBL ? Lsm[c % nS] : 0.0; }, lane);
      }
      double vmax = -INFINITY;
      #pragma unroll 1
      for (int c = lane; c < nP; c += 32) {
        double term = 0.0;
#pragma unroll
        for (int dim = 0; dim < D; ++dim) {
          const int k = (KS == 1) ? 0 : dim;
          const double q = __dadd_rn(FB[(D + k) * fbs + c], l2[k]);
          const double df = __dsub_rn(clast[dim], FB[dim * fbs + c]);
          const double tt = __dsub_rn(__dmul_rn(-0.5, k3_log(__dmul_rn(XT_TWO_PI, q))), __ddiv_rn(__dmul_rn(df, df), __dmul_rn(2.0, q)));
          term = (dim == 0) ? tt : __dadd_rn(term, tt);
        }
        double v = FB[(D + 2 * KS) * fbs + c] + term;
        if (REFINE) {
          // last entry: the unfused sequences of the last step with the end-of-track term and the initial fraction of
          // their newest state (refined_localization.py:188-194: the last stored LP is the array updated in place)
          v = __dadd_rn(FB[(D + 2 * KS) * fbs + c], __dadd_rn(term, a.LF[c % nS]));
          double* e2 = dmp + ((size_t)(L - 2) * a.capD + c) * COD;
#pragma unroll
          for (int dim = 0; dim < D; ++dim) e2[dim] = FB[dim * fbs + c];
#pragma unroll
          for (int k = 0; k < KS; ++k) e2[D + k] = have_children ? FB[(D + KS + k) * fbs + c] : __dsqrt_rn(FB[(D + k) * fbs + c]);
          e2[D + KS] = v;
          e2[D + KS + 1] = (double)(c % nS);
          continue;
        }
        if constexpr (PATH) {  // the final path score, in place of V
          K3_PATH_PTRS;
          double* fv = have_children ? pa.vC : pa.vP;
          double vs = fv[c] + term;
          if (ck.isBL) vs += Lsm[c % nS];
          fv[c] = vs;
        }
        if (ck.isBL) v += Lsm[c % nS];
        aC[c] = v;
        vmax = fmax(vmax, v);
      }
      if (REFINE) {
        if (entn && lane == 0) entn[L - 2] = nP;
        __syncwarp();
        continue;  // no posteriors in this mode
      }
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o2));
      double ssum = 0.0;
      #pragma unroll 1
      for (int c = lane; c < nP; c += 32) {
        const double e = k3_exp(aC[c] - vmax);
        aC[c] = e;
        ssum += e;
      }
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) ssum += __shfl_xor_sync(0xffffffffu, ssum, o2);
      const double inv = 1.0 / ssum;
      #pragma unroll 1
      for (int c = lane; c < nP; c += 32) aC[c] *= inv;
      __syncwarp();
      if constexpr (PATH) {
        // the best final sequence (ties: the lowest index), then the backtrack along the recorded argmax members
        K3_PATH_PTRS;
        const double* fv = have_children ? pa.vC : pa.vP;
        double pbest = -INFINITY;
        int pc = -1;
        #pragma unroll 1
        for (int c = lane; c < nP; c += 32) {
          if (pc < 0 || fv[c] > pbest) {
            pbest = fv[c];
            pc = c;
          }
        }
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
          const double ov = __shfl_xor_sync(0xffffffffu, pbest, o2);
          const int oc = __shfl_xor_sync(0xffffffffu, pc, o2);
          if (oc >= 0 && (pc < 0 || ov > pbest || (ov == pbest && oc < pc))) {
            pbest = ov;
            pc = oc;
          }
        }
        if (lane == 0) {  // the label of the chosen child at every level, then its parent's best member
          int8_t* lab = (int8_t*)a.path[0] + (size_t)ck.loc_off + (size_t)t * L;
          int c = pc;
          #pragma unroll 1
          for (int s = L - 1; s >= 2; --s) {
            lab[s] = (int8_t)label(c);
            const int p = c / K;
            c = s > 2 ? (int)pa.recArg[(size_t)(s - 1) * capP + p] : p;
          }
          lab[1] = (int8_t)(c % nS);  // initial sequence c = h0 + nS*h1: row 1 = h0, row 0 = h1
          lab[0] = (int8_t)(c / nS);
          ((double*)a.path[1])[(size_t)ck.trk_off + t] = pbest - (log(ssum) + vmax);
        }
      }

      // ---- backward sweep over the recorded lattice (deterministic warp reductions) ----
      // aC holds the posterior of the sequences *after* the expansion of `step`.
      auto emit_row = [&](int row, const double* av, int n, int mode) {
        // mode 0: label = int8-wrapped child index; 1: j % nS; 2: j / nS
        if ((NSC == 2 || NSC == 4) && mode != 2) {
          // the label of a child is the residue of its lane: one strided sum, reduced across the lanes of a residue
          double acc = 0.0;
          #pragma unroll 1
          for (int c = lane; c < n; c += 32) acc += av[c];
#pragma unroll
          for (int o2 = 16; o2 >= (NSC ? NSC : 1); o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
          if (lane < nS) out[row * nS + lane] = acc;
          return;
        }
        for (int s = 0; s < nS; ++s) {
          double acc = 0.0;
          #pragma unroll 1
          for (int c = lane; c < n; c += 32) {
            const int lab = (mode == 0) ? label(c) : ((mode == 1) ? (c % nS) : (c / nS));
            if (lab == s) acc += av[c];
          }
#pragma unroll
          for (int o2 = 16; o2 > 0; o2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o2);
          if (lane == 0) out[row * nS + s] = acc;
        }
      };
      int nC = nP;
      const double* init_src = aC;  // L == 2: the final sequences are the initial ones
      for (int step = L - 1; step >= 2; --step) {
        // the fusion records of the step before (global memory) are fetched under this level's reductions
        const int nCprev = step > 2 ? recN[step - 1] : 0;
        const bool pre = step > 2 && nCprev <= 64;
        const double* rwp = recW + (size_t)(step - 1) * cap;
        const uint16_t* rgp = recGid + (size_t)(step - 1) * cap;
        double w0 = 0.0, w1 = 0.0;
        int q0 = 0, q1 = 0;
        if (pre) {
          if (lane < nCprev) { w0 = rwp[lane]; q0 = rgp[lane]; }
          if (lane + 32 < nCprev) { w1 = rwp[lane + 32]; q1 = rgp[lane + 32]; }
        }
        emit_row(step, aC, nC, 0);  // newest row of this level: forward-time index = step
        if constexpr (PAIRS) {
          double* po = a.pairs + ((size_t)(ck.loc_off - ck.trk_off) + (size_t)t * (L - 1) + step - 1) * nS * nS;
          if (step > 2) k3_emit_pairs<NSC>(po, aC, nCprev, rwp, rgp, nS, wrap, lane);
          else k3_emit_pairs<NSC>(po, aC, nS * nS, nullptr, nullptr, nS, wrap, lane);
        }
        const int nPar = nC / K;
        for (int p = lane; p < nPar; p += 32) {
          double sacc = 0.0;
          #pragma unroll 1
          for (int r = 0; r < K; ++r) sacc += aC[p * K + r];
          aP[p] = sacc;
        }
        __syncwarp();
        if (step > 2) {  // the parents of `step` are the groups of step-1
          if (pre) {
            if (lane < nCprev) aC[lane] = aP[q0] * w0;
            if (lane + 32 < nCprev) aC[lane + 32] = aP[q1] * w1;
          } else {
            #pragma unroll 1
            for (int c = lane; c < nCprev; c += 32) aC[c] = aP[rgp[c]] * rwp[c];
          }
          nC = nCprev;
        } else {
          init_src = aP;
        }
        __syncwarp();
      }
      // initial sequences j = h0 + nS*h1: row 1 = h0 (newest of the two), row 0 = h1 (oldest)
      emit_row(1, init_src, nS * nS, 1);
      emit_row(0, init_src, nS * nS, 2);
      if constexpr (PAIRS) {  // initial sequence c = h0 + nS*h1 is the pair (h1, h0): flat index h1*nS + h0 = c
        double* po = a.pairs + ((size_t)(ck.loc_off - ck.trk_off) + (size_t)t * (L - 1)) * nS * nS;
        for (int c = lane; c < nS * nS; c += 32) po[c] = init_src[c];
      }
      __syncwarp();
    }
  }
#undef BP
#undef BC
#undef HIX
#undef HISTP
#undef HISTN
#undef DDX
#undef LROW
#undef K3_PATH_PTRS
}
