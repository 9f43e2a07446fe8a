// K4 — segment-length histogram (SURVEY.md §8(f) N2; reference extrack/histograms.py:26-258
// P_segment_len, :265-373 len_hist): the same Gaussian-product recursion as the likelihood, but with
// the *literal* top-max_nb_states pruning per track (descending sort of LP + log-density of the next
// localisation, histograms.py:183-206) and a tally of the run lengths of every surviving state sequence.
//
// One CTA per chunk of <= 50 tracks (persistent over the chunk list), one track at a time: the chunk is
// the reference's unit for the rescale of final log-probabilities above 600 (histograms.py:243-244: if
// any LP of the chunk exceeds 600, every column j is shifted by max over the chunk's tracks of LP[:, j]
// minus 600 — a per-column shift, reproduced): the CTA tallies optimistically while it tracks the column
// maxima, and repeats the chunk with the shifts if the chunk maximum exceeded 600.
// The live sequences of the track — moments,
// log-probabilities LP / LL, newest state — sit in shared memory as two sets (parents / children).
// Instead of the reference's history matrix cur_Bs[nT, nB, L], which it re-gathers at every pruning
// step, each step writes one lattice record per surviving sequence (parent slot | newest state << 16)
// to a per-CTA scratch; histories are recovered once, at the end, by walking the records back.
// Arithmetic follows the reference's operation order (no FMA contraction) so that the sort keys agree
// with numpy's to the last bit up to the library log; the sort is a bitonic network over
// (key, index) pairs with a total order: descending key, equal keys by descending index (what a stable
// ascending argsort followed by [::-1] gives; numpy's default sort leaves it unspecified).
// Reproduced quirks: LL keeps the *last* k ranks of the order while everything else keeps the first k
// (histograms.py:202); end_p_stay = p_stay[s] only if newest == previous == s, else p_stay[0] (:224);
// no transition term in the leave expansion (:220); runs of length L are not counted (:251).
#pragma once
#include "xt_common.cuh"

#define XT_SEG_THREADS 256

struct K4Args {
  const XtChunk* chunks;
  const double* soa;
  int32_t n_chunks;
  int32_t cap;              // sequence slots per set
  int32_t n2;               // power of two >= cap (sort network size)
  int32_t Lmax;
  uint32_t* lattice;        // [gridDim.x][Lmax][cap]
  double* colmax;           // [gridDim.x][cap]: per column, max over the chunk's tracks of the final LP
  double* hist;             // [n_chunks][Lmax][nS], rows (L-1) x nS of every chunk written once by its CTA
  int32_t* flags;           // [0]: bit 0 = some chunk needed the > 600 rescale (informational); [1]: next position in corder
  const int32_t* corder;    // chunk ids, longest tracks first (CTAs take the next one when they are done)
  double leave_LL[XT_MAX_HEADS];  // log(pBL + (1-e) - pBL(1-e)) per head = newest + nS * previous
  // test seam (P_segment_len outputs) for the tracks of chunk dbg_chunk, or nullptr
  double* dbg_LP;           // [nT][nBf]
  int8_t* dbg_Bs;           // [nT][nBf][L]
  int32_t dbg_chunk, dbg_nBf;
};

// two sets of (m[d], s2[KS], LP, LL), sort keys and indices, the chunk's histogram (FP64) and one track's fixed-point
// histogram (int64), reduction slots, newest states
__host__ __device__ inline size_t xt_seg_smem(int d, int KS, int cap, int n2, int Lmax, int nS) {
  return (size_t)2 * cap * (d + KS + 2) * 8 + (size_t)n2 * 12 + (size_t)2 * cap + 16 + (size_t)2 * Lmax * nS * 8 + 64;
}

// Fixed-point scale of a track's histogram: 2^(62 - bits(L)), so that L * scale < 2^62.  A track's weights sum to 1 and a
// sequence adds its weight to one bin at most L times, so a bin stays below 2^62 plus the rounding of its additions
// (< 2^15 * L of them): integer additions, exact and independent of their order.  The scale depends on the chunk's own L
// only, so a chunk's histogram does not depend on what else is uploaded.
__device__ __forceinline__ int xt_seg_fix_exp(int L) { return 62 - (32 - __clz(L)); }

// "x comes before y" in the pruning order: descending key, equal keys by descending index
__device__ __forceinline__ bool xt_seg_before(double kx, int ix, double ky, int iy) {
  return kx > ky || (kx == ky && ix > iy);
}

template <int D, int KS>
__device__ __forceinline__ double xt_seg_logdens(const double (&Cn)[D], const double* m, const double* s2, int j, int cap,
                                                 const double (&l2)[KS]) {
  // sum over dims of (-0.5 log(2 pi (s2 + l2)) - (Cn - m)^2 / (2 (s2 + l2)))  (histograms.py:187-188, :238-239)
  double acc = 0.0;
  double lg0 = 0.0, n0 = 0.0;
  if (KS == 1) {
    n0 = __dadd_rn(s2[j], l2[0]);
    lg0 = __dmul_rn(-0.5, log(__dmul_rn(XT_TWO_PI, n0)));
  }
#pragma unroll
  for (int dim = 0; dim < D; ++dim) {
    double ns, lg;
    if (KS == 1) {
      ns = n0;
      lg = lg0;
    } else {
      ns = __dadd_rn(s2[dim * cap + j], l2[dim]);
      lg = __dmul_rn(-0.5, log(__dmul_rn(XT_TWO_PI, ns)));
    }
    const double df = __dadd_rn(Cn[dim], -m[dim * cap + j]);
    const double t = __dadd_rn(lg, -__ddiv_rn(__dmul_rn(df, df), __dmul_rn(2.0, ns)));
    acc = dim == 0 ? t : __dadd_rn(acc, t);
  }
  return acc;
}

// Bitonic sort of the n2 (key, index) pairs in keys[] / ord[] into the pruning order (xt_seg_before), with the elements
// in registers: thread t holds the EPT consecutive elements EPT*t .. EPT*t + EPT - 1 for the whole network.
// Compare-exchange distances below EPT run inside the thread, distances up to 16 * EPT between the lanes of a warp with
// shuffles, and only the longer ones (thread distance >= 32) go through shared memory: for 1024 pairs on 256 threads that
// is 6 of the 55 stages (the first version passed 36 stages through shared memory with a CTA barrier each).
// All XT_SEG_THREADS threads call it; n2 is a power of two, 4 <= n2 <= EPT * XT_SEG_THREADS.  The total order (keys,
// then indices, all indices distinct) makes the result independent of the network.
template <int EPT>
__device__ __forceinline__ void xt_seg_sort(double* keys, int* ord, int n2, int tid) {
  static_assert(EPT == 4 || EPT == 8 || EPT == 16, "elements per thread");
  double kk[EPT];
  int ii[EPT];
  const int base = EPT * tid;
  const bool live = base < n2;  // (n2 is a multiple of EPT: a thread is live with all of its elements or none)
  if (live) {
#pragma unroll
    for (int e = 0; e < EPT; e += 2) {
      const double2 v = reinterpret_cast<const double2*>(keys)[(base + e) >> 1];
      kk[e] = v.x;
      kk[e + 1] = v.y;
    }
#pragma unroll
    for (int e = 0; e < EPT; e += 4) {
      const int4 v = reinterpret_cast<const int4*>(ord)[(base + e) >> 2];
      ii[e] = v.x; ii[e + 1] = v.y; ii[e + 2] = v.z; ii[e + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      kk[e] = -INFINITY;
      ii[e] = -1 - (base + e);
    }
  }
  for (int k = 2; k <= n2; k <<= 1) {
    int jj = k >> 1;
    for (; jj >= 32 * EPT; jj >>= 1) {
      // partner in another warp: through shared memory (own elements out, barrier, partner's elements in, barrier)
      if (live) {
#pragma unroll
        for (int e = 0; e < EPT; e += 2) reinterpret_cast<double2*>(keys)[(base + e) >> 1] = make_double2(kk[e], kk[e + 1]);
#pragma unroll
        for (int e = 0; e < EPT; e += 4) reinterpret_cast<int4*>(ord)[(base + e) >> 2] = make_int4(ii[e], ii[e + 1], ii[e + 2], ii[e + 3]);
      }
      __syncthreads();
      if (live) {
        const int pb = base ^ jj;  // (jj is a multiple of EPT: the partner thread's elements, slot by slot)
        const bool keep_first = ((base & jj) == 0) == ((base & k) == 0);
#pragma unroll
        for (int e = 0; e < EPT; e += 2) {
          const double2 v = reinterpret_cast<const double2*>(keys)[(pb + e) >> 1];
          const int2 w = reinterpret_cast<const int2*>(ord)[(pb + e) >> 1];
          const bool f0 = xt_seg_before(kk[e], ii[e], v.x, w.x), f1 = xt_seg_before(kk[e + 1], ii[e + 1], v.y, w.y);
          if (f0 != keep_first) { kk[e] = v.x; ii[e] = w.x; }
          if (f1 != keep_first) { kk[e + 1] = v.y; ii[e + 1] = w.y; }
        }
      }
      __syncthreads();
    }
    for (; jj >= EPT; jj >>= 1) {
      // partner in the same warp
      const int lm = jj / EPT;
      const bool keep_first = ((base & jj) == 0) == ((base & k) == 0);
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const double ok = __shfl_xor_sync(0xffffffffu, kk[e], lm);
        const int oi = __shfl_xor_sync(0xffffffffu, ii[e], lm);
        if (xt_seg_before(kk[e], ii[e], ok, oi) != keep_first) { kk[e] = ok; ii[e] = oi; }
      }
    }
    // both elements in this thread: the remaining distances, with compile-time register indices
#pragma unroll
    for (int j2 = EPT / 2; j2 >= 1; j2 >>= 1) {
      if (j2 <= jj) {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
          if ((e & j2) == 0) {
            const int x = e | j2;
            const bool up = (((base + e) & k) == 0);
            if (xt_seg_before(kk[x], ii[x], kk[e], ii[e]) == up) {
              const double tk = kk[e]; kk[e] = kk[x]; kk[x] = tk;
              const int ti = ii[e]; ii[e] = ii[x]; ii[x] = ti;
            }
          }
        }
      }
    }
  }
  if (live) {  // (only the order is read afterwards)
#pragma unroll
    for (int e = 0; e < EPT; e += 4) reinterpret_cast<int4*>(ord)[(base + e) >> 2] = make_int4(ii[e], ii[e + 1], ii[e + 2], ii[e + 3]);
  }
  __syncthreads();
}

template <int D, int KS, int EPT = 4>
__global__ void __launch_bounds__(XT_SEG_THREADS, EPT == 4 ? 2 : 1) k4_seglen(const K4Args a, const xt_params P) {
  constexpr int NT = XT_SEG_THREADS;
  const int tid = threadIdx.x;
  const int nS = P.nS, cap = a.cap, n2 = a.n2;
  extern __shared__ __align__(16) double k4_smem[];
  double* setA = k4_smem;
  double* setB = setA + (size_t)cap * (D + KS + 2);
  double* keys = setB + (size_t)cap * (D + KS + 2);
  int* ord = reinterpret_cast<int*>(keys + n2);
  double* shist = reinterpret_cast<double*>(ord + n2 + (n2 & 1));                         // the chunk's rows
  unsigned long long* sfix = reinterpret_cast<unsigned long long*>(shist + (size_t)a.Lmax * nS);  // one track's rows
  double* sred = reinterpret_cast<double*>(sfix + (size_t)a.Lmax * nS);  // [8]
  uint8_t* stA = reinterpret_cast<uint8_t*>(sred + 8);
  uint8_t* stB = stA + cap;
  uint32_t* lat = a.lattice + (size_t)blockIdx.x * a.Lmax * cap;
  double l2[KS];
#pragma unroll
  for (int k = 0; k < KS; ++k) l2[k] = P.l2[k];
  const int kmax = P.max_nb_states;

  double* colmax = a.colmax + (size_t)blockIdx.x * cap;
  __shared__ double s_part[NT / 32], s_max[NT / 32];
  __shared__ int s_again;
  __shared__ int s_next;
  for (;;) {
   if (tid == 0) s_next = atomicAdd(&a.flags[1], 1);
   __syncthreads();
   const int pos = s_next;
   __syncthreads();
   if (pos >= a.n_chunks) break;
   const int ci = a.corder[pos];
   const XtChunk ck = a.chunks[ci];
   const int L = ck.L;
   // bin i of shist / sfix belongs to thread i % NT outside the run-length tally (reset, fold, store)
   for (int i = tid; i < (L - 1) * nS; i += NT) {
     shist[i] = 0.0;
     sfix[i] = 0ull;
   }
   for (int i = tid; i < cap; i += NT) colmax[i] = -INFINITY;
   const double fix_scale = ldexp(1.0, xt_seg_fix_exp(L)), fix_inv = ldexp(1.0, -xt_seg_fix_exp(L));
   double cmax = -INFINITY;  // this thread's share of the chunk maximum of the final LP
   for (int pass = 0; pass < 2; ++pass) {
   for (int tk = 0; tk < ck.nT; ++tk) {
    struct { int32_t chunk, t0; } wk = {ci, tk};
    const size_t npad = (size_t)ck.nTpad;
    const double* Cs = a.soa + ck.xyz_off + wk.t0;
    auto loc = [&](int i, double (&c)[D]) {
#pragma unroll
      for (int dim = 0; dim < D; ++dim) c[dim] = Cs[((size_t)i * D + dim) * npad];
    };
    double* par = setA;
    double* chi = setB;
    uint8_t* stp = stA;
    uint8_t* stc = stB;
#define SEG_M(set) (set)
#define SEG_S(set) ((set) + (size_t)D * cap)
#define SEG_LP(set) ((set) + (size_t)(D + KS) * cap)
#define SEG_LL(set) ((set) + (size_t)(D + KS + 1) * cap)
    // ---- first localisation: nS^2 sequences, head = newest + nS * oldest (histograms.py:104-140) ----
    int nB = nS * nS;
    {
      double c0[D];
      loc(0, c0);
      for (int h = tid; h < nB; h += NT) {
#pragma unroll
        for (int dim = 0; dim < D; ++dim) SEG_M(par)[dim * cap + h] = c0[dim];
#pragma unroll
        for (int k = 0; k < KS; ++k) SEG_S(par)[k * cap + h] = __dadd_rn(l2[k], P.dd[h]);
        SEG_LP(par)[h] = __dadd_rn(P.LT[h], P.LF[h]);
        SEG_LL(par)[h] = (1 >= P.min_len) ? P.Lp_stay[h % nS] : 0.0;
        stp[h] = (uint8_t)(h % nS);
        lat[h] = (uint32_t)(h / nS) | ((uint32_t)(h % nS) << 16);  // record 0: "parent" = oldest state
      }
    }
    __syncthreads();
    // ---- steps 2..L-1 (histograms.py:143-209) ----
    for (int step = 2; step <= L - 1; ++step) {
      const int nC = nB * nS;
      double Ci[D], Cn[D];
      loc(step - 1, Ci);
      loc(step, Cn);  // step <= L-1
      const bool prune = step < L - 1 && nC > kmax;
      // One thread per parent: the new mean, the quadratic term and the log term of the update depend on the parent only
      // (every child of a parent consumes the same localisation from the same moments; only the diffusion length of
      // the step, hence s2, differs between the children), so they are computed once per parent instead of once per
      // child; the children then get their own s2, weights, lattice record and - in a pruning step - their sort key.
      for (int p = tid; p < nB; p += NT) {
        double q[KS], sp[KS], mc[D];
#pragma unroll
        for (int k = 0; k < KS; ++k) {
          sp[k] = SEG_S(par)[k * cap + p];
          q[k] = __dadd_rn(l2[k], sp[k]);
        }
        double quad = 0.0, lgs = 0.0;
#pragma unroll
        for (int dim = 0; dim < D; ++dim) {
          const int k = KS == 1 ? 0 : dim;
          const double mp = SEG_M(par)[dim * cap + p];
          mc[dim] = __ddiv_rn(__dadd_rn(__dmul_rn(mp, l2[k]), __dmul_rn(Ci[dim], sp[k])), q[k]);
          const double df = __dadd_rn(Ci[dim], -mp);
          const double t = __ddiv_rn(__dmul_rn(df, df), __dmul_rn(2.0, q[k]));
          quad = dim == 0 ? t : __dadd_rn(quad, t);
          if (KS > 1) {
            const double lg = __dmul_rn(-0.5, log(__dmul_rn(XT_TWO_PI, q[k])));
            lgs = dim == 0 ? lg : __dadd_rn(lgs, lg);
          }
        }
        if (KS == 1) lgs = __dmul_rn((double)D * -0.5, log(__dmul_rn(XT_TWO_PI, q[0])));
        const double LC = __dadd_rn(lgs, -quad);
        const double LPp = SEG_LP(par)[p], LLp = SEG_LL(par)[p];
        const int hb = nS * (int)stp[p];
        double dn[D];  // next localisation minus the children's common mean (sort key)
        if (prune) {
#pragma unroll
          for (int dim = 0; dim < D; ++dim) dn[dim] = __dadd_rn(Cn[dim], -mc[dim]);
        }
        for (int s = 0; s < nS; ++s) {
          const int j = p * nS + s, h = s + hb;
          const double dd = P.dd[h];
          double sc[KS];
#pragma unroll
          for (int dim = 0; dim < D; ++dim) SEG_M(chi)[dim * cap + j] = mc[dim];
#pragma unroll
          for (int k = 0; k < KS; ++k) {
            sc[k] = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(dd, l2[k]), __dmul_rn(dd, sp[k])), __dmul_rn(l2[k], sp[k])), q[k]);
            SEG_S(chi)[k * cap + j] = sc[k];
          }
          const double lpc = __dadd_rn(LPp, __dadd_rn(P.LT[h], LC));
          SEG_LP(chi)[j] = lpc;
          SEG_LL(chi)[j] = (step >= P.min_len) ? __dadd_rn(LLp, P.Lp_stay[s]) : LLp;
          stc[j] = (uint8_t)s;
          if (!prune) {
            lat[(size_t)(step - 1) * cap + j] = (uint32_t)p | ((uint32_t)s << 16);
          } else {
            // key = LP + log-density of the next localisation (histograms.py:186-196; same operations as xt_seg_logdens)
            double acc = 0.0, lg0 = 0.0, n0 = 0.0;
            if (KS == 1) {
              n0 = __dadd_rn(sc[0], l2[0]);
              lg0 = __dmul_rn(-0.5, log(__dmul_rn(XT_TWO_PI, n0)));
            }
#pragma unroll
            for (int dim = 0; dim < D; ++dim) {
              double ns, lg;
              if (KS == 1) {
                ns = n0;
                lg = lg0;
              } else {
                ns = __dadd_rn(sc[dim], l2[dim]);
                lg = __dmul_rn(-0.5, log(__dmul_rn(XT_TWO_PI, ns)));
              }
              const double t = __dadd_rn(lg, -__ddiv_rn(__dmul_rn(dn[dim], dn[dim]), __dmul_rn(2.0, ns)));
              acc = dim == 0 ? t : __dadd_rn(acc, t);
            }
            keys[j] = __dadd_rn(lpc, acc);
            ord[j] = j;
          }
        }
      }
      if (prune) {
        for (int j = nC + tid; j < n2; j += NT) {
          keys[j] = -INFINITY;
          ord[j] = -1 - j;
        }
      }
      __syncthreads();
      if (!prune) {
        double* t = par; par = chi; chi = t;
        uint8_t* u = stp; stp = stc; stc = u;
        nB = nC;
        continue;
      }
      xt_seg_sort<EPT>(keys, ord, n2, tid);
      for (int j = tid; j < kmax; j += NT) {
        const int src = ord[j];
        const int srcL = ord[nC - kmax + j];  // histograms.py:202: LL keeps the last k ranks
#pragma unroll
        for (int dim = 0; dim < D; ++dim) SEG_M(par)[dim * cap + j] = SEG_M(chi)[dim * cap + src];
#pragma unroll
        for (int k = 0; k < KS; ++k) SEG_S(par)[k * cap + j] = SEG_S(chi)[k * cap + src];
        SEG_LP(par)[j] = SEG_LP(chi)[src];
        SEG_LL(par)[j] = SEG_LL(chi)[srcL];
        stp[j] = stc[src];
        lat[(size_t)(step - 1) * cap + j] = (uint32_t)(src / nS) | ((uint32_t)(src % nS) << 16);
      }
      nB = kmax;
      __syncthreads();
    }
    // ---- end of track (histograms.py:211-246): last localisation, optional leave expansion ----
    double Cl[D];
    loc(L - 1, Cl);
    // per parent: LPf = LP + logdens(last); weights of its nS leave-children (or itself) in keys[], total in sred
    double part = 0.0, lpmax = -INFINITY;
    for (int p = tid; p < nB; p += NT) {
      double lpf = __dadd_rn(SEG_LP(par)[p], xt_seg_logdens<D, KS>(Cl, SEG_M(par), SEG_S(par), p, cap, l2));
      if (pass == 0) {
        colmax[p] = fmax(colmax[p], lpf);  // (column p of every track of the chunk belongs to this thread)
        cmax = fmax(cmax, lpf);
      } else {
        lpf = __dadd_rn(lpf, -__dadd_rn(colmax[p], -600.0));  // histograms.py:244
      }
      lpmax = fmax(lpmax, lpf);
      double w = 0.0;
      if (ck.isBL) {
        for (int s = 0; s < nS; ++s) {
          const double ll = __dadd_rn(SEG_LL(par)[p], a.leave_LL[s + nS * (int)stp[p]]);
          w += exp(__dadd_rn(lpf, ll));
        }
      } else {
        w = exp(__dadd_rn(lpf, SEG_LL(par)[p]));
      }
      keys[p] = w;
      part += w;
      if (a.dbg_LP && wk.chunk == a.dbg_chunk) {
        const int rep = ck.isBL ? nS : 1;
        for (int s = 0; s < rep; ++s) a.dbg_LP[(size_t)wk.t0 * a.dbg_nBf + (size_t)p * rep + s] = lpf;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      part += __shfl_down_sync(0xffffffffu, part, off);
      lpmax = fmax(lpmax, __shfl_down_sync(0xffffffffu, lpmax, off));
    }
    if ((tid & 31) == 0) {
      s_part[tid >> 5] = part;
      s_max[tid >> 5] = lpmax;
    }
    __syncthreads();
    double tot = 0.0, mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < NT / 32; ++k) {
      tot += s_part[k];
      mx = fmax(mx, s_max[k]);
    }
    (void)mx;
    // ---- histories by walking the lattice back; run lengths (histograms.py:248-258 restated) ----
    for (int p = tid; p < nB; p += NT) {
      const double w = keys[p] / tot;  // in [0, 1], or NaN when every weight of the track underflowed
      // weight in fixed point: integer additions into the track's bins, so the tally does not depend on thread order
      // (a NaN weight goes to the chunk's FP64 row directly: NaN in any order).  The 64-bit addition runs as two native
      // 32-bit shared atomics, the low word's carry added to the high word (a 64-bit shared atomicAdd is a CAS loop).
      const bool fin = isfinite(w);
      const unsigned long long wq = fin ? (unsigned long long)__double2ll_rn(__dmul_rn(w, fix_scale)) : 0ull;
      const unsigned wlo = (unsigned)wq, whi = (unsigned)(wq >> 32);
      auto tally = [&](int bin) {
        if (fin) {
          unsigned* f = reinterpret_cast<unsigned*>(sfix + bin);  // little-endian: [0] low word, [1] high word
          const unsigned old = atomicAdd(f, wlo);
          const unsigned hi = whi + (old + wlo < old ? 1u : 0u);
          if (hi) atomicAdd(f + 1, hi);
        } else {
          atomicAdd(&shist[bin], w);
        }
      };
      int idx = p;
      int cur = -1, run = 0, counted = 0, col = 0;
      int8_t* bs = (a.dbg_Bs && wk.chunk == a.dbg_chunk) ? a.dbg_Bs + ((size_t)wk.t0 * a.dbg_nBf + (size_t)p * (ck.isBL ? nS : 1)) * L
                                                        : nullptr;
      auto visit = [&](int st) {
        if (bs) {
          const int rep = ck.isBL ? nS : 1;
          for (int s = 0; s < rep; ++s) bs[(size_t)s * L + col] = (int8_t)st;
        }
        ++col;
        if (st == cur) {
          ++run;
        } else {
          if (cur >= 0) {
            tally((run - 1) * nS + cur);
            counted += run;
          }
          cur = st;
          run = 1;
        }
      };
      for (int rec = L - 2; rec >= 1; --rec) {
        const uint32_t e = lat[(size_t)rec * cap + idx];
        visit((int)(e >> 16));
        idx = (int)(e & 0xFFFFu);
      }
      const uint32_t e0 = lat[idx];
      visit((int)(e0 >> 16));
      visit((int)(e0 & 0xFFFFu));
      const int last = L - counted;
      if (last <= L - 1) tally((last - 1) * nS + cur);
    }
    __syncthreads();
    // fold the track's bins into the chunk's rows, track after track (the next track's tally starts after the
    // barriers of its first step)
    for (int i = tid; i < (L - 1) * nS; i += NT) {
      shist[i] = __dadd_rn(shist[i], __dmul_rn((double)(long long)sfix[i], fix_inv));
      sfix[i] = 0ull;
    }
   }  // tracks of the chunk
   if (pass == 0) {  // did any final LP of the chunk exceed 600?  then once more with the column shifts
#pragma unroll
     for (int off = 16; off > 0; off >>= 1) cmax = fmax(cmax, __shfl_down_sync(0xffffffffu, cmax, off));
     if ((tid & 31) == 0) s_max[tid >> 5] = cmax;
     __syncthreads();
     if (tid == 0) {
       double m = s_max[0];
       for (int k = 1; k < NT / 32; ++k) m = fmax(m, s_max[k]);
       s_again = m > 600.0;
       if (s_again) atomicOr(a.flags, 1);
     }
     __syncthreads();
     if (!s_again) break;
     for (int i = tid; i < (L - 1) * nS; i += NT) shist[i] = 0.0;
     __syncthreads();
   }
   }  // passes
   double* gh = a.hist + (size_t)ci * a.Lmax * nS;
   for (int i = tid; i < (L - 1) * nS; i += NT) gh[i] = shist[i];  // one CTA per chunk: plain stores
   __syncthreads();
  }
}
