/*
 * xtrack.h — C ABI of the B200-native ExTrack track-likelihood engine (libxtrack_b200.so).
 *
 * The reference (ExTrack 1.6.3, pure Python) has no FFI layer; its "operator API" for this
 * path is a set of Python call signatures in extrack/tracking.py.  Each entry point below
 * names the reference interface it stands in for (file:line relative to the reference
 * tree).  Plain pointers and sizes only; no torch / numpy types.  All functions return 0 on
 * success or a negative XT_ERR_* code; xt_last_error() gives the message.
 *
 * Threading: one caller thread per context (the reference objective is called from one
 * Python thread by lmfit, tracking.py:1371).  One context (xt_ctx) drives one GPU.  Multi-GPU:
 * either one process (and one context) per GPU, each holding a subset of the chunks, or ONE
 * process driving several GPUs through an xt_multi handle (xt_multi_* below), which is what a
 * notebook / GUI caller of param_fitting gets.
 */
#ifndef XTRACK_H
#define XTRACK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XT_MAX_HEADS 128 /* nS^(nb_substeps+1) */
#define XT_MAX_STATES 8
#define XT_MAX_DIMS 3
#define XT_MAX_SCORE_DIRS 32 /* directions of one xt_score_outer call */

#define XT_OK 0
#define XT_ERR_CUDA (-1)      /* CUDA runtime failure */
#define XT_ERR_ARG (-2)       /* malformed argument (maps to ValueError / TypeError in Python) */
#define XT_ERR_GROUPING (-3)  /* a sequence ended ungrouped: tracking.py:700-701 ValueError */
#define XT_ERR_CAPACITY (-4)  /* more live sequences than the engine's hard cap */
#define XT_ERR_STATE (-5)     /* call order (e.g. evaluate before upload) */
#define XT_ERR_UNSUPPORTED (-6) /* a documented gap of the engine (maps to NotImplementedError in Python) */

#define XT_FLAG_INT8_WRAP 1u /* reproduce the int8 wrap of history labels, tracking.py:543,619 */
#define XT_FLAG_VAR_LOC 2u   /* peak-wise localisation error from xt_upload_aux replaces l2 (input_LocErr, tracking.py:455-463) */
#define XT_FLAG_VAR_DT 4u    /* per-localisation dt from xt_upload_aux replaces dd (dt dict, tracking.py:494-499,:548-551) */
#define XT_FLAG_LOC_AFFINE 8u /* sigma' = clip(sigma*loc_slope + loc_offset, 1e-6, inf), tracking.py:926-930 */

typedef struct xt_ctx xt_ctx;

/*
 * Per-evaluation model tables.  Built on the host exactly as the reference builds them
 * (extract_params tracking.py:913-986; setup part of P_Cs_inter_bound_stats_th :474-524),
 * including p_stay via scipy.stats.norm.cdf, so that erf parity is exact.
 *
 * head id h = r + K*parent_state with K = nS^nsub and r = child index mod K; digit k of r
 * (base nS) is the state k sub-steps ago (digit 0 = newest), parent_state = newest state of
 * the sequence before the expansion.
 */
typedef struct xt_params {
  int32_t nS;            /* number of diffusive states (len(Ds), tracking.py:933-943) */
  int32_t nsub;          /* nb_substeps */
  int32_t d;             /* spatial dimensions of the uploaded tracks */
  int32_t n_loc;         /* 1: one LocErr for all dims; d: one per dim (tracking.py:920-925) */
  int32_t frame_len;     /* window length, tracking.py:679-681,714-715 */
  int32_t min_len;       /* shortest bucket length: gates the stay term, tracking.py:565-568 */
  int32_t max_nb_states; /* threshold escalation trigger, tracking.py:581-582 */
  uint32_t flags;        /* XT_FLAG_* */
  double threshold;      /* fusion threshold, tracking.py:689-691 */
  double l2[XT_MAX_DIMS];          /* LocErr^2 per dim (first n_loc entries used), :457 */
  double dd[XT_MAX_HEADS];         /* mean mid-sub-step displacement variance per head, :549-553 */
  double LT[XT_MAX_HEADS];         /* sum of log transition probabilities per head, :555,:759-767 */
  double LF[XT_MAX_HEADS];         /* log initial fraction of the oldest state of the head, :488 */
  double Lp_stay[XT_MAX_HEADS];    /* log(p_stay*(1-pBL)) per r (first K entries), :524 */
  double L_leave[XT_MAX_HEADS];    /* end-of-track leave term + LT per head, :630-631 */
  /* peak-wise LocErr / per-track dt (XT_FLAG_VAR_*): */
  double twoD[XT_MAX_STATES];      /* 2*D per state: ds = sqrt(twoD*dt[track, loc]), tracking.py:979-982 */
  double loc_slope, loc_offset;    /* XT_FLAG_LOC_AFFINE: slope_LocErr / offset_LocErr, :926-930 */
} xt_params;

/* Work counters of the last evaluation (for seq-updates/s and the algorithmic flop count,
 * SURVEY.md §8(d)). */
typedef struct xt_stats {
  int64_t n_tracks;
  int64_t track_steps;   /* sum over tracks of (L-1) */
  int64_t seq_updates;   /* sum over (chunk, step) of nT * nB_in */
  int64_t seq_groups;    /* sum over (chunk, fused step) of nT * nG */
  int32_t max_nB_in;     /* largest number of live sequences after an expansion */
  int32_t n_chunks;
  int32_t k1_launches;   /* kernels launched by the last evaluation */
  int32_t k2_launches;
  float ms_plan;         /* CUDA-event time of the plan kernel(s); pipelined evaluation: plan + replay */
  float ms_replay;       /* CUDA-event time of the replay kernel(s) incl. the reduction; pipelined: reduction */
  int32_t pipelined;     /* 1: plan and replay were launched per group of chunks on several streams */
  float ms_predict;      /* CUDA-event time of the last xt_predict kernel launch (all tracks) */
  int32_t k3_launches;   /* kernel launches of the last xt_predict call (> 1: the sequence capacity had to grow) */
  int32_t k3_cap;        /* sequence capacity of the last xt_predict launch */
  int32_t fp32;          /* 1: the last evaluation's replay ran in the optional FP32 kernel ("fp32_replay") */
  int32_t plan_verified; /* 1: the evaluation ran along the resident plan, every decision of it re-evaluated (verification mode) */
  int32_t replanned;     /* ... and this many chunks had a changed decision and were planned (and replayed) again */
} xt_stats;

/* Number of visible CUDA devices (0 without a driver or GPU; never an error). */
int xt_device_count(void);

/* Lifetime.  `device` is the CUDA ordinal this context drives. */
int xt_create(int device, xt_ctx** out);
void xt_destroy(xt_ctx* ctx);
const char* xt_last_error(xt_ctx* ctx); /* ctx may be NULL: last creation error */

/*
 * Upload the tracks this context owns — replaces the per-call pickling of every chunk to the
 * worker pool (tracking.py:1046-1063) with one upload per fit.  A *segment* s is `n[s]` tracks
 * of `L[s]` localisations in `d` dims: xyz[s] points at a C-order double[n][L][d] host buffer (a
 * whole length bucket, or a chunk-aligned slice of one when buckets are sharded over GPUs).
 * The engine cuts each segment into chunks of `chunk_size` tracks exactly like
 * `Css[n*nb_max:(n+1)*nb_max]` (tracking.py:1030-1036; 2000 for the fit, nb_max for
 * predict_Bs :866-867); chunks are numbered in upload order.  isBL[s] = 0 for segments of the
 * longest bucket (tracking.py:1037-1040).  Data are repacked on the device into a time-major
 * struct-of-arrays layout [L][d][nT_pad] per chunk.  Host buffers are not retained.
 */
int xt_upload(xt_ctx* ctx, int32_t n_segments, const int32_t* L, const int64_t* n, const int32_t* isBL,
              const double* const* xyz, int32_t d, int32_t chunk_size);

/*
 * Optional per-localisation inputs of the resident tracks (call after xt_upload, same segments):
 * sigma[s] = double[n][L][k_sigma] peak-wise localisation errors (input_LocErr of param_fitting /
 * predict_Bs, tracking.py:1351-1366,:826-836; k_sigma = 1 or d, 0 = none) and dt[s] = double[n][L]
 * per-localisation time steps (the dt dict, :1349-1368; NULL = none).  They are used by
 * evaluations whose xt_params carry XT_FLAG_VAR_LOC / XT_FLAG_VAR_DT; n_loc must then equal
 * k_sigma.  The reference reads dt with the reversed step counter on the un-reversed array
 * (:495,:549): step s uses dt[:, L-s]; the engine stores dt time-reversed to the same effect.
 */
int xt_upload_aux(xt_ctx* ctx, int32_t k_sigma, const double* const* sigma, const double* const* dt);

/*
 * Field-of-view tables when dt is per track: the reference derives p_stay from the median
 * diffusion length of each chunk (tracking.py:501-506), so Lp_stay (xt_params::Lp_stay, K = nS^nsub
 * entries) and L_leave (H = K*nS entries) become per chunk (per_track = 0, rows in upload chunk
 * order) for the objective, or per track (per_track = 1: predict_Bs with nb_max = 1 evaluates
 * one track per chunk) for xt_predict.  Used by evaluations with XT_FLAG_VAR_DT; NULL clears.
 */
int xt_set_stay_tables(xt_ctx* ctx, int32_t per_track, int32_t K, int32_t H, const double* Lp_stay, const double* L_leave);

/*
 * Objective — replaces the body of cum_Proba_Cs (tracking.py:1058-1070): plan kernel, replay
 * kernel, deterministic device reduction.  *out = sum over this context's tracks of log P
 * (the caller negates / all-reduces; parameter guards :1017 stay on the host).
 */
int xt_sum_logp(xt_ctx* ctx, const xt_params* p, double* out);

/*
 * Objective on host buffers — the call cum_Proba_Cs makes when it is handed numpy arrays on every
 * evaluation (tracking.py:991: all_tracks is an argument of the objective): same arguments as
 * xt_upload plus the model.  The copy of one segment overlaps the plan / replay kernels of the
 * segments already on the device.  The data set stays resident afterwards (xt_sum_logp,
 * xt_chunk_logp ... work on it).
 */
int xt_sum_logp_host(xt_ctx* ctx, int32_t n_segments, const int32_t* L, const int64_t* n, const int32_t* isBL,
                     const double* const* xyz, int32_t d, int32_t chunk_size, const xt_params* p, double* out);

/* Same as xt_sum_logp, but the result stays on the device: d_out is a device pointer to one double that is
 * used in the stream order of `cuda_stream` (a cudaStream_t; NULL = the legacy default stream): the
 * engine's own streams first wait for the work already enqueued on `cuda_stream` (e.g. the collective
 * of the previous call, which still reads or writes d_out), and `cuda_stream` is made to wait for the
 * result, so a collective can be chained without a host round trip. */
int xt_sum_logp_async(xt_ctx* ctx, const xt_params* p, double* d_out, void* cuda_stream);

/*
 * Evaluations along the frozen grouping plan — the plan of the last successful xt_sum_logp / _host / _async evaluation
 * (or of the one xt_chunk_logp ran).  The plan records hold only integers (groups, members, heads), so along them log P
 * of every track is a smooth function of the parameters; finite differences of it give per-track scores and the
 * observed information (tracking.param_uncertainty).  No plan kernel and no verification run: the replay kernel of the
 * plan's own evaluation (fused, VAR, or the two-phase linear / log-domain kernel) runs once per parameter set, sized
 * from the resident chunk summaries.  Nothing the objective keeps is changed: the next xt_sum_logp, xt_chunk_logp,
 * xt_plan_dump, the verification state and the speculation counters return what they would have without these calls.
 * Errors: XT_ERR_STATE without a resident plan (none yet, or discarded by xt_upload, xt_upload_aux,
 * xt_set_stay_tables, xt_set_option or a failed evaluation); XT_ERR_ARG if a parameter set differs in structure (nS,
 * nsub, d, n_loc, frame_len, flags) from the plan's evaluation; XT_ERR_UNSUPPORTED while "fp32_replay" is set (finite
 * differences need FP64).
 *
 * xt_eval_frozen: n evaluations.  sums[k] = sum of log P over this context's tracks for ps[k], added in the fixed order
 * xt_sum_logp uses (so at the plan's own parameters it has xt_sum_logp's bits).  track_logp (NULL = none):
 * track_logp[k] = double[n_tracks], log P per track in upload order.
 */
int xt_eval_frozen(xt_ctx* ctx, int32_t n, const xt_params* ps, double* sums, double* const* track_logp);

/*
 * xt_score_outer: 2*n_dir evaluations along the same plan (1 <= n_dir <= XT_MAX_SCORE_DIRS).  With
 * g[t][i] = (log P_t(p_plus[i]) - log P_t(p_minus[i])) * inv_2h[i]:  gsum[i] = sum_t g[t][i] and
 * gram[i * n_dir + j] = sum_t g[t][i] g[t][j] (double[n_dir * n_dir], symmetric); sum_plus[i] / sum_minus[i] are the totals
 * of the two evaluations.  The per-track vectors stay on the device: kernel k_score_gram forms g on the fly and
 * accumulates per chunk in a fixed order; the chunk partials are added in chunk order.
 */
int xt_score_outer(xt_ctx* ctx, int32_t n_dir, const xt_params* p_plus, const xt_params* p_minus, const double* inv_2h,
                   double* sum_plus, double* sum_minus, double* gsum, double* gram);

/* Test seam = Proba_Cs (tracking.py:769-787): log P per track of chunk `chunk` after the last
 * xt_sum_logp call's parameters `p`.  out has nT[chunk] entries. */
int xt_chunk_logp(xt_ctx* ctx, int32_t chunk, const xt_params* p, double* out);

/* Test seam = instrumented fuse_tracks_th (tracking.py:652-701): grouping of fusion step
 * `step` (2 <= step <= L-2, the reference's current_step) of chunk `chunk` from the last
 * evaluation.  gid[c] = group of incoming sequence c.  Returns XT_ERR_ARG if cap < nB_in. */
int xt_plan_dump(xt_ctx* ctx, int32_t chunk, int32_t step, int32_t* nB_in, int32_t* nG, int32_t* gid,
                 int32_t cap, double* threshold_used);

/*
 * State annotation — replaces the chunk loop of predict_Bs (tracking.py:860-896) for the
 * uploaded tracks.  Default (reference default nb_max = 1): every track gets its own grouping plan, whatever the
 * upload's chunk size.  With xt_set_option("predict_shared_plans", 1) the chunks of the upload (chunk_size = the
 * caller's nb_max, tracking.py:866-867) share one plan each, decided from the chunk's first 30 tracks with per-track
 * weighted histories (fuse_tracks_th with do_preds = 1); scalar LocErr / dt models (else XT_ERR_UNSUPPORTED).
 * out[s] receives double[n[s]][L[s]][nS] posteriors of segment s in forward time
 * (tracking.py:641-649).
 */
int xt_predict(xt_ctx* ctx, const xt_params* p, double* const* out);

/*
 * State annotation with transition posteriors: xt_predict (same options, plans and errors, same out[s]) that also fills
 * out_pairs[s] with double[n[s]][L[s] - 1][nS][nS], entry [t][k][i][j] = P(state i at localisation k, state j at
 * localisation k + 1 | track t) in forward time (the two-slice posteriors of the same recursion; summing over j gives
 * out[s][t][k], over i out[s][t][k + 1]).
 */
int xt_predict_pairs(xt_ctx* ctx, const xt_params* p, double* const* out, double* const* out_pairs);

/*
 * State annotation with one-step-ahead residuals: xt_predict (same options, plans and errors, same out[s]) that also
 * fills logpred[s] with double[n[s]][L[s]] and pit[s] with double[n[s]][L[s]][d].  For localisation k >= 1 of track t,
 * the recursion's live sequences j at the step that consumes c_k form the predictive mixture sum_j w_j N(m_j, q_j) of
 * c_k given c_0..c_k-1 (w = softmax of their log-weights without the Gaussian term of c_k):
 *   logpred[t][k]   = log of that mixture's density at c_k
 *   pit[t][k][x]    = sum_j w_j Phi((c_k,x - m_j,x) / sqrt(q_j,x))   (Uniform(0, 1) when the model is right)
 * Entry k = 0 is NaN (no predictive for the first localisation).
 */
int xt_predict_residuals(xt_ctx* ctx, const xt_params* p, double* const* out, double* const* logpred, double* const* pit);

/*
 * State annotation with the most probable state path (MAP / Viterbi path): xt_predict (same options, plans and errors,
 * same out[s]) that also fills path[s] with int8_t[n[s]][L[s]] and path_logp[s] with double[n[s]].  The recursion is a
 * lattice: every expansion gives each child one parent, every fusion gives each member a normalised merge weight w inside
 * its group, the final sequences get softmax(LP).  A route from an initial to a final sequence weighs its final softmax
 * weight times the product of the w along it; the route weights sum to 1 and, summed by label, give out[s].
 *   path[s][t][k]   = the state label at localisation k of track t's heaviest route (ties: lowest member / index)
 *   path_logp[s][t] = log of that route's weight (<= 0, and <= log out[s][t][k][path[s][t][k]] for every k)
 * Labels are those of out[s] (the int8 wrap included unless disabled).  Without fusion the path is the exact argmax over
 * all state sequences and path_logp its posterior log-probability.
 */
int xt_predict_path(xt_ctx* ctx, const xt_params* p, double* const* out, int8_t* const* path, double* const* path_logp);

/*
 * Position refinement — replaces extrack/refined_localization.py:207-338 (get_pos_PDF + the weighted means of
 * position_refinement) for the uploaded tracks.  Upload every length bucket as ONE chunk (chunk_size >= its track
 * count): the reference hands whole buckets to get_LC_Km_Ks (:48-204), whose grouping plan comes from the bucket's first
 * 30 tracks.  p_rev holds the tables of the pass that consumes a track from its last to its first localisation
 * (get_pos_PDF's first call: ds, Fs, TrMat), p_fwd those of the pass in forward time (second call: neutral fractions,
 * transposed transition matrix); both with nb_substeps = 1 and scalar or per-dimension LocErr; threshold, frame_len and
 * max_nb_states as in the reference call.  mu_out[s] receives double[n[s]][L[s]][d] refined positions, sigma_out[s]
 * double[n[s]][L[s]] their standard deviations (:329-337).
 */
int xt_refine_positions(xt_ctx* ctx, const xt_params* p_rev, const xt_params* p_fwd, double* const* mu_out,
                        double* const* sigma_out);

int xt_get_stats(xt_ctx* ctx, xt_stats* out);

/*
 * Segment-length histogram of the uploaded tracks — replaces extrack/histograms.py:26-258
 * (P_segment_len: literal top-`max_nb_states` pruning per track, :183-206, and the run-length tally
 * :248-258) as called per chunk of 50 tracks by len_hist (:265-373; upload with chunk_size = 50).
 * Uses p->nS, d, n_loc, l2, dd, LT, LF, Lp_stay, min_len (= min_l, :274), max_nb_states; nb_substeps
 * must be 1 and LocErr / dt scalar (or per dimension).  leave_LL[newest + nS * previous] =
 * log(pBL + (1 - e) - pBL (1 - e)) with e = p_stay[s] if newest == previous == s else p_stay[0] (:224-232).
 * hist receives double[n_chunks][Lmax][nS] (row k-1 = segments of k localisations, rows >= L-1 of a
 * chunk of L-localisation tracks stay zero); len_hist = sum over chunks.  Test seam (P_segment_len's
 * other outputs) for the tracks of chunk dbg_chunk >= 0: dbg_LP[nT][nBf] final log-probabilities and
 * dbg_Bs[nT][nBf][L] state histories (column 0 = newest), *n_final = nBf; pass -1 / NULL otherwise.
 * The rescale of final log-probabilities above 600 (per column over the tracks of a chunk, :243-244) is
 * applied on the device.  Returns XT_ERR_CAPACITY if the live sequences of one track
 * (max_nb_states * nS) do not fit in shared memory.
 */
int xt_seglen_hist(xt_ctx* ctx, const xt_params* p, const double* leave_LL, double* hist, int32_t Lmax,
                   int32_t dbg_chunk, double* dbg_LP, int8_t* dbg_Bs, int32_t* n_final);
int xt_seglen_last_ms(xt_ctx* ctx, float* ms); /* CUDA-event time of the last xt_seglen_hist kernel */

/* Engine options (tests / diagnostics).
 *  "force_global_replay" = 1: run the log-domain replay kernel with its state in global memory (the
 *      path taken when the live sequences of a track do not fit in shared memory);
 *  "k2_variant" = 1: first-generation linear-domain replay kernel instead of the fused one;
 *  "k2_wpc" (2|4|8), "k2_tpt" (1|2): warps per tile / tracks per thread of the fused replay kernel;
 *  "pipeline" = 0: always evaluate in two phases (plan for all chunks, then replay) instead of
 *      per-group launches on several streams; "n_groups": number of groups of the pipelined path;
 *  "fp32_replay" = 1: optional single-precision replay (north star: FP32 path, total log-likelihood
 *      within 1e-4 relative of the FP64 result).  The plan stays FP64 (same fusion decisions as the
 *      reference); the per-sequence moments and weight mantissas are FP32 with the same 32-bit extended
 *      exponent.  Applies to scalar LocErr / dt models whose state fits in shared memory and whose
 *      tables are representable in FP32; otherwise the FP64 kernel runs (xt_stats::fp32 tells which);
 *  "plan_verify" = 0: plan every evaluation from scratch instead of verifying the resident plan (same bits);
 *  "k2_lpt" = 0, "k2_cost0".."k2_cost3", "k2_cost_w0": schedule of the groups of a step over the replay warps
 *      (longest-processing-time-first on a cost model; 0 = round-robin); "k1_threads" (256|512|1024): threads per chunk
 *      of the plan kernel (0 = by the number of chunks);
 *  "predict_shared_plans" = 1: see xt_predict; "k3_cap0": sequence capacity of the first launch of xt_predict (tracks
 *      that outgrow it run again with twice as much); "k3_pieces": launches the first round of xt_predict is cut into on
 *      a large data set (the read-back of a piece runs under the kernels of the next); "k3_hot_smem", "k3_ctas_per_sm":
 *      placement of the per-warp scratch of the annotation kernel. */
int xt_set_option(xt_ctx* ctx, const char* name, int value);

/* Measured FP64 FMA throughput of this GPU in TFLOP/s (2 flops per DFMA), used as the
 * compute-roofline denominator by bench.py. */
int xt_fp64_peak_tflops(xt_ctx* ctx, double* out);

/*
 * In-process multi-GPU objective — stands in for the reference's process pool over chunks
 * (`Pool(workers).map(pool_star_proba, args_prod)`, tracking.py:1061-1063) behind the single-threaded
 * objective callback (lmfit.minimize, tracking.py:1371): one handle drives the devices `dev_ids[0..n_dev)`.
 * xt_multi_upload takes the same segment list as xt_upload (whole length buckets); the chunk list
 * (numbered in upload order) is dealt to the devices longest-processing-time-first on nT*(L-1) —
 * chunks are the atomic unit because the grouping plan is per chunk (tracking.py:677-691) — and every
 * device uploads only its chunks.  xt_multi_sum_logp evaluates all devices concurrently (one host
 * worker thread per device) and adds the per-chunk sums of log P in global chunk order, so the result
 * has the same bits for every n_dev (and equals xt_sum_logp of a single context holding all chunks).
 * SURVEY.md §8(b) proposed `xt_create(dev_ids, n_dev)`; a separate handle type keeps the one-GPU
 * context the unit that torchrun-style deployments use.
 */
typedef struct xt_multi xt_multi;
int xt_multi_create(const int32_t* dev_ids, int32_t n_dev, xt_multi** out);
void xt_multi_destroy(xt_multi* m);
const char* xt_multi_last_error(xt_multi* m); /* m may be NULL: last creation error */
int xt_multi_n_devices(xt_multi* m);
int xt_multi_upload(xt_multi* m, int32_t n_segments, const int32_t* L, const int64_t* n, const int32_t* isBL,
                    const double* const* xyz, int32_t d, int32_t chunk_size);
/* peak-wise sigma / per-localisation dt of the same segments (see xt_upload_aux) */
int xt_multi_upload_aux(xt_multi* m, int32_t n_segments, const int32_t* L, const int64_t* n, int32_t k_sigma,
                        const double* const* sigma, const double* const* dt);
/* per-chunk field-of-view tables, rows in global chunk order (see xt_set_stay_tables, per_track = 0) */
int xt_multi_set_stay_tables(xt_multi* m, int32_t K, int32_t H, const double* Lp_stay, const double* L_leave);
int xt_multi_sum_logp(xt_multi* m, const xt_params* p, double* out);
/* test seam: log P per track of global chunk `chunk` (see xt_chunk_logp) */
int xt_multi_chunk_logp(xt_multi* m, int32_t chunk, const xt_params* p, double* out);
int xt_multi_set_option(xt_multi* m, const char* name, int value);
/* share of device slot g (0 <= g < n_dev): CUDA ordinal, chunks and track-steps it owns */
int xt_multi_device_load(xt_multi* m, int32_t g, int32_t* device, int32_t* n_chunks, int64_t* track_steps);
/* xt_eval_frozen (sums only) / xt_score_outer over the devices: every device evaluates its chunks along its resident plan,
 * the chunk partials are added in global chunk order (same bits for every n_dev, and as one context holding all chunks) */
int xt_multi_eval_frozen(xt_multi* m, int32_t n, const xt_params* ps, double* sums);
int xt_multi_score_outer(xt_multi* m, int32_t n_dir, const xt_params* p_plus, const xt_params* p_minus, const double* inv_2h,
                         double* sum_plus, double* sum_minus, double* gsum, double* gram);
/* counters of the last evaluation: sums over the devices; times and maxima are the max over the devices */
int xt_multi_get_stats(xt_multi* m, xt_stats* out);

/* Pinned host memory helpers for end-to-end timing with host buffers. */
int xt_host_alloc(void** out, uint64_t bytes);
int xt_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* XTRACK_H */
