// Host side of libxtrack_b200.so: context, upload + device repack, evaluation driver, C ABI.
// See include/xtrack.h for the contract of every entry point.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <cstring>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "xt_common.cuh"
#include "xt_launch.h"
#include "xt_plan.cuh"
#include "xt_replay.cuh"
#include "xt_replay_lin.cuh"
#include "xt_replay_fused.cuh"
#include "xt_replay_f32.cuh"
#include "xt_seglen.cuh"
#include "xt_predict.cuh"
#include "xt_predict_shared.cuh"
#include "xt_refine.cuh"

struct xt_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  // data
  int d = 0;
  int64_t n_tracks = 0, track_steps = 0, n_locs = 0;
  std::vector<int> seg_chunk0;
  std::vector<int64_t> upload_sig;  // shapes of the resident data set (allocation reuse)
  double* stage[2] = {nullptr, nullptr};
  double* stage_all = nullptr;          // host-buffer objective: one staging area per segment (no reuse, no host waits)
  size_t stage_all_elems = 0;
  std::vector<size_t> seg_stage_off;
  cudaEvent_t stage_done[2] = {nullptr, nullptr};
  size_t stage_elems = 0;
  std::vector<int64_t> seg_n;
  std::vector<int> seg_L;
  std::vector<XtChunk> chunks;
  std::vector<XtWork> work;
  int nrec_total = 0;
  int maxL = 0;
  double* d_soa = nullptr;
  XtChunk* d_chunks = nullptr;
  XtWork* d_work = nullptr;
  XtWork* d_workf[2] = {nullptr, nullptr};  // fused replay: tiles of 32 / 64 tracks, chunk order
  int n_workf[2] = {0, 0};
  std::vector<int> corder;                  // chunk ids sorted by track length, longest first (stable)
  int32_t* d_corder = nullptr;
  std::vector<int> seg_pos0, seg_pos1;      // position range of every segment's chunks in corder
  std::vector<int> chunk_w0[2];             // first tile of every corder position in d_workf (+ one past the end)
  // pipelined evaluation: plan + replay launched per group of chunks on several streams, sized
  // speculatively with the parent-slot count of the previous evaluation, verified afterwards
  static constexpr int NCS = 32;  // streams created; n_streams of them are used
  cudaStream_t cs[NCS] = {};
  int n_streams = 8;
  cudaStream_t up_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join[NCS] = {};
  std::vector<cudaEvent_t> ev_seg;
  int* d_spec = nullptr;
  int* h_spec = nullptr;  // pinned
  int* d_spec_own = nullptr;  // the word of a context without data; after an upload d_spec / h_spec point into the tail block
  int* h_spec_own = nullptr;
  // one device block [chunk sums f64[n] | verification flags i32[n] | speculation word i32] and its pinned mirror: what
  // the host reads after a verified evaluation comes back in one copy
  unsigned char* d_tail = nullptr;
  unsigned char* h_tail = nullptr;
  size_t tail_bytes = 0;
  int spec_Pmax = 0;      // 0: unknown (first evaluation of a data set runs the two-phase path)
  int spec_maxP = 0, spec_maxC = 0;  // most parents / children of the previous evaluation: sizes the plan kernel's
                                     // shared-memory scratch (0: global-memory scratch)
  int k1_smem_scratch = 1;
  int k2_global_ctas = 32;    // one-warp CTAs per SM of the global-memory replay kernel (latency-bound: as many as fit)
  int k3_shared = 0;          // state annotation: 1 = the tracks of an uploaded chunk share one plan (predict_Bs with nb_max > 1)
  int k3_cap0 = 48;           // state annotation: sequence capacity of the first launch (tracks that outgrow it run again with more)
  int k3_pieces = 8;          // state annotation of a large data set: launches of the first round (read-back of a piece under the next)
  int verify_fork_k2 = 0;     // verified evaluation: 1 = the replay on a stream of its own (0: on the context's main stream)
  int k3_hot_smem = 1;        // state-annotation kernel: forward-pass state of every warp in shared memory
  int k3_ctas_per_sm = 4;     // resident CTAs per SM of the state-annotation kernel (its per-warp scratch should stay in L2)
  int k1_threads = 0;         // plan kernel threads per chunk: 0 = automatic (256, or 1024 for <= n_sm chunks)
  int k2_lpt = 1;             // replay schedule of the plan records: longest-processing-time-first (0: round-robin)
  int k2_cost[4] = {4, 7, 6, 2};  // its cost model: single-member group, pair, member list (base, per member)
  int k2_cost_w0 = 0;         // per-step extra work of replay warp 0 (record staging), same units
  int k1_batch = 1;           // plan kernel, > 64 sequences: batched candidate leaders (0: one leader at a time)
  int pipeline = 1;
  int n_groups = 6;
  // plan verification (k1_plan<.., VERIFY>): the resident plan stays valid across evaluations as long as every
  // floating-point decision behind it is reproduced with the new parameters
  bool plan_valid = false;      // the resident plan + records describe the resident data for plan_sig
  xt_params plan_sig{};         // structural fields of the parameters the plan was built with
  int plan_verify = 1;          // option: 0 = always plan from scratch
  int32_t* d_vflag = nullptr;   // [n_chunks] verification outcome per chunk
  int32_t* h_vflag = nullptr;   // pinned
  int32_t* d_redo = nullptr;    // [n_chunks] chunk ids to plan again
  std::vector<int> corder_pos;  // position of every chunk in corder
  double* d_logp = nullptr;
  double* d_partial = nullptr;
  double* d_out = nullptr;
  // per-chunk sums of log P (fixed order over the chunk's tiles): the objective is their sum in chunk order
  // on the host, so its bits do not depend on how the chunks are spread over GPUs (xt_multi_*)
  double* d_csum = nullptr;
  double* h_csum = nullptr;                 // pinned
  bool csum_fetched = false;                // h_csum already holds the chunk sums of the last evaluation
  bool spec_dirty = true;                   // d_spec may be non-zero (set by a replay launch, or never cleared yet)
  int32_t* d_cw0[3] = {nullptr, nullptr, nullptr};  // first tile of every position: [0],[1] fused tables (corder), [2] plain table
  XtChunkSummary* d_summ = nullptr;
  std::vector<XtChunkSummary> summ;
  XtChunkSummary* h_summ = nullptr;  // pinned
  double* h_out = nullptr;           // pinned
  // plan storage / K1 scratch (sized by cap and the model)
  int cap = 0, RH = 0, nS_alloc = 0, CO1_alloc = 0;
  XtPlanPtrs plan{};
  double* d_state1 = nullptr;
  double* d_hist1 = nullptr;
  // K2 global-state fallback
  double* d_gstate = nullptr;
  size_t gstate_bytes = 0;
  // fused replay kernel with its state in global memory (GST): state blocks + per-SM slot bitmaps
  char* d_fstate = nullptr;
  size_t fstate_bytes = 0;
  unsigned* d_fslots = nullptr;
  int k2_gst_below_ctas = 3;  // prefer the GST instantiation when fewer than this many shared-memory CTAs fit on an SM
  int k2_gst = 1;             // 0: never use the GST instantiation (falls back to the log-domain kernel)
  int k2_fp32 = 0;            // 1: optional single-precision replay (xt_replay_f32.cuh) where it applies
  int smem_optin = 0, n_sm = 0;
  bool have_eval = false;
  bool force_global = false;  // test hook: run the log-domain global-memory replay variant
  int k2_wpc = 4;             // warps cooperating on one 32-track tile in the fast replay kernel
  int k2_tpt = 1;             // tracks per thread of the fused replay kernel (tile = 32 * k2_tpt tracks)
  int k2_variant = 0;         // 0: fused merge+update kernel (default), 1: first-generation linear-domain kernel
  bool last_fused = false;    // the previous evaluation ran the fused replay kernel
  bool plan_has_grec = false; // the resident plan carries the first-generation kernel's inline group records
  xt_params last_p{};
  xt_stats stats{};
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_k3[2] = {nullptr, nullptr};
  float ms_predict = 0.f;
  float ms_seglen = 0.f;
  bool seglen_rescaled = false;  // the last xt_seglen_hist call applied the > 600 rescale to some chunk
  int k3_launches = 0, k3_cap = 0;
  // optional per-localisation inputs (xt_upload_aux) and field-of-view tables (xt_set_stay_tables)
  double* d_aux = nullptr;
  int aux_R = 0, aux_ka = 0, aux_has_dt = 0;
  int64_t soa_elems = 0;
  double* d_stay[2] = {nullptr, nullptr};   // [0] per chunk, [1] per track: Lp_stay [rows][K]
  double* d_leave[2] = {nullptr, nullptr};  // [0] per chunk: linear sums [rows][nS]; [1] per track: log-sums [rows][nS]
  int stay_K[2] = {0, 0}, stay_H[2] = {0, 0};
  // frozen evaluations (xt_eval_frozen / xt_score_outer): the replay launch of the last evaluation, repeated with other
  // parameters along its plan.  Outputs go to buffers of their own, so the state above is never touched.
  int frozen_kind = 0;          // 0: no plan resident; XT_FROZEN_FUSED / XT_FROZEN_OLD: the replay kernel that plan's evaluation ran
  int frozen_Pcap = 0;          // parent slots that launch was sized with (>= max_nP of every chunk summary)
  xt_params frozen_sig{};       // the parameters of that evaluation (structure check)
  double* d_flogp = nullptr;    // [slots][n_tracks] per-track log P
  size_t flogp_elems = 0;
  double* d_fpartial = nullptr; // per-tile partial sums
  double* d_fcsum = nullptr;    // [n_eval][n_chunks] chunk sums, and its pinned mirror
  double* h_fcsum = nullptr;
  size_t fcsum_elems = 0;
  double* d_fgram = nullptr;    // [n_chunks][E] score / outer-product partials of k_score_gram, and its pinned mirror
  double* h_fgram = nullptr;
  size_t fgram_elems = 0;
  int* d_fspec = nullptr;       // speculation word of the frozen launches (never set: their sizes come from the summaries)
};

static std::string g_create_error;
static void set_error(xt_ctx* ctx, const std::string& s) {
  if (ctx) ctx->err = s; else g_create_error = s;
}

// ------------------------------------------------------------------------------------------
// repack: AoS [n][L][d] (host order) -> per-chunk SoA [L][d][nTpad]
// ------------------------------------------------------------------------------------------
__global__ void k_pack(const double* __restrict__ src, double* __restrict__ soa, const XtChunk* __restrict__ chunks,
                       int chunk0, int chunk_size, int n, int L, int d) {
  // one thread per (row = k*d+dim, track i) with i fastest => coalesced writes
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int rows = L * d;
  if (idx >= (long long)n * rows) return;
  const int i = (int)(idx % n);
  const int row = (int)(idx / n);
  const int c = i / chunk_size, t = i - c * chunk_size;
  const XtChunk ck = chunks[chunk0 + c];
  soa[ck.xyz_off + (size_t)row * ck.nTpad + t] = src[(size_t)i * rows + row];
}

// aux repack: src [n][L][kin] -> rows row0..row0+kin-1 of the per-chunk blocks [L][R][nTpad] at
// (xyz_off / d) * R; `reverse` stores localisation j at row block L-1-j (dt, see XtAux)
__global__ void k_pack_aux(const double* __restrict__ src, double* __restrict__ aux, const XtChunk* __restrict__ chunks,
                           int chunk0, int chunk_size, int n, int L, int kin, int R, int row0, int d, int reverse) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int rows = L * kin;
  if (idx >= (long long)n * rows) return;
  const int i = (int)(idx % n);
  const int row = (int)(idx / n);
  const int j = row / kin, k = row - j * kin;
  const int c = i / chunk_size, t = i - c * chunk_size;
  const XtChunk ck = chunks[chunk0 + c];
  const int jo = reverse ? (L - 1 - j) : j;
  aux[(size_t)(ck.xyz_off / d) * R + ((size_t)jo * R + row0 + k) * ck.nTpad + t] = src[(size_t)i * rows + row];
}

__global__ void k_fp64_peak(double* out, int iters) {
  double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
  double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
  const double b = 0.999999, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
    a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

static void free_plan(xt_ctx* ctx) {
  cudaFree(ctx->plan.hdr); cudaFree(ctx->plan.goff); cudaFree(ctx->plan.ent);
  cudaFree(ctx->plan.curG); cudaFree(ctx->plan.gid); cudaFree(ctx->plan.grec); cudaFree(ctx->plan.blob);
  cudaFree(ctx->plan.vrec); cudaFree(ctx->plan.vok);
  ctx->plan_valid = false;
  cudaFree(ctx->d_state1); cudaFree(ctx->d_hist1);
  ctx->plan = XtPlanPtrs{};
  ctx->d_state1 = ctx->d_hist1 = nullptr;
  ctx->cap = 0;
  ctx->frozen_kind = 0;
}

static void free_data(xt_ctx* ctx) {
  cudaFree(ctx->d_aux);
  ctx->d_aux = nullptr;
  ctx->aux_R = ctx->aux_ka = ctx->aux_has_dt = 0;
  for (int i = 0; i < 2; ++i) {
    cudaFree(ctx->d_stay[i]); cudaFree(ctx->d_leave[i]);
    ctx->d_stay[i] = ctx->d_leave[i] = nullptr;
    ctx->stay_K[i] = ctx->stay_H[i] = 0;
  }
  cudaFree(ctx->d_soa); cudaFree(ctx->d_chunks); cudaFree(ctx->d_work); cudaFree(ctx->d_logp);
  cudaFree(ctx->d_partial); cudaFree(ctx->d_summ); cudaFree(ctx->d_gstate);
  cudaFree(ctx->d_fstate); cudaFree(ctx->d_fslots);
  ctx->d_fstate = nullptr; ctx->d_fslots = nullptr; ctx->fstate_bytes = 0;
  cudaFree(ctx->d_workf[0]); cudaFree(ctx->d_workf[1]); cudaFree(ctx->d_corder);
  ctx->d_corder = nullptr;
  cudaFree(ctx->d_redo);
  ctx->d_redo = nullptr;
  ctx->plan_valid = false;
  cudaFree(ctx->d_flogp); cudaFree(ctx->d_fpartial); cudaFree(ctx->d_fcsum); cudaFree(ctx->d_fgram); cudaFree(ctx->d_fspec);
  if (ctx->h_fcsum) cudaFreeHost(ctx->h_fcsum);
  if (ctx->h_fgram) cudaFreeHost(ctx->h_fgram);
  ctx->d_flogp = ctx->d_fpartial = ctx->d_fcsum = ctx->h_fcsum = ctx->d_fgram = ctx->h_fgram = nullptr;
  ctx->d_fspec = nullptr;
  ctx->flogp_elems = ctx->fcsum_elems = ctx->fgram_elems = 0;
  cudaFree(ctx->d_tail);
  if (ctx->h_tail) cudaFreeHost(ctx->h_tail);
  ctx->d_tail = ctx->h_tail = nullptr;
  ctx->tail_bytes = 0;
  ctx->d_vflag = ctx->h_vflag = nullptr;
  ctx->d_csum = ctx->h_csum = nullptr;
  ctx->d_spec = ctx->d_spec_own;
  ctx->h_spec = ctx->h_spec_own;
  ctx->spec_dirty = true;
  for (int v = 0; v < 3; ++v) { cudaFree(ctx->d_cw0[v]); ctx->d_cw0[v] = nullptr; }
  ctx->d_workf[0] = ctx->d_workf[1] = nullptr;
  if (ctx->h_summ) cudaFreeHost(ctx->h_summ);
  ctx->d_soa = ctx->d_logp = ctx->d_partial = ctx->d_gstate = nullptr;
  ctx->d_chunks = nullptr; ctx->d_work = nullptr; ctx->d_summ = nullptr; ctx->h_summ = nullptr;
  ctx->gstate_bytes = 0;
  ctx->chunks.clear(); ctx->work.clear(); ctx->summ.clear(); ctx->upload_sig.clear();
  ctx->have_eval = false;
  ctx->spec_Pmax = 0;
  ctx->spec_maxP = ctx->spec_maxC = 0;
  free_plan(ctx);
}

static int create_resources(xt_ctx* ctx, int device) {
  xt_ctx* c = ctx;
  XT_CUDA_OK(cudaSetDevice(device));
  XT_CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  XT_CUDA_OK(cudaMalloc(&c->d_out, sizeof(double)));
  XT_CUDA_OK(cudaMallocHost(&c->h_out, sizeof(double)));
  for (int i = 0; i < 3; ++i) XT_CUDA_OK(cudaEventCreate(&c->ev[i]));
  for (int i = 0; i < 2; ++i) XT_CUDA_OK(cudaEventCreate(&c->ev_k3[i]));
  for (int i = 0; i < xt_ctx::NCS; ++i) {
    XT_CUDA_OK(cudaStreamCreateWithFlags(&c->cs[i], cudaStreamNonBlocking));
    XT_CUDA_OK(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
  }
  XT_CUDA_OK(cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking));
  XT_CUDA_OK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  XT_CUDA_OK(cudaMalloc(&c->d_spec_own, sizeof(int)));
  XT_CUDA_OK(cudaMallocHost(&c->h_spec_own, sizeof(int)));
  c->d_spec = c->d_spec_own;
  c->h_spec = c->h_spec_own;
  XT_CUDA_OK(cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  c->smem_optin -= 256;  // the kernels' static shared memory counts against the same limit (<= 144 B; the plan kernel: k1_scratch_caps)
  XT_CUDA_OK(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device));
  return XT_OK;
}

extern "C" void xt_destroy(xt_ctx* ctx);

extern "C" int xt_create(int device, xt_ctx** out) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(nullptr, std::string("no CUDA device: ") + cudaGetErrorString(e));
    return XT_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) {
    set_error(nullptr, "device ordinal out of range");
    return XT_ERR_ARG;
  }
  xt_ctx* c = new xt_ctx();
  c->device = device;
  const int rc = create_resources(c, device);
  if (rc) {  // the message goes where xt_last_error(NULL) finds it; nothing of the half-built context is kept
    g_create_error = c->err;
    xt_destroy(c);
    return rc;
  }
  *out = c;
  return XT_OK;
}

extern "C" void xt_destroy(xt_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  free_data(ctx);
  for (int b = 0; b < 2; ++b) {
    cudaFree(ctx->stage[b]);
    if (ctx->stage_done[b]) cudaEventDestroy(ctx->stage_done[b]);
  }
  cudaFree(ctx->stage_all);
  cudaFree(ctx->d_out);
  if (ctx->h_out) cudaFreeHost(ctx->h_out);
  for (int i = 0; i < 3; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  for (int i = 0; i < 2; ++i) if (ctx->ev_k3[i]) cudaEventDestroy(ctx->ev_k3[i]);
  for (int i = 0; i < xt_ctx::NCS; ++i) {
    if (ctx->cs[i]) cudaStreamDestroy(ctx->cs[i]);
    if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
  }
  if (ctx->up_stream) cudaStreamDestroy(ctx->up_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  for (cudaEvent_t e : ctx->ev_seg) cudaEventDestroy(e);
  cudaFree(ctx->d_spec_own);
  if (ctx->h_spec_own) cudaFreeHost(ctx->h_spec_own);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  cudaGetLastError();
  delete ctx;
}

extern "C" int xt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" const char* xt_last_error(xt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int xt_host_alloc(void** out, uint64_t bytes) {
  return cudaMallocHost(out, bytes) == cudaSuccess ? XT_OK : XT_ERR_CUDA;
}
extern "C" int xt_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? XT_OK : XT_ERR_CUDA; }

// Validate the segment list and (re)build the chunk / work tables and the device allocations.
// Same shapes as the resident data set (a re-upload of new coordinates, e.g. one objective call
// per host buffer): every allocation, table and the plan storage are kept.
static int setup_layout(xt_ctx* ctx, int32_t n_seg, const int32_t* L, const int64_t* n, const int32_t* isBL, int32_t d,
                        int32_t chunk_size) {
  if (n_seg <= 0 || d < 1 || d > XT_MAX_DIMS || chunk_size < 1) {
    set_error(ctx, "xt_upload: need n_seg >= 1, 1 <= d <= 3, chunk_size >= 1");
    return XT_ERR_ARG;
  }
  for (int s = 0; s < n_seg; ++s) {
    if (L[s] < 2) {
      set_error(ctx, "minimal track length = 2, here track length = " + std::to_string(L[s]));
      return XT_ERR_ARG;
    }
    if (n[s] < 1) {
      set_error(ctx, "xt_upload: empty segment");
      return XT_ERR_ARG;
    }
  }
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  std::vector<int64_t> sig;
  sig.push_back(n_seg); sig.push_back(d); sig.push_back(chunk_size);
  for (int s = 0; s < n_seg; ++s) { sig.push_back(L[s]); sig.push_back(n[s]); sig.push_back(isBL[s]); }
  const bool reuse = !ctx->chunks.empty() && sig == ctx->upload_sig;
  int64_t max_seg_elems = 0;
  for (int s = 0; s < n_seg; ++s) max_seg_elems = std::max<int64_t>(max_seg_elems, n[s] * L[s] * d);
  if (!reuse) {
    free_data(ctx);
    ctx->upload_sig = sig;
    ctx->d = d;
    ctx->n_tracks = 0;
    ctx->n_locs = 0;
    ctx->track_steps = 0;
    ctx->maxL = 0;
    int64_t soa_elems = 0;
    int rec = 0;
    ctx->seg_chunk0.assign(n_seg + 1, 0);
    for (int s = 0; s < n_seg; ++s) {
      ctx->seg_chunk0[s] = (int)ctx->chunks.size();
      ctx->maxL = std::max(ctx->maxL, (int)L[s]);
      for (int64_t a = 0; a < n[s]; a += chunk_size) {
        XtChunk ck{};
        ck.L = L[s];
        ck.nT = (int)std::min<int64_t>(chunk_size, n[s] - a);
        ck.nTpad = (ck.nT + 31) & ~31;
        ck.isBL = isBL[s];
        ck.xyz_off = soa_elems;
        ck.trk_off = ctx->n_tracks;
        ck.loc_off = ctx->n_locs;
        ck.rec0 = rec;
        ck.nrec = std::max(0, ck.L - 3);
        ck.seg = s;
        ck.seg_t0 = (int)a;
        rec += ck.nrec;
        soa_elems += (int64_t)ck.L * d * ck.nTpad;
        ctx->n_tracks += ck.nT;
        ctx->n_locs += (int64_t)ck.nT * ck.L;
        ctx->track_steps += (int64_t)ck.nT * (ck.L - 1);
        for (int t0 = 0; t0 < ck.nT; t0 += 32) ctx->work.push_back(XtWork{(int)ctx->chunks.size(), t0});
        ctx->chunks.push_back(ck);
      }
    }
    ctx->seg_chunk0[n_seg] = (int)ctx->chunks.size();
    ctx->soa_elems = soa_elems;
    ctx->nrec_total = rec;
    ctx->seg_n.assign(n, n + n_seg);
    ctx->seg_L.assign(L, L + n_seg);
    const size_t nch = ctx->chunks.size();
    XT_CUDA_OK(cudaMalloc(&ctx->d_soa, sizeof(double) * (size_t)soa_elems));
    XT_CUDA_OK(cudaMemsetAsync(ctx->d_soa, 0, sizeof(double) * (size_t)soa_elems, ctx->stream));  // padding lanes
    XT_CUDA_OK(cudaMalloc(&ctx->d_chunks, sizeof(XtChunk) * nch));
    XT_CUDA_OK(cudaMalloc(&ctx->d_work, sizeof(XtWork) * ctx->work.size()));
    XT_CUDA_OK(cudaMalloc(&ctx->d_logp, sizeof(double) * (size_t)ctx->n_tracks));
    XT_CUDA_OK(cudaMalloc(&ctx->d_partial, sizeof(double) * ctx->work.size()));
    XT_CUDA_OK(cudaMalloc(&ctx->d_summ, sizeof(XtChunkSummary) * nch));
    XT_CUDA_OK(cudaMallocHost(&ctx->h_summ, sizeof(XtChunkSummary) * nch));
    ctx->summ.resize(nch);
    XT_CUDA_OK(cudaMemcpyAsync(ctx->d_chunks, ctx->chunks.data(), sizeof(XtChunk) * nch, cudaMemcpyHostToDevice,
                               ctx->stream));
    XT_CUDA_OK(cudaMemcpyAsync(ctx->d_work, ctx->work.data(), sizeof(XtWork) * ctx->work.size(),
                               cudaMemcpyHostToDevice, ctx->stream));
    // chunk order of the kernels: longest tracks first (their plan is the critical path and their
    // replay CTAs run longest); the work tables of the fused replay kernel (tiles of 32 and 64
    // tracks) follow that order, so a range of positions is a range of tiles
    ctx->corder.resize(nch);
    for (size_t c = 0; c < nch; ++c) ctx->corder[c] = (int)c;
    std::stable_sort(ctx->corder.begin(), ctx->corder.end(),
                     [&](int x, int y) { return ctx->chunks[x].L > ctx->chunks[y].L; });
    ctx->seg_pos0.assign(n_seg, (int)nch);
    ctx->seg_pos1.assign(n_seg, 0);
    for (size_t q = 0; q < nch; ++q) {
      const int sg = ctx->chunks[ctx->corder[q]].seg;
      ctx->seg_pos0[sg] = std::min(ctx->seg_pos0[sg], (int)q);
      ctx->seg_pos1[sg] = std::max(ctx->seg_pos1[sg], (int)q + 1);
    }
    XT_CUDA_OK(cudaMalloc(&ctx->d_corder, sizeof(int32_t) * nch));
    XT_CUDA_OK(cudaMemcpy(ctx->d_corder, ctx->corder.data(), sizeof(int32_t) * nch, cudaMemcpyHostToDevice));
    for (int v = 0; v < 2; ++v) {
      const int tile = 32 << v;
      std::vector<XtWork> wf;
      ctx->chunk_w0[v].assign(nch + 1, 0);
      for (size_t q = 0; q < nch; ++q) {
        const int c = ctx->corder[q];
        ctx->chunk_w0[v][q] = (int)wf.size();
        for (int t0 = 0; t0 < ctx->chunks[c].nT; t0 += tile) wf.push_back(XtWork{c, t0});
      }
      ctx->chunk_w0[v][nch] = (int)wf.size();
      ctx->n_workf[v] = (int)wf.size();
      XT_CUDA_OK(cudaMalloc(&ctx->d_workf[v], sizeof(XtWork) * wf.size()));
      XT_CUDA_OK(cudaMemcpy(ctx->d_workf[v], wf.data(), sizeof(XtWork) * wf.size(), cudaMemcpyHostToDevice));
      XT_CUDA_OK(cudaMalloc(&ctx->d_cw0[v], sizeof(int32_t) * (nch + 1)));
      XT_CUDA_OK(cudaMemcpy(ctx->d_cw0[v], ctx->chunk_w0[v].data(), sizeof(int32_t) * (nch + 1), cudaMemcpyHostToDevice));
    }
    {  // plain work table (first-generation / log-domain replay kernels): 32-track tiles in chunk order
      std::vector<int32_t> w0(nch + 1, 0);
      for (size_t c = 0; c < nch; ++c) w0[c + 1] = w0[c] + (ctx->chunks[c].nT + 31) / 32;
      XT_CUDA_OK(cudaMalloc(&ctx->d_cw0[2], sizeof(int32_t) * (nch + 1)));
      XT_CUDA_OK(cudaMemcpy(ctx->d_cw0[2], w0.data(), sizeof(int32_t) * (nch + 1), cudaMemcpyHostToDevice));
    }
    ctx->tail_bytes = sizeof(double) * nch + sizeof(int32_t) * (nch + 1);
    XT_CUDA_OK(cudaMalloc(&ctx->d_tail, ctx->tail_bytes));
    XT_CUDA_OK(cudaMallocHost(&ctx->h_tail, ctx->tail_bytes));
    XT_CUDA_OK(cudaMemsetAsync(ctx->d_tail, 0, ctx->tail_bytes, ctx->stream));
    std::memset(ctx->h_tail, 0, ctx->tail_bytes);
    ctx->d_csum = (double*)ctx->d_tail;
    ctx->h_csum = (double*)ctx->h_tail;
    ctx->d_vflag = (int32_t*)(ctx->d_tail + sizeof(double) * nch);
    ctx->h_vflag = (int32_t*)(ctx->h_tail + sizeof(double) * nch);
    ctx->d_spec = (int*)(ctx->d_vflag + nch);
    ctx->h_spec = (int*)(ctx->h_vflag + nch);
    ctx->spec_dirty = true;
    XT_CUDA_OK(cudaMalloc(&ctx->d_redo, sizeof(int32_t) * nch));
    ctx->corder_pos.assign(nch, 0);
    for (size_t q = 0; q < nch; ++q) ctx->corder_pos[ctx->corder[q]] = (int)q;
    while ((int)ctx->ev_seg.size() < n_seg) {
      cudaEvent_t e;
      XT_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ctx->ev_seg.push_back(e);
    }
    XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  }
  ctx->have_eval = false;
  ctx->plan_valid = false;  // new coordinates: the resident plan describes the previous data set
  ctx->frozen_kind = 0;
  // two staging buffers (AoS as on the host) overlap the copy of one segment with the repack of another
  if ((size_t)max_seg_elems > ctx->stage_elems) {
    for (int b = 0; b < 2; ++b) {
      cudaFree(ctx->stage[b]);
      ctx->stage[b] = nullptr;
      XT_CUDA_OK(cudaMalloc(&ctx->stage[b], sizeof(double) * (size_t)max_seg_elems));
      if (!ctx->stage_done[b]) XT_CUDA_OK(cudaEventCreateWithFlags(&ctx->stage_done[b], cudaEventDisableTiming));
    }
    ctx->stage_elems = (size_t)max_seg_elems;
  }
  return XT_OK;
}

// Copy segment s to the device and repack it into the SoA blocks of its chunks, on `stream`;
// `slot` alternates between the two staging buffers.
static int enqueue_segment(xt_ctx* ctx, int s, const double* xyz, int slot, cudaStream_t stream) {
  const int b = slot & 1;
  const int64_t n = ctx->seg_n[s];
  const int L = ctx->seg_L[s], d = ctx->d;
  const size_t elems = (size_t)n * L * d;
  const int chunk_size = (int)ctx->upload_sig[2];
  XT_CUDA_OK(cudaEventSynchronize(ctx->stage_done[b]));
  XT_CUDA_OK(cudaMemcpyAsync(ctx->stage[b], xyz, sizeof(double) * elems, cudaMemcpyHostToDevice, stream));
  const int threads = 256;
  const long long blocks = ((long long)elems + threads - 1) / threads;
  k_pack<<<(unsigned)blocks, threads, 0, stream>>>(ctx->stage[b], ctx->d_soa, ctx->d_chunks, ctx->seg_chunk0[s], chunk_size,
                                                   (int)n, L, d);
  XT_CUDA_OK(cudaEventRecord(ctx->stage_done[b], stream));
  return XT_OK;
}

// Host-buffer objective: every segment has its own staging area, so the copies run back to back on
// the upload stream (the PCIe link never waits for a repack kernel or for the host) and the repack
// is done on the compute stream that consumes the segment.
static int ensure_stage_all(xt_ctx* ctx) {
  const int n_seg = (int)ctx->seg_L.size();
  size_t total = 0;
  ctx->seg_stage_off.assign(n_seg, 0);
  for (int s = 0; s < n_seg; ++s) {
    ctx->seg_stage_off[s] = total;
    total += (size_t)ctx->seg_n[s] * ctx->seg_L[s] * ctx->d;
  }
  if (total > ctx->stage_all_elems) {
    cudaFree(ctx->stage_all);
    ctx->stage_all = nullptr;
    ctx->stage_all_elems = 0;
    XT_CUDA_OK(cudaMalloc(&ctx->stage_all, sizeof(double) * total));
    ctx->stage_all_elems = total;
  }
  return XT_OK;
}

static int enqueue_pack(xt_ctx* ctx, int s, cudaStream_t stream) {
  const int64_t n = ctx->seg_n[s];
  const int L = ctx->seg_L[s], d = ctx->d;
  const size_t elems = (size_t)n * L * d;
  const int threads = 256;
  const long long blocks = ((long long)elems + threads - 1) / threads;
  k_pack<<<(unsigned)blocks, threads, 0, stream>>>(ctx->stage_all + ctx->seg_stage_off[s], ctx->d_soa, ctx->d_chunks,
                                                   ctx->seg_chunk0[s], (int)ctx->upload_sig[2], (int)n, L, d);
  XT_CUDA_OK(cudaGetLastError());
  return XT_OK;
}

extern "C" int xt_upload(xt_ctx* ctx, int32_t n_seg, const int32_t* L, const int64_t* n, const int32_t* isBL,
                         const double* const* xyz, int32_t d, int32_t chunk_size) {
  if (!ctx) return XT_ERR_ARG;
  int rc = setup_layout(ctx, n_seg, L, n, isBL, d, chunk_size);
  if (rc) return rc;
  for (int s = 0; s < n_seg; ++s) {
    rc = enqueue_segment(ctx, s, xyz[s], s, ctx->stream);
    if (rc) return rc;
  }
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  XT_CUDA_OK(cudaGetLastError());
  return XT_OK;
}

extern "C" int xt_upload_aux(xt_ctx* ctx, int32_t k_sigma, const double* const* sigma, const double* const* dt) {
  if (!ctx) return XT_ERR_ARG;
  if (ctx->chunks.empty()) {
    set_error(ctx, "xt_upload_aux: upload the tracks first");
    return XT_ERR_STATE;
  }
  if (k_sigma < 0 || (k_sigma != 0 && k_sigma != 1 && k_sigma != ctx->d) || (k_sigma > 0 && !sigma) ||
      (k_sigma == 0 && !dt)) {
    set_error(ctx, "Localization error is not specified correctly: peak-wise errors must have 1 or d components per localisation");
    return XT_ERR_ARG;
  }
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  const int R = k_sigma + (dt ? 1 : 0);
  cudaFree(ctx->d_aux);
  ctx->d_aux = nullptr;
  const size_t elems = (size_t)(ctx->soa_elems / ctx->d) * R;
  XT_CUDA_OK(cudaMalloc(&ctx->d_aux, sizeof(double) * elems));
  XT_CUDA_OK(cudaMemsetAsync(ctx->d_aux, 0, sizeof(double) * elems, ctx->stream));
  ctx->aux_R = R;
  ctx->aux_ka = k_sigma;
  ctx->aux_has_dt = dt ? 1 : 0;
  ctx->have_eval = false;
  ctx->plan_valid = false;
  ctx->frozen_kind = 0;
  const int chunk_size = (int)ctx->upload_sig[2];
  int slot = 0;
  for (int pass = 0; pass < 2; ++pass) {
    const double* const* src = pass == 0 ? sigma : dt;
    const int kin = pass == 0 ? k_sigma : 1;
    if (!src || kin == 0) continue;
    for (int s = 0; s < (int)ctx->seg_L.size(); ++s, ++slot) {
      const int b = slot & 1;
      const int64_t n = ctx->seg_n[s];
      const int L = ctx->seg_L[s];
      const size_t cnt = (size_t)n * L * kin;
      XT_CUDA_OK(cudaEventSynchronize(ctx->stage_done[b]));
      XT_CUDA_OK(cudaMemcpyAsync(ctx->stage[b], src[s], sizeof(double) * cnt, cudaMemcpyHostToDevice, ctx->stream));
      const long long blocks = ((long long)cnt + 255) / 256;
      k_pack_aux<<<(unsigned)blocks, 256, 0, ctx->stream>>>(ctx->stage[b], ctx->d_aux, ctx->d_chunks, ctx->seg_chunk0[s],
                                                             chunk_size, (int)n, L, kin, R, pass == 0 ? 0 : k_sigma, ctx->d,
                                                             pass == 1);
      XT_CUDA_OK(cudaEventRecord(ctx->stage_done[b], ctx->stream));
    }
  }
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  XT_CUDA_OK(cudaGetLastError());
  return XT_OK;
}

extern "C" int xt_set_stay_tables(xt_ctx* ctx, int32_t per_track, int32_t K, int32_t H, const double* Lp_stay,
                                  const double* L_leave) {
  if (!ctx) return XT_ERR_ARG;
  const int i = per_track ? 1 : 0;
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  cudaFree(ctx->d_stay[i]); cudaFree(ctx->d_leave[i]);
  ctx->d_stay[i] = ctx->d_leave[i] = nullptr;
  ctx->stay_K[i] = ctx->stay_H[i] = 0;
  ctx->have_eval = false;
  ctx->plan_valid = false;
  ctx->frozen_kind = 0;  // (per-chunk tables are context state the frozen launches would read)
  if (!Lp_stay || !L_leave) return XT_OK;
  if (ctx->chunks.empty() || K < 1 || H < K || H % K != 0) {
    set_error(ctx, "xt_set_stay_tables: upload the tracks first; need K >= 1 and H a multiple of K");
    return XT_ERR_ARG;
  }
  const size_t rows = per_track ? (size_t)ctx->n_tracks : ctx->chunks.size();
  const int nS = H / K;
  std::vector<double> lv(rows * nS);
  for (size_t r = 0; r < rows; ++r)
    for (int s = 0; s < nS; ++s) {  // end-of-track expansion folded: sum over r of exp(L_leave[r + K*s])
      const double* v = L_leave + r * H + (size_t)K * s;
      double mx = -INFINITY;
      for (int q = 0; q < K; ++q) mx = std::max(mx, v[q]);
      double acc = 0;
      for (int q = 0; q < K; ++q) acc += std::exp(v[q] - mx);
      lv[r * nS + s] = per_track ? std::log(acc) + mx : std::exp(std::log(acc) + mx);
    }
  XT_CUDA_OK(cudaMalloc(&ctx->d_stay[i], sizeof(double) * rows * K));
  XT_CUDA_OK(cudaMalloc(&ctx->d_leave[i], sizeof(double) * rows * nS));
  XT_CUDA_OK(cudaMemcpy(ctx->d_stay[i], Lp_stay, sizeof(double) * rows * K, cudaMemcpyHostToDevice));
  XT_CUDA_OK(cudaMemcpy(ctx->d_leave[i], lv.data(), sizeof(double) * rows * nS, cudaMemcpyHostToDevice));
  ctx->stay_K[i] = K;
  ctx->stay_H[i] = H;
  return XT_OK;
}

// ------------------------------------------------------------------------------------------
// evaluation
// ------------------------------------------------------------------------------------------
static int ipow(int b, int e) { int r = 1; for (int i = 0; i < e; ++i) r *= b; return r; }

static bool is_var(const xt_params* p) { return (p->flags & (XT_FLAG_VAR_LOC | XT_FLAG_VAR_DT)) != 0; }

static XtAux make_aux(xt_ctx* ctx, const xt_params* p, int per_track) {
  XtAux ax{};
  ax.aux = ctx->d_aux;
  ax.R = ctx->aux_R;
  ax.ka = ctx->aux_ka;
  ax.d = ctx->d;
  if ((p->flags & XT_FLAG_VAR_DT) && ctx->d_stay[per_track]) {
    ax.stay = ctx->d_stay[per_track];
    ax.leave = ctx->d_leave[per_track];
  }
  return ax;
}

// dd per unit time of every head (replay kernels: dd = ddu * dt[track, loc] up to rounding)
static void dd_unit(const xt_params* p, double* ddu) {
  const int nS = p->nS, nsub = p->nsub, H = ipow(nS, nsub + 1);
  for (int h = 0; h < H; ++h) {
    int x = h;
    double prev = p->twoD[x % nS], sum = 0;
    x /= nS;
    for (int k = 0; k < nsub; ++k) {
      const double cur = p->twoD[x % nS];
      x /= nS;
      sum += (cur + prev) * 0.5;
      prev = cur;
    }
    ddu[h] = sum / nsub;
  }
}

static int check_params(xt_ctx* ctx, const xt_params* p, int* bits_out) {
  if (!p || p->nS < 1 || p->nS > XT_MAX_STATES || p->nsub < 1 || p->d != ctx->d ||
      (p->n_loc != 1 && p->n_loc != p->d) || p->frame_len < 1) {
    set_error(ctx, "xt_params: inconsistent model (nS, nsub, d, n_loc or frame_len)");
    return XT_ERR_ARG;
  }
  long long heads = 1;
  for (int i = 0; i <= p->nsub; ++i) heads *= p->nS;
  if (heads > XT_MAX_HEADS) {
    set_error(ctx, "xt_params: nS^(nb_substeps+1) exceeds XT_MAX_HEADS");
    return XT_ERR_ARG;
  }
  const int bits = p->nS <= 2 ? 1 : (p->nS <= 4 ? 2 : 3);
  if ((long long)bits * std::max(p->frame_len, p->nsub + 1) > 64) {
    set_error(ctx, "xt_params: frame_len too large for the window code (bits*frame_len must be <= 64)");
    return XT_ERR_ARG;
  }
  if (is_var(p)) {
    if (!ctx->d_aux || ((p->flags & XT_FLAG_VAR_LOC) && ctx->aux_ka != p->n_loc) ||
        ((p->flags & XT_FLAG_VAR_DT) && !ctx->aux_has_dt)) {
      set_error(ctx, "xt_params: XT_FLAG_VAR_LOC / XT_FLAG_VAR_DT need matching xt_upload_aux data (n_loc = k_sigma)");
      return XT_ERR_STATE;
    }
    bool bad_tables = false;
    for (int i = 0; i < 2; ++i)  // [0] per chunk (objective), [1] per track (xt_predict)
      bad_tables = bad_tables || (ctx->d_stay[i] && (ctx->stay_K[i] != ipow(p->nS, p->nsub) || ctx->stay_H[i] != ipow(p->nS, p->nsub + 1)));
    if ((p->flags & XT_FLAG_VAR_DT) && bad_tables) {
      set_error(ctx, "xt_set_stay_tables: K / H do not match the model");
      return XT_ERR_ARG;
    }
  }
  *bits_out = bits;
  return XT_OK;
}

static int ensure_plan(xt_ctx* ctx, const xt_params* p, int cap) {
  const int KS = p->n_loc;
  const int CO1 = p->d + 2 * KS + 1;
  const int RH = p->frame_len + p->nsub + 1;
  if (ctx->cap >= cap && ctx->RH >= RH && ctx->nS_alloc >= p->nS && ctx->CO1_alloc >= CO1) return XT_OK;
  cap = std::max(cap, ctx->cap);
  free_plan(ctx);
  const size_t nrec = (size_t)std::max(1, ctx->nrec_total), nch = ctx->chunks.size();
  XT_CUDA_OK(cudaMalloc(&ctx->plan.hdr, sizeof(XtRecHdr) * nrec));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.goff, sizeof(uint16_t) * nrec * (cap + 1)));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.ent, sizeof(uint32_t) * nrec * cap));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.curG, sizeof(uint8_t) * nrec * cap));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.gid, sizeof(uint16_t) * nrec * cap));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.grec, sizeof(unsigned long long) * nrec * cap));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.blob, sizeof(uint4) * nrec * xt_blob_stride16(cap)));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.vrec, sizeof(XtVRec) * nrec * XT_VREC_PER_STEP));
  XT_CUDA_OK(cudaMalloc(&ctx->plan.vok, nrec));
  XT_CUDA_OK(cudaMemset(ctx->plan.vok, 0, nrec));
  ctx->plan.cap = cap;
  XT_CUDA_OK(cudaMalloc(&ctx->d_state1, sizeof(double) * nch * 2 * cap * CO1 * 32));
  XT_CUDA_OK(cudaMalloc(&ctx->d_hist1, sizeof(double) * nch * 2 * cap * RH * p->nS));
  ctx->cap = cap;
  ctx->RH = RH;
  ctx->nS_alloc = p->nS;
  ctx->CO1_alloc = CO1;
  return XT_OK;
}

#ifdef XT_K1_PROF
static long long* g_k1_prof = nullptr;
extern "C" int xt_debug_k1_prof(long long* out, int n_chunks) {
  return cudaMemcpy(out, g_k1_prof, sizeof(long long) * 12 * n_chunks, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -1;
}
#endif
static K1Args make_k1_args(xt_ctx* ctx, int bits) {
  K1Args a{};
  a.chunks = ctx->d_chunks;
  a.soa = ctx->d_soa;
  a.state = ctx->d_state1;
  a.hist = ctx->d_hist1;
  a.plan = ctx->plan;
  a.summ = ctx->d_summ;
  a.cap = ctx->cap;
  a.RH = ctx->RH;
  a.bits = bits;
  a.wpc = ctx->k2_wpc;
  // inline group records are only read by the first-generation linear-domain kernel (k2_variant 1, or
  // the shared-memory fallback when the fused kernel's staging limits are exceeded)
  a.want_grec = ctx->k2_variant == 1 || !ctx->last_fused;
  ctx->plan_has_grec = a.want_grec != 0;
  a.corder = ctx->d_corder;
  a.batch_mode = ctx->k1_batch;
  a.lpt = ctx->k2_lpt;
  for (int i = 0; i < 4; ++i) a.cost[i] = ctx->k2_cost[i];
  a.cost_w0 = ctx->k2_cost_w0;
#ifdef XT_K1_PROF
  if (!g_k1_prof) cudaMalloc(&g_k1_prof, sizeof(long long) * 12 * 65536);
  a.prof = g_k1_prof;
#endif
  return a;
}
// shared-memory scratch of the plan kernel: used when the previous evaluation tells how many
// parents / children to expect and 3 CTAs per SM still fit
// threads per chunk of the plan kernel: 1024 when every chunk can have an SM of its own
static int k1_threads(xt_ctx* ctx) {
  if (ctx->k1_threads) return ctx->k1_threads;
  if ((int)ctx->chunks.size() > ctx->n_sm) return XT_K1_THREADS;
  // a chunk per SM: 512 threads (up to 128 registers each) cover the <= 64 live sequences of the matrix-mode grouping,
  // 1024 threads when the previous evaluation saw more
  return (ctx->spec_maxC > 0 && ctx->spec_maxC <= 64) ? 512 : 1024;
}

static void k1_scratch_caps(xt_ctx* ctx, const xt_params* p, bool use_smem, int* scapP, int* scapC) {
  *scapP = *scapC = 0;
  if (!use_smem || !ctx->k1_smem_scratch || ctx->spec_maxC <= 0) return;
  const int CO1 = p->d + 2 * p->n_loc + 1;
  const int nt = k1_threads(ctx);
  const size_t b = xt_k1_smem(ctx->cap, CO1, ctx->RH, p->nS, ctx->spec_maxP, ctx->spec_maxC,
                              is_var(p) ? ipow(p->nS, p->nsub + 1) : 0, nt);
  // static shared memory of the kernel (bit rows, byte lists: 1.6 / 2.2 / 3.4 KB at 256 / 512 / 1024 threads; it counts
  // against the opt-in maximum of a block together with the dynamic part) and the 1 KB the system reserves per CTA
  const size_t stat = nt >= 1024 ? 3584 : (nt >= 512 ? 2304 : 1792);
  const int ctas = nt == XT_K1_THREADS ? XT_K1_MIN_CTAS : 1;
  if (b + stat + 1024 > (size_t)(228 * 1024) / ctas || b + stat > (size_t)ctx->smem_optin) return;
  *scapP = ctx->spec_maxP;
  *scapC = ctx->spec_maxC;
}

static int enqueue_k1(xt_ctx* ctx, const xt_params* p, int bits, int c0, int nc, cudaStream_t stream, bool smem_scratch) {
  K1Args a = make_k1_args(ctx, bits);
  a.chunk0 = c0;
  k1_scratch_caps(ctx, p, smem_scratch, &a.scapP, &a.scapC);
  const bool var = is_var(p);
  const int varH = var ? ipow(p->nS, p->nsub + 1) : 0;
  const int nt = k1_threads(ctx);
  const size_t smem = xt_k1_smem(ctx->cap, p->d + 2 * p->n_loc + 1, ctx->RH, p->nS, a.scapP, a.scapC, varH, nt);
  if (var) a.ax = make_aux(ctx, p, 0);
  const cudaError_t e = xt_launch_k1(a, *p, smem, nc, stream, nt);
  if (e != cudaSuccess) {
    set_error(ctx, std::string("plan kernel launch (") + std::to_string(nc) + " chunks, " + std::to_string(nt) + " threads, " +
                       std::to_string(smem) + " B shared memory, scratch " + std::to_string(a.scapP) + "/" + std::to_string(a.scapC) +
                       ", cap " + std::to_string(ctx->cap) + "): " + cudaGetErrorString(e));
    return XT_ERR_CUDA;
  }
  ctx->stats.k1_launches++;
  return XT_OK;
}

static int initial_cap(xt_ctx* ctx, const xt_params* p) {
  const int K = ipow(p->nS, p->nsub);
  return std::max(ctx->cap, std::max(128, K * K * p->nS));
}

// scan the per-chunk summaries in h_summ: returns an error, or *need = capacity wanted (0: fine)
static int scan_summaries(xt_ctx* ctx, int* need) {
  *need = 0;
  bool smem_short = false;
  for (size_t c = 0; c < ctx->chunks.size(); ++c) {
    const XtChunkSummary& s = ctx->h_summ[c];
    if (s.err == 1) {
      set_error(ctx, "problem with grouping: a state sequence ended ungrouped in chunk " + std::to_string(c) +
                         " (threshold must be > 0 and the model finite)");
      return XT_ERR_GROUPING;
    }
    if (s.err == 2) *need = std::max(*need, s.need_cap);
    if (s.err == 3) smem_short = true;  // shared-memory scratch too small: rerun with the global one
  }
  if (!*need && smem_short) *need = -1;
  return XT_OK;
}

static int run_plan(xt_ctx* ctx, const xt_params* p, int bits) {
  // run K1 over all chunks, growing the sequence capacity on overflow
  int cap = initial_cap(ctx, p);
  bool smem_scratch = true;
  for (;;) {
    if (cap > XT_HARD_CAP) {
      set_error(ctx, "more than " + std::to_string(XT_HARD_CAP) + " live state sequences; lower frame_len or raise threshold");
      return XT_ERR_CAPACITY;
    }
    int rc = ensure_plan(ctx, p, cap);
    if (rc) return rc;
    cap = ctx->cap;
    rc = enqueue_k1(ctx, p, bits, 0, (int)ctx->chunks.size(), ctx->stream, smem_scratch);
    if (rc) return rc;
    XT_CUDA_OK(cudaMemcpyAsync(ctx->h_summ, ctx->d_summ, sizeof(XtChunkSummary) * ctx->chunks.size(),
                               cudaMemcpyDeviceToHost, ctx->stream));
    XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    int need = 0;
    rc = scan_summaries(ctx, &need);
    if (rc) return rc;
    if (need < 0) {  // the shared-memory scratch (sized from the previous evaluation) was too small
      smem_scratch = false;
      continue;
    }
    if (need == 0) break;
    int ncap = cap;
    while (ncap < need) ncap *= 2;
    cap = ncap;
  }
  std::copy(ctx->h_summ, ctx->h_summ + ctx->chunks.size(), ctx->summ.begin());
  return XT_OK;
}

// Deterministic final reduction of the per-CTA partial sums (second level of tracking.py:1069).
__global__ void __launch_bounds__(1024) k_reduce(const double* __restrict__ partial, int n, double* out) {
  __shared__ double sh[1024];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 1024) acc += partial[i];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
}

// per-tile partial sums -> per-chunk sums (one warp per chunk, fixed order) -> device total (fixed tree over the
// chunk sums).  `table`: 0 / 1 = fused work tables (tiles of 32 / 64 tracks, corder), 2 = plain work table.
__global__ void k_reduce_chunks(const double* __restrict__ partial, const int32_t* __restrict__ w0,
                                const int32_t* __restrict__ cid, double* __restrict__ csum) {
  const int q = blockIdx.x, lane = threadIdx.x;
  double acc = 0.0;
  for (int i = w0[q] + lane; i < w0[q + 1]; i += 32) acc += partial[i];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  if (lane == 0) csum[cid ? cid[q] : q] = acc;
}
static int enqueue_reduce(xt_ctx* ctx, int table, double* d_out) {
  const int nch = (int)ctx->chunks.size();
  k_reduce_chunks<<<nch, 32, 0, ctx->stream>>>(ctx->d_partial, ctx->d_cw0[table], table < 2 ? ctx->d_corder : nullptr,
                                               ctx->d_csum);
  ctx->stats.k2_launches += 1;
  if (d_out) {  // device-resident total (xt_sum_logp_async); the synchronous entry points add the chunk sums on the host
    k_reduce<<<1, 1024, 0, ctx->stream>>>(ctx->d_csum, nch, d_out);
    ctx->stats.k2_launches += 1;
  }
  XT_CUDA_OK(cudaGetLastError());
  return XT_OK;
}
// objective of this context: the chunk sums added in chunk order on the host (after the evaluation)
static int read_total(xt_ctx* ctx, double* out) {
  const size_t nch = ctx->chunks.size();
  if (!ctx->csum_fetched) {
    XT_CUDA_OK(cudaMemcpyAsync(ctx->h_csum, ctx->d_csum, sizeof(double) * nch, cudaMemcpyDeviceToHost, ctx->stream));
    XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  }
  double acc = 0.0;
  for (size_t c = 0; c < nch; ++c) acc += ctx->h_csum[c];
  *out = acc;
  return XT_OK;
}

static int finish_eval(xt_ctx* ctx, const xt_params* p, int table, double* d_out, int64_t su, int64_t sg, int maxC) {
  int rcr = enqueue_reduce(ctx, table, d_out);
  if (rcr) return rcr;
  XT_CUDA_OK(cudaEventRecord(ctx->ev[2], ctx->stream));
  ctx->stats.n_tracks = ctx->n_tracks;
  ctx->stats.track_steps = ctx->track_steps;
  ctx->stats.seq_updates = su;
  ctx->stats.seq_groups = sg;
  ctx->stats.max_nB_in = maxC;
  ctx->stats.n_chunks = (int)ctx->chunks.size();
  ctx->last_p = *p;
  ctx->have_eval = true;
  return XT_OK;
}

// work counters of an evaluation from the chunk summaries in ctx->summ
static void work_counters(xt_ctx* ctx, const xt_params* p, int* Pmax, int* maxC, int64_t* su, int64_t* sg) {
  *Pmax = 1;
  *maxC = 0;
  *su = *sg = 0;
  for (size_t c = 0; c < ctx->chunks.size(); ++c) {
    const XtChunkSummary& s = ctx->summ[c];
    *Pmax = std::max(*Pmax, s.max_nP);
    *maxC = std::max(*maxC, s.max_nC);
    *su += s.sum_nC * ctx->chunks[c].nT;
    *sg += s.sum_nG * ctx->chunks[c].nT;
  }
  const int K = ipow(p->nS, p->nsub);
  *maxC = std::max(*maxC, K * p->nS);
  ctx->spec_maxP = *Pmax;
  ctx->spec_maxC = *maxC;
  *Pmax = std::max(*Pmax, 4);  // the fused kernel parks its end-of-track partial sums in an idle state buffer
}

struct FusedLaunch {  // everything a fused replay launch needs besides its tile range
  K2Tab tab;
  K2FArgs fa;
  size_t smem;
  int wpc, tpt;
  bool var;
  bool gst;  // state in global memory (the live sequences of a tile exceed shared memory)
  bool f32;  // single-precision replay kernel
};

// FP32 replay applies when every table entry is zero or comfortably inside the FP32 range (the weights
// themselves carry an extended exponent, the per-step factors do not)
static bool f32_tables_ok(const xt_params* p, const double* Lsum) {
  const int K = ipow(p->nS, p->nsub), H = K * p->nS;
  auto fac_ok = [](double v) { return v == 0.0 || (v >= 1e-20 && v <= 1e3); };
  for (int h = 0; h < H; ++h) {
    if (!fac_ok(std::exp(p->LT[h])) || !fac_ok(std::exp(p->LT[h] + p->Lp_stay[h % K])) ||
        !fac_ok(std::exp(p->LT[h] + p->LF[h])))
      return false;
    if (!(p->dd[h] >= 0.0 && p->dd[h] <= 1e6)) return false;
  }
  for (int s = 0; s < p->nS; ++s)
    if (!fac_ok(std::exp(Lsum[s]))) return false;
  for (int k = 0; k < p->n_loc; ++k)
    if (!(p->l2[k] >= 1e-12 && p->l2[k] <= 1e6)) return false;
  return true;
}

static void leave_sums(const xt_params* p, double* Lsum) {
  const int K = ipow(p->nS, p->nsub);
  for (int s = 0; s < p->nS; ++s) {
    double mx = -INFINITY;
    for (int r = 0; r < K; ++r) mx = std::max(mx, p->L_leave[r + K * s]);
    double acc = 0;
    for (int r = 0; r < K; ++r) acc += std::exp(p->L_leave[r + K * s] - mx);
    Lsum[s] = std::log(acc) + mx;
  }
}

// returns false if the fused kernel cannot run with Pmax parent slots (shared memory / staging limits)
static bool prepare_fused(xt_ctx* ctx, const xt_params* p, int Pmax, FusedLaunch* fl) {
  const int K = ipow(p->nS, p->nsub), KS = p->n_loc, H = K * p->nS;
  fl->wpc = ctx->k2_wpc;
  fl->tpt = ctx->k2_tpt;
  fl->var = is_var(p);
  if (fl->var) fl->tpt = 1;
  if (fl->tpt == 2 && xt_fused_smem(p->d, KS, Pmax, K, H, fl->wpc, 2) > (size_t)ctx->smem_optin) fl->tpt = 1;
  fl->smem = xt_fused_smem(p->d, KS, Pmax, K, H, fl->wpc, fl->tpt, fl->var);
  fl->gst = false;
  fl->f32 = false;
  if (ctx->k2_variant != 0 || ctx->force_global || (fl->var && fl->wpc != 4)) return false;
  double Lsum[XT_MAX_STATES];
  leave_sums(p, Lsum);
  if (ctx->k2_fp32 && !fl->var && fl->wpc == 4 && xt_f32_smem(p->d, KS, Pmax, K, H) <= (size_t)ctx->smem_optin &&
      xt_fused_blob16(Pmax, K) <= 256 && f32_tables_ok(p, Lsum)) {
    fl->f32 = true;
    fl->wpc = 4;
    fl->tpt = 1;
    fl->smem = xt_f32_smem(p->d, KS, Pmax, K, H);
  }
  const int smem_ctas = fl->smem ? (int)(((size_t)228 * 1024) / (fl->smem + 1024)) : 0;
  if (!fl->f32 && (fl->smem > (size_t)ctx->smem_optin || xt_fused_blob16(Pmax, K) > 64 * fl->wpc ||
                   (!fl->var && fl->wpc == 4 && smem_ctas < ctx->k2_gst_below_ctas))) {
    // the live sequences of a tile do not fit in shared memory: same kernel with its state in global memory
    const size_t stride = xt_fused_gstride(p->d, KS, Pmax);
    const size_t need = stride * 32 * (size_t)ctx->n_sm;
    if (!ctx->k2_gst || fl->var || fl->wpc != 4 || Pmax > 4095 || need > ((size_t)8 << 30) ||
        xt_fused_smem_gst(Pmax, K, H) > (size_t)ctx->smem_optin)
      return false;
    if (need > ctx->fstate_bytes) {
      cudaFree(ctx->d_fstate);
      ctx->d_fstate = nullptr;
      ctx->fstate_bytes = 0;
      if (cudaMalloc(&ctx->d_fstate, need) != cudaSuccess) {
        cudaGetLastError();
        return false;
      }
      ctx->fstate_bytes = need;
    }
    if (!ctx->d_fslots) {
      if (cudaMalloc(&ctx->d_fslots, sizeof(unsigned) * ctx->n_sm) != cudaSuccess) return false;
      cudaMemset(ctx->d_fslots, 0, sizeof(unsigned) * ctx->n_sm);
    }
    fl->gst = true;
    fl->tpt = 1;
    fl->smem = xt_fused_smem_gst(Pmax, K, H);
  }
  K2Tab& tab = fl->tab;
  tab = K2Tab{};
  // constant folded into the weight factors of the FP64 kernel (K2Tab::lnc): c = prod over dims of sqrt(l2)
  double cfold = 1.0;
  if (!fl->var && !fl->f32)
    for (int dim = 0; dim < p->d; ++dim) cfold *= std::sqrt(p->l2[KS == 1 ? 0 : dim]);
  if (!(cfold > 1e-30 && cfold < 1e30)) cfold = 1.0;  // (keeps every intermediate product far from the exponent limits)
  tab.lnc = std::log(cfold);
  for (int h = 0; h < H; ++h) {
    tab.tau0[h] = std::exp(p->LT[h]) * cfold;
    tab.tau1[h] = std::exp(p->LT[h] + p->Lp_stay[h % K]) * cfold;
    tab.dd[h] = p->dd[h];
    tab.winit[h] = std::exp(p->LT[h] + p->LF[h]) * cfold;
  }
  for (int s = 0; s < p->nS; ++s) tab.leave[s] = std::exp(Lsum[s]);
  for (int k = 0; k < KS; ++k) tab.l2[k] = p->l2[k];
  for (int j = 0; j < 16; ++j) tab.e2[j] = std::exp2((double)j / 16.0);
  tab.nS = p->nS;
  tab.nsub = p->nsub;
  tab.K = K;
  tab.min_len = p->min_len;
  {
    const double kc[6] = XT_EXP_CONSTS;
    for (int i = 0; i < 6; ++i) tab.kc[i] = kc[i];
  }
  tab.flags = p->flags;
  tab.loc_slope = p->loc_slope;
  tab.loc_offset = p->loc_offset;
  if (p->flags & XT_FLAG_VAR_DT) dd_unit(p, tab.dd);
  K2FArgs& fa = fl->fa;
  fa = K2FArgs{};
  if (fl->var) fa.ax = make_aux(ctx, p, 0);
  if (fl->gst) {
    fa.gstate = ctx->d_fstate;
    fa.gslots = ctx->d_fslots;
    fa.gstride = xt_fused_gstride(p->d, KS, Pmax);
  }
  fa.chunks = ctx->d_chunks;
  fa.work = ctx->d_workf[fl->tpt - 1];
  fa.soa = ctx->d_soa;
  fa.plan = ctx->plan;
  fa.logp = ctx->d_logp;
  fa.partial = ctx->d_partial;
  fa.summ = ctx->d_summ;
  fa.spec_fail = ctx->d_spec;
  fa.Pcap = Pmax;
  return true;
}

// fused replay of the chunks at positions [c0, c1) of corder on `stream`
static int enqueue_fused(xt_ctx* ctx, const xt_params* p, const FusedLaunch& fl, int c0, int c1, cudaStream_t stream) {
  K2FArgs fa = fl.fa;
  const std::vector<int>& w0 = ctx->chunk_w0[fl.tpt - 1];
  fa.work0 = w0[c0];
  fa.n_work = w0[c1] - w0[c0];
  if (fa.n_work <= 0) return XT_OK;
  const cudaError_t ef = fl.f32 ? xt_launch_k2_f32(p->d, p->n_loc, fa, fl.tab, fl.smem, stream)
                                : xt_launch_k2_fused(p->d, p->n_loc, fa, fl.tab, fl.smem, fl.wpc, fl.tpt, stream, fl.var);
  XT_CUDA_OK(ef);
  ctx->stats.k2_launches++;
  ctx->stats.fp32 = fl.f32 ? 1 : 0;
  return XT_OK;
}

// shape of the model: a resident plan can only be verified for parameters of the same shape
static bool same_structure(const xt_params& a, const xt_params& b) {
  return a.nS == b.nS && a.nsub == b.nsub && a.d == b.d && a.n_loc == b.n_loc && a.frame_len == b.frame_len && a.flags == b.flags;
}
static void mark_plan_valid(xt_ctx* ctx, const xt_params* p) {
  ctx->plan_valid = true;
  ctx->plan_sig = *p;
}
#define XT_FROZEN_FUSED 1  // fused replay kernel (shared- or global-memory state, VAR instantiation included)
#define XT_FROZEN_OLD 2    // first-generation linear-domain / log-domain kernel of the two-phase path
// the evaluation that just succeeded left a plan for the frozen entry points: which replay launch it ran
static void mark_frozen(xt_ctx* ctx, const xt_params* p, int kind, int Pcap) {
  ctx->frozen_kind = kind;
  ctx->frozen_Pcap = Pcap;
  ctx->frozen_sig = *p;
}

#define XT_RETRY 1        // internal: the speculative single-pass evaluation has to be redone in two phases
#define XT_RETRY_EARLY 2  // same, and nothing was enqueued yet (host buffers not copied)

// Pipelined evaluation: for every group of chunks, plan and replay are enqueued back to back on
// one of NCS streams, so the (latency-bound) plan kernel of one group overlaps the replay of
// another.  The replay launches are sized with the parent-slot count of the previous evaluation
// and check it against the plan's summary; the host verifies afterwards (one synchronisation per
// evaluation) and falls back to the two-phase path if the guess was too small.
// `xyz` != nullptr: the segments are first copied from these host buffers (upload stream) and
// each segment is its own group, so that the copy of one segment overlaps the kernels of another.
static int evaluate_pipelined(xt_ctx* ctx, const xt_params* p, int bits, double* d_out, const double* const* xyz) {
  int rc = ensure_plan(ctx, p, initial_cap(ctx, p));
  if (rc) return rc;
  FusedLaunch fl;
  if (!prepare_fused(ctx, p, ctx->spec_Pmax, &fl)) return XT_RETRY_EARLY;
  const int nch = (int)ctx->chunks.size(), n_seg = (int)ctx->seg_L.size();
  XT_CUDA_OK(cudaMemsetAsync(ctx->d_spec, 0, sizeof(int), ctx->stream));
  XT_CUDA_OK(cudaEventRecord(ctx->ev[0], ctx->stream));
  XT_CUDA_OK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  const int NS = ctx->n_streams;
  for (int i = 0; i < NS; ++i) XT_CUDA_OK(cudaStreamWaitEvent(ctx->cs[i], ctx->ev_fork, 0));
  // host buffers: segments are copied longest tracks first
  std::vector<int> order(n_seg);
  for (int s = 0; s < n_seg; ++s) order[s] = s;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return ctx->seg_L[x] > ctx->seg_L[y]; });
  if (xyz) {
    rc = ensure_stage_all(ctx);
    if (rc) return rc;
    XT_CUDA_OK(cudaStreamWaitEvent(ctx->up_stream, ctx->ev_fork, 0));
    for (int i = 0; i < n_seg; ++i) {  // all copies first: the link stays busy while the host enqueues the kernels
      const int s = order[i];
      XT_CUDA_OK(cudaMemcpyAsync(ctx->stage_all + ctx->seg_stage_off[s], xyz[s],
                                 sizeof(double) * (size_t)ctx->seg_n[s] * ctx->seg_L[s] * ctx->d, cudaMemcpyHostToDevice,
                                 ctx->up_stream));
      XT_CUDA_OK(cudaEventRecord(ctx->ev_seg[s], ctx->up_stream));
    }
    for (int i = 0; i < n_seg; ++i) {
      const int s = order[i];
      cudaStream_t st = ctx->cs[i % NS];
      XT_CUDA_OK(cudaStreamWaitEvent(st, ctx->ev_seg[s], 0));
      rc = enqueue_pack(ctx, s, st);
      if (rc) return rc;
      const int c0 = ctx->seg_pos0[s], c1 = ctx->seg_pos1[s];
      rc = enqueue_k1(ctx, p, bits, c0, c1 - c0, st, true);
      if (rc) return rc;
      rc = enqueue_fused(ctx, p, fl, c0, c1, st);
      if (rc) return rc;
    }
  } else {
    // resident data: n_groups contiguous ranges of corder (longest tracks first) with about equal
    // replay work
    const int G = std::max(1, std::min(ctx->n_groups, nch));
    int q0 = 0, g = 0;
    int64_t done = 0;
    std::vector<int> gq;  // group boundaries in corder
    gq.push_back(0);
    for (int q = 0; q < nch; ++q) {
      const XtChunk& ck = ctx->chunks[ctx->corder[q]];
      done += (int64_t)ck.nT * (ck.L - 1);
      const bool last = q + 1 == nch;
      if (last || (g + 1 < G && done * G >= ctx->track_steps * (int64_t)(g + 1))) {
        gq.push_back(q + 1);
        q0 = q + 1;
        ++g;
      }
    }
    (void)q0;
    // all plan kernels first (they are latency-bound and run concurrently), then each group's
    // replay behind its own plan
    for (int pass = 0; pass < 2; ++pass)
      for (int k = 0; k + 1 < (int)gq.size(); ++k) {
        cudaStream_t st = ctx->cs[k % NS];
        rc = pass == 0 ? enqueue_k1(ctx, p, bits, gq[k], gq[k + 1] - gq[k], st, true)
                       : enqueue_fused(ctx, p, fl, gq[k], gq[k + 1], st);
        if (rc) return rc;
      }
  }
  for (int i = 0; i < NS; ++i) {
    XT_CUDA_OK(cudaEventRecord(ctx->ev_join[i], ctx->cs[i]));
    XT_CUDA_OK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[i], 0));
  }
  XT_CUDA_OK(cudaEventRecord(ctx->ev[1], ctx->stream));
  rc = enqueue_reduce(ctx, fl.tpt - 1, d_out);
  if (rc) return rc;
  XT_CUDA_OK(cudaEventRecord(ctx->ev[2], ctx->stream));
  XT_CUDA_OK(cudaMemcpyAsync(ctx->h_summ, ctx->d_summ, sizeof(XtChunkSummary) * nch, cudaMemcpyDeviceToHost, ctx->stream));
  XT_CUDA_OK(cudaMemcpyAsync(ctx->h_spec, ctx->d_spec, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  int need = 0;
  rc = scan_summaries(ctx, &need);
  if (rc) return rc;
  if (need || *ctx->h_spec) return XT_RETRY;
  std::copy(ctx->h_summ, ctx->h_summ + nch, ctx->summ.begin());
  int Pmax, maxC;
  int64_t su, sg;
  work_counters(ctx, p, &Pmax, &maxC, &su, &sg);
  ctx->spec_Pmax = Pmax;
  ctx->stats.pipelined = 1;
  ctx->stats.n_tracks = ctx->n_tracks;
  ctx->stats.track_steps = ctx->track_steps;
  ctx->stats.seq_updates = su;
  ctx->stats.seq_groups = sg;
  ctx->stats.max_nB_in = maxC;
  ctx->stats.n_chunks = nch;
  ctx->last_p = *p;
  ctx->have_eval = true;
  ctx->last_fused = true;
  mark_plan_valid(ctx, p);
  mark_frozen(ctx, p, XT_FROZEN_FUSED, fl.fa.Pcap);
  return XT_OK;
}

// Evaluation along the RESIDENT plan: the replay kernel runs on the resident records while the plan kernel, in
// verification mode, re-evaluates every floating-point decision those records rest on with the new parameters (both
// only read the plan, so they run concurrently).  Chunks with a changed decision are planned again from scratch and
// replayed again before the sums are formed; everything else of the result is already final.  Returns XT_RETRY when
// the evaluation has to take the construction path instead.
static double xt_now_us() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

static int evaluate_verified(xt_ctx* ctx, const xt_params* p, int bits, double* d_out) {
  const int nch = (int)ctx->chunks.size();
  static const bool trace = std::getenv("XT_TRACE") != nullptr;  // host-side timeline of the call (diagnostic)
  const double t_in = trace ? xt_now_us() : 0.0;
  double t_k1 = 0, t_k2 = 0, t_enq = 0;
  FusedLaunch fl;
  if (is_var(p) || ctx->spec_maxC <= 0 || ctx->spec_maxC > 64 || !prepare_fused(ctx, p, ctx->spec_Pmax, &fl)) return XT_RETRY_EARLY;
  int nt = k1_threads(ctx);
  if (nt == 1024) nt = 512;
  K1Args a = make_k1_args(ctx, bits);
  a.chunk0 = 0;
  a.vflag = ctx->d_vflag;
  k1_scratch_caps(ctx, p, true, &a.scapP, &a.scapC);
  if (a.scapC <= 0) return XT_RETRY_EARLY;
  const size_t smem = xt_k1_smem(ctx->cap, p->d + 2 * p->n_loc + 1, ctx->RH, p->nS, a.scapP, a.scapC, 0, nt);
  if (ctx->spec_dirty) {  // (the replay kernel only ever sets the flag: it is cleared here after it was seen set)
    XT_CUDA_OK(cudaMemsetAsync(ctx->d_spec, 0, sizeof(int), ctx->stream));
    ctx->spec_dirty = false;
  }
  // (every CTA of the verification launch writes its chunk's flag, 0 included: no clearing pass)
  // the replay stays on the main stream; only the verification kernel forks off (and joins before the reduction)
  XT_CUDA_OK(cudaEventRecord(ctx->ev[0], ctx->stream));
  XT_CUDA_OK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  XT_CUDA_OK(cudaStreamWaitEvent(ctx->cs[0], ctx->ev_fork, 0));
  {
    const cudaError_t e = xt_launch_k1_verify(a, *p, smem, nch, ctx->cs[0], nt);
    if (e != cudaSuccess) {
      set_error(ctx, std::string("plan verification launch: ") + cudaGetErrorString(e));
      return XT_ERR_CUDA;
    }
    ctx->stats.k1_launches++;
  }
  if (trace) t_k1 = xt_now_us();
  int rc;
  if (ctx->verify_fork_k2) {  // (option "verify_fork_k2": the replay on a stream of its own, joined before the reduction)
    XT_CUDA_OK(cudaStreamWaitEvent(ctx->cs[1], ctx->ev_fork, 0));
    rc = enqueue_fused(ctx, p, fl, 0, nch, ctx->cs[1]);
    if (rc) return rc;
    XT_CUDA_OK(cudaEventRecord(ctx->ev_join[1], ctx->cs[1]));
    XT_CUDA_OK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[1], 0));
  } else {
    rc = enqueue_fused(ctx, p, fl, 0, nch, ctx->stream);
    if (rc) return rc;
  }
  if (trace) t_k2 = xt_now_us();
  XT_CUDA_OK(cudaEventRecord(ctx->ev_join[0], ctx->cs[0]));
  XT_CUDA_OK(cudaEventRecord(ctx->ev[1], ctx->stream));
  rc = enqueue_reduce(ctx, fl.tpt - 1, d_out);
  if (rc) return rc;
  XT_CUDA_OK(cudaEventRecord(ctx->ev[2], ctx->stream));
  XT_CUDA_OK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));  // (the flags of the verification kernel)
  // chunk sums, verification flags and the speculation word in one copy (one round trip)
  XT_CUDA_OK(cudaMemcpyAsync(ctx->h_tail, ctx->d_tail, ctx->tail_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (trace) t_enq = xt_now_us();
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  if (trace) {
    const double t_sync = xt_now_us();
    float g01 = 0.f, g12 = 0.f;
    cudaEventElapsedTime(&g01, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&g12, ctx->ev[1], ctx->ev[2]);
    std::fprintf(stderr, "xt trace: host us: prepare+fork+K1v launch %.1f, K2 launch %.1f, join+reduce+copy enqueue %.1f, wait %.1f, total %.1f"
                         " | device us: replay %.1f, reduce %.1f\n",
                 t_k1 - t_in, t_k2 - t_k1, t_enq - t_k2, t_sync - t_enq, t_sync - t_in, g01 * 1e3, g12 * 1e3);
  }
  if (*ctx->h_spec) {
    ctx->spec_dirty = true;
    return XT_RETRY;
  }
  ctx->csum_fetched = true;
  std::vector<int32_t> redo;
  for (int c = 0; c < nch; ++c)
    if (ctx->h_vflag[c]) redo.push_back(c);
  ctx->stats.plan_verified = 1;
  ctx->stats.replanned = (int)redo.size();
  if (!redo.empty()) {
    ctx->csum_fetched = false;
    // a decision changed in some chunks: new plans for those (construction mode), their tiles replayed again
    if ((int)redo.size() > 64 || (int)redo.size() * 4 > nch + 3) return XT_RETRY;
    std::stable_sort(redo.begin(), redo.end(), [&](int x, int y) { return ctx->chunks[x].L > ctx->chunks[y].L; });
    XT_CUDA_OK(cudaMemcpyAsync(ctx->d_redo, redo.data(), sizeof(int32_t) * redo.size(), cudaMemcpyHostToDevice, ctx->stream));
    K1Args b = make_k1_args(ctx, bits);
    b.chunk0 = 0;
    b.corder = ctx->d_redo;
    k1_scratch_caps(ctx, p, true, &b.scapP, &b.scapC);
    const int ntc = k1_threads(ctx);
    const size_t smem_c = xt_k1_smem(ctx->cap, p->d + 2 * p->n_loc + 1, ctx->RH, p->nS, b.scapP, b.scapC, 0, ntc);
    const cudaError_t e = xt_launch_k1(b, *p, smem_c, (int)redo.size(), ctx->stream, ntc);
    if (e != cudaSuccess) {
      set_error(ctx, std::string("plan kernel launch (changed chunks): ") + cudaGetErrorString(e));
      return XT_ERR_CUDA;
    }
    ctx->stats.k1_launches++;
    XT_CUDA_OK(cudaMemcpyAsync(ctx->h_summ, ctx->d_summ, sizeof(XtChunkSummary) * nch, cudaMemcpyDeviceToHost, ctx->stream));
    XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    for (int c : redo) {  // anything but a plain new plan within the sizes of this launch: full construction path
      const XtChunkSummary& sm = ctx->h_summ[c];
      if (sm.err != 0 || sm.max_nP > ctx->spec_Pmax) return XT_RETRY;
    }
    for (int c : redo) {
      rc = enqueue_fused(ctx, p, fl, ctx->corder_pos[c], ctx->corder_pos[c] + 1, ctx->stream);
      if (rc) return rc;
    }
    XT_CUDA_OK(cudaEventRecord(ctx->ev[1], ctx->stream));
    rc = enqueue_reduce(ctx, fl.tpt - 1, d_out);
    if (rc) return rc;
    XT_CUDA_OK(cudaEventRecord(ctx->ev[2], ctx->stream));
    XT_CUDA_OK(cudaMemcpyAsync(ctx->h_spec, ctx->d_spec, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    if (*ctx->h_spec) {
      ctx->spec_dirty = true;
      return XT_RETRY;
    }
    for (int c : redo) ctx->summ[c] = ctx->h_summ[c];
  }
  int Pmax, maxC;
  int64_t su, sg;
  work_counters(ctx, p, &Pmax, &maxC, &su, &sg);
  ctx->spec_Pmax = std::max(ctx->spec_Pmax, Pmax);
  ctx->stats.pipelined = 1;
  ctx->stats.n_tracks = ctx->n_tracks;
  ctx->stats.track_steps = ctx->track_steps;
  ctx->stats.seq_updates = su;
  ctx->stats.seq_groups = sg;
  ctx->stats.max_nB_in = maxC;
  ctx->stats.n_chunks = nch;
  ctx->last_p = *p;
  ctx->have_eval = true;
  mark_plan_valid(ctx, p);
  mark_frozen(ctx, p, XT_FROZEN_FUSED, fl.fa.Pcap);
  return XT_OK;
}

// first-generation linear-domain replay kernel (k2_variant 1) or its log-domain global-memory variant, over all chunks
// with Pmax parent slots; per-track log P to `logp`, per-tile partial sums to `partial` (plain work table)
static int enqueue_old(xt_ctx* ctx, const xt_params* p, int Pmax, double* logp, double* partial) {
  const int K = ipow(p->nS, p->nsub);
  const int KS = p->n_loc, CO = p->d + KS + 1;
  K2Args a{};
  a.chunks = ctx->d_chunks;
  a.work = ctx->d_work;
  a.soa = ctx->d_soa;
  a.plan = ctx->plan;
  a.summ = ctx->d_summ;
  a.logp = logp;
  a.partial = partial;
  a.Pcap = Pmax;
  a.n_work = (int)ctx->work.size();
  leave_sums(p, a.Lsum);
  K2Lin lin{};
  for (int h = 0; h < K * p->nS; ++h) {
    lin.winit[h] = std::exp(p->LT[h] + p->LF[h]);
    lin.tau0[h] = std::exp(p->LT[h]);
    lin.tau1[h] = std::exp(p->LT[h] + p->Lp_stay[h % K]);
  }
  for (int s = 0; s < p->nS; ++s) lin.leave[s] = std::exp(a.Lsum[s]);
  const int wpc = ctx->k2_wpc;
  const size_t state_bytes = (size_t)2 * Pmax * CO * 32 * sizeof(double);
  const size_t smem = state_bytes + (size_t)2 * wpc * 32 * sizeof(double);
  const bool use_smem = smem <= (size_t)ctx->smem_optin && !ctx->force_global && !is_var(p);
  if (is_var(p)) {
    a.ax = make_aux(ctx, p, 0);
    if (p->flags & XT_FLAG_VAR_DT) dd_unit(p, a.ddu);
  }
  int grid = a.n_work;
  if (!use_smem) {
    grid = std::min(a.n_work, ctx->n_sm * ctx->k2_global_ctas);
    const size_t need = (size_t)grid * state_bytes;
    if (need > ctx->gstate_bytes) {
      cudaFree(ctx->d_gstate);
      ctx->d_gstate = nullptr;
      ctx->gstate_bytes = 0;
      XT_CUDA_OK(cudaMalloc(&ctx->d_gstate, need));
      ctx->gstate_bytes = need;
    }
    a.gstate = ctx->d_gstate;
  }
  const cudaError_t e = xt_launch_k2_old(a, *p, lin, smem, use_smem, grid, wpc, ctx->stream);
  XT_CUDA_OK(e);
  ctx->stats.k2_launches++;
  return XT_OK;
}

static int evaluate(xt_ctx* ctx, const xt_params* p, double* d_out, const double* const* xyz) {
  if (!ctx) return XT_ERR_ARG;
  if (ctx->chunks.empty()) {
    set_error(ctx, "no tracks uploaded");
    return XT_ERR_STATE;
  }
  int bits = 0;
  int rc = check_params(ctx, p, &bits);
  if (rc) return rc;
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  ctx->stats = xt_stats{};
  ctx->csum_fetched = false;
  ctx->frozen_kind = 0;  // (set again when this evaluation succeeds)
  if (!xyz && ctx->pipeline && ctx->plan_verify && ctx->plan_valid && ctx->last_fused && same_structure(*p, ctx->plan_sig)) {
    rc = evaluate_verified(ctx, p, bits, d_out);
    if (rc != XT_RETRY && rc != XT_RETRY_EARLY) return rc;
    ctx->stats = xt_stats{};
    ctx->plan_valid = false;
  }
  ctx->spec_dirty = true;  // (the construction paths clear the flag themselves and may leave it set)
  if (ctx->pipeline && ctx->spec_Pmax > 0) {
    rc = evaluate_pipelined(ctx, p, bits, d_out, xyz);
    if (rc != XT_RETRY && rc != XT_RETRY_EARLY) return rc;
    if (rc == XT_RETRY) xyz = nullptr;  // the data are resident now
    ctx->stats = xt_stats{};
  }
  if (xyz) {  // host buffers, no history to size the launches with: plain upload first
    for (int s = 0; s < (int)ctx->seg_L.size(); ++s) {
      rc = enqueue_segment(ctx, s, xyz[s], s, ctx->stream);
      if (rc) return rc;
    }
  }
  // two-phase path: plan for all chunks, read the summaries back, then the replay
  XT_CUDA_OK(cudaEventRecord(ctx->ev[0], ctx->stream));
  rc = run_plan(ctx, p, bits);
  if (rc) return rc;
  XT_CUDA_OK(cudaEventRecord(ctx->ev[1], ctx->stream));
  int Pmax, maxC;
  int64_t su, sg;
  work_counters(ctx, p, &Pmax, &maxC, &su, &sg);
  ctx->spec_Pmax = Pmax;
  const int nch = (int)ctx->chunks.size();
  FusedLaunch fl;
  if (prepare_fused(ctx, p, Pmax, &fl)) {
    XT_CUDA_OK(cudaMemsetAsync(ctx->d_spec, 0, sizeof(int), ctx->stream));
    rc = enqueue_fused(ctx, p, fl, 0, nch, ctx->stream);
    if (rc) return rc;
    ctx->last_fused = true;
    rc = finish_eval(ctx, p, fl.tpt - 1, d_out, su, sg, maxC);
    if (rc == XT_OK) {
      mark_plan_valid(ctx, p);
      mark_frozen(ctx, p, XT_FROZEN_FUSED, Pmax);
    }
    return rc;
  }
  if (ctx->last_fused || !ctx->plan_has_grec) {  // the plan was written without the records this path reads
    ctx->last_fused = false;
    rc = run_plan(ctx, p, bits);
    if (rc) return rc;
  }
  // first-generation linear-domain kernel (k2_variant 1) or log-domain global-memory fallback
  rc = enqueue_old(ctx, p, Pmax, ctx->d_logp, ctx->d_partial);
  if (rc) return rc;
  rc = finish_eval(ctx, p, 2, d_out, su, sg, maxC);
  if (rc == XT_OK) mark_frozen(ctx, p, XT_FROZEN_OLD, Pmax);
  return rc;
}

extern "C" int xt_sum_logp(xt_ctx* ctx, const xt_params* p, double* out) {
  int rc = evaluate(ctx, p, nullptr, nullptr);
  if (rc) return rc;
  return read_total(ctx, out);
}

extern "C" int xt_sum_logp_host(xt_ctx* ctx, int32_t n_seg, const int32_t* L, const int64_t* n, const int32_t* isBL,
                                const double* const* xyz, int32_t d, int32_t chunk_size, const xt_params* p, double* out) {
  if (!ctx) return XT_ERR_ARG;
  int rc = setup_layout(ctx, n_seg, L, n, isBL, d, chunk_size);
  if (rc) return rc;
  rc = evaluate(ctx, p, nullptr, xyz);
  if (rc) return rc;
  return read_total(ctx, out);
}

extern "C" int xt_sum_logp_async(xt_ctx* ctx, const xt_params* p, double* d_out, void* cuda_stream) {
  // The result lands in d_out in stream order of the context's stream; if the caller passes its
  // own stream it is made to wait for the result.
  if (!ctx) return XT_ERR_ARG;
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  XT_CUDA_OK(cudaEventRecord(ctx->ev_fork, (cudaStream_t)cuda_stream));  // (ev_fork is re-recorded by the evaluation)
  XT_CUDA_OK(cudaStreamWaitEvent(ctx->stream, ctx->ev_fork, 0));
  int rc = evaluate(ctx, p, d_out, nullptr);
  if (rc) return rc;
  XT_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)cuda_stream, ctx->ev[2], 0));
  return XT_OK;
}

extern "C" int xt_set_option(xt_ctx* ctx, const char* name, int value) {
  if (!ctx || !name) return XT_ERR_ARG;
  ctx->plan_valid = false;  // (records and schedules depend on the options: the next evaluation plans from scratch)
  ctx->frozen_kind = 0;
  if (std::strcmp(name, "plan_verify") == 0) {
    ctx->plan_verify = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "force_global_replay") == 0) {
    ctx->force_global = value != 0;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_variant") == 0) {
    if (value != 0 && value != 1) {
      set_error(ctx, "xt_set_option: k2_variant must be 0 (fused) or 1 (first-generation linear)");
      return XT_ERR_ARG;
    }
    ctx->k2_variant = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k1_threads") == 0) {
    if (value != 0 && value != 256 && value != 512 && value != 1024) {
      set_error(ctx, "xt_set_option: k1_threads must be 0 (automatic), 256, 512 or 1024");
      return XT_ERR_ARG;
    }
    ctx->k1_threads = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_gst_below_ctas") == 0) {
    ctx->k2_gst_below_ctas = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "fp32_replay") == 0) {
    ctx->k2_fp32 = value != 0;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_gst") == 0) {
    ctx->k2_gst = value != 0;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_global_ctas") == 0) {
    if (value < 1 || value > 32) {
      set_error(ctx, "xt_set_option: k2_global_ctas must be in 1..32");
      return XT_ERR_ARG;
    }
    ctx->k2_global_ctas = value;
    return XT_OK;
  }
  if (std::strcmp(name, "predict_shared_plans") == 0) {
    ctx->k3_shared = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "k3_cap0") == 0) {
    if (value < 8 || value > XT_HARD_CAP) {
      set_error(ctx, "xt_set_option: k3_cap0 must be in 8..XT_HARD_CAP");
      return XT_ERR_ARG;
    }
    ctx->k3_cap0 = value;
    return XT_OK;
  }
  if (std::strcmp(name, "k3_pieces") == 0) {
    ctx->k3_pieces = value < 1 ? 1 : (value > 64 ? 64 : value);
    return XT_OK;
  }
  if (std::strcmp(name, "verify_fork_k2") == 0) {
    ctx->verify_fork_k2 = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "k3_hot_smem") == 0) {
    ctx->k3_hot_smem = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "k3_ctas_per_sm") == 0) {
    if (value < 1 || value > 8) {
      set_error(ctx, "xt_set_option: k3_ctas_per_sm must be in 1..8");
      return XT_ERR_ARG;
    }
    ctx->k3_ctas_per_sm = value;
    return XT_OK;
  }
  if (std::strncmp(name, "k2_cost", 7) == 0 && name[7] >= '0' && name[7] <= '3' && name[8] == 0) {
    if (value < 1 || value > 1000) {
      set_error(ctx, "xt_set_option: k2_cost0..3 must be in 1..1000");
      return XT_ERR_ARG;
    }
    ctx->k2_cost[name[7] - '0'] = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_cost_w0") == 0) {
    ctx->k2_cost_w0 = value < 0 ? 0 : value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_lpt") == 0) {
    ctx->k2_lpt = value != 0;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k1_batch") == 0) {
    ctx->k1_batch = value != 0;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k1_smem_scratch") == 0) {
    ctx->k1_smem_scratch = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "pipeline") == 0) {
    ctx->pipeline = value != 0;
    return XT_OK;
  }
  if (std::strcmp(name, "n_groups") == 0) {
    if (value < 1 || value > 64) {
      set_error(ctx, "xt_set_option: n_groups must be in 1..64");
      return XT_ERR_ARG;
    }
    ctx->n_groups = value;
    return XT_OK;
  }
  if (std::strcmp(name, "n_streams") == 0) {
    if (value < 1 || value > xt_ctx::NCS) {
      set_error(ctx, "xt_set_option: n_streams must be in 1..32");
      return XT_ERR_ARG;
    }
    ctx->n_streams = value;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_tpt") == 0) {
    if (value != 1 && value != 2) {
      set_error(ctx, "xt_set_option: k2_tpt must be 1 or 2");
      return XT_ERR_ARG;
    }
    ctx->k2_tpt = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  if (std::strcmp(name, "k2_wpc") == 0) {
    if (value != 2 && value != 4 && value != 8) {
      set_error(ctx, "xt_set_option: k2_wpc must be 2, 4 or 8");
      return XT_ERR_ARG;
    }
    ctx->k2_wpc = value;
    ctx->have_eval = false;
    return XT_OK;
  }
  set_error(ctx, std::string("xt_set_option: unknown option ") + name);
  return XT_ERR_ARG;
}

extern "C" int xt_get_stats(xt_ctx* ctx, xt_stats* out) {
  if (!ctx || !out) return XT_ERR_ARG;
  if (ctx->have_eval) {
    XT_CUDA_OK(cudaSetDevice(ctx->device));
    XT_CUDA_OK(cudaEventSynchronize(ctx->ev[2]));
    cudaEventElapsedTime(&ctx->stats.ms_plan, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->stats.ms_replay, ctx->ev[1], ctx->ev[2]);
  }
  ctx->stats.ms_predict = ctx->ms_predict;
  ctx->stats.k3_launches = ctx->k3_launches;
  ctx->stats.k3_cap = ctx->k3_cap;
  *out = ctx->stats;
  return XT_OK;
}

extern "C" int xt_chunk_logp(xt_ctx* ctx, int32_t chunk, const xt_params* p, double* out) {
  if (!ctx || chunk < 0 || chunk >= (int)ctx->chunks.size()) {
    set_error(ctx, "xt_chunk_logp: bad chunk index");
    return XT_ERR_ARG;
  }
  if (!ctx->have_eval || std::memcmp(&ctx->last_p, p, sizeof(xt_params)) != 0) {
    int rc = evaluate(ctx, p, nullptr, nullptr);
    if (rc) return rc;
  }
  const XtChunk& ck = ctx->chunks[chunk];
  XT_CUDA_OK(cudaMemcpyAsync(out, ctx->d_logp + ck.trk_off, sizeof(double) * ck.nT, cudaMemcpyDeviceToHost,
                             ctx->stream));
  XT_CUDA_OK(cudaStreamSynchronize(ctx->stream));
  return XT_OK;
}

extern "C" int xt_plan_dump(xt_ctx* ctx, int32_t chunk, int32_t step, int32_t* nB_in, int32_t* nG, int32_t* gid,
                            int32_t cap, double* threshold_used) {
  if (!ctx || !ctx->have_eval || chunk < 0 || chunk >= (int)ctx->chunks.size()) {
    set_error(ctx, "xt_plan_dump: no evaluation yet or bad chunk index");
    return XT_ERR_ARG;
  }
  const XtChunk& ck = ctx->chunks[chunk];
  if (step < 2 || step > ck.L - 2) {
    set_error(ctx, "xt_plan_dump: step must satisfy 2 <= step <= L-2");
    return XT_ERR_ARG;
  }
  const int rec = ck.rec0 + (step - 2);
  XtRecHdr h;
  XT_CUDA_OK(cudaMemcpy(&h, ctx->plan.hdr + rec, sizeof(h), cudaMemcpyDeviceToHost));
  *nB_in = h.nC;
  *nG = h.nG;
  if (threshold_used) *threshold_used = h.th;
  if (cap < h.nC) {
    set_error(ctx, "xt_plan_dump: gid buffer too small");
    return XT_ERR_ARG;
  }
  std::vector<uint16_t> tmp(h.nC);
  XT_CUDA_OK(cudaMemcpy(tmp.data(), ctx->plan.gid + (size_t)rec * ctx->plan.cap, sizeof(uint16_t) * h.nC,
                        cudaMemcpyDeviceToHost));
  for (int i = 0; i < h.nC; ++i) gid[i] = tmp[i];
  return XT_OK;
}

extern "C" int xt_fp64_peak_tflops(xt_ctx* ctx, double* out) {
  if (!ctx) return XT_ERR_ARG;
  XT_CUDA_OK(cudaSetDevice(ctx->device));
  const int blocks = ctx->n_sm * 8, threads = 256, iters = 1 << 15;
  double* buf = nullptr;
  XT_CUDA_OK(cudaMalloc(&buf, sizeof(double) * blocks * threads));
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(a, ctx->stream);
    k_fp64_peak<<<blocks, threads, 0, ctx->stream>>>(buf, iters);
    cudaEventRecord(b, ctx->stream);
    cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    if (rep > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(buf);
  XT_CUDA_OK(cudaGetLastError());
  const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
  *out = flops / (best * 1e-3) / 1e12;
  return XT_OK;
}

#include "xt_predict_host.inl"
#include "xt_refine_host.inl"
#include "xt_seglen_host.inl"
#include "xt_multi.inl"
#include "xt_frozen_host.inl"
