// common.cuh — internal definitions shared by the sm_100a kernels of libsfmgpu.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <vector>

#include "../../include/sfmgpu.h"

#define SFM_MAXL 8        // pyramid levels supported by the by-value views
#define SFM_NSM_FALLBACK 148

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

// By-value view of a frame batch handed to kernels: level l of frame f starts at base[l] + f*fstride[l].
struct PyrView {
  const uint8_t* base[SFM_MAXL];
  int w[SFM_MAXL], h[SFM_MAXL], pitch[SFM_MAXL];
  size_t fstride[SFM_MAXL];
  int levels;
};

struct sfmgpu_frames {
  int w = 0, h = 0, n = 0, levels = 0;
  int lw[SFM_MAXL], lh[SFM_MAXL], pitch[SFM_MAXL];
  size_t fstride[SFM_MAXL];
  uint8_t* lvl[SFM_MAXL];
  PyrView view() const {
    PyrView v;
    for (int l = 0; l < SFM_MAXL; l++) {
      v.base[l] = l < levels ? lvl[l] : nullptr;
      v.w[l] = l < levels ? lw[l] : 0;
      v.h[l] = l < levels ? lh[l] : 0;
      v.pitch[l] = l < levels ? pitch[l] : 0;
      v.fstride[l] = l < levels ? fstride[l] : 0;
    }
    v.levels = levels;
    return v;
  }
};

struct sfmgpu_ctx {
  int device = 0;
  int n_sm = SFM_NSM_FALLBACK;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr, back_stream = nullptr;  // H2D / D2H legs of the streaming front end
  cudaStream_t sel_stream = nullptr, klt_stream = nullptr;  // stage streams of the chunk pipeline (frontend.cu)
  int pipe_chunk = 0;                 // resident batches: pairs per chunk of the stage pipeline, 0 = sequential
  std::vector<cudaEvent_t> pipe_evs;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  long long launches = 0;
  // scratch, grown on demand (never shrunk)
  DevBuf flush;
  DevBuf klt_in, klt_p1, klt_pb, klt_nit, klt_keep, klt_defer;
  int klt_mode = 0;  // 0 auto, 1 warp-per-feature, 2 lane-per-feature (tests / profiling)
  int select_mode = 0;  // 0 bucket selection + tie fallback, 1 introsort emulation only, 12..34 bucket selection with that many code bits, 1064..5096 bucket selection with a gather of (mode - 1000) words (tests / profiling)
  DevBuf cs_work;    // corner-score work area for single-frame calls
  DevBuf sel_work;   // corner-select work area
  DevBuf misc;       // small scalars
  DevBuf rs_xi, rs_xj, rs_E, rs_counts, rs_inl, rs_best, rs_idx8;
  DevBuf rs_raw;     // std::mt19937(12345) outputs for single-call sampling (two_view.cu: raw_stream)
  int rs_raw_n = 0;
  DevBuf sv_list;    // screening solver: [0] count, [64...] hypotheses left to the Jacobi emulation (repeated index)
  DevBuf pk_stage[2];  // packed input (codec.cu): staged blob bytes (two: the streaming call uploads one while it decodes the other)
  DevBuf pk_fo, pk_flag;  // packed input: frame offsets of the staged range, "a tile record did not decode" flag
  DevBuf pk_tmp, pk_enc;  // encoder: record sizes / tile tables / frame offsets, and the records of one batch of frames
  int rs_n = 0, rs_H = 0;
  bool rs_screened = false;  // rs_E holds screening hypotheses of the octets in rs_idx8: the winner is re-solved when scored
  int solver_mode = 1;       // device 8-point solver: 1 screening solver for the counts of launches beyond one wave + Jacobi emulation for the winner, 0 Jacobi emulation for every hypothesis, 2 the same by the warp kernel, 3 screening always (2, 3: tests)
  int rs_early = 1;          // batched RANSAC stage: stop scoring a pair once a hypothesis explains all of its points (two_view.cu)
  bool profile = false;
  struct StageEv { int stage; cudaEvent_t a, b; };
  std::vector<StageEv> stage_evs;
  float stage_ms[7] = {0, 0, 0, 0, 0, 0, 0};  // corner score, corner select, KLT, compaction, RANSAC stage, list-call gather, packed decode
  void* pinned = nullptr;  // staging for small D2H results
  size_t pinned_cap = 0;
  // kernels whose >48 KB dynamic shared memory opt-in has been set ON THIS CONTEXT'S DEVICE (the attribute is per device)
  std::vector<bool> smem_cfg;
};

// One id per call site / template instantiation that opts a kernel into large dynamic shared memory.
int sfm_next_cfg_id();
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (context, kernel): `id` comes from a function-local
// `static const int id = sfm_next_cfg_id();`
#define SFM_SMEM_OPTIN(ctx, id, kernel, bytes)                                                                    \
  do {                                                                                                            \
    if ((int)(ctx)->smem_cfg.size() <= (id)) (ctx)->smem_cfg.resize((id) + 1, false);                             \
    if (!(ctx)->smem_cfg[(id)]) {                                                                                 \
      SFM_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)));     \
      (ctx)->smem_cfg[(id)] = true;                                                                               \
    }                                                                                                             \
  } while (0)

// Device-resident results of a batch of frame pairs (frontend.cu) and of their RANSAC stage (two_view.cu).
struct TwoViewState;  // two_view.cu
struct sfmgpu_pairs {
  int max_pairs = 0, cap = 0;
  double2 *xy0 = nullptr, *p1 = nullptr, *pb = nullptr, *li = nullptr, *lj = nullptr;
  int *ncorn = nullptr, *nkept = nullptr, *nit = nullptr;
  uint8_t* keep = nullptr;
  unsigned long long* totals = nullptr;
  DevBuf work[2];  // corner work areas (two, so that the stage pipeline can score one chunk while it selects another)
  DevBuf gather;   // list call: the pyramids of both frames of every pair of a chunk
  DevBuf idx;      // list call: frame_a, frame_b (device copies for the gather)
  int last_npairs = 0;
  TwoViewState* tv = nullptr;  // allocated by the first sfmgpu_pairs_ransac call
  int* ids = nullptr;          // segment call: track ids [max_pairs][cap] (allocated by its first use)
  bool ids_valid = false;      // the last batch came from the segment call (other batches carry no ids)
  sfmgpu_multitracker* seg = nullptr;  // segment call: the lock-step tracker it drives (kept for the next call)
};
// The stage works on result sets of `cap` rows: the pairs of a batch, or the sequences of the lock-step tracker.
void sfm_two_view_free(sfmgpu_ctx* ctx, TwoViewState** tv);
bool sfm_two_view_enabled(const TwoViewState* tv);
int sfm_two_view_configure(sfmgpu_ctx* ctx, TwoViewState** tv, int max_sets, int cap, const double* K, const sfmgpu_ransac_cfg* rc,
                           const char* who);
// Same with one camera per set: K [max_sets][9], set s normalised with the inverse of K + 9 s.
int sfm_two_view_configure_sets(sfmgpu_ctx* ctx, TwoViewState** tv, int max_sets, int cap, const double* K, const sfmgpu_ransac_cfg* rc,
                                const char* who);
int sfm_two_view_stage(sfmgpu_ctx* ctx, TwoViewState* tv, const double2* li, const double2* lj, const int* nkept, int cap, int set_off,
                       int nsets, const double* E_host);
int sfm_two_view_skip(sfmgpu_ctx* ctx, TwoViewState* tv, const int* n_in, int nsets);
int sfm_two_view_download(sfmgpu_ctx* ctx, TwoViewState* tv, int cap, int set_off, int nsets, cudaStream_t s);
int sfm_two_view_download_all(sfmgpu_ctx* ctx, TwoViewState* tv, int cap, int nsets, int32_t* status, int32_t* best_n, int32_t* inliers,
                              double* R, double* t, const char* who);
int sfm_two_view_early(sfmgpu_ctx* ctx, TwoViewState* tv, long long* stopped);

// codec.cu: packed frame input
int sfm_pk_check(sfmgpu_ctx* ctx, const sfmgpu_frames* f, const uint8_t* blob, size_t blob_bytes, int blob_first, int count,
                 std::vector<uint64_t>& fo, const char* who);
int sfm_pk_decode(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* stage, const unsigned long long* d_fo,
                  unsigned long long base, int* d_bad);
int sfm_pk_prepare(sfmgpu_ctx* ctx, const uint8_t* blob, int blob_first, const std::vector<uint64_t>& fo, size_t stage_bytes, int nstage);
// Level-0 destination of one frame of a decode over frames of different sizes (sfm_pk_decode_table).
struct PkDst {
  uint8_t* lvl0;  // the frame's level-0 base
  int pitch, w, h, tiles_x, ntiles;
};
PkDst sfm_pk_dst(const sfmgpu_frames* f, int frame);
int sfm_pk_decode_table(sfmgpu_ctx* ctx, const PkDst* d_dst, int count, int max_tiles, const uint8_t* stage,
                        const unsigned long long* d_fo, int* d_bad);
size_t sfm_pk_frame_bound(int w, int h);
size_t sfm_pk_max_chunk_bytes(const std::vector<uint64_t>& fo, int chunk);
int sfm_pk_read_flag(sfmgpu_ctx* ctx, const char* who);

int sfm_fail(sfmgpu_ctx* ctx, int code, const char* fmt, ...);
int sfm_reserve(sfmgpu_ctx* ctx, DevBuf& b, size_t bytes);
int sfm_pinned(sfmgpu_ctx* ctx, size_t bytes);

#define SFM_CUDA(ctx, expr)                                                                          \
  do {                                                                                               \
    cudaError_t e__ = (expr);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      return sfm_fail(ctx, SFMGPU_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),   \
                      __FILE__, __LINE__);                                                           \
  } while (0)

// Every extern "C" entry point that takes a context makes the context's device current first (one context = one device;
// the caller's thread may have another device selected).
#define SFM_ENTER(ctx)                                                                                \
  do {                                                                                                \
    if (ctx) {                                                                                        \
      cudaError_t e__ = cudaSetDevice((ctx)->device);                                                 \
      if (e__ != cudaSuccess)                                                                         \
        return sfm_fail(ctx, SFMGPU_E_CUDA, "cudaSetDevice(%d) failed: %s", (ctx)->device, cudaGetErrorString(e__)); \
    }                                                                                                 \
  } while (0)
#define SFM_ENTER_VOID(ctx)                  \
  do {                                       \
    if (ctx) cudaSetDevice((ctx)->device);   \
  } while (0)

#define SFM_TRY(expr)        \
  do {                       \
    int r__ = (expr);        \
    if (r__ != 0) return r__; \
  } while (0)

// Launch a kernel on the context stream, count it, and surface launch errors.
#define SFM_LAUNCH(ctx, kernel, grid, block, smem, ...)                                  \
  do {                                                                                   \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                     \
    (ctx)->launches++;                                                                   \
    SFM_CUDA(ctx, cudaGetLastError());                                                   \
  } while (0)

// Stage timing (only when ctx->profile): records a CUDA event pair around a stage on the context stream.
struct StageTimer {
  sfmgpu_ctx* ctx;
  int idx = -1;
  StageTimer(sfmgpu_ctx* c, int stage) : ctx(c) {
    if (!c->profile) return;
    sfmgpu_ctx::StageEv e;
    e.stage = stage;
    if (cudaEventCreate(&e.a) != cudaSuccess || cudaEventCreate(&e.b) != cudaSuccess) return;
    cudaEventRecord(e.a, c->stream);
    c->stage_evs.push_back(e);
    idx = (int)c->stage_evs.size() - 1;
  }
  ~StageTimer() {
    if (idx >= 0) cudaEventRecord(ctx->stage_evs[idx].b, ctx->stream);
  }
};

// The LK early exit `std::hypot(step) < 1e-3` (:413-416).  The squared norm decides everything outside a 1 % band around
// the threshold (its rounding error is ~1e-16 relative); inside the band the reference's own form is evaluated, so the
// discontinuity sits where the reference has it (up to hypot's last-ulp differences between libm implementations).
#ifdef __CUDACC__
__device__ __forceinline__ bool sfm_lk_step_small(double sx, double sy) {
  const double q = sx * sx + sy * sy;
  if (q < 0.98e-6) return true;
  if (q > 1.02e-6) return false;
  return hypot(sx, sy) < 1e-3;  // also reached by NaN steps: false, as in the reference
}
#endif

static inline int sfm_align16(int v) { return v <= 0 ? 16 : ((v + 15) / 16) * 16; }
static inline unsigned sfm_cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

// ---- internal cross-file entry points (device-pointer level) --------------------------------------------
// klt.cu
// Geometry of one list (pair) of a KLT launch whose lists have their own image sizes (the lock-step tracker over sequences of
// different sizes): level l of image A starts at lv[l].a, of image B at lv[l].b; both are w x h with row pitch `pitch`.
struct KltGeoLevel {
  const uint8_t* a;
  const uint8_t* b;
  int w, h, pitch, pad;
};
struct KltGeo {
  KltGeoLevel lv[SFM_MAXL];
};
struct KltLaunch {
  PyrView pv;            // image A: frame fa0 + k*fa_step of this batch
  const double2* p0;     // [npairs*cap] (or [n] when npairs == 1)
  const int* counts;     // per-pair valid count, or nullptr (all cap valid)
  int npairs, cap;
  int fa0, fa_step, fb0, fb_step;  // frame indices of image A / B for pair k: fa0 + k*fa_step ...
  int radius, iters;
  double fb_thresh;
  double2* p1;           // forward result
  double2* pb;           // backward result
  int* nit;              // optional
  uint8_t* keep;         // optional: !(fb >= fb_thresh)
  // Image B: frame fb0 + k*fb_step of this batch.  Callers that track within one batch set it equal to pv.  A launch whose
  // two views differ (two batches, of any sizes, with equal level counts) always runs the two-geometry warp-per-feature
  // kernel; the lane kernels and the context's KLT mode only apply to one-batch launches.
  PyrView pvb;
  // Optional device table [npairs]: list k reads its images from geo[k] instead of pv / pvb and the frame indices (pv gives
  // the level count; pvb must equal pv).  Such launches take the same kernel family as one-batch launches, through
  // instantiations of their own.
  const KltGeo* geo = nullptr;
};
int sfm_klt_launch(sfmgpu_ctx* ctx, const KltLaunch& k);

// corner_score.cu / corner_select.cu
struct CornerWork;  // opaque per-batch work area
size_t sfm_corner_work_bytes_md(int w, int h, int nframes, int cand_cap, int min_dist);
// Detect corners for frames [first, first+count): out_xy [count][max_corners] (double2, integer valued),
// out_n[count].  cand_cap = per-frame candidate capacity (overflow -> E_CAPACITY, reported via status word).
int sfm_corners_batch(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, int max_corners, double quality,
                      int min_dist, int cand_cap, void* work, size_t work_bytes, double2* out_xy, int* out_n);
int sfm_corners_score_stage(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, double quality, int min_dist, int cand_cap,
                            void* work, size_t work_bytes);
int sfm_corners_select_stage(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, int max_corners, double quality, int min_dist,
                             int cand_cap, void* work, size_t work_bytes, double2* out_xy, int* out_n);
int sfm_candidates_single(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int frame, double quality, int32_t* xy,
                          double* score, int cap, int* n_out, double* max_score);
int sfm_sort_perm(sfmgpu_ctx* ctx, const double* keys, int n, int32_t* perm);
// solver.cu / ransac.cu: batched over correspondence sets
int sfm_eight_point_batched(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_single,
                            int npairs, const int* idx8, int H, double* Eout, int screen);
int sfm_eight_point_range(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_single,
                          int npairs, const int* idx8, int H, int h0, int h1, double* Eout, int screen);
bool sfm_solver_screens(const sfmgpu_ctx* ctx, int npairs, int H);
int sfm_sample_octets(sfmgpu_ctx* ctx, int n, int H, int* d_idx8, int* d_flag);
int sfm_eight_point_winners(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_single,
                            int npairs, const int* idx8, int H, const int* best, double* E);
int sfm_pose_batched(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, int npairs, const int* status,
                     const int* best, const int* inl, const double* bestE, double* R, double* t);
int sfm_ransac_score_batched(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_max,
                             int npairs, double* E, int H, double thr, int* counts, int* best, int* inl, const int* refine_idx8);
int sfm_ransac_count_range(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_max,
                           int npairs, const double* E, int H, int h0, int h1, double thr, int* counts);
int sfm_ransac_finish(sfmgpu_ctx* ctx, const double2* xi, const double2* xj, size_t pt_stride, const int* npts, int n_max, int npairs,
                      double* E, int H, double thr, const int* counts, int* best, int* inl, const int* refine_idx8);
