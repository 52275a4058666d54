/* sfmgpu.h — C ABI of libsfmgpu.so: the B200 (sm_100a) front end of the SfM pipeline.
 *
 * Drop-in boundary for the data-parallel front end of RoozbehSanaei/Structure-from-Motion-3D-Reconstruction
 * (reference citations are relative to cpp/src/templering_sfm.cpp unless a header is named):
 *   build_pyr :224-232, shi_tomasi :237-302, KLTTracker :323-466, sampson_err/find_E_ransac scoring loop
 *   :629-638 / :664-677, two-view front end :1836-1857.
 * The reference has no FFI: its hot functions are file-static.  These entry points are what a binding
 * for that path would call; the C++ source-compatible shim that re-creates the reference's own names on
 * top of them is host/sfmgpu_shim.hpp (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns 0 on success or a negative sfmgpu_status;
 *     sfmgpu_last_error(ctx) gives the message.  No exceptions cross the boundary.
 *   - the caller owns host buffers; the library owns device memory and pinned staging.
 *   - one context = one CUDA device + one stream; calls on a context are stream-ordered; functions that
 *     take host output pointers return after the results are in those buffers.
 *   - there is no CPU fallback anywhere: without a usable B200 every call fails with SFMGPU_E_CUDA.
 *   - images are 8-bit, row-major, stride = w on the host side (GrayImage, cpp/include/pgm_io.hpp:10-15);
 *     points are (x, y) double pairs (Vec2, cpp/include/linalg.hpp:15-17); 3x3 matrices are 9 doubles
 *     row-major (Mat33, linalg.hpp:25-35).
 */
#ifndef SFMGPU_H_
#define SFMGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFMGPU_VERSION 100

typedef enum sfmgpu_status {
  SFMGPU_OK = 0,
  SFMGPU_E_ARG = -1,      /* invalid argument */
  SFMGPU_E_CUDA = -2,     /* CUDA runtime / driver failure (including "no device") */
  SFMGPU_E_CAPACITY = -3, /* a caller- or batch-sized buffer was too small; nothing was truncated silently */
  SFMGPU_E_STATE = -4     /* call sequence error (e.g. pyramid not built) */
} sfmgpu_status;

typedef struct sfmgpu_ctx sfmgpu_ctx;
typedef struct sfmgpu_frames sfmgpu_frames;   /* F frames of one size + their pyramids, resident in HBM */
typedef struct sfmgpu_pairs sfmgpu_pairs;     /* device-resident results of a batch of frame pairs */
typedef struct sfmgpu_tracker sfmgpu_tracker; /* stateful KLTTracker twin */
typedef struct sfmgpu_multitracker sfmgpu_multitracker; /* S KLTTracker twins advanced in lock step */

/* LKConfig, :307-316 (same field meaning and defaults). */
typedef struct sfmgpu_lkcfg {
  int max_tracks;    /* 2200 */
  int min_tracks;    /* 900  */
  double quality;    /* 0.01 */
  int min_distance;  /* 8    */
  int pyr_levels;    /* 3    */
  int win_radius;    /* 5    */
  int iters;         /* 10   */
  double fb_thresh;  /* 1.0  */
} sfmgpu_lkcfg;

void sfmgpu_lkcfg_default(sfmgpu_lkcfg* cfg);

/* ---- context ------------------------------------------------------------------------------------ */
int sfmgpu_version(void);
int sfmgpu_create(int device, sfmgpu_ctx** out);
void sfmgpu_destroy(sfmgpu_ctx* ctx);
const char* sfmgpu_last_error(sfmgpu_ctx* ctx);
int sfmgpu_sync(sfmgpu_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
long long sfmgpu_launch_count(sfmgpu_ctx* ctx);
/* CUDA-event timer on the context's stream: start, ..., stop -> elapsed milliseconds. */
int sfmgpu_timer_start(sfmgpu_ctx* ctx);
int sfmgpu_timer_stop(sfmgpu_ctx* ctx, float* ms);
/* Write `bytes` of device memory (L2 flush between timed iterations). */
int sfmgpu_flush_l2(sfmgpu_ctx* ctx, size_t bytes);
/* Per-stage device times of pair_frontend calls: enable, run, then read the accumulated milliseconds
 * ms[0] corner score (max, candidates, scan, order), ms[1] corner select (sort + NMS), ms[2] KLT, ms[3] compaction.
 * Reading synchronises the stream and resets the accumulators. */
int sfmgpu_profile(sfmgpu_ctx* ctx, int enable);
int sfmgpu_stage_times(sfmgpu_ctx* ctx, float* ms4);
/* Same with n values: ms[4] = the RANSAC stage of the two-view unit (sfmgpu_pairs_set_ransac, sfmgpu_multitracker_set_ransac),
 * ms[5] = the frame gather of sfmgpu_pair_frontend_list. */
int sfmgpu_stage_times_n(sfmgpu_ctx* ctx, float* ms, int n);
/* Measured non-tensor FP64 throughput of this GPU (DFMA micro-benchmark, ~10 ms): the KLT / RANSAC roofline. */
int sfmgpu_fp64_peak(sfmgpu_ctx* ctx, double* tflops);
/* Pinned host memory for callers that want asynchronous uploads. */
int sfmgpu_host_alloc(sfmgpu_ctx* ctx, size_t bytes, void** out);
int sfmgpu_host_free(sfmgpu_ctx* ctx, void* p);

/* ---- frames + pyramid: GrayImage / Pyramid / build_pyr / downsample2 (:200-232) ------------------ */
/* Storage for `nframes` images of w x h with `levels` pyramid levels (level 0 = the image itself). */
int sfmgpu_frames_create(sfmgpu_ctx* ctx, int w, int h, int nframes, int levels, sfmgpu_frames** out);
void sfmgpu_frames_destroy(sfmgpu_ctx* ctx, sfmgpu_frames* f);
/* Host -> level 0 of frames [first, first+count); host_pix = count images, each w*h bytes, stride w.  Here and in the
 * tracker / multitracker / streaming entry points an image pointer may also be DEVICE memory of the context's GPU
 * (unified addressing: the copy is then device to device). */
int sfmgpu_frames_upload(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* host_pix);
/* Same from device memory (row pitch in bytes). */
int sfmgpu_frames_upload_device(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* dev_pix,
                                size_t pitch);
/* Integer synthetic generator (sfmgpu/synth.py twin): frame first+k gets time index t0+k of sequence seed. */
int sfmgpu_frames_synth(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, uint32_t seed, int t0);
/* build_pyr for frames [first, first+count): fills levels 1..levels-1 (one fused launch per 2 levels). */
int sfmgpu_pyramid_build(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count);
/* Level geometry and download (parity checks): out = w_l*h_l bytes, stride w_l. */
int sfmgpu_frames_level_size(const sfmgpu_frames* f, int level, int* w, int* h);
int sfmgpu_frames_download(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, int level, uint8_t* host_out);
/* Device address of a level (frame k starts at ptr + k * frame_stride, rows are pitch bytes apart): interop with the
 * caller's own kernels, NCCL, or as an image source for the entry points that accept device pointers. */
int sfmgpu_frames_device_ptr(const sfmgpu_frames* f, int level, void** ptr, size_t* pitch, size_t* frame_stride);

/* ---- corners: shi_tomasi (:237-302) ---------------------------------------------------------------- */
/* Raster-ordered candidate list {s >= max*quality} of one frame (:274-285): pixel (x,y) and exact score.
 * Returns SFMGPU_E_CAPACITY (with *n_out = required size) when cap is too small. */
int sfmgpu_corner_candidates(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, double quality, int32_t* xy,
                             double* score, int cap, int* n_out, double* max_score);
/* Full shi_tomasi: corners in acceptance order, integer-valued doubles; xy_out holds max_corners pairs. */
int sfmgpu_corners(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, int max_corners, double quality, int min_dist,
                   double* xy_out, int* n_out);
/* The libstdc++ std::sort permutation (:286) of n keys sorted descending, computed on the device:
 * perm[i] = original index of the element that std::sort leaves at position i. */
int sfmgpu_sort_perm_desc(sfmgpu_ctx* ctx, const double* keys, int n, int32_t* perm);
/* How every later corner selection of this context orders its candidates (results are bit-identical either way):
 * 0 = bucket selection (candidates grouped by score bucket, blocked ones dropped unsorted, the survivors sorted and
 * selected bucket group by bucket group), and the exact introsort emulation only for frames where two candidates with
 * identical scores are both still selectable (default); 1 = introsort emulation for every frame; 2 = full radix sort by
 * score + selection over the sorted list; 12..34 = bucket selection with that many order-code bits (tests: short codes
 * exercise the equal-code path); 1064..5096 = bucket selection with gathers of (mode - 1000) words (tests: small gathers
 * exercise the walk of an oversized bucket by sub-buckets). */
int sfmgpu_select_set_mode(sfmgpu_ctx* ctx, int mode);

/* ---- KLT: track_one / lk_step / sample_bilinear (:183-198, :396-460) ------------------------------- */
/* Forward track frame a -> b and backward b -> a for n points (what :356-361 and :1846-1848 do per
 * track).  p1 = forward result, p0_back = backward result (NULL: forward only, i.e. one track_one_public call
 * per point); n_iters (optional) = LK iterations executed. */
int sfmgpu_klt_track(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame_a, int frame_b, const double* p0_xy, int n,
                     int win_radius, int iters, double* p1_xy, double* p0_back_xy, int32_t* n_iters);
/* Kernel selection for every KLT launch of this context (tests and profiling; results agree within the parity
 * budget either way): 0 = automatic (lane-per-feature kernel for batches of >= 6000 features with win_radius 5,
 * warp-per-feature otherwise), 1 = warp-per-feature only, 2 = lane-per-feature whenever win_radius is 5. */
int sfmgpu_klt_set_mode(sfmgpu_ctx* ctx, int mode);

/* ---- stateless two-view front end over a batch of pairs (:1836-1857) -------------------------------- */
/* For every pair (first_frame+k, first_frame+k+1), k < npairs: pyramids must be built; detect up to
 * cfg->max_tracks corners on the first frame, track fwd/bwd, keep iff !(fb >= fb_thresh).
 * Results stay on the device in `out` (create once, reuse).  The call returns when the batch has finished: candidate
 * lists are sized for w*h/6 entries per frame, and frames that need more (flat / weak-texture images, where up to every
 * pixel is a candidate, :274-285) are redone with the full capacity before the call returns, so every frame carries the
 * reference's result; an error (SFMGPU_E_CAPACITY included) is reported by this call, not by a later download. */
int sfmgpu_pairs_create(sfmgpu_ctx* ctx, int max_pairs, int max_corners, sfmgpu_pairs** out);
void sfmgpu_pairs_destroy(sfmgpu_ctx* ctx, sfmgpu_pairs* p);
int sfmgpu_pair_frontend(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first_frame, int npairs, const sfmgpu_lkcfg* cfg,
                         sfmgpu_pairs* out);
/* The same unit over an explicit list of frame pairs (loop-closure verification: old keyframe, current frame).  Pair k =
 * (frame_a[k], frame_b[k]) of f, k < npairs: any indices, repeats, a == b and a > b allowed; pyramids built.  Detect on
 * frame_a[k], track a -> b and back, fb filter, compaction - and the RANSAC stage when sfmgpu_pairs_set_ransac is on - into
 * slot k of `out`: per pair the results sfmgpu_pair_frontend gives for (a, b) when they are adjacent, bit for bit, including
 * the redo of frames that overflow the candidate lists.  Every reader of a pairs object (download(_all), totals,
 * ransac_download(_all), ransac_early, device_ptrs, sfmgpu_sched_gather_pairs) works on the result unchanged.
 * The pyramids of both frames of every pair of a chunk are copied into a scratch batch (about 2.7*W*H bytes per pair with 3
 * levels; chunks follow sfmgpu_pair_frontend's rule, <= 1024 pairs); chunks run back to back on the context stream
 * (sfmgpu_pipeline_set does not apply).  An index outside [0, f->n), npairs > max_pairs,
 * NULL arrays with npairs > 0, or a cfg that does not match `out` / `f` is SFMGPU_E_ARG, reported before any work is queued.
 * Returns when the batch has finished. */
int sfmgpu_pair_frontend_list(sfmgpu_ctx* ctx, sfmgpu_frames* f, const int32_t* frame_a, const int32_t* frame_b, int npairs,
                              const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out);
/* Stage pipeline: with pairs_per_chunk > 0, a resident batch of at least 2*pairs_per_chunk pairs is cut into chunks
 * that flow through three streams (score -> select on a high-priority stream -> KLT), so the latency-bound corner
 * selection of one chunk shares the SMs with the score / KLT kernels of its neighbours (results are identical).
 * 0 (default) = one stream, stages back to back.  The host-streaming call below always pipelines per upload chunk. */
int sfmgpu_pipeline_set(sfmgpu_ctx* ctx, int pairs_per_chunk);
/* Streaming variant for frames that live in HOST memory (pinned for full speed; nframes images of w*h bytes, stride
 * w).  Frames [0, nframes) of `f` are overwritten; pairs (k, k+1), k < nframes-1.  The upload of chunk c+1 overlaps
 * pyramid + corners + KLT of chunk c and the download of chunk c-1 (separate streams); chunk_frames <= 0 picks
 * about 100 frames (at least 8, at most 20 chunks).  li/lj are [nframes-1][max_corners] (x,y) pairs, n_kept/n_corners [nframes-1]; any of the
 * four may be NULL.  Returns after everything has landed in host memory. */
int sfmgpu_pair_frontend_host(sfmgpu_ctx* ctx, sfmgpu_frames* f, const uint8_t* host_pix, int nframes,
                              const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out, int chunk_frames, double* li_xy, double* lj_xy,
                              int32_t* n_kept, int32_t* n_corners);
/* Totals over the last batch: corners detected (= tracks attempted), survivors, LK iterations. */
int sfmgpu_pairs_totals(sfmgpu_ctx* ctx, sfmgpu_pairs* p, long long* n_corners, long long* n_kept,
                        long long* n_lk_iters);
/* One pair's results: survivors in corner order.  li/lj = (x,y) in first/second frame, cap pairs each. */
int sfmgpu_pairs_download(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int pair, double* li_xy, double* lj_xy, int cap,
                          int* n_kept, int* n_corners);

/* All pairs of the last batch at once: li/lj are [npairs][max_corners] (x,y) pairs, n_kept/n_corners [npairs].
 * Any pointer may be NULL.  Use pinned buffers (sfmgpu_host_alloc) for full-speed copies. */
int sfmgpu_pairs_download_all(sfmgpu_ctx* ctx, sfmgpu_pairs* p, double* li_xy, double* lj_xy, int32_t* n_kept,
                              int32_t* n_corners);
/* Correspondences that do not come from the tracker (e.g. the keyframe observations of :1784-1793): li/lj are
 * [npairs][max_corners] (x,y) pairs, the first n_kept[k] of pair k valid.  They become "the last batch", ready for
 * sfmgpu_pairs_ransac. */
int sfmgpu_pairs_set_matches(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int npairs, const double* li_xy, const double* lj_xy,
                             const int32_t* n_kept);
/* Device addresses of the same arrays (for NCCL gathers by the scheduler); valid until pairs_destroy. */
int sfmgpu_pairs_device_ptrs(sfmgpu_pairs* p, void** li_xy, void** lj_xy, void** n_kept, void** n_corners);

/* ---- RANSAC stage of the two-view unit, batched over the pairs of a batch (:1855-1857; find_E_ransac :640-761) -----------
 * What the loop-closure block does with the survivors of a pair:
 *     if (li.size() >= 120) { auto lopt = find_E_ransac(K, li, lj, 4000, 2e-3, 80); ... }
 * for every pair of a batch in one launch set per stage: K^-1 normalisation (:649-655), the seeded sampling (:657-665:
 * std::mt19937(12345) + uniform_int_distribution, bit-exact index octets incl. the distribution's rejection loop),
 * eight_point_E per octet (device solver: hypotheses equal to the reference's to ~1e-9, see sfmgpu_ransac_hypotheses),
 * the scoring loop (:667-676: counts, winner, ascending inlier list - bit-exact for the hypotheses scored), the
 * min_inliers test (:678) and the pose tail (:680-760; device arithmetic, R and t agree to ~1e-10).
 * Passing the caller's own hypotheses (E_host, e.g. from the reference's solver) makes counts, winner and inlier lists
 * bit-identical to find_E_ransac's. */
typedef struct sfmgpu_ransac_cfg {
  int iters;        /* hypotheses per pair: 4000 at :1856, 2500 at :1739 */
  double thr;       /* Sampson threshold: 2e-3 / 1e-3 */
  int min_inliers;  /* fewer inliers: no pose, std::nullopt (:678): 80 / 60 */
  int min_points;   /* the caller's guard li.size() >= 120 (:1855); pairs below it are skipped; 0: none */
} sfmgpu_ransac_cfg;
/* Per-pair status after the stage. */
#define SFMGPU_TV_SKIPPED 0 /* fewer than min_points survivors: find_E_ransac was not called */
#define SFMGPU_TV_NONE 1    /* std::nullopt: fewer than 8 points, or the winner has fewer than min_inliers inliers */
#define SFMGPU_TV_OK 2      /* R, t and the inlier list are valid */
/* Make the stage part of sfmgpu_pair_frontend / sfmgpu_pair_frontend_host for this pairs object (rc == NULL: off again).
 * K: 9 doubles row-major; a singular K is SFMGPU_E_ARG ("Singular K", :474). */
int sfmgpu_pairs_set_ransac(sfmgpu_ctx* ctx, sfmgpu_pairs* p, const double* K, const sfmgpu_ransac_cfg* rc);
/* Host arrays the streaming front end fills chunk by chunk when the stage is on: status / best_n [npairs], inliers
 * [npairs][max_corners] (first best_n valid), R [npairs][9], t [npairs][3]; any may be NULL; pinned memory for overlap. */
int sfmgpu_pairs_ransac_host_outputs(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int32_t* status, int32_t* best_n, int32_t* inliers,
                                     double* R, double* t);
/* Early stop of the stage (default on; exact).  The scoring loop keeps the FIRST hypothesis with the largest count (:673,
 * strict >) and a count cannot exceed the number of correspondences, so once a hypothesis explains ALL points of a pair
 * nothing after it can win: the stage scores the first 128 hypotheses of every pair and takes the pairs that already hold
 * a full count out of the remaining launches - same winner, inlier list, count and pose.  With the reference's thresholds
 * (1e-3 / 2e-3 on the Sampson error in normalised coordinates) that is the common case.  Applies to the device solver's
 * own hypotheses (not E_host) and iters > 256.  on = 0: every hypothesis of every pair is solved and scored.
 * sfmgpu_pairs_ransac_early: pairs stopped early since the last call of it (reads and resets; synchronises). */
int sfmgpu_ransac_set_early_stop(sfmgpu_ctx* ctx, int on);
int sfmgpu_pairs_ransac_early(sfmgpu_ctx* ctx, sfmgpu_pairs* p, long long* pairs_stopped);
/* Run the stage now on the pairs of the last batch.  E_host: NULL (device solver) or [npairs][iters][9] hypotheses. */
int sfmgpu_pairs_ransac(sfmgpu_ctx* ctx, sfmgpu_pairs* p, const double* K, const sfmgpu_ransac_cfg* rc, const double* E_host);
/* One pair: status, winner (-1: none), its count, inlier indices ascending (into the pair's survivor list; cap entries of
 * room), the winning hypothesis, R_ji, t_ji.  Any output may be NULL. */
int sfmgpu_pairs_ransac_download(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int pair, int* status, int* best_h, int* best_n,
                                 int32_t* inliers, int cap, double* E9, double* R9, double* t3);
/* All pairs of the last batch (layout as in sfmgpu_pairs_ransac_host_outputs). */
int sfmgpu_pairs_ransac_download_all(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int32_t* status, int32_t* best_n, int32_t* inliers,
                                     double* R, double* t);
/* Device addresses for NCCL gathers: status int32 [npairs], best int32 [npairs][2] = (winner, count), inliers int32
 * [npairs][max_corners], R double [npairs][9], t double [npairs][3]. */
int sfmgpu_pairs_ransac_device_ptrs(sfmgpu_pairs* p, void** status, void** best, void** inliers, void** R, void** t);
/* `count` draws of std::uniform_int_distribution<int>(0, n-1) on std::mt19937(12345), produced by the device sampler. */
int sfmgpu_ransac_sample(sfmgpu_ctx* ctx, int n, int count, int32_t* out);

/* ---- multi-GPU frame-pair scheduler (SURVEY.md §8e): one rank (process or thread) per GPU ---------------------------------
 * The two-view unit (:1836-1857) is stateless per frame pair: ONE sequence shards by contiguous blocks of pairs plus one
 * halo frame per rank (whole sequences shard the same way), with no data-path collective; the only communication is the
 * gather of the per-pair results to one rank, ncclSend / ncclRecv grouped into one launch.  NCCL is bound at run time
 * (dlopen of libnccl.so.2, or SFMGPU_NCCL_LIB): a single-GPU user never needs it. */
typedef struct sfmgpu_sched sfmgpu_sched;
#define SFMGPU_SCHED_ID_BYTES 128 /* sizeof(ncclUniqueId) */
/* Contiguous block [begin, end) of n_items for `rank` of `world` (sizes differ by at most one, lower ranks get the extra). */
int sfmgpu_sched_shard(int n_items, int world, int rank, int* begin, int* end);
/* Rank 0 creates the id (ncclGetUniqueId) and hands it to the other ranks out of band (file, MPI, socket ...). */
int sfmgpu_sched_unique_id(void* id128);
/* One scheduler per rank, on the context's device.  Either id128 (SFMGPU_SCHED_ID_BYTES from sfmgpu_sched_unique_id:
 * the communicator is created here, collectively) or nccl_comm (the caller's ncclComm_t, adopted, not destroyed);
 * world == 1 needs neither. */
int sfmgpu_sched_create(sfmgpu_ctx* ctx, int world, int rank, const void* id128, void* nccl_comm, sfmgpu_sched** out);
void sfmgpu_sched_destroy(sfmgpu_ctx* ctx, sfmgpu_sched* s);
/* Pair-mode shard of a sequence of n_frames for this rank: pairs [pair_begin, pair_end) and the frames
 * [frame_begin, frame_end) it must hold (frame_end = pair_end + 1: one halo frame). */
int sfmgpu_sched_pair_shard(const sfmgpu_sched* s, int n_frames, int* pair_begin, int* pair_end, int* frame_begin,
                            int* frame_end);
/* Collective: every rank passes its pairs object, whose last batch is its block of the n_pairs_total pairs (in order).
 * On `root` the host arrays receive the whole sequence: li / lj [n_pairs_total][max_corners][2], n_kept / n_corners
 * [n_pairs_total]; with_ransac != 0 adds status / best_n [n_pairs_total], inliers [n_pairs_total][max_corners],
 * R [n_pairs_total][9], t [n_pairs_total][3] (sfmgpu_pairs_ransac*).  Host pointers are ignored on other ranks and may
 * be NULL on the root.  Returns after the data has landed. */
int sfmgpu_sched_gather_pairs(sfmgpu_ctx* ctx, sfmgpu_sched* s, sfmgpu_pairs* p, int n_pairs_total, int root, int with_ransac,
                              double* li_xy, double* lj_xy, int32_t* n_kept, int32_t* n_corners, int32_t* status,
                              int32_t* best_n, int32_t* inliers, double* R, double* t);

/* ---- stateful tracker: KLTTracker (:323-391) ----------------------------------------------------------
 * A track list never holds more than ROWS = max(max_tracks, min_tracks, 1) + 1 entries; `cap` arguments of that size
 * always suffice. */
int sfmgpu_tracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, sfmgpu_tracker** out);
void sfmgpu_tracker_destroy(sfmgpu_ctx* ctx, sfmgpu_tracker* t);
/* reset(gray) :327-332 */
int sfmgpu_tracker_reset(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h);
/* step(gray) :340-391.  Survivors (prev, cur, id) in track order; *n_out = 0 on the first frame. */
int sfmgpu_tracker_step(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h,
                        double* prev_xy, double* cur_xy, int32_t* ids, int cap, int* n_out);
/* Same with the frame already resident (frame index into `f`, pyramid built): no H2D in the step. */
int sfmgpu_tracker_step_frames(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame, double* prev_xy,
                               double* cur_xy, int32_t* ids, int cap, int* n_out);
/* tracks() :393 */
int sfmgpu_tracker_tracks(sfmgpu_ctx* ctx, sfmgpu_tracker* t, double* xy, int32_t* ids, int cap, int* n_out);
/* Sum of track-list sizes entering step() so far, and LK iterations executed. */
int sfmgpu_tracker_totals(sfmgpu_ctx* ctx, sfmgpu_tracker* t, long long* n_track_steps, long long* n_lk_iters);

/* ---- S independent KLTTrackers advanced in lock step (several sequences per GPU) ------------------------ */
/* Per sequence exactly KLTTracker::step (:340-391); one batched launch per stage for all sequences.  All images are
 * w x h.  The first step resets every sequence (n_out = 0 everywhere). */
int sfmgpu_multitracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, int n_sequences, int w, int h, sfmgpu_multitracker** out);
void sfmgpu_multitracker_destroy(sfmgpu_ctx* ctx, sfmgpu_multitracker* t);
/* host_pix: [n_sequences][h][w], the next frame of every sequence.  With ROWS = max(max_tracks, min_tracks, 1) + 1 (the
 * longest a track list can get: replenish appends before it tests the cap, :386-387): prev_xy / cur_xy are
 * [n_sequences][ROWS][2], ids [n_sequences][ROWS], n_out [n_sequences] survivors per sequence (any output may be NULL). */
int sfmgpu_multitracker_step(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix, double* prev_xy, double* cur_xy,
                             int32_t* ids, int32_t* n_out);
/* Pipelined form: next_host_pix (may be NULL) = the frames of the FOLLOWING step; they are uploaded and their pyramids built
 * on a second stream while this step computes, and the next call passes host_pix = NULL to consume them.  Page-locked
 * host memory (sfmgpu_host_alloc) is needed for the overlap.  sfmgpu_multitracker_prefetch primes the pipeline before
 * the first step.  Results are identical to the plain step. */
int sfmgpu_multitracker_prefetch(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix);
int sfmgpu_multitracker_step_pipelined(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix, const uint8_t* next_host_pix,
                                       double* prev_xy, double* cur_xy, int32_t* ids, int32_t* n_out);
/* Back to the state after create (the next step resets every sequence, ids restart at 0). */
int sfmgpu_multitracker_reset(sfmgpu_ctx* ctx, sfmgpu_multitracker* t);
int sfmgpu_multitracker_tracks(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int sequence, double* xy, int32_t* ids, int cap, int* n_out);
int sfmgpu_multitracker_totals(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* n_track_steps, long long* n_lk_iters);
/* find_E_ransac(K, prev_pts, cur_pts, iters, thr, min_inliers) (:1739) on every sequence's survivors, inside every later
 * step; rc == NULL: off.  rc->min_points = 1 is the reference's `prev_pts.empty()` guard (:1715).  Singular K: SFMGPU_E_ARG.
 * The stage is the one of sfmgpu_pairs_set_ransac (same results for the same survivors; early stop and solver mode follow
 * the context) and runs before the step's one synchronisation.  A sequence that the step resets instead of tracking (the
 * first step, the first after sfmgpu_multitracker_reset, a sequence without tracks) is SFMGPU_TV_SKIPPED. */
int sfmgpu_multitracker_set_ransac(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const double* K, const sfmgpu_ransac_cfg* rc);
/* Results of the last step: status / best_n [S], inliers [S][ROWS] (indices into that step's survivor list, ascending),
 * R [S][9], t [S][3] (valid for SFMGPU_TV_OK); any may be NULL.  SFMGPU_E_STATE when the last step ran without the stage
 * (never enabled, switched off, or no step since set_ransac / reset). */
int sfmgpu_multitracker_ransac_download_all(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int32_t* status, int32_t* best_n,
                                            int32_t* inliers, double* R, double* t3);
/* Sets stopped early since the last call (reads and resets). */
int sfmgpu_multitracker_ransac_early(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* sets_stopped);

/* ---- RANSAC scoring: sampson_err + the loop at :667-676 ------------------------------------------------- */
/* xi/xj: n normalised correspondences; E: H hypotheses, 9 doubles each.  counts[h] = #{i : e_i < thr};
 * best_h = lowest h with the largest count (-1 when every count is 0); best_inl = its inlier indices
 * ascending (n ints of room), best_n their number.  counts may be NULL. */
int sfmgpu_ransac_score(sfmgpu_ctx* ctx, const double* xi_xy, const double* xj_xy, int n, const double* E, int H,
                        double thr, int32_t* counts, int* best_h, int32_t* best_inl, int* best_n);
/* Device-resident variant for throughput runs: upload once, score many times. */
int sfmgpu_ransac_upload(sfmgpu_ctx* ctx, const double* xi_xy, const double* xj_xy, int n, const double* E, int H);
int sfmgpu_ransac_score_resident(sfmgpu_ctx* ctx, double thr, int* best_h, int* best_n);
int sfmgpu_ransac_download(sfmgpu_ctx* ctx, int32_t* counts, int32_t* best_inl, int cap_inl);


/* ---- minimal solver on the device (opt-in): eight_point_E :609-627 + jacobi_eig_sym (linalg.hpp:133-201) ------------
 * One hypothesis per sampled index octet idx8[H][8] (the host keeps the reference's seeded sampling :657-665).  Leaves
 * the points and the H hypotheses resident, ready for sfmgpu_ransac_score_resident / sfmgpu_ransac_download; E_out
 * (optional) receives the hypotheses, 9 doubles each.  NOT bit-identical to the reference's solver (CUDA vs glibc
 * atan2 / sin / cos in the Jacobi rotations; ~1e-12 relative, eigenvector sign may differ): the default path of the
 * drop-in keeps the host solver, whose hypotheses are bit-identical.  With E_out == NULL (hypotheses resident for scoring
 * only) the context's solver mode applies, see sfmgpu_ransac_solve_score. */
int sfmgpu_ransac_hypotheses(sfmgpu_ctx* ctx, const double* xi_xy, const double* xj_xy, int n, const int32_t* idx8, int H,
                             double* E_out);
/* Solver + scoring loop of find_E_ransac (:657-677) in one call: hypotheses of the octets idx8[H][8] (NULL: the reference's
 * seeded sampling for n correspondences, std::mt19937(12345) + uniform_int_distribution, on the device), counts, winner
 * (largest count, lowest index), its hypothesis best_E[9] (zero matrix when no hypothesis has an inlier, as the reference's
 * Mat33{}) and ascending inlier list best_inl (room for n).  In solver mode 1 (default) the COUNTS come from a screening
 * solver - the unit null vector of the 8 x 9 design matrix by Householder QR, i.e. the vector the reference's Jacobi
 * iteration converges to, ~50x cheaper - and the winner is solved again by the Jacobi emulation of
 * sfmgpu_ransac_hypotheses before its inlier list and count are taken: best_E, best_n and best_inl are the emulation's.
 * Mode 0 runs the emulation for every octet (mode 2: the same through the warp-per-hypothesis kernel that re-solves the
 * winners - bit-identical, for tests; mode 3: screening for every launch, for tests).  The batched RANSAC stage (sfmgpu_pairs_set_ransac) follows the same mode. */
int sfmgpu_ransac_solve_score(sfmgpu_ctx* ctx, const double* xi_xy, const double* xj_xy, int n, const int32_t* idx8, int H,
                              double thr, int* best_h, int* best_n, double* best_E, int32_t* best_inl);
int sfmgpu_solver_set_mode(sfmgpu_ctx* ctx, int mode);


/* ---- batched two-view DLT triangulation (opt-in): triangulate_dlt :1477-1516 -----------------------------------------------
 * poses: P camera-to-world poses (PoseCW :157-168), 12 doubles each = R row-major + camera centre.  Track k observes
 * pixel ui[k] in pose ia[k] and uj[k] in pose ib[k]; X_out [n][3] are the world points.  Same formulas as the
 * reference; the 4x4 Jacobi uses CUDA's trig, so results agree to ~1e-10 relative, not bit for bit (the shim's
 * single-track triangulate_dlt stays on the host and IS bit-identical). */
int sfmgpu_triangulate_dlt(sfmgpu_ctx* ctx, const double* K, const double* poses, int P, const int32_t* ia, const int32_t* ib,
                           const double* ui_xy, const double* uj_xy, int n, double* X_out);

/* ---- loop-closure descriptor and candidate search: global_desc_32 :1100-1122, dot_desc :1124-1129, :1823-1831 ---------
 * desc_out: count descriptors of 1024 floats (host) for frames [first, first+count) (level 0 is read; bit-exact). */
int sfmgpu_global_desc32(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, float* desc_out);
/* Dot product of `query` with each of the first n_search stored descriptors (host arrays): scores (optional),
 * best_id = first index with the strictly largest score above 0 (-1: none), best_score (0 when none). */
int sfmgpu_desc_search(sfmgpu_ctx* ctx, const float* descs, int n_search, const float* query, float* scores, int* best_id,
                       float* best_score);

/* ---- device-resident descriptor bank and batched candidate search (loop closure for a whole sequence) ----------------
 * A bank holds `capacity` descriptors of 1024 floats in HBM, zero-filled at create: a zero descriptor scores 0 against
 * anything, so an unfilled slot can never become a candidate. */
typedef struct sfmgpu_descs sfmgpu_descs;
int sfmgpu_descs_create(sfmgpu_ctx* ctx, int capacity, sfmgpu_descs** out);
void sfmgpu_descs_destroy(sfmgpu_ctx* ctx, sfmgpu_descs* d);
/* global_desc_32 (:1100-1122) of frames [first, first+count) of f into slots [slot, slot+count), without a host round trip
 * (same values as sfmgpu_global_desc32).  Stream-ordered: returns before the kernels finish. */
int sfmgpu_descs_compute(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, sfmgpu_frames* f, int first, int count);
/* Host <-> slots [slot, slot+count): count * 1024 floats.  Both return when the copy is done. */
int sfmgpu_descs_upload(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, int count, const float* host);
int sfmgpu_descs_download(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, int count, float* host);
/* For every query q: the loop of :1823-1831 with query = slot query_slot[q] over slots [0, n_search[q]):
 * best_id[q] = first slot with the strictly largest score above 0 (-1: none), best_score[q] (0 when none).
 * scores (optional): [nq][ld], ld = max n_search; entries k >= n_search[q] are 0.  Every score is dot_desc (:1124-1129)
 * bit for bit.  The caller keeps the reference's keyframe gap (n_search = k - gap for keyframe k) and its gate (a
 * comparison on best_score).  query_slot outside [0, capacity) or n_search outside [0, capacity] is SFMGPU_E_ARG.
 * best_id / best_score may be NULL; returns when the outputs are in host memory. */
int sfmgpu_descs_search(sfmgpu_ctx* ctx, sfmgpu_descs* d, const int32_t* query_slot, const int32_t* n_search, int nq,
                        int32_t* best_id, float* best_score, float* scores);

#ifdef __cplusplus
}
#endif
#endif /* SFMGPU_H_ */
