// frontend.cu — the two callers of the kernels that the reference has:
//   * the stateless two-view front end (cpp/src/templering_sfm.cpp:1836-1857), batched over frame pairs;
//   * the stateful KLTTracker (:323-391): reset / step / tracks, with the replenish rule (:374-389).
// Everything stays on the device between stages; only survivors / counts are copied back when the caller asks.
#include <stdlib.h>

#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "common.cuh"

// ---- small kernels -----------------------------------------------------------------------------------------------
namespace {

// Rank of this thread's element among the kept elements of its 1024-element tile, in block order; *total receives the tile's
// count.  Called by every thread of a 1024-thread block, once per tile: the next call's shared writes come after a barrier
// that every thread reaches only once it has read this call's results.
__device__ __forceinline__ int tile_rank(bool k, int* total) {
  __shared__ int wcnt[32], wpre[32], tile_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned m = __ballot_sync(0xffffffffu, k);
  if (lane == 0) wcnt[warp] = __popc(m);
  __syncthreads();
  if (warp == 0) {
    const int a = wcnt[lane];
    int ia = a;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, ia, o);
      if (lane >= o) ia += u;
    }
    wpre[lane] = ia - a;
    if (lane == 31) tile_total = ia;
  }
  __syncthreads();
  *total = tile_total;
  return wpre[warp] + __popc(m & ((1u << lane) - 1u));
}

// Ordered compaction of the survivors of one pair / one tracker step: block = one pair.
// keep == nullptr keeps everything.  Outputs (any may be null): a/b = p0/p1 of survivors, ids_out, n_out.
__global__ void __launch_bounds__(1024) compact_kernel(const double2* __restrict__ p0, const double2* __restrict__ p1,
                                                      const uint8_t* __restrict__ keep, const int* __restrict__ ids,
                                                      const int* __restrict__ counts, int cap, double2* __restrict__ oa,
                                                      double2* __restrict__ ob, int* __restrict__ oid,
                                                      int* __restrict__ n_out) {
  const int pair = blockIdx.x;
  int n = counts ? counts[pair] : cap;
  n = n < 0 ? 0 : (n > cap ? cap : n);
  const size_t off = (size_t)pair * cap;
  int base = 0;
  for (int s = 0; s < n; s += 1024) {
    const int i = s + threadIdx.x;
    const bool k = i < n && (keep ? keep[off + i] != 0 : true);
    int total;
    const int r = base + tile_rank(k, &total);
    if (k) {
      if (oa) oa[off + r] = p0[off + i];
      if (ob) ob[off + r] = p1[off + i];
      if (oid) oid[off + r] = ids[off + i];
    }
    base += total;
  }
  if (threadIdx.x == 0 && n_out) n_out[pair] = base;
}

// totals[0] += sum max(ncorn,0); totals[1] += sum nkept; totals[2] += sum nit; totals[3] += #frames with ncorn < 0
// (ncorn == nullptr: cap for every pair)
__global__ void __launch_bounds__(256) totals_kernel(const int* __restrict__ ncorn, const int* __restrict__ nkept,
                                                    const int* __restrict__ nit, int npairs, int cap,
                                                    unsigned long long* __restrict__ totals) {
  unsigned long long c = 0, k = 0, it = 0, bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)npairs * cap;
       i += (long long)gridDim.x * blockDim.x) {
    const int pair = (int)(i / cap), slot = (int)(i - (long long)pair * cap);
    const int n = ncorn ? ncorn[pair] : cap;
    if (slot == 0) {
      if (n < 0) bad++;
      c += n > 0 ? n : 0;
      k += nkept[pair];
    }
    if (slot < n) it += nit[i];
  }
  c = __reduce_add_sync(0xffffffffu, (unsigned)c);  // per-warp partials fit 32 bits
  k = __reduce_add_sync(0xffffffffu, (unsigned)k);
  bad = __reduce_add_sync(0xffffffffu, (unsigned)bad);
  // nit can exceed 32 bits per warp only for absurd sizes; reduce in two halves to be safe
  unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(it & 0xFFFFu));
  unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(it >> 16));
  if ((threadIdx.x & 31) == 0) {  // zero partials are skipped: only the warps holding slot 0 of a pair count corners
    if (c) atomicAdd(&totals[0], c);
    if (k) atomicAdd(&totals[1], k);
    if (lo | hi) atomicAdd(&totals[2], (unsigned long long)lo + ((unsigned long long)hi << 16));
    if (bad) atomicAdd(&totals[3], bad);
  }
}

// Replenish filter (:378-388): new corner i survives iff no LIVE track lies at squared distance < d^2
// (FP64, no contraction: this file is built with -fmad=false).  Corners are pairwise >= d apart already,
// so tracks appended earlier in the same loop can never reject a later corner; the test is independent per corner.
__global__ void __launch_bounds__(256) replenish_filter_kernel(const double2* __restrict__ fresh, const int* __restrict__ n_fresh,
                                                              const double2* __restrict__ tracks, int n_tracks, double d2,
                                                              uint8_t* __restrict__ ok) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int nf = *n_fresh;
  if (i >= nf) return;
  const double2 p = fresh[i];
  bool good = true;
  for (int j = 0; j < n_tracks; j++) {
    const double2 t = tracks[j];
    const double dx = t.x - p.x, dy = t.y - p.y;
    if (dx * dx + dy * dy < d2) {
      good = false;
      break;
    }
  }
  ok[i] = good ? 1 : 0;
}

// Append up to `room` surviving fresh corners to the track list with consecutive ids (one block).
__global__ void __launch_bounds__(1024) replenish_append_kernel(const double2* __restrict__ fresh, const int* __restrict__ n_fresh,
                                                               const uint8_t* __restrict__ ok, double2* __restrict__ tracks,
                                                               int* __restrict__ ids, int n_tracks, int room, int next_id,
                                                               int* __restrict__ n_added) {
  const int nf = *n_fresh;
  int base = 0;
  for (int s = 0; s < nf && base < room; s += 1024) {
    const int i = s + threadIdx.x;
    const bool k = i < nf && ok[i];
    int total;
    const int r = base + tile_rank(k, &total);
    if (k && r < room) {
      tracks[n_tracks + r] = fresh[i];
      ids[n_tracks + r] = next_id + r;
    }
    base += total;
  }
  if (threadIdx.x == 0) *n_added = base < room ? base : room;
}

// After a detection into `fresh` (row stride fresh_stride): row s of the track lists = the first n[s] corners with ids
// first_id[s]...
__global__ void take_corners_kernel(const double2* __restrict__ fresh, int fresh_stride, const int* __restrict__ n,
                                    const int* __restrict__ first_id, double2* __restrict__ trk, int* __restrict__ ids, int rows) {
  const int s = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n[s] || i >= rows) return;
  trk[(size_t)s * rows + i] = fresh[(size_t)s * fresh_stride + i];
  ids[(size_t)s * rows + i] = first_id[s] + i;
}

// Rows of a track list: after reset at most max(max_tracks, 1) entries; replenish appends first and tests the cap afterwards
// (:386-387), so a list below min_tracks grows to max_tracks, or by ONE entry when it is already at / above max_tracks
// (min_tracks > max_tracks): the list never exceeds max(max_tracks, min_tracks, 1), plus one overshoot entry.
int track_rows(const sfmgpu_lkcfg& c) {
  int m = c.max_tracks < 1 ? 1 : c.max_tracks;
  if (c.min_tracks > m) m = c.min_tracks;
  return m + 1;
}

// List call, one pyramid level: frame idx_a[y] of src -> frame y of dst and frame idx_b[y] -> frame b_off + y (grid.z = 0 / 1),
// whole frames with their row padding, 16 B per thread and step.
__global__ void __launch_bounds__(256) gather_frames_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, size_t fstride,
                                                           const int* __restrict__ idx_a, const int* __restrict__ idx_b, int b_off) {
  const size_t n16 = fstride / 16;  // pitch is a multiple of 16
  const int y = blockIdx.y, sf = blockIdx.z ? idx_b[y] : idx_a[y], df = blockIdx.z ? b_off + y : y;
  const uint4* s = reinterpret_cast<const uint4*>(src + (size_t)sf * fstride);
  uint4* d = reinterpret_cast<uint4*>(dst + (size_t)df * fstride);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) d[i] = s[i];
}

// One whole-frame copy of a pyramid level: n16 16-byte words from src to dst.
struct FrameCopy {
  const uint4* src;
  uint4* dst;
  unsigned long long n16;
};

// Lock-step tracker, resident input: copy tab[blockIdx.y] for every (sequence, level) entry of the table in one launch, 16 B per
// thread and step.
__global__ void __launch_bounds__(256) copy_frames_kernel(const FrameCopy* __restrict__ tab) {
  const FrameCopy c = tab[blockIdx.y];
#pragma unroll 4
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < c.n16; i += (size_t)gridDim.x * blockDim.x) c.dst[i] = c.src[i];
}

int default_cand_cap(int w, int h) {
  long long px = (long long)w * h;
  long long cap = px / 6;
  if (cap < 65536) cap = 65536;
  if (cap > px) cap = px;
  return (int)cap;
}

int abs_min_distance(const sfmgpu_lkcfg& c) { return c.min_distance < 0 ? -c.min_distance : c.min_distance; }

// Corners of frames [first, first + count) with the work area sized for the worst case, W*H candidates per frame (a flat image
// makes every pixel one), so that no frame overflows: out [count][max(max_corners, 1)], counts d_n[count].
int detect_full(sfmgpu_ctx* ctx, const sfmgpu_lkcfg& cfg, sfmgpu_frames* f, int first, int count, int max_corners, double2* out,
                int* d_n) {
  const int cand_cap = f->w * f->h;
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sfm_corner_work_bytes_md(f->w, f->h, count, cand_cap, abs_min_distance(cfg))));
  return sfm_corners_batch(ctx, f, first, count, max_corners, cfg.quality, cfg.min_distance, cand_cap, ctx->cs_work.p,
                           ctx->cs_work.cap, out, d_n);
}

}  // namespace

// ---- batched pair front end -------------------------------------------------------------------------------------------
extern "C" {

int sfmgpu_pairs_create(sfmgpu_ctx* ctx, int max_pairs, int max_corners, sfmgpu_pairs** out) {
  SFM_ENTER(ctx);
  if (!ctx || !out || max_pairs <= 0) return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_create: bad arguments");
  sfmgpu_pairs* p = new sfmgpu_pairs();
  p->max_pairs = max_pairs;
  p->cap = max_corners < 1 ? 1 : max_corners;
  const size_t n = (size_t)max_pairs * p->cap;
  cudaError_t e = cudaSuccess;
  auto al = [&](void** q, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(q, bytes + 256);
  };
  al((void**)&p->xy0, n * 16);
  al((void**)&p->p1, n * 16);
  al((void**)&p->pb, n * 16);
  al((void**)&p->li, n * 16);
  al((void**)&p->lj, n * 16);
  al((void**)&p->nit, n * 4);
  al((void**)&p->keep, n);
  al((void**)&p->ncorn, (size_t)max_pairs * 4);
  al((void**)&p->nkept, (size_t)max_pairs * 4);
  al((void**)&p->totals, 64);
  if (e != cudaSuccess) {
    sfmgpu_pairs_destroy(ctx, p);
    return sfm_fail(ctx, SFMGPU_E_CUDA, "pairs_create: cudaMalloc failed: %s", cudaGetErrorString(e));
  }
  *out = p;
  return 0;
}

void sfmgpu_pairs_destroy(sfmgpu_ctx* ctx, sfmgpu_pairs* p) {
  SFM_ENTER_VOID(ctx);
  if (!p) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  sfm_two_view_free(ctx, &p->tv);
  if (p->seg) sfmgpu_multitracker_destroy(ctx, p->seg);
  void* ptrs[] = {p->xy0, p->p1, p->pb, p->li, p->lj, p->nit, p->keep, p->ncorn, p->nkept, p->totals, p->work[0].p, p->work[1].p,
                  p->gather.p, p->idx.p, p->ids};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  delete p;
}

// ---- the three stages of a chunk of pairs --------------------------------------------------------------------------
// Pairs (first_frame + k, first_frame + k + 1), k < npairs, go to slots [pair_off, pair_off + npairs) of `out`;
// totals are accumulated (the caller zeroes them).  A chunk is at most 1024 frames (the corner work area).
// The stages read the pairs' frames from `cf`: image A of pair k is frame cfirst + k, image B frame cfirst + b_off + k.  The
// consecutive calls use cf = f, cfirst = first_frame, b_off = 1; the list call (explicit frame pairs) a gathered copy of
// both frames' pyramids, A frames first, B frames b_off later.
struct ChunkArgs {
  sfmgpu_frames* f;
  int first_frame, pair_off, npairs;
  const sfmgpu_lkcfg* cfg;
  sfmgpu_pairs* out;
  DevBuf* work;
  int cand_cap, md;
  const sfmgpu_frames* cf;
  int cfirst, b_off;
};

static int stage_score(sfmgpu_ctx* ctx, const ChunkArgs& c) {
  return sfm_corners_score_stage(ctx, c.cf, c.cfirst, c.npairs, c.cfg->quality, c.md, c.cand_cap, c.work->p, c.work->cap);
}

static int stage_select(sfmgpu_ctx* ctx, const ChunkArgs& c) {
  const size_t so = (size_t)c.pair_off * c.out->cap;
  return sfm_corners_select_stage(ctx, c.cf, c.cfirst, c.npairs, c.cfg->max_tracks, c.cfg->quality, c.md, c.cand_cap, c.work->p, c.work->cap, c.out->xy0 + so,
                                  c.out->ncorn + c.pair_off);
}

static int stage_klt(sfmgpu_ctx* ctx, const ChunkArgs& c) {
  sfmgpu_pairs* out = c.out;
  const size_t so = (size_t)c.pair_off * out->cap;
  KltLaunch k;
  k.pv = c.cf->view();
  k.pvb = k.pv;
  k.p0 = out->xy0 + so;
  k.counts = out->ncorn + c.pair_off;
  k.npairs = c.npairs;
  k.cap = out->cap;
  k.fa0 = c.cfirst;
  k.fa_step = 1;
  k.fb0 = c.cfirst + c.b_off;
  k.fb_step = 1;
  k.radius = c.cfg->win_radius;
  k.iters = c.cfg->iters;
  k.fb_thresh = c.cfg->fb_thresh;
  k.p1 = out->p1 + so;
  k.pb = out->pb + so;
  k.nit = out->nit + so;
  k.keep = out->keep + so;
  {
    StageTimer st(ctx, 2);
    SFM_TRY(sfm_klt_launch(ctx, k));
  }
  {
    StageTimer st(ctx, 3);
    SFM_LAUNCH(ctx, compact_kernel, c.npairs, 1024, 0, out->xy0 + so, out->p1 + so, out->keep + so, (const int*)nullptr,
               out->ncorn + c.pair_off, out->cap, out->li + so, out->lj + so, (int*)nullptr, out->nkept + c.pair_off);
    SFM_LAUNCH(ctx, totals_kernel, 256, 256, 0, out->ncorn + c.pair_off, out->nkept + c.pair_off, out->nit + so, c.npairs, out->cap,
               out->totals);
  }
  if (sfm_two_view_enabled(out->tv)) {  // the unit's last step: find_E_ransac on the survivors of every pair (:1855-1857)
    StageTimer rt(ctx, 4);
    SFM_TRY(sfm_two_view_stage(ctx, out->tv, out->li, out->lj, out->nkept, out->cap, c.pair_off, c.npairs, nullptr));
  }
  return 0;
}

static ChunkArgs chunk_args(sfmgpu_frames* f, int first_frame, int pair_off, int npairs, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out,
                            DevBuf* work) {
  ChunkArgs c;
  c.f = f;
  c.first_frame = first_frame;
  c.pair_off = pair_off;
  c.npairs = npairs;
  c.cfg = cfg;
  c.out = out;
  c.work = work;
  c.cand_cap = default_cand_cap(f->w, f->h);
  c.md = abs_min_distance(*cfg);
  c.cf = f;
  c.cfirst = first_frame;
  c.b_off = 1;
  return c;
}

// Pairs per corner launch: >= 4 blocks per SM keeps the one-block-per-frame selection kernels busy; large frames are
// limited by the work area instead (47 MB per 4K frame at min_distance 8: 16 GiB hold 362 of them, ~2.4 blocks per SM)
static int pair_chunk(sfmgpu_ctx* ctx, sfmgpu_frames* f, int npairs, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out) {
  ChunkArgs c1 = chunk_args(f, 0, 0, 1, cfg, out, &out->work[0]);
  const size_t per_frame = sfm_corner_work_bytes_md(f->w, f->h, 1, c1.cand_cap, c1.md);
  long long by_mem = (long long)(((size_t)16 << 30) / (per_frame ? per_frame : 1));
  if (by_mem < 2 * ctx->n_sm) by_mem = 2 * ctx->n_sm;
  int chunk = npairs < 1024 ? npairs : 1024;
  if (chunk > by_mem) chunk = (int)by_mem;
  return chunk;
}

// Everything back to back on the context stream (chunks of <= 1024 frames).
static int pair_range(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first_frame, int pair_off, int npairs, const sfmgpu_lkcfg* cfg,
                      sfmgpu_pairs* out) {
  if (npairs == 0) return 0;
  const int chunk = pair_chunk(ctx, f, npairs, cfg, out);
  ChunkArgs c0 = chunk_args(f, first_frame, pair_off, chunk, cfg, out, &out->work[0]);
  SFM_TRY(sfm_reserve(ctx, out->work[0], sfm_corner_work_bytes_md(f->w, f->h, chunk, c0.cand_cap, c0.md)));
  for (int p = 0; p < npairs; p += chunk) {
    const int cnt = npairs - p < chunk ? npairs - p : chunk;
    ChunkArgs c = chunk_args(f, first_frame + p, pair_off + p, cnt, cfg, out, &out->work[0]);
    SFM_TRY(stage_score(ctx, c));
    SFM_TRY(stage_select(ctx, c));
    SFM_TRY(stage_klt(ctx, c));
  }
  return 0;
}

// ---- stage pipeline over chunks -------------------------------------------------------------------------------------
// The corner-select kernel is latency bound: one block per frame walks the introsort tree and the greedy selection,
// ~4.8 ms for a launch no matter how few frames it holds, at a fraction of the SM's issue rate.  Chunks of pairs
// therefore flow through three streams, one per stage: score (context stream) -> select (HIGH-priority stream: its
// few blocks are placed as soon as they are ready) -> KLT + compaction.  select(c) then shares the SMs with
// score(c+1) and KLT(c-1).  Two corner work areas alternate; score(c+2) waits for select(c).  Results are identical
// to the sequential order (chunks are independent).
struct StageScope {  // run a piece of work on another stream: SFM_LAUNCH and friends use ctx->stream
  sfmgpu_ctx* ctx;
  cudaStream_t saved;
  StageScope(sfmgpu_ctx* c, cudaStream_t s) : ctx(c), saved(c->stream) { c->stream = s; }
  ~StageScope() { ctx->stream = saved; }
};

static cudaEvent_t pipe_event(sfmgpu_ctx* ctx, size_t i) {
  while (ctx->pipe_evs.size() <= i) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ctx->pipe_evs.push_back(e);
  }
  return ctx->pipe_evs[i];
}

static int pipe_streams(sfmgpu_ctx* ctx) {
  if (!ctx->sel_stream) {
    int lo = 0, hi = 0;
    SFM_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = numerically lowest = greatest priority
    SFM_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->sel_stream, cudaStreamNonBlocking, hi));
    SFM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->klt_stream, cudaStreamNonBlocking));
    SFM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    SFM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->back_stream, cudaStreamNonBlocking));
  }
  return 0;
}

// Scratch is sized before any work is queued (growing a buffer frees and reallocates it).
static int pipe_reserve(sfmgpu_ctx* ctx, sfmgpu_frames* f, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out, int chunk) {
  const ChunkArgs c = chunk_args(f, 0, 0, chunk, cfg, out, nullptr);
  const size_t wb = sfm_corner_work_bytes_md(f->w, f->h, chunk, c.cand_cap, c.md);
  SFM_TRY(sfm_reserve(ctx, out->work[0], wb));
  SFM_TRY(sfm_reserve(ctx, out->work[1], wb));
  SFM_TRY(sfm_reserve(ctx, ctx->klt_defer, 2 * ((size_t)chunk * out->cap + 2) * sizeof(int)));
  return 0;
}

// Pipeline state of one call: event indices are handed out sequentially from ctx->pipe_evs.
struct Pipe {
  sfmgpu_ctx* ctx;
  size_t ev = 0;
  int nchunk = 0;
  cudaEvent_t sel_done[2] = {nullptr, nullptr};  // select of the chunk that last used work area 0 / 1
  cudaEvent_t next() { return pipe_event(ctx, ev++); }
  // SFMGPU_PIPE_TRACE=1: timestamps around every stage of every chunk, printed by trace_dump() (diagnostics only)
  bool trace = getenv("SFMGPU_PIPE_TRACE") != nullptr;
  std::vector<cudaEvent_t> tev;
  cudaEvent_t t0 = nullptr;
  void mark(cudaStream_t s) {
    if (!trace) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    tev.push_back(e);
  }
  void trace_dump() {
    if (!trace || tev.empty()) return;
    static const char* nm[3] = {"score", "select", "klt"};
    for (size_t i = 0; i + 1 < tev.size(); i += 2) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, tev[0], tev[i]);
      cudaEventElapsedTime(&b, tev[0], tev[i + 1]);
      fprintf(stderr, "[pipe] chunk %zu %-6s %8.3f -> %8.3f ms\n", i / 6, nm[(i / 2) % 3], a, b);
    }
    for (cudaEvent_t e : tev) cudaEventDestroy(e);
    tev.clear();
  }
};

// Queue one chunk: score on the context stream (after `ready`, if given), select on the priority stream, KLT on its
// stream; *done (if given) is recorded behind the chunk's last kernel.
static int pipe_chunk(Pipe& p, sfmgpu_frames* f, int first_frame, int pair_off, int npairs, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out,
                      cudaEvent_t ready, cudaEvent_t* done) {
  sfmgpu_ctx* ctx = p.ctx;
  const int wa = p.nchunk & 1;
  p.nchunk++;
  ChunkArgs c = chunk_args(f, first_frame, pair_off, npairs, cfg, out, &out->work[wa]);
  cudaEvent_t e_score = p.next(), e_sel = p.next(), e_done = p.next();
  if (!e_score || !e_sel || !e_done) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend: cudaEventCreate failed");
  if (ready) SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ready, 0));
  if (p.sel_done[wa]) SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, p.sel_done[wa], 0));  // work area free again
  p.mark(ctx->stream);
  SFM_TRY(stage_score(ctx, c));
  p.mark(ctx->stream);
  SFM_CUDA(ctx, cudaEventRecord(e_score, ctx->stream));
  {
    StageScope sc(ctx, ctx->sel_stream);
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, e_score, 0));
    p.mark(ctx->stream);
    SFM_TRY(stage_select(ctx, c));
    p.mark(ctx->stream);
    SFM_CUDA(ctx, cudaEventRecord(e_sel, ctx->stream));
  }
  p.sel_done[wa] = e_sel;
  {
    StageScope sc(ctx, ctx->klt_stream);
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, e_sel, 0));
    p.mark(ctx->stream);
    SFM_TRY(stage_klt(ctx, c));
    p.mark(ctx->stream);
    SFM_CUDA(ctx, cudaEventRecord(e_done, ctx->stream));
  }
  if (done) *done = e_done;
  return 0;
}

static int pair_cfg_ok(sfmgpu_ctx* ctx, sfmgpu_frames* f, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out) {
  const int cap_out = cfg->max_tracks < 1 ? 1 : cfg->max_tracks;
  if (cap_out != out->cap) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend: cfg->max_tracks != pairs capacity");
  if (cfg->pyr_levels != f->levels) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend: cfg->pyr_levels != frames levels");
  return 0;
}

static int pair_args_ok(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first_frame, int npairs, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out) {
  if (npairs < 0 || npairs > out->max_pairs || first_frame < 0 || first_frame + npairs + (npairs > 0 ? 1 : 0) > f->n)
    return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend: pair range [%d,%d) does not fit (frames %d, max_pairs %d)", first_frame,
                    first_frame + npairs, f->n, out->max_pairs);
  return pair_cfg_ok(ctx, f, cfg, out);
}

// Batch calls size the candidate lists for W*H/6 entries per frame.  A frame whose FINAL list is longer (flat or
// weak-texture image: thr = 0 makes every pixel a candidate, :274-285) comes back with n_corners < 0; it is redone here
// through the single-frame path, whose work area holds the worst case (W*H candidates), so the batch returns what the
// reference returns for every frame.  Synchronises the context stream (the overflow flags are read on the host).
// redone (optional) receives the pair slots that were recomputed.  The list call passes its frame pairs (h_fa, h_fb: host);
// the consecutive calls pass none (pair p = (first_frame + p, first_frame + p + 1)).  Either way the frames are read from f.
static int pair_fix_overflow(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first_frame, int npairs, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out,
                             std::vector<int>* redone, const int* h_fa = nullptr, const int* h_fb = nullptr) {
  if (npairs <= 0) return 0;
  SFM_TRY(sfm_pinned(ctx, (size_t)npairs * sizeof(int)));
  int* hn = (int*)ctx->pinned;
  SFM_CUDA(ctx, cudaMemcpyAsync(hn, out->ncorn, (size_t)npairs * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  std::vector<int> bad;
  for (int p = 0; p < npairs; p++)
    if (hn[p] < 0) bad.push_back(p);
  if (bad.empty()) return 0;
  for (int p : bad) {
    SFM_TRY(detect_full(ctx, *cfg, f, h_fa ? h_fa[p] : first_frame + p, 1, cfg->max_tracks, out->xy0 + (size_t)p * out->cap, out->ncorn + p));
    ChunkArgs c = chunk_args(f, first_frame + p, p, 1, cfg, out, nullptr);
    if (h_fa) {
      c.cfirst = h_fa[p];
      c.b_off = h_fb[p] - h_fa[p];
    }
    SFM_TRY(stage_klt(ctx, c));  // adds this pair's corners / survivors / iterations to the totals
  }
  SFM_CUDA(ctx, cudaMemcpyAsync(hn, out->ncorn, (size_t)npairs * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals + 3, 0, sizeof(unsigned long long), ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int p : bad)
    if (hn[p] < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pair_frontend: pair %d exceeded the full candidate capacity", p);
  if (redone) *redone = bad;
  return 0;
}

int sfmgpu_pipeline_set(sfmgpu_ctx* ctx, int pairs_per_chunk) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  if (pairs_per_chunk < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "pipeline_set: negative chunk");
  ctx->pipe_chunk = pairs_per_chunk > 1024 ? 1024 : pairs_per_chunk;
  return 0;
}

int sfmgpu_pair_frontend(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first_frame, int npairs, const sfmgpu_lkcfg* cfg,
                         sfmgpu_pairs* out) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out) return SFMGPU_E_ARG;
  SFM_TRY(pair_args_ok(ctx, f, first_frame, npairs, cfg, out));
  out->last_npairs = npairs;
  out->ids_valid = false;
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals, 0, 64, ctx->stream));
  const int sub = ctx->pipe_chunk;
  if (sub <= 0 || ctx->profile || npairs < 2 * sub) {  // stage profiling wants the stages back to back on one stream
    SFM_TRY(pair_range(ctx, f, first_frame, 0, npairs, cfg, out));
    return pair_fix_overflow(ctx, f, first_frame, npairs, cfg, out, nullptr);
  }
  SFM_TRY(pipe_streams(ctx));
  SFM_TRY(pipe_reserve(ctx, f, cfg, out, sub));
  Pipe p;
  p.ctx = ctx;
  cudaEvent_t fork = p.next();
  if (!fork) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend: cudaEventCreate failed");
  SFM_CUDA(ctx, cudaEventRecord(fork, ctx->stream));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->sel_stream, fork, 0));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->klt_stream, fork, 0));
  cudaEvent_t last = nullptr;
  for (int p0 = 0; p0 < npairs; p0 += sub) {
    const int cnt = npairs - p0 < sub ? npairs - p0 : sub;
    SFM_TRY(pipe_chunk(p, f, first_frame + p0, p0, cnt, cfg, out, nullptr, &last));
  }
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, last, 0));  // the KLT stream is in order: its last event covers all chunks
  return pair_fix_overflow(ctx, f, first_frame, npairs, cfg, out, nullptr);
}

// Explicit frame pairs (loop-closure verification): pair k = (frame_a[k], frame_b[k]) of resident frames.  Per chunk, the
// pyramids of both frames of every pair are gathered into a scratch batch (A frames, then B frames) and the three stages run
// on it unchanged, as they run on consecutive frames; chunks run back to back on the context stream.
int sfmgpu_pair_frontend_list(sfmgpu_ctx* ctx, sfmgpu_frames* f, const int32_t* frame_a, const int32_t* frame_b, int npairs,
                              const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out) return SFMGPU_E_ARG;
  if (npairs < 0 || npairs > out->max_pairs)
    return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_list: %d pairs, room for %d", npairs, out->max_pairs);
  if (npairs > 0 && (!frame_a || !frame_b)) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_list: null frame index array");
  for (int k = 0; k < npairs; k++)
    if (frame_a[k] < 0 || frame_a[k] >= f->n || frame_b[k] < 0 || frame_b[k] >= f->n)
      return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_list: pair %d = (%d, %d) outside frames [0,%d)", k, frame_a[k], frame_b[k], f->n);
  SFM_TRY(pair_cfg_ok(ctx, f, cfg, out));
  const int chunk = npairs > 0 ? pair_chunk(ctx, f, npairs, cfg, out) : 0;
  // scratch batch of 2 * chunk frames with f's geometry: level l at gather + lofs[l]
  size_t lofs[SFM_MAXL], gbytes = 0;
  for (int l = 0; l < f->levels; l++) {
    lofs[l] = gbytes;
    gbytes += (f->fstride[l] * 2 * chunk + 255) & ~(size_t)255;
  }
  if (npairs > 0) {  // scratch is sized before any work is queued
    const ChunkArgs c0 = chunk_args(f, 0, 0, chunk, cfg, out, nullptr);
    SFM_TRY(sfm_reserve(ctx, out->idx, 2 * (size_t)npairs * sizeof(int)));
    SFM_TRY(sfm_reserve(ctx, out->work[0], sfm_corner_work_bytes_md(f->w, f->h, chunk, c0.cand_cap, c0.md)));
    SFM_TRY(sfm_reserve(ctx, out->gather, gbytes));
  }
  out->last_npairs = npairs;
  out->ids_valid = false;
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals, 0, 64, ctx->stream));
  if (npairs == 0) return 0;
  int* d_fa = (int*)out->idx.p;
  int* d_fb = d_fa + npairs;
  SFM_CUDA(ctx, cudaMemcpyAsync(d_fa, frame_a, (size_t)npairs * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(d_fb, frame_b, (size_t)npairs * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  sfmgpu_frames g = *f;  // same geometry and levels, 2 * chunk frames in the scratch
  g.n = 2 * chunk;
  for (int l = 0; l < f->levels; l++) g.lvl[l] = (uint8_t*)out->gather.p + lofs[l];
  for (int p = 0; p < npairs; p += chunk) {
    const int cnt = npairs - p < chunk ? npairs - p : chunk;
    {
      StageTimer st(ctx, 5);
      for (int l = 0; l < f->levels; l++) {
        if (f->fstride[l] == 0) continue;  // level of zero size
        const unsigned gx = sfm_cdiv((long long)(f->fstride[l] / 16), 256 * 8);
        SFM_LAUNCH(ctx, gather_frames_kernel, dim3(gx, cnt, 2), 256, 0, f->lvl[l], g.lvl[l], f->fstride[l], (const int*)(d_fa + p),
                   (const int*)(d_fb + p), chunk);
      }
    }
    ChunkArgs c = chunk_args(f, 0, p, cnt, cfg, out, &out->work[0]);
    c.cf = &g;
    c.cfirst = 0;
    c.b_off = chunk;
    SFM_TRY(stage_score(ctx, c));
    SFM_TRY(stage_select(ctx, c));
    SFM_TRY(stage_klt(ctx, c));
  }
  return pair_fix_overflow(ctx, f, 0, npairs, cfg, out, nullptr, frame_a, frame_b);
}

// Frames per upload chunk of the streaming calls (chunk_frames <= 0: the default rule).
static int host_chunk(const sfmgpu_frames* f, int nframes, int chunk_frames) {
  // default: about 100 frames (50 for large frames), at least 8 chunks for short sequences, at most 20 (40) for long ones.  Smaller chunks shorten the
  // pipeline fill (the first upload and the last chunk's compute are not overlapped), too small ones under-fill the
  // one-block-per-frame kernels.  Measured end to end: C2 (1000 x 1080p) chunks of 84-125 frames 43.0 ms, 167: 44.1, 250: 46.3,
  // 50: 47.8; C3 with the RANSAC stage (2000 x 4K) 50: 372 ms, 100: 358, 150: 385, 200: 390.  (Tried and dropped: halving the
  // last chunks - 50, 25, 13, 12 frames, or 50 + 25 + 25 - so that less compute is left behind the last upload: 325 / 322 ms
  // against 321 ms on C3; the one-block-per-frame kernels of a 12-frame chunk still take their full latency and the short
  // uploads ran at 37 instead of 54 GB/s.)
  int chunk = chunk_frames;
  if (chunk <= 0) {
    // what is left behind the last upload is the compute of the last chunk, which grows with the frame size: about 100 frames
    // up to 4 Mpixel, about 50 above (C3 with the uploads back to back on the copy stream: 100 frames 315 ms, 64: 314, 50: 309,
    // 40: 311; C2: 100-125 frames 47.8 ms, 50: 52.6, 32: 64.1)
    const bool big = (size_t)f->w * f->h > 4000000u;
    const int base = big ? 48 : 96, most = big ? 40 : 20;
    const int by8 = (nframes + 7) / 8, bym = (nframes + most - 1) / most;
    chunk = by8 < base ? by8 : base;
    if (chunk < bym) chunk = bym;
  }
  if (chunk < 2) chunk = 2;
  if (chunk > 1024) chunk = 1024;
  return chunk;
}

// Queues level 0 of frames [a, b) (upload chunk c) on the copy stream and makes ctx->stream wait for it; whatever else the
// frames need before their pyramids (a decode) goes on ctx->stream behind that wait.
struct ChunkFill {
  virtual int fill(Pipe& p, sfmgpu_frames* f, int c, int a, int b) = 0;
};

// The streaming front end: frames [0, nframes) of `f` are filled chunk by chunk by `src` on a copy stream; every chunk's
// pyramids are built on the score stream, the chunk flows through the stage pipeline and its results go back on a fifth
// stream.  Argument checks are the caller's.
static int host_stream(sfmgpu_ctx* ctx, sfmgpu_frames* f, int nframes, int chunk, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out,
                       ChunkFill& src, double* li_xy, double* lj_xy, int32_t* n_kept, int32_t* n_corners) {
  const int npairs = nframes > 0 ? nframes - 1 : 0;
  out->last_npairs = npairs;
  out->ids_valid = false;
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals, 0, 64, ctx->stream));
  if (nframes == 0) return 0;
  SFM_TRY(pipe_streams(ctx));
  const int nchunks = (nframes + chunk - 1) / chunk;
  SFM_TRY(pipe_reserve(ctx, f, cfg, out, chunk));
  Pipe p;
  p.ctx = ctx;
  cudaEvent_t fork = p.next();
  if (!fork) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend_host: cudaEventCreate failed");
  // nothing may overwrite frames / results that an earlier call on the context stream still uses
  SFM_CUDA(ctx, cudaEventRecord(fork, ctx->stream));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, fork, 0));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->back_stream, fork, 0));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->sel_stream, fork, 0));
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->klt_stream, fork, 0));
  const size_t cap = (size_t)out->cap;
  for (int c = 0; c < nchunks; c++) {
    const int a = c * chunk, b = a + chunk < nframes ? a + chunk : nframes;
    SFM_TRY(src.fill(p, f, c, a, b));
    SFM_TRY(sfmgpu_pyramid_build(ctx, f, a, b - a));
    // pairs whose second frame arrived with this chunk
    const int P0 = a > 0 ? a - 1 : 0, P1 = b - 1;
    if (P1 <= P0) continue;
    cudaEvent_t done = nullptr;
    SFM_TRY(pipe_chunk(p, f, P0, P0, P1 - P0, cfg, out, nullptr, &done));
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->back_stream, done, 0));
    const size_t np_ = (size_t)(P1 - P0), o = (size_t)P0;
    if (li_xy)
      SFM_CUDA(ctx, cudaMemcpyAsync(li_xy + 2 * o * cap, out->li + o * cap, np_ * cap * 16, cudaMemcpyDeviceToHost, ctx->back_stream));
    if (lj_xy)
      SFM_CUDA(ctx, cudaMemcpyAsync(lj_xy + 2 * o * cap, out->lj + o * cap, np_ * cap * 16, cudaMemcpyDeviceToHost, ctx->back_stream));
    if (n_kept) SFM_CUDA(ctx, cudaMemcpyAsync(n_kept + o, out->nkept + o, np_ * 4, cudaMemcpyDeviceToHost, ctx->back_stream));
    if (n_corners) SFM_CUDA(ctx, cudaMemcpyAsync(n_corners + o, out->ncorn + o, np_ * 4, cudaMemcpyDeviceToHost, ctx->back_stream));
    if (sfm_two_view_enabled(out->tv)) SFM_TRY(sfm_two_view_download(ctx, out->tv, out->cap, P0, P1 - P0, ctx->back_stream));
  }
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->back_stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->klt_stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->sel_stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  p.trace_dump();
  std::vector<int> redone;
  SFM_TRY(pair_fix_overflow(ctx, f, 0, npairs, cfg, out, &redone));
  for (int q : redone) {  // rare: frames redone with the full candidate capacity go back once more
    const size_t o = (size_t)q;
    if (li_xy) SFM_CUDA(ctx, cudaMemcpyAsync(li_xy + 2 * o * cap, out->li + o * cap, cap * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (lj_xy) SFM_CUDA(ctx, cudaMemcpyAsync(lj_xy + 2 * o * cap, out->lj + o * cap, cap * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_kept) SFM_CUDA(ctx, cudaMemcpyAsync(n_kept + o, out->nkept + o, 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_corners) SFM_CUDA(ctx, cudaMemcpyAsync(n_corners + o, out->ncorn + o, 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (sfm_two_view_enabled(out->tv)) SFM_TRY(sfm_two_view_download(ctx, out->tv, out->cap, q, 1, ctx->stream));
  }
  if (!redone.empty()) SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

struct RawFill : ChunkFill {
  const uint8_t* pix;
  int fill(Pipe& p, sfmgpu_frames* f, int, int a, int b) override {
    sfmgpu_ctx* ctx = p.ctx;
    SFM_CUDA(ctx, cudaMemcpy2DAsync(f->lvl[0] + (size_t)a * f->fstride[0], f->pitch[0], pix + (size_t)a * f->w * f->h, f->w, f->w,
                                    (size_t)f->h * (b - a), cudaMemcpyDefault, ctx->copy_stream));
    cudaEvent_t up = p.next();
    if (!up) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend_host: cudaEventCreate failed");
    // The copy stream carries NOTHING but the uploads, back to back: the call is bound by them.  The chunk's pyramid is built
    // on the score stream behind the upload's event (on the copy stream it sat between two uploads and, waiting for SMs
    // behind the running KLT / RANSAC kernels, kept the copy engine idle ~0.35 ms per chunk).
    SFM_CUDA(ctx, cudaEventRecord(up, ctx->copy_stream));
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, up, 0));
    return 0;
  }
};

// Packed chunks: one cudaMemcpyAsync of the chunk's blob bytes into staging buffer c % 2 on the copy stream, then the decode on
// the score stream behind the upload's event.  A staging buffer is overwritten only after the decode that read it (chunk c - 2).
struct PackedFill : ChunkFill {
  const uint8_t* blob;
  const std::vector<uint64_t>* fo;  // absolute offsets of the call's frames in the blob
  const unsigned long long* d_fo;   // the same on the device
  cudaEvent_t decoded[2] = {nullptr, nullptr};
  int fill(Pipe& p, sfmgpu_frames* f, int c, int a, int b) override {
    sfmgpu_ctx* ctx = p.ctx;
    const int s = c & 1;
    cudaEvent_t up = p.next(), dec = p.next();
    if (!up || !dec) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend_host_packed: cudaEventCreate failed");
    if (decoded[s]) SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, decoded[s], 0));
    const uint64_t o0 = (*fo)[a], o1 = (*fo)[b];
    SFM_CUDA(ctx, cudaMemcpyAsync(ctx->pk_stage[s].p, blob + o0, o1 - o0, cudaMemcpyHostToDevice, ctx->copy_stream));
    SFM_CUDA(ctx, cudaEventRecord(up, ctx->copy_stream));
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, up, 0));
    SFM_TRY(sfm_pk_decode(ctx, f, a, b - a, (const uint8_t*)ctx->pk_stage[s].p, d_fo + a, o0, (int*)ctx->pk_flag.p));
    SFM_CUDA(ctx, cudaEventRecord(dec, ctx->stream));
    decoded[s] = dec;
    return 0;
  }
};

static int host_args_ok(sfmgpu_ctx* ctx, sfmgpu_frames* f, int nframes, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out, const char* who) {
  if (nframes < 0 || nframes > f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: %d frames do not fit (%d)", who, nframes, f->n);
  return pair_args_ok(ctx, f, 0, nframes > 0 ? nframes - 1 : 0, cfg, out);
}

int sfmgpu_pair_frontend_host(sfmgpu_ctx* ctx, sfmgpu_frames* f, const uint8_t* host_pix, int nframes, const sfmgpu_lkcfg* cfg,
                              sfmgpu_pairs* out, int chunk_frames, double* li_xy, double* lj_xy, int32_t* n_kept,
                              int32_t* n_corners) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out || !host_pix) return SFMGPU_E_ARG;
  SFM_TRY(host_args_ok(ctx, f, nframes, cfg, out, "pair_frontend_host"));
  RawFill src;
  src.pix = host_pix;
  return host_stream(ctx, f, nframes, host_chunk(f, nframes, chunk_frames), cfg, out, src, li_xy, lj_xy, n_kept, n_corners);
}

int sfmgpu_pair_frontend_host_packed(sfmgpu_ctx* ctx, sfmgpu_frames* f, const uint8_t* blob, size_t blob_bytes, int blob_first,
                                     int nframes, const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out, int chunk_frames, double* li_xy,
                                     double* lj_xy, int32_t* n_kept, int32_t* n_corners) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out) return SFMGPU_E_ARG;
  const char* who = "pair_frontend_host_packed";
  SFM_TRY(host_args_ok(ctx, f, nframes, cfg, out, who));
  std::vector<uint64_t> fo;
  SFM_TRY(sfm_pk_check(ctx, f, blob, blob_bytes, blob_first, nframes, fo, who));
  const int chunk = host_chunk(f, nframes, chunk_frames);
  if (nframes > 0) SFM_TRY(sfm_pk_prepare(ctx, blob, blob_first, fo, sfm_pk_max_chunk_bytes(fo, chunk), 2));
  PackedFill src;
  src.blob = blob;
  src.fo = &fo;
  src.d_fo = (const unsigned long long*)ctx->pk_fo.p;
  SFM_TRY(host_stream(ctx, f, nframes, chunk, cfg, out, src, li_xy, lj_xy, n_kept, n_corners));
  return nframes > 0 ? sfm_pk_read_flag(ctx, who) : 0;
}

int sfmgpu_pairs_totals(sfmgpu_ctx* ctx, sfmgpu_pairs* p, long long* n_corners, long long* n_kept, long long* n_lk_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !p) return SFMGPU_E_ARG;
  unsigned long long t[4];
  SFM_CUDA(ctx, cudaMemcpyAsync(t, p->totals, sizeof t, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_corners) *n_corners = (long long)t[0];
  if (n_kept) *n_kept = (long long)t[1];
  if (n_lk_iters) *n_lk_iters = (long long)t[2];
  if (t[3])
    return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pair_frontend: %llu frame(s) exceeded the candidate capacity", t[3]);
  return 0;
}

int sfmgpu_pairs_download_all(sfmgpu_ctx* ctx, sfmgpu_pairs* p, double* li_xy, double* lj_xy, int32_t* n_kept,
                              int32_t* n_corners) {
  SFM_ENTER(ctx);
  if (!ctx || !p) return SFMGPU_E_ARG;
  const size_t np_ = (size_t)p->last_npairs;
  if (np_ == 0) return 0;
  if (li_xy) SFM_CUDA(ctx, cudaMemcpyAsync(li_xy, p->li, np_ * p->cap * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (lj_xy) SFM_CUDA(ctx, cudaMemcpyAsync(lj_xy, p->lj, np_ * p->cap * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (n_kept) SFM_CUDA(ctx, cudaMemcpyAsync(n_kept, p->nkept, np_ * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (n_corners) SFM_CUDA(ctx, cudaMemcpyAsync(n_corners, p->ncorn, np_ * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

int sfmgpu_pairs_set_matches(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int npairs, const double* li_xy, const double* lj_xy,
                             const int32_t* n_kept) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !n_kept || (npairs > 0 && (!li_xy || !lj_xy))) return SFMGPU_E_ARG;
  if (npairs < 0 || npairs > p->max_pairs) return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_set_matches: %d pairs, room for %d", npairs, p->max_pairs);
  for (int k = 0; k < npairs; k++)
    if (n_kept[k] < 0 || n_kept[k] > p->cap)
      return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_set_matches: pair %d has %d matches, room for %d", k, n_kept[k], p->cap);
  const size_t n = (size_t)npairs * p->cap;
  if (npairs > 0) {
    SFM_CUDA(ctx, cudaMemcpyAsync(p->li, li_xy, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(p->lj, lj_xy, n * 16, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(p->nkept, n_kept, (size_t)npairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(p->ncorn, n_kept, (size_t)npairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the caller's arrays may be pageable / reused
  }
  p->last_npairs = npairs;
  p->ids_valid = false;
  return 0;
}

int sfmgpu_pairs_device_ptrs(sfmgpu_pairs* p, void** li_xy, void** lj_xy, void** n_kept, void** n_corners) {
  if (!p) return SFMGPU_E_ARG;
  if (li_xy) *li_xy = p->li;
  if (lj_xy) *lj_xy = p->lj;
  if (n_kept) *n_kept = p->nkept;
  if (n_corners) *n_corners = p->ncorn;
  return 0;
}

int sfmgpu_pairs_ids_device_ptr(sfmgpu_pairs* p, void** ids) {
  if (!p || !ids) return SFMGPU_E_ARG;
  if (!p->ids_valid) return SFMGPU_E_STATE;
  *ids = p->ids;
  return 0;
}

int sfmgpu_pairs_ids_download_all(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int32_t* ids) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !ids) return SFMGPU_E_ARG;
  if (!p->ids_valid) return sfm_fail(ctx, SFMGPU_E_STATE, "pairs_ids_download_all: the last batch carries no track ids (not a segment call)");
  const size_t np_ = (size_t)p->last_npairs;
  if (np_ == 0) return 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(ids, p->ids, np_ * p->cap * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

int sfmgpu_pairs_download(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int pair, double* li_xy, double* lj_xy, int cap, int* n_kept,
                          int* n_corners) {
  SFM_ENTER(ctx);
  if (!ctx || !p || pair < 0 || pair >= p->last_npairs) return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_download: bad pair index");
  int nk = 0, nc = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&nk, p->nkept + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(&nc, p->ncorn + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (nc < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pairs_download: pair %d exceeded the candidate capacity", pair);
  if (n_kept) *n_kept = nk;
  if (n_corners) *n_corners = nc;
  if (nk > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pairs_download: %d survivors, room for %d", nk, cap);
  if (nk > 0) {
    if (li_xy) SFM_CUDA(ctx, cudaMemcpyAsync(li_xy, p->li + (size_t)pair * p->cap, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (lj_xy) SFM_CUDA(ctx, cudaMemcpyAsync(lj_xy, p->lj + (size_t)pair * p->cap, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

}  // extern "C"

// ---- track lists: the state and the operations of KLTTracker (:323-391) ------------------------------------------------------
// Both tracker objects run on this one core: sfmgpu_tracker holds one track list, sfmgpu_multitracker S lists that are stepped
// together.  What differs between them is where the frames come from, how the KLT launch is sized, and what is downloaded.
namespace {

// S track lists of `rows` entries, list s at entry s * rows, with the device scratch of their steps.
struct TrackLists {
  int S = 0, rows = 0, fresh_cap = 0;
  double2 *trk = nullptr, *p1 = nullptr, *pb = nullptr, *oa = nullptr, *ob = nullptr, *fresh = nullptr;
  int *ids = nullptr, *oid = nullptr, *nit = nullptr;
  int *dn = nullptr, *dnk = nullptr;  // per list: tracks entering the last step (KLT_BY_ROWS), its survivors
  int* rst = nullptr;                 // a reset's per-list corner counts [S] and first ids [S]
  int* scal = nullptr;                // a replenishment's [1] n_fresh, [2] n_added
  uint8_t *keep = nullptr, *ok = nullptr;
  unsigned long long* tot = nullptr;  // totals_kernel's sums over all steps ([2]: LK iterations)
  std::vector<int> n, next_id;        // host: live tracks and the next id of every list
  long long track_steps = 0;
};

int lkcfg_ok(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, const char* who) {
  if (cfg->pyr_levels < 1 || cfg->pyr_levels > SFM_MAXL || cfg->max_tracks > (1 << 24) || cfg->min_tracks > (1 << 24))
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: bad configuration", who);
  return 0;
}

cudaError_t lists_alloc(sfmgpu_ctx* ctx, TrackLists& L, const sfmgpu_lkcfg& cfg, int S) {
  L.S = S;
  L.rows = track_rows(cfg);
  L.fresh_cap = 3 * (cfg.max_tracks < 1 ? 1 : cfg.max_tracks);
  L.n.assign(S, 0);
  L.next_id.assign(S, 0);
  cudaError_t e = cudaSuccess;
  auto al = [&](void** q, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(q, bytes + 256);
  };
  const size_t n = (size_t)L.rows * S;
  al((void**)&L.trk, n * 16);
  al((void**)&L.p1, n * 16);
  al((void**)&L.pb, n * 16);
  al((void**)&L.oa, n * 16);
  al((void**)&L.ob, n * 16);
  al((void**)&L.ids, n * 4);
  al((void**)&L.oid, n * 4);
  al((void**)&L.nit, n * 4);
  al((void**)&L.keep, n);
  al((void**)&L.fresh, (size_t)L.fresh_cap * 16 * S);
  al((void**)&L.ok, (size_t)L.fresh_cap);
  al((void**)&L.dn, (size_t)S * 4);
  al((void**)&L.dnk, (size_t)S * 4);
  al((void**)&L.rst, (size_t)S * 8);
  al((void**)&L.scal, 64);
  al((void**)&L.tot, 64);
  if (e == cudaSuccess) e = cudaMemsetAsync(L.tot, 0, 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(L.scal, 0, 64, ctx->stream);
  return e;
}

void lists_free(TrackLists& L) {
  void* ptrs[] = {L.trk, L.p1, L.pb, L.oa, L.ob, L.fresh, L.ids, L.oid, L.nit, L.dn, L.dnk, L.rst, L.scal, L.keep, L.ok, L.tot};
  for (void* q : ptrs)
    if (q) cudaFree(q);
}

// reset(gray) (:327-332) of lists [s0, s0 + count) on frames first + s0, ...: list s = the first corners of its frame
// (shi_tomasi(gray, max_tracks, ...)) with ids next_id[s]++.  Synchronises the context stream.
int lists_reset(sfmgpu_ctx* ctx, TrackLists& L, const sfmgpu_lkcfg& cfg, sfmgpu_frames* f, int first, int s0, int count,
                const char* who) {
  const int stride = cfg.max_tracks < 1 ? 1 : cfg.max_tracks;
  int *d_n = L.rst + s0, *d_id = L.rst + L.S + s0;
  SFM_TRY(detect_full(ctx, cfg, f, first + s0, count, cfg.max_tracks, L.fresh, d_n));
  std::vector<int> n(count);
  SFM_CUDA(ctx, cudaMemcpyAsync(n.data(), d_n, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(d_id, L.next_id.data() + s0, (size_t)count * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int j = 0; j < count; j++)
    if (n[j] < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "%s: candidate capacity exceeded (sequence %d)", who, s0 + j);
  SFM_LAUNCH(ctx, take_corners_kernel, dim3(sfm_cdiv(stride, 256), count), 256, 0, (const double2*)L.fresh, stride, (const int*)d_n,
             (const int*)d_id, L.trk + (size_t)s0 * L.rows, L.ids + (size_t)s0 * L.rows, L.rows);
  for (int j = 0; j < count; j++) {
    L.n[s0 + j] = n[j];
    L.next_id[s0 + j] += n[j];
  }
  return 0;
}

// How a step's launches are sized.  sfm_klt_launch picks the kernel family from npairs * cap, and the two families agree to
// within 1e-6 px, not bit for bit, so each tracker keeps its own rule: the single tracker by its live tracks, the lock-step
// tracker by all S x rows entries with the live counts uploaded to dn.
enum KltSizing { KLT_BY_LIVE, KLT_BY_ROWS };

// One step of every list from frame fa0 + s of fa to frame fb0 + s of fb (:346-371): the survivors of list s in track order,
// (p0, p1, id), go to row s of oa / ob / oid and their count to dnk[s]; the step's sums are added to tot.  fa != fb (the single
// tracker across an image-size change) runs the two-geometry KLT kernel.  geo != nullptr (the lock-step tracker over sequences of
// different sizes): list s reads its two images from geo[s], fa only gives the level count.
int lists_track(sfmgpu_ctx* ctx, TrackLists& L, const sfmgpu_lkcfg& cfg, sfmgpu_frames* fa, sfmgpu_frames* fb, int fa0, int fb0,
                KltSizing sizing, const KltGeo* geo = nullptr) {
  KltLaunch k;
  k.pv = fa->view();
  k.pvb = fb->view();
  k.geo = geo;
  k.p0 = L.trk;
  if (sizing == KLT_BY_LIVE) {  // one list
    k.counts = nullptr;
    k.npairs = 1;
    k.cap = L.n[0];
  } else {
    SFM_CUDA(ctx, cudaMemcpyAsync(L.dn, L.n.data(), (size_t)L.S * 4, cudaMemcpyHostToDevice, ctx->stream));
    k.counts = L.dn;
    k.npairs = L.S;
    k.cap = L.rows;
  }
  k.fa0 = fa0;
  k.fa_step = 1;
  k.fb0 = fb0;
  k.fb_step = 1;
  k.radius = cfg.win_radius;
  k.iters = cfg.iters;
  k.fb_thresh = cfg.fb_thresh;
  k.p1 = L.p1;
  k.pb = L.pb;
  k.nit = L.nit;
  k.keep = L.keep;
  {
    StageTimer st(ctx, 2);
    SFM_TRY(sfm_klt_launch(ctx, k));
  }
  for (int s = 0; s < L.S; s++) L.track_steps += L.n[s];
  SFM_LAUNCH(ctx, compact_kernel, L.S, 1024, 0, L.trk, L.p1, L.keep, (const int*)L.ids, k.counts, k.cap, L.oa, L.ob, L.oid, L.dnk);
  const unsigned tb = sfm_cdiv((long long)k.npairs * k.cap, 256);  // no more blocks (and atomics) than entries
  SFM_LAUNCH(ctx, totals_kernel, tb < 64 ? tb : 64, 256, 0, k.counts, (const int*)L.dnk, (const int*)L.nit, L.S, k.cap, L.tot);
  return 0;
}

// tracks_ = kept (:371): the first `entries` entries of the survivor rows become the track lists (the caller sets n).
// Synchronises the context stream, so downloads queued before it have landed when it returns.
int lists_commit(sfmgpu_ctx* ctx, TrackLists& L, size_t entries) {
  if (entries == 0) return 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(L.trk, L.ob, entries * 16, cudaMemcpyDeviceToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(L.ids, L.oid, entries * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

// Replenish list s (:374-389): detect need*3 corners on its current frame, drop those within min_distance of a live track,
// append survivors with consecutive ids until max_tracks (tested after the append: at least one is added).
int replenish_row(sfmgpu_ctx* ctx, TrackLists& L, const sfmgpu_lkcfg& cfg, sfmgpu_frames* f, int frame, int s) {
  int &n = L.n[s], &next_id = L.next_id[s];
  double2* trk = L.trk + (size_t)s * L.rows;
  const int need = cfg.max_tracks - n;
  long long want = (long long)need * 3;
  if (want > L.fresh_cap) want = L.fresh_cap;  // fresh_cap = 3*max_tracks >= need*3
  SFM_TRY(detect_full(ctx, cfg, f, frame, 1, (int)want, L.fresh, L.scal + 1));
  int nf = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&nf, L.scal + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (nf < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker: candidate capacity exceeded");
  if (nf > 0) {
    const double d2 = (double)cfg.min_distance * cfg.min_distance;
    SFM_LAUNCH(ctx, replenish_filter_kernel, sfm_cdiv(nf, 256), 256, 0, L.fresh, (const int*)(L.scal + 1), trk, n, d2, L.ok);
    // the reference appends first and tests the cap afterwards (:386-387): at least one corner is added
    int room = cfg.max_tracks - n;
    if (room < 1) room = 1;
    if (n + room > L.rows)  // cannot happen with rows sized by track_rows(); never write past the row
      return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker: track list of %d + %d exceeds its %d rows", n, room, L.rows);
    SFM_LAUNCH(ctx, replenish_append_kernel, 1, 1024, 0, L.fresh, (const int*)(L.scal + 1), L.ok, trk, L.ids + (size_t)s * L.rows, n,
               room, next_id, L.scal + 2);
    int na = 0;
    SFM_CUDA(ctx, cudaMemcpyAsync(&na, L.scal + 2, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    n += na;
    next_id += na;
  }
  return 0;
}

// After a commit, list by list on its current frame (where(s, &batch, &index)): a list that entered the step without tracks
// (empty[s]; empty == nullptr: none did) is reset on its frame instead of stepped (:341-344), one frame at a time; a list below
// min_tracks is replenished.
template <class Where>
int lists_refill(sfmgpu_ctx* ctx, TrackLists& L, const sfmgpu_lkcfg& cfg, Where where, const std::vector<char>* empty, const char* who) {
  for (int s = 0; s < L.S; s++) {
    sfmgpu_frames* f = nullptr;
    int frame = 0;
    where(s, &f, &frame);
    if (empty && (*empty)[s])
      SFM_TRY(lists_reset(ctx, L, cfg, f, frame - s, s, 1, who));
    else if (L.n[s] < cfg.min_tracks)
      SFM_TRY(replenish_row(ctx, L, cfg, f, frame, s));
  }
  return 0;
}

// tracks() of list s: its first n entries into the caller's cap.
int lists_tracks(sfmgpu_ctx* ctx, const TrackLists& L, int s, double* xy, int32_t* ids, int cap, int* n_out, const char* who) {
  const int n = L.n[s];
  if (n_out) *n_out = n;
  if (n > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "%s: %d tracks, room for %d", who, n, cap);
  if (n > 0) {
    if (xy) SFM_CUDA(ctx, cudaMemcpyAsync(xy, L.trk + (size_t)s * L.rows, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, L.ids + (size_t)s * L.rows, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

int lists_totals(sfmgpu_ctx* ctx, const TrackLists& L, long long* n_track_steps, long long* n_lk_iters) {
  unsigned long long tt[4];
  SFM_CUDA(ctx, cudaMemcpyAsync(tt, L.tot, sizeof tt, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_track_steps) *n_track_steps = L.track_steps;
  if (n_lk_iters) *n_lk_iters = (long long)tt[2];
  return 0;
}

}  // namespace

// ---- stateful tracker: one track list; its frames are read in place from the caller's batch ---------------------------------
struct sfmgpu_tracker {
  sfmgpu_lkcfg cfg;
  sfmgpu_frames* own = nullptr;     // 2-slot ping-pong used by the host-image entry points
  sfmgpu_frames* prev_frames = nullptr;
  int prev_index = -1;
  bool size_change = false;         // host images of a new size: followed (sfmgpu_tracker_set_size_change) or refused
  TrackLists L;                     // S = 1
};

namespace {

int tracker_reset_on(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame) {
  SFM_TRY(lists_reset(ctx, t->L, t->cfg, f, frame, 0, 1, "tracker"));
  t->prev_frames = f;
  t->prev_index = frame;
  return 0;
}

// Steps from the previous frame, which must live in fprev, to frame `frame` of f: fprev == f except across an image-size change
// of the host-image entry points, where fprev is the tracker's old batch and f its new one.
int tracker_step_on(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* fprev, sfmgpu_frames* f, int frame, double* prev_xy,
                    double* cur_xy, int32_t* ids, int cap, int* n_out) {
  TrackLists& L = t->L;
  if (n_out) *n_out = 0;
  if (t->prev_index < 0 || L.n[0] == 0) return tracker_reset_on(ctx, t, f, frame);  // :341-344
  if (t->prev_frames != fprev) return sfm_fail(ctx, SFMGPU_E_STATE, "tracker: previous frame lives in another frame batch");
  SFM_TRY(lists_track(ctx, L, t->cfg, fprev, f, t->prev_index, frame, KLT_BY_LIVE));
  int nk = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&nk, L.dnk, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (nk > cap && (prev_xy || cur_xy || ids))
    return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker_step: %d survivors, room for %d", nk, cap);
  if (nk > 0) {
    if (prev_xy) SFM_CUDA(ctx, cudaMemcpyAsync(prev_xy, L.oa, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (cur_xy) SFM_CUDA(ctx, cudaMemcpyAsync(cur_xy, L.ob, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, L.oid, (size_t)nk * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  // the header's promise: results are in the caller's (possibly pinned) buffers when the call returns
  SFM_TRY(lists_commit(ctx, L, (size_t)nk));
  L.n[0] = nk;
  t->prev_frames = f;
  t->prev_index = frame;
  if (n_out) *n_out = nk;
  auto where = [&](int, sfmgpu_frames** wf, int* wi) {
    *wf = f;
    *wi = frame;
  };
  return lists_refill(ctx, L, t->cfg, where, nullptr, "tracker");
}

// A host image of the tracker's size goes to the slot of its 2-slot batch that does not hold the previous frame.
int tracker_own_slot(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h, int* slot) {
  if (!t->own) SFM_TRY(sfmgpu_frames_create(ctx, w, h, 2, t->cfg.pyr_levels, &t->own));
  *slot = (t->prev_frames == t->own && t->prev_index == 0) ? 1 : 0;
  SFM_TRY(sfmgpu_frames_upload(ctx, t->own, *slot, 1, host_pix));
  return sfmgpu_pyramid_build(ctx, t->own, *slot, 1);
}

// A host image of another size (:345-346 build the two pyramids at their own sizes): it goes to slot 0 of a new 2-slot batch,
// the tracker resets or steps onto it (the step tracks from the old batch), and the new batch replaces the old one once it
// holds the previous frame.  So no more than two batches are alive, and a call that fails before the step commits keeps the
// tracker on its old batch.
int tracker_resized(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h, bool reset, double* prev_xy,
                    double* cur_xy, int32_t* ids, int cap, int* n_out) {
  if (!t->size_change)
    return sfm_fail(ctx, SFMGPU_E_ARG, "tracker: image size changed from %dx%d to %dx%d (sfmgpu_tracker_set_size_change not set)",
                    t->own->w, t->own->h, w, h);
  sfmgpu_frames* nb = nullptr;
  SFM_TRY(sfmgpu_frames_create(ctx, w, h, 2, t->cfg.pyr_levels, &nb));
  int r = sfmgpu_frames_upload(ctx, nb, 0, 1, host_pix);
  if (r == 0) r = sfmgpu_pyramid_build(ctx, nb, 0, 1);
  if (r == 0)
    r = reset ? tracker_reset_on(ctx, t, nb, 0) : tracker_step_on(ctx, t, t->own, nb, 0, prev_xy, cur_xy, ids, cap, n_out);
  if (t->prev_frames == nb) std::swap(t->own, nb);
  sfmgpu_frames_destroy(ctx, nb);  // synchronises the context stream first
  return r;
}

}  // namespace

extern "C" {

int sfmgpu_tracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, sfmgpu_tracker** out) {
  SFM_ENTER(ctx);
  if (!ctx || !cfg || !out) return SFMGPU_E_ARG;
  SFM_TRY(lkcfg_ok(ctx, cfg, "tracker_create"));
  sfmgpu_tracker* t = new sfmgpu_tracker();
  t->cfg = *cfg;
  const cudaError_t e = lists_alloc(ctx, t->L, *cfg, 1);
  if (e != cudaSuccess) {
    sfmgpu_tracker_destroy(ctx, t);
    return sfm_fail(ctx, SFMGPU_E_CUDA, "tracker_create: CUDA allocation failed: %s", cudaGetErrorString(e));
  }
  *out = t;
  return 0;
}

void sfmgpu_tracker_destroy(sfmgpu_ctx* ctx, sfmgpu_tracker* t) {
  SFM_ENTER_VOID(ctx);
  if (!t) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  lists_free(t->L);
  if (t->own) sfmgpu_frames_destroy(ctx, t->own);
  delete t;
}

int sfmgpu_tracker_set_size_change(sfmgpu_ctx* ctx, sfmgpu_tracker* t, int follow) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (follow != 0 && follow != 1) return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_set_size_change: %d not in {0,1}", follow);
  t->size_change = follow == 1;
  return 0;
}

int sfmgpu_tracker_reset(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !host_pix) return SFMGPU_E_ARG;
  if (t->own && (t->own->w != w || t->own->h != h))
    return tracker_resized(ctx, t, host_pix, w, h, true, nullptr, nullptr, nullptr, 0, nullptr);
  int slot = 0;
  SFM_TRY(tracker_own_slot(ctx, t, host_pix, w, h, &slot));
  return tracker_reset_on(ctx, t, t->own, slot);
}

int sfmgpu_tracker_step(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h, double* prev_xy,
                        double* cur_xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !host_pix) return SFMGPU_E_ARG;
  if (t->own && (t->own->w != w || t->own->h != h))
    return tracker_resized(ctx, t, host_pix, w, h, false, prev_xy, cur_xy, ids, cap, n_out);
  int slot = 0;
  SFM_TRY(tracker_own_slot(ctx, t, host_pix, w, h, &slot));
  return tracker_step_on(ctx, t, t->own, t->own, slot, prev_xy, cur_xy, ids, cap, n_out);
}

int sfmgpu_tracker_step_frames(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame, double* prev_xy,
                               double* cur_xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !f) return SFMGPU_E_ARG;
  if (frame < 0 || frame >= f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_step_frames: bad frame index");
  if (f->levels != t->cfg.pyr_levels) return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_step_frames: pyramid levels differ from cfg");
  return tracker_step_on(ctx, t, f, f, frame, prev_xy, cur_xy, ids, cap, n_out);
}

int sfmgpu_tracker_tracks(sfmgpu_ctx* ctx, sfmgpu_tracker* t, double* xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  return lists_tracks(ctx, t->L, 0, xy, ids, cap, n_out, "tracker_tracks");
}

int sfmgpu_tracker_totals(sfmgpu_ctx* ctx, sfmgpu_tracker* t, long long* n_track_steps, long long* n_lk_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  return lists_totals(ctx, t->L, n_track_steps, n_lk_iters);
}

}  // extern "C"

// ---- lock-step tracker over S independent sequences (BASELINE.json C5: several sequences per GPU) -------------------------------
// The same KLTTracker semantics per sequence (:323-391) on the same track-list core, but ONE batched launch per stage and step for
// all of them: frame t of every sequence arrives together, the S x max_tracks feature-tracks share a KLT launch (large enough
// for the lane-per-feature kernels), survivors are compacted per sequence.  Results are identical to S separate sfmgpu_tracker
// objects.  Resets after a total track loss and replenishment (rare) run list by list.
//
// Sequences may have different image sizes (sfmgpu_multitracker_create_sized).  The sequences of one size form a size class with
// its own frame batch; the KLT chain still runs once over all S lists, reading every list's images through a per-list geometry
// table, and everything after it (compaction, totals, commit, the RANSAC stage) works on the [S][ROWS] lists as before.
struct sfmgpu_multitracker {
  sfmgpu_lkcfg cfg;
  int w = 0, h = 0;                 // class 0's size (every sequence's, unless the tracker is mixed)
  sfmgpu_frames* frames = nullptr;  // class 0's batch
  // Size class: 3*n slots, group g of its i-th sequence in slot g*n + i (previous / current / prefetched).  With one class,
  // sequence s is its s-th: group g of sequence s lives in slot g*S + s.
  struct SizeClass {
    int w, h, n;
    sfmgpu_frames* frames;
    size_t pk_bound;  // the largest packed record of a w x h frame (sfm_pk_frame_bound)
  };
  // Adjacent sequences of one class: one upload.  host_off: where sequence s0's frame starts in the caller's S frames.
  struct Run {
    int s0, count, cls, i0;
    size_t host_off;
  };
  std::vector<SizeClass> cls;
  std::vector<Run> runs;
  std::vector<int> cls_of, idx_in;  // per sequence: its class and its index in that class
  KltGeo* geo = nullptr;            // mixed: [3][S] geometry tables, steps from group g to group (g+1)%3 read entries g*S ...
  PkDst* pkdst = nullptr;           // mixed: [3][S] packed-decode destinations, group g of sequence s at g*S + s
  int pk_tiles = 0;                 // mixed: the largest tile count of a sequence's frame
  bool mixed() const { return cls.size() > 1; }
  int parity = -1;                  // slot group of the previous frames, -1: nothing tracked yet
  bool prefetched = false;          // group (parity+1)%3 holds the next frames (uploaded + pyramids), ready at pf_done
  cudaEvent_t pf_done = nullptr;
  TrackLists L;                     // list s: sequence s
  FrameCopy* gtab = nullptr;        // resident input: the gather's (sequence, level) table, [S][levels] entries at most
  TwoViewState* tv = nullptr;       // find_E_ransac on every sequence's survivors inside the step (sfmgpu_multitracker_set_ransac)
  bool tv_fresh = false;            // the last step ran the stage: its results can be downloaded
  // packed input (sfmgpu_multitracker_step_packed): the tracker's own device buffer [decode flag | staged frame offsets [S+1] |
  // S frame records back to back, sum over s of the bound of a w[s] x h[s] record], allocated by the first packed call, so that
  // no other call on the context can overwrite a pending prefetch.  pk_done follows the last decode that read the staging;
  // pk_bad receives the flag.
  uint8_t* pk = nullptr;
  int* pk_bad = nullptr;            // page-locked host copy of the decode flag
  cudaEvent_t pk_done = nullptr;
  bool pk_used = false;             // pk_done has been recorded
  bool pf_packed = false;           // the prefetched frames were decoded: their flag is checked before they are stepped
};

extern "C" {

}  // extern "C"

// Per-list geometry of the KLT launches of a mixed tracker: table g, entry s = sequence s from group g to group (g+1)%3.
static std::vector<KltGeo> multi_geo_tables(const sfmgpu_multitracker* t) {
  const int S = t->L.S;
  std::vector<KltGeo> geo((size_t)3 * S);
  for (int g = 0; g < 3; g++)
    for (int s = 0; s < S; s++) {
      const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
      const sfmgpu_frames* f = c.frames;
      const size_t sa = (size_t)g * c.n + t->idx_in[s], sb = (size_t)((g + 1) % 3) * c.n + t->idx_in[s];
      KltGeo& e = geo[(size_t)g * S + s];
      for (int l = 0; l < SFM_MAXL; l++) {
        const bool in = l < f->levels;
        e.lv[l].a = in ? f->lvl[l] + sa * f->fstride[l] : nullptr;
        e.lv[l].b = in ? f->lvl[l] + sb * f->fstride[l] : nullptr;
        e.lv[l].w = in ? f->lw[l] : 0;
        e.lv[l].h = in ? f->lh[l] : 0;
        e.lv[l].pitch = in ? f->pitch[l] : 0;
        e.lv[l].pad = 0;
      }
    }
  return geo;
}

// Sequence s has images of w[s] x h[s] (checked by the caller).
static int multi_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, int S, const int32_t* w, const int32_t* h, sfmgpu_multitracker** out,
                        const char* who) {
  SFM_TRY(lkcfg_ok(ctx, cfg, who));
  sfmgpu_multitracker* t = new sfmgpu_multitracker();
  t->cfg = *cfg;
  t->cls_of.resize(S);
  t->idx_in.resize(S);
  size_t off = 0;
  for (int s = 0; s < S; s++) {
    int c = 0;
    while (c < (int)t->cls.size() && (t->cls[c].w != w[s] || t->cls[c].h != h[s])) c++;
    if (c == (int)t->cls.size()) t->cls.push_back({w[s], h[s], 0, nullptr, sfm_pk_frame_bound(w[s], h[s])});
    t->cls_of[s] = c;
    t->idx_in[s] = t->cls[c].n++;
    if (s > 0 && t->cls_of[s - 1] == c)
      t->runs.back().count++;
    else
      t->runs.push_back({s, 1, c, t->idx_in[s], off});
    off += (size_t)w[s] * h[s];
  }
  for (sfmgpu_multitracker::SizeClass& c : t->cls) {
    const int rc = sfmgpu_frames_create(ctx, c.w, c.h, 3 * c.n, cfg->pyr_levels, &c.frames);
    if (rc != 0) {
      sfmgpu_multitracker_destroy(ctx, t);
      return rc;
    }
  }
  t->frames = t->cls[0].frames;
  t->w = t->cls[0].w;
  t->h = t->cls[0].h;
  cudaError_t e = lists_alloc(ctx, t->L, *cfg, S);
  if (e == cudaSuccess) e = cudaMalloc((void**)&t->gtab, (size_t)S * SFM_MAXL * sizeof(FrameCopy));
  if (e == cudaSuccess && t->mixed()) {
    const std::vector<KltGeo> geo = multi_geo_tables(t);
    e = cudaMalloc((void**)&t->geo, geo.size() * sizeof(KltGeo));
    if (e == cudaSuccess) e = cudaMemcpy(t->geo, geo.data(), geo.size() * sizeof(KltGeo), cudaMemcpyHostToDevice);
    // packed input: level 0 of group g of sequence s, decoded by one launch over all S frames of a step
    std::vector<PkDst> dst((size_t)3 * S);
    for (int g = 0; g < 3; g++)
      for (int s = 0; s < S; s++) {
        const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
        dst[(size_t)g * S + s] = sfm_pk_dst(c.frames, g * c.n + t->idx_in[s]);
        if (dst[(size_t)g * S + s].ntiles > t->pk_tiles) t->pk_tiles = dst[(size_t)g * S + s].ntiles;
      }
    if (e == cudaSuccess) e = cudaMalloc((void**)&t->pkdst, dst.size() * sizeof(PkDst));
    if (e == cudaSuccess) e = cudaMemcpy(t->pkdst, dst.data(), dst.size() * sizeof(PkDst), cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) {
    sfmgpu_multitracker_destroy(ctx, t);
    return sfm_fail(ctx, SFMGPU_E_CUDA, "%s: CUDA allocation failed: %s", who, cudaGetErrorString(e));
  }
  *out = t;
  return 0;
}

extern "C" {

int sfmgpu_multitracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, int n_sequences, int w, int h, sfmgpu_multitracker** out) {
  SFM_ENTER(ctx);
  if (!ctx || !cfg || !out) return SFMGPU_E_ARG;
  if (n_sequences < 1 || n_sequences > 512 || w < 1 || h < 1) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_create: bad configuration");
  const std::vector<int32_t> ws(n_sequences, w), hs(n_sequences, h);
  return multi_create(ctx, cfg, n_sequences, ws.data(), hs.data(), out, "multitracker_create");
}

int sfmgpu_multitracker_create_sized(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, int n_sequences, const int32_t* w, const int32_t* h,
                                     sfmgpu_multitracker** out) {
  SFM_ENTER(ctx);
  const char* who = "multitracker_create_sized";
  if (!ctx || !cfg || !out) return SFMGPU_E_ARG;
  if (!w || !h) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null size array", who);
  if (n_sequences < 1 || n_sequences > 512) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: %d sequences, not in [1, 512]", who, n_sequences);
  for (int s = 0; s < n_sequences; s++)
    if (w[s] < 1 || w[s] > 32767 || h[s] < 1 || h[s] > 32767)
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequence %d is %d x %d, sizes must lie in [1, 32767]", who, s, w[s], h[s]);
  return multi_create(ctx, cfg, n_sequences, w, h, out, who);
}

void sfmgpu_multitracker_destroy(sfmgpu_ctx* ctx, sfmgpu_multitracker* t) {
  SFM_ENTER_VOID(ctx);
  if (!t) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  if (t->pf_done) cudaEventSynchronize(t->pf_done);  // a prefetch still running on the copy stream
  sfm_two_view_free(ctx, &t->tv);
  lists_free(t->L);
  if (t->gtab) cudaFree(t->gtab);
  if (t->geo) cudaFree(t->geo);
  if (t->pkdst) cudaFree(t->pkdst);
  for (sfmgpu_multitracker::SizeClass& c : t->cls)
    if (c.frames) sfmgpu_frames_destroy(ctx, c.frames);
  if (t->pk) cudaFree(t->pk);
  if (t->pk_bad) cudaFreeHost(t->pk_bad);
  if (t->pf_done) cudaEventDestroy(t->pf_done);
  if (t->pk_done) cudaEventDestroy(t->pk_done);
  delete t;
}

// Slot group of the next step's frames.
static int multi_next_group(const sfmgpu_multitracker* t) { return t->parity < 0 ? 0 : (t->parity + 1) % 3; }
static int multi_step_on(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int par, double* prev_xy, double* cur_xy, int32_t* ids, int32_t* n_out);

// The pyramids of slot group g (level 0 written), one build per size class, on ctx->stream.
static int multi_pyramids(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int g) {
  for (const sfmgpu_multitracker::SizeClass& c : t->cls) SFM_TRY(sfmgpu_pyramid_build(ctx, c.frames, g * c.n, c.n));
  return 0;
}

// The S frames of one step (back to back in sequence order, frame s of w[s] x h[s] bytes) into slot group g, one copy per run of
// adjacent sequences of one size, then the pyramids, on ctx->stream.
static int multi_upload(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int g, const uint8_t* host_pix) {
  for (const sfmgpu_multitracker::Run& r : t->runs) {
    const sfmgpu_multitracker::SizeClass& c = t->cls[r.cls];
    SFM_TRY(sfmgpu_frames_upload(ctx, c.frames, g * c.n + r.i0, r.count, host_pix + r.host_off));
  }
  return multi_pyramids(ctx, t, g);
}

// Upload + pyramids of the frames of a LATER step on the copy stream, into the slot group after `after_group`.
static int multi_prefetch(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int after_group, const uint8_t* host_pix) {
  SFM_TRY(pipe_streams(ctx));
  if (!t->pf_done && cudaEventCreateWithFlags(&t->pf_done, cudaEventDisableTiming) != cudaSuccess)
    return sfm_fail(ctx, SFMGPU_E_CUDA, "multitracker: cudaEventCreate failed");
  const int g = (after_group + 1) % 3;
  {
    StageScope sc(ctx, ctx->copy_stream);
    SFM_TRY(multi_upload(ctx, t, g, host_pix));
    SFM_CUDA(ctx, cudaEventRecord(t->pf_done, ctx->stream));
  }
  t->prefetched = true;
  t->pf_packed = false;
  return 0;
}

// Packed input: blob frame blob_frame[s] of blobs[s] for every sequence s, checked against the frames of sequence s's size.  The
// records are staged back to back in sequence order (fo: their offsets in the staging), with one copy per run of records that
// are adjacent in host memory (a step-major blob: one copy per step).
struct PkPlan {
  struct Copy {
    const uint8_t* src;
    size_t dst, bytes;
  };
  std::vector<unsigned long long> fo;
  std::vector<Copy> copies;
};

static int multi_pk_plan(sfmgpu_ctx* ctx, const sfmgpu_multitracker* t, const uint8_t* const* blobs, const size_t* blob_bytes,
                         const int32_t* blob_frame, PkPlan& p, const char* who) {
  if (!blobs || !blob_bytes) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null blob array", who);
  if (t->mixed()) {  // a blob's header holds one size: one blob read by sequences of two sizes is never valid
    std::unordered_map<const uint8_t*, int> first;  // blob -> the first sequence that reads it
    for (int s = 0; s < t->L.S; s++) {
      if (!blobs[s]) continue;
      const int s0 = first.emplace(blobs[s], s).first->second;
      if (t->cls_of[s0] != t->cls_of[s])
        return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequences %d and %d have different image sizes (%dx%d, %dx%d) but read one blob", who, s0,
                        s, t->cls[t->cls_of[s0]].w, t->cls[t->cls_of[s0]].h, t->cls[t->cls_of[s]].w, t->cls[t->cls_of[s]].h);
    }
  }
  std::vector<uint64_t> fo;
  p.fo.assign(1, 0);
  p.copies.clear();
  for (int s = 0; s < t->L.S; s++) {
    const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
    if (sfm_pk_check(ctx, c.frames, blobs[s], blob_bytes[s], blob_frame[s], 1, fo, who) != 0) {
      const std::string m = ctx->err;
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s (sequence %d, %dx%d)", m.c_str(), s, c.w, c.h);
    }
    const size_t bytes = fo[1] - fo[0];
    if (bytes > c.pk_bound)
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequence %d: frame record of %zu bytes, a %dx%d frame holds at most %zu", who, s, bytes,
                      c.w, c.h, c.pk_bound);
    const uint8_t* src = blobs[s] + fo[0];
    if (!p.copies.empty() && p.copies.back().src + p.copies.back().bytes == src)
      p.copies.back().bytes += bytes;
    else
      p.copies.push_back({src, (size_t)p.fo.back(), bytes});
    p.fo.push_back(p.fo.back() + bytes);
  }
  return 0;
}

// Copy and decode planned records into slot group g on ctx->stream (the caller may scope it to the copy stream); the flag is
// copied to t->pk_bad behind the decode.  The staging is refilled only after the decode that last read it, on any stream.
static int multi_pk_decode(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int g, const PkPlan& p) {
  const int S = t->L.S;
  const size_t o_fo = 16, o_stage = (o_fo + 8 * ((size_t)S + 1) + 15) & ~(size_t)15;
  // each piece on its own: a call after a failed allocation completes what is missing
  if (!t->pk) {
    size_t records = 0;
    for (const sfmgpu_multitracker::SizeClass& c : t->cls) records += (size_t)c.n * c.pk_bound;
    SFM_CUDA(ctx, cudaMalloc(&t->pk, o_stage + records));
  }
  if (!t->pk_bad) SFM_CUDA(ctx, cudaMallocHost(&t->pk_bad, sizeof(int)));
  if (!t->pk_done) SFM_CUDA(ctx, cudaEventCreateWithFlags(&t->pk_done, cudaEventDisableTiming));
  int* d_bad = (int*)t->pk;
  unsigned long long* d_fo = (unsigned long long*)(t->pk + o_fo);
  uint8_t* stage = t->pk + o_stage;
  if (t->pk_used) SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, t->pk_done, 0));
  SFM_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(int), ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(d_fo, p.fo.data(), 8 * p.fo.size(), cudaMemcpyHostToDevice, ctx->stream));
  for (const PkPlan::Copy& c : p.copies)
    SFM_CUDA(ctx, cudaMemcpyAsync(stage + c.dst, c.src, c.bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (t->mixed())  // all S frames in one launch, each into its own size class's slot
    SFM_TRY(sfm_pk_decode_table(ctx, t->pkdst + (size_t)g * S, S, t->pk_tiles, stage, d_fo, d_bad));
  else
    SFM_TRY(sfm_pk_decode(ctx, t->frames, g * S, S, stage, d_fo, 0, d_bad));
  SFM_CUDA(ctx, cudaEventRecord(t->pk_done, ctx->stream));
  t->pk_used = true;
  SFM_CUDA(ctx, cudaMemcpyAsync(t->pk_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  return 0;
}

// multi_prefetch for packed frames: copy, decode and pyramids on the copy stream.
static int multi_prefetch_packed(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int after_group, const PkPlan& p) {
  SFM_TRY(pipe_streams(ctx));
  if (!t->pf_done && cudaEventCreateWithFlags(&t->pf_done, cudaEventDisableTiming) != cudaSuccess)
    return sfm_fail(ctx, SFMGPU_E_CUDA, "multitracker: cudaEventCreate failed");
  const int g = (after_group + 1) % 3;
  {
    StageScope sc(ctx, ctx->copy_stream);
    SFM_TRY(multi_pk_decode(ctx, t, g, p));
    SFM_TRY(multi_pyramids(ctx, t, g));
    SFM_CUDA(ctx, cudaEventRecord(t->pf_done, ctx->stream));
  }
  t->prefetched = true;
  t->pf_packed = true;
  return 0;
}

// Hand the prefetched frames to the step on ctx->stream.  Decoded frames are waited for on the host first: records that do not
// decode fail the call before the step queues anything, and drop the prefetch.
static int multi_take_prefetch(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const char* who) {
  t->prefetched = false;
  if (t->pf_packed) {
    t->pf_packed = false;
    SFM_CUDA(ctx, cudaEventSynchronize(t->pf_done));
    if (*t->pk_bad) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: a tile record of the prefetched frames does not decode", who);
  }
  SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, t->pf_done, 0));
  return 0;
}

// Back to the state after create: the next step resets every sequence again (ids restart at 0).
int sfmgpu_multitracker_reset(sfmgpu_ctx* ctx, sfmgpu_multitracker* t) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->copy_stream) SFM_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  t->parity = -1;
  t->prefetched = false;
  t->pf_packed = false;
  t->tv_fresh = false;
  t->L.n.assign(t->L.S, 0);
  t->L.next_id.assign(t->L.S, 0);
  t->L.track_steps = 0;
  SFM_CUDA(ctx, cudaMemsetAsync(t->L.tot, 0, 64, ctx->stream));
  return 0;
}

int sfmgpu_multitracker_prefetch(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !host_pix) return SFMGPU_E_ARG;
  if (t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_prefetch: the prefetched frames have not been stepped yet");
  return multi_prefetch(ctx, t, t->parity < 0 ? 2 : t->parity, host_pix);
}

int sfmgpu_multitracker_step(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix, double* prev_xy, double* cur_xy,
                             int32_t* ids, int32_t* n_out) {
  SFM_ENTER(ctx);
  return sfmgpu_multitracker_step_pipelined(ctx, t, host_pix, nullptr, prev_xy, cur_xy, ids, n_out);
}

int sfmgpu_multitracker_step_pipelined(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* host_pix, const uint8_t* next_host_pix,
                                       double* prev_xy, double* cur_xy, int32_t* ids, int32_t* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (!host_pix && !t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_step: no frames given and none prefetched");
  if (host_pix && t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_step: frames given but others are prefetched");
  const int par = multi_next_group(t);
  if (!host_pix) SFM_TRY(multi_take_prefetch(ctx, t, "multitracker_step"));
  t->tv_fresh = false;
  if (host_pix) SFM_TRY(multi_upload(ctx, t, par, host_pix));
  // the frames of the NEXT step travel while this one computes (their slot group is neither previous nor current)
  if (next_host_pix) SFM_TRY(multi_prefetch(ctx, t, par, next_host_pix));
  return multi_step_on(ctx, t, par, prev_xy, cur_xy, ids, n_out);
}

int sfmgpu_multitracker_prefetch_packed(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* const* blobs, const size_t* blob_bytes,
                                        const int32_t* blob_frame) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  const char* who = "multitracker_prefetch_packed";
  if (!blob_frame) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null frame index array", who);
  if (t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "%s: the prefetched frames have not been stepped yet", who);
  PkPlan p;
  SFM_TRY(multi_pk_plan(ctx, t, blobs, blob_bytes, blob_frame, p, who));
  return multi_prefetch_packed(ctx, t, t->parity < 0 ? 2 : t->parity, p);
}

int sfmgpu_multitracker_step_packed(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const uint8_t* const* blobs, const size_t* blob_bytes,
                                    const int32_t* blob_frame, const int32_t* next_blob_frame, double* prev_xy, double* cur_xy,
                                    int32_t* ids, int32_t* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  const char* who = "multitracker_step_packed";
  if (!blob_frame && !t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "%s: no frames given and none prefetched", who);
  if (blob_frame && t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "%s: frames given but others are prefetched", who);
  PkPlan cur, next;
  if (blob_frame) SFM_TRY(multi_pk_plan(ctx, t, blobs, blob_bytes, blob_frame, cur, who));
  if (next_blob_frame) SFM_TRY(multi_pk_plan(ctx, t, blobs, blob_bytes, next_blob_frame, next, who));
  const int par = multi_next_group(t);
  if (blob_frame) {  // decoded and checked before the step queues anything; the pyramids only for frames that decoded
    SFM_TRY(multi_pk_decode(ctx, t, par, cur));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*t->pk_bad) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: a tile record of the frames does not decode", who);
    SFM_TRY(multi_pyramids(ctx, t, par));
  } else {
    SFM_TRY(multi_take_prefetch(ctx, t, who));
  }
  t->tv_fresh = false;
  if (next_blob_frame) SFM_TRY(multi_prefetch_packed(ctx, t, par, next));
  return multi_step_on(ctx, t, par, prev_xy, cur_xy, ids, n_out);
}

}  // extern "C"

// Resident frames: the pyramid of frame idx[s] of f[s] (checked by the caller: sequence s's size, the tracker's levels, an index
// inside f[s]) is copied into sequence s's slot of the current group by one launch over a (sequence, level) table, so that every
// kernel of the step reads its frames exactly as it reads uploaded ones.  Batches of one size and level count have one layout,
// so every entry is a whole-frame copy.
static int multi_step_resident(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, sfmgpu_frames* const* f, const int32_t* idx, double* prev_xy,
                               double* cur_xy, int32_t* ids, int32_t* n_out) {
  const int S = t->L.S, par = multi_next_group(t);
  std::vector<FrameCopy> tab;
  tab.reserve((size_t)S * t->cfg.pyr_levels);
  unsigned long long most = 0;
  for (int s = 0; s < S; s++) {
    const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
    const sfmgpu_frames* g = c.frames;
    const size_t slot = (size_t)par * c.n + t->idx_in[s];
    for (int l = 0; l < g->levels; l++) {
      if (g->fstride[l] == 0) continue;  // level of zero size
      const unsigned long long n16 = g->fstride[l] / 16;  // pitch is a multiple of 16
      tab.push_back({reinterpret_cast<const uint4*>(f[s]->lvl[l] + (size_t)idx[s] * g->fstride[l]),
                     reinterpret_cast<uint4*>(g->lvl[l] + slot * g->fstride[l]), n16});
      if (n16 > most) most = n16;
    }
  }
  t->tv_fresh = false;
  SFM_CUDA(ctx, cudaMemcpyAsync(t->gtab, tab.data(), tab.size() * sizeof(FrameCopy), cudaMemcpyHostToDevice, ctx->stream));
  {
    StageTimer st(ctx, 5);
    if (!tab.empty())
      SFM_LAUNCH(ctx, copy_frames_kernel, dim3(sfm_cdiv((long long)most, 256 * 8), (unsigned)tab.size(), 1), 256, 0,
                 (const FrameCopy*)t->gtab);
  }
  return multi_step_on(ctx, t, par, prev_xy, cur_xy, ids, n_out);
}

extern "C" {

int sfmgpu_multitracker_step_frames(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, sfmgpu_frames* f, const int32_t* frame_idx, double* prev_xy,
                                    double* cur_xy, int32_t* ids, int32_t* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !f) return SFMGPU_E_ARG;
  if (t->mixed())
    return sfm_fail(ctx, SFMGPU_E_ARG,
                    "multitracker_step_frames: the sequences have different image sizes; packed and resident input take one size");
  if (!frame_idx) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_step_frames: null frame index array");
  if (t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_step_frames: frames are prefetched; step them first");
  const sfmgpu_frames* g = t->frames;
  if (f->w != g->w || f->h != g->h || f->levels != g->levels)
    return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_step_frames: frames are %dx%d with %d levels, the tracker %dx%d with %d", f->w, f->h,
                    f->levels, g->w, g->h, g->levels);
  const int S = t->L.S;
  for (int s = 0; s < S; s++)
    if (frame_idx[s] < 0 || frame_idx[s] >= f->n)
      return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_step_frames: sequence %d: frame %d outside [0,%d)", s, frame_idx[s], f->n);
  const std::vector<sfmgpu_frames*> fs(S, f);
  return multi_step_resident(ctx, t, fs.data(), frame_idx, prev_xy, cur_xy, ids, n_out);
}

int sfmgpu_multitracker_step_frames_sized(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, sfmgpu_frames* const* f, const int32_t* frame_idx,
                                          double* prev_xy, double* cur_xy, int32_t* ids, int32_t* n_out) {
  SFM_ENTER(ctx);
  const char* who = "multitracker_step_frames_sized";
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (!f || !frame_idx) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null frame batch or index array", who);
  const int S = t->L.S;
  for (int s = 0; s < S; s++)
    if (!f[s]) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequence %d: null frame batch", who, s);
  if (t->prefetched) return sfm_fail(ctx, SFMGPU_E_STATE, "%s: frames are prefetched; step them first", who);
  for (int s = 0; s < S; s++) {
    const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
    if (f[s]->w != c.w || f[s]->h != c.h || f[s]->levels != t->cfg.pyr_levels)
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequence %d: frames are %dx%d with %d levels, the sequence %dx%d with %d", who, s, f[s]->w,
                      f[s]->h, f[s]->levels, c.w, c.h, t->cfg.pyr_levels);
    if (frame_idx[s] < 0 || frame_idx[s] >= f[s]->n)
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s: sequence %d: frame %d outside [0,%d)", who, s, frame_idx[s], f[s]->n);
  }
  return multi_step_resident(ctx, t, f, frame_idx, prev_xy, cur_xy, ids, n_out);
}

}  // extern "C"

// One step of every sequence on the frames in slot group `par` (uploaded, prefetched or gathered there).
static int multi_step_on(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int par, double* prev_xy, double* cur_xy, int32_t* ids, int32_t* n_out) {
  TrackLists& L = t->L;
  const int S = L.S;
  const bool stage = sfm_two_view_enabled(t->tv);
  if (n_out)
    for (int s = 0; s < S; s++) n_out[s] = 0;
  if (t->parity < 0) {  // first frames: reset every sequence (:341-344); find_E_ransac is not called (:1715)
    for (const sfmgpu_multitracker::Run& r : t->runs) {
      const sfmgpu_multitracker::SizeClass& c = t->cls[r.cls];
      SFM_TRY(lists_reset(ctx, L, t->cfg, c.frames, par * c.n + r.i0 - r.s0, r.s0, r.count, "multitracker"));
    }
    t->parity = par;
    if (stage) SFM_TRY(sfm_two_view_skip(ctx, t->tv, nullptr, S));
    t->tv_fresh = stage;
    return 0;
  }
  std::vector<char> empty(S);  // sequences without tracks are reset on this frame instead of stepped (:341-344)
  bool any_empty = false;
  for (int s = 0; s < S; s++) {
    empty[s] = L.n[s] == 0;
    any_empty = any_empty || empty[s];
  }
  SFM_TRY(lists_track(ctx, L, t->cfg, t->frames, t->frames, t->parity * S, par * S, KLT_BY_ROWS,
                      t->mixed() ? t->geo + (size_t)t->parity * S : nullptr));
  if (stage) {  // find_E_ransac(K, prev_pts, cur_pts, ...) on every sequence's survivors (:1739), inside the step's one synchronisation
    StageTimer rt(ctx, 4);
    SFM_TRY(sfm_two_view_stage(ctx, t->tv, L.oa, L.ob, L.dnk, L.rows, 0, S, nullptr));
    // sequences reset on this frame instead of stepped (dn == 0) return no step: SKIPPED whatever min_points says
    if (any_empty) SFM_TRY(sfm_two_view_skip(ctx, t->tv, L.dn, S));
  }
  SFM_CUDA(ctx, cudaMemcpyAsync(L.n.data(), L.dnk, (size_t)S * 4, cudaMemcpyDeviceToHost, ctx->stream));
  const size_t rows = (size_t)S * L.rows;
  if (prev_xy) SFM_CUDA(ctx, cudaMemcpyAsync(prev_xy, L.oa, rows * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (cur_xy) SFM_CUDA(ctx, cudaMemcpyAsync(cur_xy, L.ob, rows * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, L.oid, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_TRY(lists_commit(ctx, L, rows));
  t->parity = par;
  t->tv_fresh = stage;
  if (n_out)
    for (int s = 0; s < S; s++) n_out[s] = L.n[s];
  auto where = [&](int s, sfmgpu_frames** f, int* frame) {
    const sfmgpu_multitracker::SizeClass& c = t->cls[t->cls_of[s]];
    *f = c.frames;
    *frame = par * c.n + t->idx_in[s];
  };
  return lists_refill(ctx, L, t->cfg, where, &empty, "multitracker");
}

extern "C" {

int sfmgpu_multitracker_set_ransac(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const double* K, const sfmgpu_ransac_cfg* rc) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  t->tv_fresh = false;  // results of earlier steps are not those of this configuration
  return sfm_two_view_configure(ctx, &t->tv, t->L.S, t->L.rows, K, rc, "multitracker_set_ransac");
}

int sfmgpu_multitracker_set_ransac_cameras(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const double* K, const sfmgpu_ransac_cfg* rc) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  SFM_TRY(sfm_two_view_configure_sets(ctx, &t->tv, t->L.S, t->L.rows, K, rc, "multitracker_set_ransac_cameras"));
  t->tv_fresh = false;  // results of earlier steps are not those of this configuration (a refused call keeps them)
  return 0;
}

int sfmgpu_multitracker_ransac_download_all(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int32_t* status, int32_t* best_n, int32_t* inliers,
                                            double* R, double* tr) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (!t->tv || !t->tv_fresh)
    return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_ransac_download_all: the last step ran without the RANSAC stage");
  return sfm_two_view_download_all(ctx, t->tv, t->L.rows, t->L.S, status, best_n, inliers, R, tr, "multitracker_ransac");
}

int sfmgpu_multitracker_ransac_early(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* sets_stopped) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !sets_stopped) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_ransac_early: null pointer");
  return sfm_two_view_early(ctx, t->tv, sets_stopped);
}

int sfmgpu_multitracker_tracks(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int sequence, double* xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (sequence < 0 || sequence >= t->L.S) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_tracks: bad sequence index");
  return lists_tracks(ctx, t->L, sequence, xy, ids, cap, n_out, "multitracker_tracks");
}

int sfmgpu_multitracker_totals(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* n_track_steps, long long* n_lk_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  return lists_totals(ctx, t->L, n_track_steps, n_lk_iters);
}

}  // extern "C"

// ---- segment mode: contiguous segments of one resident sequence, each a fresh KLTTracker (SURVEY.md §8e) -------------------
// A chunk of segments is one lock step: slot s of the tracker runs segment j0 + s, reset on its first frame and stepped through
// the next `steps` frames, read from the resident batch by sfmgpu_multitracker_step_frames.  Every segment of a call has the
// same length, so the slots start and finish together.  Step k of segment j is written to row j * steps + (k - 1) of the pairs
// object; the RANSAC stage then runs once over all rows, as it does after the other batch calls.
namespace {

// Survivors (the first n_kept of slot s), their ids and the counts of slot s -> row row0 + s * row_stride of the pairs arrays.
__global__ void __launch_bounds__(256) segment_rows_kernel(const double2* __restrict__ oa, const double2* __restrict__ ob,
                                                          const int* __restrict__ oid, const int* __restrict__ n_in,
                                                          const int* __restrict__ n_kept, int src_cap, double2* __restrict__ li,
                                                          double2* __restrict__ lj, int* __restrict__ ids, int* __restrict__ ncorn,
                                                          int* __restrict__ nkept, int dst_cap, long long row0, int row_stride) {
  const int s = blockIdx.y, n = n_kept[s];
  const long long row = row0 + (long long)s * row_stride;
  const size_t so = (size_t)s * src_cap, d = (size_t)row * dst_cap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    li[d + i] = oa[so + i];
    lj[d + i] = ob[so + i];
    ids[d + i] = oid[so + i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ncorn[row] = n_in[s];
    nkept[row] = n;
  }
}

bool same_lkcfg(const sfmgpu_lkcfg& a, const sfmgpu_lkcfg& b) {
  return a.max_tracks == b.max_tracks && a.min_tracks == b.min_tracks && a.quality == b.quality && a.min_distance == b.min_distance &&
         a.pyr_levels == b.pyr_levels && a.win_radius == b.win_radius && a.iters == b.iters && a.fb_thresh == b.fb_thresh;
}

}  // namespace

extern "C" int sfmgpu_pair_frontend_segments(sfmgpu_ctx* ctx, sfmgpu_frames* f, const int32_t* seg_first, int nseg, int steps,
                                             const sfmgpu_lkcfg* cfg, sfmgpu_pairs* out) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out) return SFMGPU_E_ARG;
  if (steps < 1) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: %d steps per segment (at least 1)", steps);
  if (nseg < 0 || (long long)nseg * steps > out->max_pairs)
    return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: %d segments x %d steps, room for %d rows", nseg, steps, out->max_pairs);
  if (nseg > 0 && !seg_first) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: null seg_first");
  for (int j = 0; j < nseg; j++)
    if (seg_first[j] < 0 || (long long)seg_first[j] + steps >= f->n)
      return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: segment %d = frames [%d, %lld] outside [0,%d)", j, seg_first[j],
                      (long long)seg_first[j] + steps, f->n);
  if (cfg->pyr_levels != f->levels) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: cfg->pyr_levels != frames levels");
  SFM_TRY(lkcfg_ok(ctx, cfg, "pair_frontend_segments"));
  const int rows = track_rows(*cfg);
  if (out->cap < rows)
    return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_segments: pairs rows hold %d points, a track list up to %d (max(max_tracks, min_tracks, 1) + 1)",
                    out->cap, rows);
  // Slots per lock step: the reset's corner work area holds W*H candidates per slot (~265 MB at 4K); 16 GiB bound it as
  // they bound the pair calls' chunks.  Chunks are balanced; the last one's spare slots repeat its last segment (unread).
  int S = 0;
  if (nseg > 0) {
    const size_t per = sfm_corner_work_bytes_md(f->w, f->h, 1, f->w * f->h, abs_min_distance(*cfg));
    long long most = (long long)(((size_t)16 << 30) / (per ? per : 1));
    if (most > 512) most = 512;  // sfmgpu_multitracker_create's limit
    if (most < 1) most = 1;
    const int nchunk = (int)((nseg + most - 1) / most);
    S = (nseg + nchunk - 1) / nchunk;
  }
  sfmgpu_multitracker* mt = out->seg;
  if (mt && S > 0 && (mt->L.S != S || mt->w != f->w || mt->h != f->h || !same_lkcfg(mt->cfg, *cfg))) {
    sfmgpu_multitracker_destroy(ctx, mt);
    out->seg = mt = nullptr;
  }
  if (!mt && S > 0) {
    SFM_TRY(sfmgpu_multitracker_create(ctx, cfg, S, f->w, f->h, &out->seg));
    mt = out->seg;
  }
  if (!out->ids) SFM_CUDA(ctx, cudaMalloc((void**)&out->ids, (size_t)out->max_pairs * out->cap * 4 + 256));
  const int npairs = nseg * steps;
  out->last_npairs = npairs;
  out->ids_valid = true;
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals, 0, 64, ctx->stream));
  std::vector<int32_t> idx(S);
  for (int j0 = 0; j0 < nseg; j0 += S) {
    const int cnt = nseg - j0 < S ? nseg - j0 : S;
    SFM_TRY(sfmgpu_multitracker_reset(ctx, mt));
    for (int k = 0; k <= steps; k++) {  // k = 0: reset on the segment's first frame, no result (:341-344)
      for (int s = 0; s < S; s++) idx[s] = seg_first[j0 + (s < cnt ? s : cnt - 1)] + k;
      SFM_TRY(sfmgpu_multitracker_step_frames(ctx, mt, f, idx.data(), nullptr, nullptr, nullptr, nullptr));
      if (k == 0) continue;
      const TrackLists& L = mt->L;
      SFM_LAUNCH(ctx, segment_rows_kernel, dim3(sfm_cdiv(rows, 256), cnt), 256, 0, (const double2*)L.oa, (const double2*)L.ob,
                 (const int*)L.oid, (const int*)L.dn, (const int*)L.dnk, L.rows, out->li, out->lj, out->ids, out->ncorn, out->nkept,
                 out->cap, (long long)j0 * steps + (k - 1), steps);
      SFM_LAUNCH(ctx, totals_kernel, 64, 256, 0, (const int*)L.dn, (const int*)L.dnk, (const int*)L.nit, cnt, L.rows, out->totals);
    }
  }
  if (sfm_two_view_enabled(out->tv) && npairs > 0) {  // find_E_ransac(K, prev_pts, cur_pts, ...) on every step's survivors (:1739)
    StageTimer rt(ctx, 4);
    SFM_TRY(sfm_two_view_stage(ctx, out->tv, out->li, out->lj, out->nkept, out->cap, 0, npairs, nullptr));
    // a step that reset its segment (no tracks entering it) returns no step: SKIPPED whatever min_points says
    SFM_TRY(sfm_two_view_skip(ctx, out->tv, out->ncorn, npairs));
  }
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}
