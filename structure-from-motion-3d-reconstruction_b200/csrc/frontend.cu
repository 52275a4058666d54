// frontend.cu — the two callers of the kernels that the reference has:
//   * the stateless two-view front end (cpp/src/templering_sfm.cpp:1836-1857), batched over frame pairs;
//   * the stateful KLTTracker (:323-391): reset / step / tracks, with the replenish rule (:374-389).
// Everything stays on the device between stages; only survivors / counts are copied back when the caller asks.
#include <stdlib.h>

#include <utility>
#include <vector>

#include "common.cuh"

// ---- small kernels -----------------------------------------------------------------------------------------------
namespace {

// Ordered compaction of the survivors of one pair / one tracker step: block = one pair.
// keep == nullptr keeps everything.  Outputs (any may be null): a/b = p0/p1 of survivors, ids_out, n_out.
__global__ void __launch_bounds__(1024) compact_kernel(const double2* __restrict__ p0, const double2* __restrict__ p1,
                                                      const uint8_t* __restrict__ keep, const int* __restrict__ ids,
                                                      const int* __restrict__ counts, int cap, double2* __restrict__ oa,
                                                      double2* __restrict__ ob, int* __restrict__ oid,
                                                      int* __restrict__ n_out) {
  __shared__ int wcnt[32], wpre[32];
  __shared__ int base, total;
  const int pair = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int n = counts ? counts[pair] : cap;
  n = n < 0 ? 0 : (n > cap ? cap : n);
  const size_t off = (size_t)pair * cap;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int s = 0; s < n; s += 1024) {
    const int i = s + tid;
    const bool k = i < n && (keep ? keep[off + i] != 0 : true);
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
      if (lane == 31) total = ia;
    }
    __syncthreads();
    if (k) {
      const int r = base + wpre[warp] + __popc(m & ((1u << lane) - 1u));
      if (oa) oa[off + r] = p0[off + i];
      if (ob) ob[off + r] = p1[off + i];
      if (oid) oid[off + r] = ids[off + i];
    }
    __syncthreads();
    if (tid == 0) base += total;
    __syncthreads();
  }
  if (tid == 0 && n_out) n_out[pair] = base;
}

// totals[0] += sum max(ncorn,0); totals[1] += sum nkept; totals[2] += sum nit; totals[3] += #frames with ncorn < 0
__global__ void __launch_bounds__(256) totals_kernel(const int* __restrict__ ncorn, const int* __restrict__ nkept,
                                                    const int* __restrict__ nit, int npairs, int cap,
                                                    unsigned long long* __restrict__ totals) {
  unsigned long long c = 0, k = 0, it = 0, bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)npairs * cap;
       i += (long long)gridDim.x * blockDim.x) {
    const int pair = (int)(i / cap), slot = (int)(i - (long long)pair * cap);
    const int n = ncorn[pair];
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
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&totals[0], c);
    atomicAdd(&totals[1], k);
    atomicAdd(&totals[2], (unsigned long long)lo + ((unsigned long long)hi << 16));
    atomicAdd(&totals[3], bad);
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
  __shared__ int wcnt[32], wpre[32];
  __shared__ int base, total;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nf = *n_fresh;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int s = 0; s < nf; s += 1024) {
    const int i = s + tid;
    const bool k = i < nf && ok[i];
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
      if (lane == 31) total = ia;
    }
    __syncthreads();
    if (k) {
      const int r = base + wpre[warp] + __popc(m & ((1u << lane) - 1u));
      if (r < room) {
        tracks[n_tracks + r] = fresh[i];
        ids[n_tracks + r] = next_id + r;
      }
    }
    __syncthreads();
    if (tid == 0) base += total;
    __syncthreads();
    if (base >= room) break;
  }
  if (tid == 0) *n_added = base < room ? base : room;
}

// out[0] += sum v[0..n)
__global__ void __launch_bounds__(256) sum_int_kernel(const int* __restrict__ v, int n, unsigned long long* __restrict__ out) {
  unsigned s = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += (unsigned)v[i];
  s = __reduce_add_sync(0xffffffffu, s);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, (unsigned long long)s);
}

__global__ void iota_ids_kernel(int* ids, const int* n, int next_id) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < *n) ids[i] = next_id + i;
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

int default_cand_cap(int w, int h) {
  long long px = (long long)w * h;
  long long cap = px / 6;
  if (cap < 65536) cap = 65536;
  if (cap > px) cap = px;
  return (int)cap;
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
  void* ptrs[] = {p->xy0, p->p1, p->pb, p->li, p->lj, p->nit, p->keep, p->ncorn, p->nkept, p->totals, p->work[0].p, p->work[1].p,
                  p->gather.p, p->idx.p};
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
  c.md = cfg->min_distance < 0 ? -cfg->min_distance : cfg->min_distance;
  c.cf = f;
  c.cfirst = first_frame;
  c.b_off = 1;
  return c;
}

// Pairs per corner launch: >= 4 blocks per SM keeps the one-block-per-frame selection kernels busy; large frames are
// limited by the work area instead (57 MB per 4K frame: 16 GiB hold 280 of them - still two waves of blocks)
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
  const int full_cap = f->w * f->h, md = cfg->min_distance < 0 ? -cfg->min_distance : cfg->min_distance;
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sfm_corner_work_bytes_md(f->w, f->h, 1, full_cap, md)));
  for (int p : bad) {
    SFM_TRY(sfm_corners_batch(ctx, f, h_fa ? h_fa[p] : first_frame + p, 1, cfg->max_tracks, cfg->quality, cfg->min_distance, full_cap,
                              ctx->cs_work.p, ctx->cs_work.cap, out->xy0 + (size_t)p * out->cap, out->ncorn + p));
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

// Streaming variant for frames that live in HOST memory: frames [0, nframes) of `f` are filled from host_pix in
// chunks on a copy stream (which also builds their pyramids); every chunk then flows through the stage pipeline and
// its results go back on a fifth stream.
int sfmgpu_pair_frontend_host(sfmgpu_ctx* ctx, sfmgpu_frames* f, const uint8_t* host_pix, int nframes, const sfmgpu_lkcfg* cfg,
                              sfmgpu_pairs* out, int chunk_frames, double* li_xy, double* lj_xy, int32_t* n_kept,
                              int32_t* n_corners) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !cfg || !out || !host_pix) return SFMGPU_E_ARG;
  if (nframes < 0 || nframes > f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "pair_frontend_host: %d frames do not fit (%d)", nframes, f->n);
  const int npairs = nframes > 0 ? nframes - 1 : 0;
  SFM_TRY(pair_args_ok(ctx, f, 0, npairs, cfg, out));
  out->last_npairs = npairs;
  SFM_CUDA(ctx, cudaMemsetAsync(out->totals, 0, 64, ctx->stream));
  if (nframes == 0) return 0;
  SFM_TRY(pipe_streams(ctx));
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
    SFM_CUDA(ctx, cudaMemcpy2DAsync(f->lvl[0] + (size_t)a * f->fstride[0], f->pitch[0], host_pix + (size_t)a * f->w * f->h, f->w,
                                    f->w, (size_t)f->h * (b - a), cudaMemcpyDefault, ctx->copy_stream));
    cudaEvent_t up = p.next();
    if (!up) return sfm_fail(ctx, SFMGPU_E_CUDA, "pair_frontend_host: cudaEventCreate failed");
    // The copy stream carries NOTHING but the uploads, back to back: the call is bound by them.  The chunk's pyramid is built
    // on the score stream behind the upload's event (on the copy stream it sat between two uploads and, waiting for SMs
    // behind the running KLT / RANSAC kernels, kept the copy engine idle ~0.35 ms per chunk).
    SFM_CUDA(ctx, cudaEventRecord(up, ctx->copy_stream));
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, up, 0));
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

// ---- stateful tracker -------------------------------------------------------------------------------------------------
struct sfmgpu_tracker {
  sfmgpu_lkcfg cfg;
  sfmgpu_frames* own = nullptr;     // 2-slot ping-pong used by the host-image entry points
  sfmgpu_frames* prev_frames = nullptr;
  int prev_index = -1;
  int n = 0;                        // live tracks (host copy)
  int next_id = 0;
  int cap = 0;
  double2 *trk = nullptr, *p1 = nullptr, *pb = nullptr, *oa = nullptr, *ob = nullptr, *fresh = nullptr;
  int *ids = nullptr, *oid = nullptr, *nit = nullptr, *scal = nullptr;  // scal: [0] n_out, [1] n_fresh, [2] n_added
  uint8_t *keep = nullptr, *ok = nullptr;
  int fresh_cap = 0;
  long long track_steps = 0;
  unsigned long long* tot = nullptr;
};

namespace {

int tracker_detect(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame, int max_corners, double2* out, int* d_n) {
  const int cand_cap = f->w * f->h;  // single frame: always room for the worst case
  const int md = t->cfg.min_distance < 0 ? -t->cfg.min_distance : t->cfg.min_distance;
  const size_t wb = sfm_corner_work_bytes_md(f->w, f->h, 1, cand_cap, md);
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, wb));
  return sfm_corners_batch(ctx, f, frame, 1, max_corners, t->cfg.quality, t->cfg.min_distance, cand_cap, ctx->cs_work.p,
                           ctx->cs_work.cap, out, d_n);
}

// Replenish one track list (:374-389): detect need*3 corners on the current frame, drop those within min_distance of a live
// track, append survivors with consecutive ids until max_tracks (tested after the append: at least one is added).
int replenish_row(sfmgpu_ctx* ctx, const sfmgpu_lkcfg& cfg, sfmgpu_frames* f, int frame, double2* trk, int* ids, int* n_io, int* next_id_io,
                  double2* fresh, int fresh_cap, uint8_t* ok, int* scal, int row_cap) {
  const int need = cfg.max_tracks - *n_io;
  long long want = (long long)need * 3;
  if (want > fresh_cap) want = fresh_cap;  // fresh_cap = 3*max_tracks >= need*3
  const int cand_cap = f->w * f->h;        // single frame: always room for the worst case
  const int md = cfg.min_distance < 0 ? -cfg.min_distance : cfg.min_distance;
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sfm_corner_work_bytes_md(f->w, f->h, 1, cand_cap, md)));
  SFM_TRY(sfm_corners_batch(ctx, f, frame, 1, (int)want, cfg.quality, cfg.min_distance, cand_cap, ctx->cs_work.p, ctx->cs_work.cap, fresh,
                            scal + 1));
  int nf = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&nf, scal + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (nf < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker: candidate capacity exceeded");
  if (nf > 0) {
    const double d2 = (double)cfg.min_distance * cfg.min_distance;
    SFM_LAUNCH(ctx, replenish_filter_kernel, sfm_cdiv(nf, 256), 256, 0, fresh, (const int*)(scal + 1), trk, *n_io, d2, ok);
    // the reference appends first and tests the cap afterwards (:386-387): at least one corner is added
    int room = cfg.max_tracks - *n_io;
    if (room < 1) room = 1;
    if (*n_io + room > row_cap)  // cannot happen with rows sized by track_rows(); never write past the row
      return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker: track list of %d + %d exceeds its %d rows", *n_io, room, row_cap);
    SFM_LAUNCH(ctx, replenish_append_kernel, 1, 1024, 0, fresh, (const int*)(scal + 1), ok, trk, ids, *n_io, room, *next_id_io, scal + 2);
    int na = 0;
    SFM_CUDA(ctx, cudaMemcpyAsync(&na, scal + 2, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_io += na;
    *next_id_io += na;
  }
  return 0;
}

int tracker_reset_on(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame) {
  // reset(gray) :327-332: prev_ = gray; tracks_ = shi_tomasi(...) with ids next_id_++
  SFM_TRY(tracker_detect(ctx, t, f, frame, t->cfg.max_tracks, t->trk, t->scal + 1));
  int n = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&n, t->scal + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker: candidate capacity exceeded");
  if (n > 0) SFM_LAUNCH(ctx, iota_ids_kernel, sfm_cdiv(n, 256), 256, 0, t->ids, (const int*)(t->scal + 1), t->next_id);
  t->n = n;
  t->next_id += n;
  t->prev_frames = f;
  t->prev_index = frame;
  return 0;
}

int tracker_step_on(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame, double* prev_xy, double* cur_xy,
                    int32_t* ids, int cap, int* n_out) {
  if (n_out) *n_out = 0;
  if (t->prev_index < 0 || t->n == 0) return tracker_reset_on(ctx, t, f, frame);  // :341-344
  if (t->prev_frames != f) return sfm_fail(ctx, SFMGPU_E_STATE, "tracker: previous frame lives in another frame batch");
  KltLaunch k;
  k.pv = f->view();
  k.p0 = t->trk;
  k.counts = nullptr;
  k.npairs = 1;
  k.cap = t->n;
  k.fa0 = t->prev_index;
  k.fa_step = 0;
  k.fb0 = frame;
  k.fb_step = 0;
  k.radius = t->cfg.win_radius;
  k.iters = t->cfg.iters;
  k.fb_thresh = t->cfg.fb_thresh;
  k.p1 = t->p1;
  k.pb = t->pb;
  k.nit = t->nit;
  k.keep = t->keep;
  SFM_TRY(sfm_klt_launch(ctx, k));
  t->track_steps += t->n;
  SFM_LAUNCH(ctx, sum_int_kernel, 8, 256, 0, (const int*)t->nit, t->n, t->tot + 2);
  // survivors in track order: (p0, p1, id); tracks_ = kept (:364-371)
  SFM_LAUNCH(ctx, compact_kernel, 1, 1024, 0, t->trk, t->p1, t->keep, t->ids, (const int*)nullptr, t->n, t->oa, t->ob, t->oid,
             t->scal);
  int nk = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&nk, t->scal, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (nk > cap && (prev_xy || cur_xy || ids))
    return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker_step: %d survivors, room for %d", nk, cap);
  if (nk > 0) {
    if (prev_xy) SFM_CUDA(ctx, cudaMemcpyAsync(prev_xy, t->oa, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (cur_xy) SFM_CUDA(ctx, cudaMemcpyAsync(cur_xy, t->ob, (size_t)nk * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, t->oid, (size_t)nk * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(t->trk, t->ob, (size_t)nk * 16, cudaMemcpyDeviceToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(t->ids, t->oid, (size_t)nk * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    // the header's promise: results are in the caller's (possibly pinned) buffers when the call returns
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  t->n = nk;
  t->prev_frames = f;
  t->prev_index = frame;
  if (n_out) *n_out = nk;
  // replenish (:374-389)
  if (t->n < t->cfg.min_tracks)
    SFM_TRY(replenish_row(ctx, t->cfg, f, frame, t->trk, t->ids, &t->n, &t->next_id, t->fresh, t->fresh_cap, t->ok, t->scal, t->cap));
  return 0;
}

int tracker_own_frames(sfmgpu_ctx* ctx, sfmgpu_tracker* t, int w, int h) {
  if (t->own && (t->own->w != w || t->own->h != h))
    return sfm_fail(ctx, SFMGPU_E_ARG, "tracker: image size changed from %dx%d to %dx%d (not supported)", t->own->w, t->own->h, w,
                    h);
  if (!t->own) SFM_TRY(sfmgpu_frames_create(ctx, w, h, 2, t->cfg.pyr_levels, &t->own));
  return 0;
}

}  // namespace

extern "C" {

int sfmgpu_tracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, sfmgpu_tracker** out) {
  SFM_ENTER(ctx);
  if (!ctx || !cfg || !out) return SFMGPU_E_ARG;
  if (cfg->pyr_levels < 1 || cfg->pyr_levels > SFM_MAXL || cfg->max_tracks > (1 << 24) || cfg->min_tracks > (1 << 24))
    return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_create: bad configuration");
  sfmgpu_tracker* t = new sfmgpu_tracker();
  t->cfg = *cfg;
  t->cap = track_rows(*cfg);
  t->fresh_cap = 3 * (cfg->max_tracks < 1 ? 1 : cfg->max_tracks);
  cudaError_t e = cudaSuccess;
  auto al = [&](void** q, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(q, bytes + 256);
  };
  const size_t n = (size_t)t->cap;
  al((void**)&t->trk, n * 16);
  al((void**)&t->p1, n * 16);
  al((void**)&t->pb, n * 16);
  al((void**)&t->oa, n * 16);
  al((void**)&t->ob, n * 16);
  al((void**)&t->ids, n * 4);
  al((void**)&t->oid, n * 4);
  al((void**)&t->nit, n * 4);
  al((void**)&t->keep, n);
  al((void**)&t->fresh, (size_t)t->fresh_cap * 16);
  al((void**)&t->ok, (size_t)t->fresh_cap);
  al((void**)&t->scal, 64);
  al((void**)&t->tot, 64);
  if (e == cudaSuccess) e = cudaMemsetAsync(t->tot, 0, 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(t->scal, 0, 64, ctx->stream);
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
  void* ptrs[] = {t->trk, t->p1, t->pb, t->oa, t->ob, t->ids, t->oid, t->nit, t->keep, t->fresh, t->ok, t->scal, t->tot};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  if (t->own) sfmgpu_frames_destroy(ctx, t->own);
  delete t;
}

int sfmgpu_tracker_reset(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !host_pix) return SFMGPU_E_ARG;
  SFM_TRY(tracker_own_frames(ctx, t, w, h));
  const int slot = (t->prev_frames == t->own && t->prev_index == 0) ? 1 : 0;
  SFM_TRY(sfmgpu_frames_upload(ctx, t->own, slot, 1, host_pix));
  SFM_TRY(sfmgpu_pyramid_build(ctx, t->own, slot, 1));
  return tracker_reset_on(ctx, t, t->own, slot);
}

int sfmgpu_tracker_step(sfmgpu_ctx* ctx, sfmgpu_tracker* t, const uint8_t* host_pix, int w, int h, double* prev_xy,
                        double* cur_xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !host_pix) return SFMGPU_E_ARG;
  SFM_TRY(tracker_own_frames(ctx, t, w, h));
  const int slot = (t->prev_frames == t->own && t->prev_index == 0) ? 1 : 0;
  SFM_TRY(sfmgpu_frames_upload(ctx, t->own, slot, 1, host_pix));
  SFM_TRY(sfmgpu_pyramid_build(ctx, t->own, slot, 1));
  return tracker_step_on(ctx, t, t->own, slot, prev_xy, cur_xy, ids, cap, n_out);
}

int sfmgpu_tracker_step_frames(sfmgpu_ctx* ctx, sfmgpu_tracker* t, sfmgpu_frames* f, int frame, double* prev_xy,
                               double* cur_xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !f) return SFMGPU_E_ARG;
  if (frame < 0 || frame >= f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_step_frames: bad frame index");
  if (f->levels != t->cfg.pyr_levels) return sfm_fail(ctx, SFMGPU_E_ARG, "tracker_step_frames: pyramid levels differ from cfg");
  return tracker_step_on(ctx, t, f, frame, prev_xy, cur_xy, ids, cap, n_out);
}

int sfmgpu_tracker_tracks(sfmgpu_ctx* ctx, sfmgpu_tracker* t, double* xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (n_out) *n_out = t->n;
  if (t->n > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "tracker_tracks: %d tracks, room for %d", t->n, cap);
  if (t->n > 0) {
    if (xy) SFM_CUDA(ctx, cudaMemcpyAsync(xy, t->trk, (size_t)t->n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, t->ids, (size_t)t->n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

int sfmgpu_tracker_totals(sfmgpu_ctx* ctx, sfmgpu_tracker* t, long long* n_track_steps, long long* n_lk_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  unsigned long long tt[4];
  SFM_CUDA(ctx, cudaMemcpyAsync(tt, t->tot, sizeof tt, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_track_steps) *n_track_steps = t->track_steps;
  if (n_lk_iters) *n_lk_iters = (long long)tt[2];
  return 0;
}

}  // extern "C"

// ---- lock-step tracker over S independent sequences (BASELINE.json C5: several sequences per GPU) -------------------------------
// The same KLTTracker semantics per sequence (:323-391), but ONE batched launch per stage and step for all of them: frame t of
// every sequence arrives together, the S x max_tracks feature-tracks share a KLT launch (large enough for the lane-per-feature
// kernels), survivors are compacted per sequence.  Results are identical to S separate sfmgpu_tracker objects.  Replenishment
// (rare: a track list below min_tracks) is done sequence by sequence with the single-tracker code.
struct sfmgpu_multitracker {
  sfmgpu_lkcfg cfg;
  int S = 0, w = 0, h = 0, cap = 0, fresh_cap = 0;
  sfmgpu_frames* frames = nullptr;  // 3*S slots: group g of sequence s lives in slot g*S + s (previous / current / prefetched)
  int parity = -1;                  // slot group of the previous frames, -1: nothing tracked yet
  bool prefetched = false;          // group (parity+1)%3 holds the next frames (uploaded + pyramids), ready at pf_done
  cudaEvent_t pf_done = nullptr;
  std::vector<int> n, next_id;      // host copies
  double2 *trk = nullptr, *p1 = nullptr, *pb = nullptr, *oa = nullptr, *ob = nullptr, *fresh = nullptr;
  int *ids = nullptr, *oid = nullptr, *nit = nullptr, *dn = nullptr, *dnk = nullptr, *scal = nullptr;
  uint8_t *keep = nullptr, *ok = nullptr;
  long long track_steps = 0;
  unsigned long long* tot = nullptr;
  TwoViewState* tv = nullptr;       // find_E_ransac on every sequence's survivors inside the step (sfmgpu_multitracker_set_ransac)
  bool tv_fresh = false;            // the last step ran the stage: its results can be downloaded
};

namespace {

// after a batched detection: row s of the track list = the first n[s] corners with ids next_id[s]..
__global__ void multi_take_corners_kernel(const double2* __restrict__ fresh, int fresh_stride, const int* __restrict__ n,
                                          const int* __restrict__ next_id, double2* __restrict__ trk, int* __restrict__ ids, int cap) {
  const int s = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n[s] || i >= cap) return;
  trk[(size_t)s * cap + i] = fresh[(size_t)s * fresh_stride + i];
  ids[(size_t)s * cap + i] = next_id[s] + i;
}

int multi_reset(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int par) {
  const int S = t->S, mc = t->cfg.max_tracks, cap_out = mc < 1 ? 1 : mc;
  const int cand_cap = t->w * t->h;
  const int md = t->cfg.min_distance < 0 ? -t->cfg.min_distance : t->cfg.min_distance;
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sfm_corner_work_bytes_md(t->w, t->h, S, cand_cap, md)));
  SFM_TRY(sfm_corners_batch(ctx, t->frames, par * S, S, mc, t->cfg.quality, t->cfg.min_distance, cand_cap, ctx->cs_work.p,
                            ctx->cs_work.cap, t->fresh, t->dn));
  SFM_CUDA(ctx, cudaMemcpyAsync(t->n.data(), t->dn, (size_t)S * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(t->dnk, t->next_id.data(), (size_t)S * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int s = 0; s < S; s++)
    if (t->n[s] < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "multitracker: candidate capacity exceeded (sequence %d)", s);
  SFM_LAUNCH(ctx, multi_take_corners_kernel, dim3(sfm_cdiv(cap_out, 256), S), 256, 0, t->fresh, cap_out, (const int*)t->dn,
             (const int*)t->dnk, t->trk, t->ids, t->cap);
  for (int s = 0; s < S; s++) t->next_id[s] += t->n[s];
  t->parity = par;
  return 0;
}

}  // namespace

extern "C" {

int sfmgpu_multitracker_create(sfmgpu_ctx* ctx, const sfmgpu_lkcfg* cfg, int n_sequences, int w, int h, sfmgpu_multitracker** out) {
  SFM_ENTER(ctx);
  if (!ctx || !cfg || !out) return SFMGPU_E_ARG;
  if (n_sequences < 1 || n_sequences > 512 || w < 1 || h < 1 || cfg->pyr_levels < 1 || cfg->pyr_levels > SFM_MAXL ||
      cfg->max_tracks > (1 << 24) || cfg->min_tracks > (1 << 24))
    return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_create: bad configuration");
  sfmgpu_multitracker* t = new sfmgpu_multitracker();
  t->cfg = *cfg;
  t->S = n_sequences;
  t->w = w;
  t->h = h;
  t->cap = track_rows(*cfg);  // as in sfmgpu_tracker
  t->fresh_cap = 3 * (cfg->max_tracks < 1 ? 1 : cfg->max_tracks);
  t->n.assign(n_sequences, 0);
  t->next_id.assign(n_sequences, 0);
  int rc = sfmgpu_frames_create(ctx, w, h, 3 * n_sequences, cfg->pyr_levels, &t->frames);
  if (rc != 0) {
    delete t;
    return rc;
  }
  cudaError_t e = cudaSuccess;
  auto al = [&](void** q, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(q, bytes + 256);
  };
  const size_t n = (size_t)t->cap * n_sequences;
  al((void**)&t->trk, n * 16);
  al((void**)&t->p1, n * 16);
  al((void**)&t->pb, n * 16);
  al((void**)&t->oa, n * 16);
  al((void**)&t->ob, n * 16);
  al((void**)&t->ids, n * 4);
  al((void**)&t->oid, n * 4);
  al((void**)&t->nit, n * 4);
  al((void**)&t->keep, n);
  al((void**)&t->fresh, (size_t)t->fresh_cap * 16 * n_sequences);
  al((void**)&t->ok, (size_t)t->fresh_cap);
  al((void**)&t->dn, (size_t)n_sequences * 4);
  al((void**)&t->dnk, (size_t)n_sequences * 4);
  al((void**)&t->scal, 64);
  al((void**)&t->tot, 64);
  if (e == cudaSuccess) e = cudaMemsetAsync(t->tot, 0, 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(t->scal, 0, 64, ctx->stream);
  if (e != cudaSuccess) {
    sfmgpu_multitracker_destroy(ctx, t);
    return sfm_fail(ctx, SFMGPU_E_CUDA, "multitracker_create: CUDA allocation failed: %s", cudaGetErrorString(e));
  }
  *out = t;
  return 0;
}

void sfmgpu_multitracker_destroy(sfmgpu_ctx* ctx, sfmgpu_multitracker* t) {
  SFM_ENTER_VOID(ctx);
  if (!t) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  sfm_two_view_free(ctx, &t->tv);
  void* ptrs[] = {t->trk, t->p1, t->pb, t->oa, t->ob, t->ids, t->oid, t->nit, t->keep, t->fresh, t->ok, t->dn, t->dnk, t->scal, t->tot};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  if (t->frames) sfmgpu_frames_destroy(ctx, t->frames);
  if (t->pf_done) cudaEventDestroy(t->pf_done);
  delete t;
}

// Upload + pyramids of the frames of a LATER step on the copy stream, into the slot group after `after_group`.
static int multi_prefetch(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int after_group, const uint8_t* host_pix) {
  SFM_TRY(pipe_streams(ctx));
  if (!t->pf_done && cudaEventCreateWithFlags(&t->pf_done, cudaEventDisableTiming) != cudaSuccess)
    return sfm_fail(ctx, SFMGPU_E_CUDA, "multitracker: cudaEventCreate failed");
  const int S = t->S, g = (after_group + 1) % 3;
  sfmgpu_frames* f = t->frames;
  SFM_CUDA(ctx, cudaMemcpy2DAsync(f->lvl[0] + (size_t)g * S * f->fstride[0], f->pitch[0], host_pix, f->w, f->w, (size_t)f->h * S,
                                  cudaMemcpyDefault, ctx->copy_stream));
  {
    StageScope sc(ctx, ctx->copy_stream);
    SFM_TRY(sfmgpu_pyramid_build(ctx, f, g * S, S));
    SFM_CUDA(ctx, cudaEventRecord(t->pf_done, ctx->stream));
  }
  t->prefetched = true;
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
  t->tv_fresh = false;
  t->n.assign(t->S, 0);
  t->next_id.assign(t->S, 0);
  t->track_steps = 0;
  SFM_CUDA(ctx, cudaMemsetAsync(t->tot, 0, 64, ctx->stream));
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
  const int S = t->S, cap = t->cap;
  const int par = t->parity < 0 ? 0 : (t->parity + 1) % 3;
  const bool stage = sfm_two_view_enabled(t->tv);
  t->tv_fresh = false;
  if (host_pix) {
    SFM_TRY(sfmgpu_frames_upload(ctx, t->frames, par * S, S, host_pix));
    SFM_TRY(sfmgpu_pyramid_build(ctx, t->frames, par * S, S));
  } else {
    SFM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, t->pf_done, 0));
    t->prefetched = false;
  }
  // the frames of the NEXT step travel while this one computes (their slot group is neither previous nor current)
  if (next_host_pix) SFM_TRY(multi_prefetch(ctx, t, par, next_host_pix));
  if (n_out)
    for (int s = 0; s < S; s++) n_out[s] = 0;
  if (t->parity < 0) {  // first frames: reset every sequence (:341-344); find_E_ransac is not called (:1715)
    SFM_TRY(multi_reset(ctx, t, par));
    if (stage) SFM_TRY(sfm_two_view_skip(ctx, t->tv, nullptr, S));
    t->tv_fresh = stage;
    return 0;
  }
  std::vector<int> empties;  // sequences without tracks are reset on this frame instead of stepped (:341-344)
  for (int s = 0; s < S; s++)
    if (t->n[s] == 0) empties.push_back(s);
  SFM_CUDA(ctx, cudaMemcpyAsync(t->dn, t->n.data(), (size_t)S * 4, cudaMemcpyHostToDevice, ctx->stream));
  KltLaunch k;
  k.pv = t->frames->view();
  k.p0 = t->trk;
  k.counts = t->dn;
  k.npairs = S;
  k.cap = cap;
  k.fa0 = t->parity * S;
  k.fa_step = 1;
  k.fb0 = par * S;
  k.fb_step = 1;
  k.radius = t->cfg.win_radius;
  k.iters = t->cfg.iters;
  k.fb_thresh = t->cfg.fb_thresh;
  k.p1 = t->p1;
  k.pb = t->pb;
  k.nit = t->nit;
  k.keep = t->keep;
  SFM_TRY(sfm_klt_launch(ctx, k));
  for (int s = 0; s < S; s++) t->track_steps += t->n[s];
  // survivors per sequence in track order: (p0, p1, id) (:364-371); LK iterations into the totals
  SFM_LAUNCH(ctx, compact_kernel, S, 1024, 0, t->trk, t->p1, t->keep, (const int*)t->ids, (const int*)t->dn, cap, t->oa, t->ob, t->oid,
             t->dnk);
  SFM_LAUNCH(ctx, totals_kernel, 64, 256, 0, (const int*)t->dn, (const int*)t->dnk, (const int*)t->nit, S, cap, t->tot);
  if (stage) {  // find_E_ransac(K, prev_pts, cur_pts, ...) on every sequence's survivors (:1739), inside the step's one synchronisation
    StageTimer rt(ctx, 4);
    SFM_TRY(sfm_two_view_stage(ctx, t->tv, t->oa, t->ob, t->dnk, cap, 0, S, nullptr));
    // sequences reset on this frame instead of stepped (dn == 0) return no step: SKIPPED whatever min_points says
    if (!empties.empty()) SFM_TRY(sfm_two_view_skip(ctx, t->tv, t->dn, S));
  }
  SFM_CUDA(ctx, cudaMemcpyAsync(t->n.data(), t->dnk, (size_t)S * 4, cudaMemcpyDeviceToHost, ctx->stream));
  const size_t rows = (size_t)S * cap;
  if (prev_xy) SFM_CUDA(ctx, cudaMemcpyAsync(prev_xy, t->oa, rows * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (cur_xy) SFM_CUDA(ctx, cudaMemcpyAsync(cur_xy, t->ob, rows * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, t->oid, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(t->trk, t->ob, rows * 16, cudaMemcpyDeviceToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(t->ids, t->oid, rows * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  t->parity = par;
  t->tv_fresh = stage;
  if (n_out)
    for (int s = 0; s < S; s++) n_out[s] = t->n[s];
  for (int s : empties) {
    // reset(gray): tracks_ = shi_tomasi(gray, max_tracks, ...) with ids next_id_++; the step returns nothing for it
    const int cand_cap = t->w * t->h;
    const int md = t->cfg.min_distance < 0 ? -t->cfg.min_distance : t->cfg.min_distance;
    SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sfm_corner_work_bytes_md(t->w, t->h, 1, cand_cap, md)));
    SFM_TRY(sfm_corners_batch(ctx, t->frames, par * S + s, 1, t->cfg.max_tracks, t->cfg.quality, t->cfg.min_distance, cand_cap,
                              ctx->cs_work.p, ctx->cs_work.cap, t->trk + (size_t)s * cap, t->scal + 1));
    int n = 0;
    SFM_CUDA(ctx, cudaMemcpyAsync(&n, t->scal + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (n < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "multitracker: candidate capacity exceeded (sequence %d)", s);
    if (n > 0) SFM_LAUNCH(ctx, iota_ids_kernel, sfm_cdiv(n, 256), 256, 0, t->ids + (size_t)s * cap, (const int*)(t->scal + 1), t->next_id[s]);
    t->n[s] = n;
    t->next_id[s] += n;
    if (n_out) n_out[s] = 0;
  }
  for (int s = 0; s < S; s++) {
    bool was_empty = false;
    for (int e : empties) was_empty = was_empty || e == s;
    if (!was_empty && t->n[s] < t->cfg.min_tracks)
      SFM_TRY(replenish_row(ctx, t->cfg, t->frames, par * S + s, t->trk + (size_t)s * cap, t->ids + (size_t)s * cap, &t->n[s],
                            &t->next_id[s], t->fresh, t->fresh_cap, t->ok, t->scal, cap));
  }
  return 0;
}

int sfmgpu_multitracker_set_ransac(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, const double* K, const sfmgpu_ransac_cfg* rc) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  t->tv_fresh = false;  // results of earlier steps are not those of this configuration
  return sfm_two_view_configure(ctx, &t->tv, t->S, t->cap, K, rc, "multitracker_set_ransac");
}

int sfmgpu_multitracker_ransac_download_all(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int32_t* status, int32_t* best_n, int32_t* inliers,
                                            double* R, double* tr) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (!t->tv || !t->tv_fresh)
    return sfm_fail(ctx, SFMGPU_E_STATE, "multitracker_ransac_download_all: the last step ran without the RANSAC stage");
  return sfm_two_view_download_all(ctx, t->tv, t->cap, t->S, status, best_n, inliers, R, tr, "multitracker_ransac");
}

int sfmgpu_multitracker_ransac_early(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* sets_stopped) {
  SFM_ENTER(ctx);
  if (!ctx || !t || !sets_stopped) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_ransac_early: null pointer");
  return sfm_two_view_early(ctx, t->tv, sets_stopped);
}

int sfmgpu_multitracker_tracks(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, int sequence, double* xy, int32_t* ids, int cap, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  if (sequence < 0 || sequence >= t->S) return sfm_fail(ctx, SFMGPU_E_ARG, "multitracker_tracks: bad sequence index");
  const int n = t->n[sequence];
  if (n_out) *n_out = n;
  if (n > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "multitracker_tracks: %d tracks, room for %d", n, cap);
  if (n > 0) {
    if (xy) SFM_CUDA(ctx, cudaMemcpyAsync(xy, t->trk + (size_t)sequence * t->cap, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (ids) SFM_CUDA(ctx, cudaMemcpyAsync(ids, t->ids + (size_t)sequence * t->cap, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

int sfmgpu_multitracker_totals(sfmgpu_ctx* ctx, sfmgpu_multitracker* t, long long* n_track_steps, long long* n_lk_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !t) return SFMGPU_E_ARG;
  unsigned long long tt[4];
  SFM_CUDA(ctx, cudaMemcpyAsync(tt, t->tot, sizeof tt, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_track_steps) *n_track_steps = t->track_steps;
  if (n_lk_iters) *n_lk_iters = (long long)tt[2];
  return 0;
}

}  // extern "C"
