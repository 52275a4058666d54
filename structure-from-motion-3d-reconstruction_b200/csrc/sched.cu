// sched.cu — the multi-GPU frame-pair scheduler behind the C ABI (SURVEY.md §8e): one rank (process or thread) per GPU.
//
// The two-view unit (cpp/src/templering_sfm.cpp:1836-1857) is stateless per frame pair, so ONE sequence shards by
// contiguous blocks of pairs plus one halo frame per rank, with no data-path collective; whole sequences shard the same
// way (sfmgpu_sched_shard).  The only communication is the gather of the per-pair results (survivors, counts and, when the
// RANSAC stage ran, status / winner count / inlier lists / poses) to one root rank: ncclSend / ncclRecv grouped into one
// launch (NCCL has no gatherv), straight out of the pairs object's device arrays into a device staging area on the root,
// then one D2H per array.  No fused compute+collective kernel is warranted: ~260 KB per 8k-track pair against NVLink.
//
// NCCL is bound at run time (dlopen of libnccl.so.2, or SFMGPU_NCCL_LIB): libsfmgpu.so itself has no NCCL dependency, a
// single-GPU drop-in never loads it, and inside a PyTorch process the already-loaded library is found by its soname.
#include <dlfcn.h>
#include <stddef.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
};

// Bound once per process (C++11 function-local static: thread-safe - ranks may be threads of one process).
NcclApi* nccl_api() {
  static NcclApi api = [] {
    NcclApi a;
    const char* names[] = {getenv("SFMGPU_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (a.lib) break;
    }
    if (!a.lib) {
      a.err = "NCCL library not found (libnccl.so.2; set SFMGPU_NCCL_LIB)";
      return a;
    }
    bool ok = true;
    auto sym = [&](const char* name) {
      void* p = dlsym(a.lib, name);
      if (!p) {
        ok = false;
        a.err = std::string("NCCL symbol missing: ") + name;
      }
      return p;
    };
    a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
    a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
    a.Send = (decltype(a.Send))sym("ncclSend");
    a.Recv = (decltype(a.Recv))sym("ncclRecv");
    a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
    a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
    if (!ok) {
      dlclose(a.lib);
      a.lib = nullptr;
    }
    return a;
  }();
  return &api;
}

void shard(int n_items, int world, int rank, int* begin, int* end) {
  if (n_items < 0) n_items = 0;
  const int base = n_items / world, extra = n_items % world;
  const int b = rank * base + (rank < extra ? rank : extra);
  *begin = b;
  *end = b + base + (rank < extra ? 1 : 0);
}

}  // namespace

struct sfmgpu_sched {
  int world = 1, rank = 0;
  ncclComm_t comm = nullptr;
  bool own_comm = false;
  DevBuf stage;  // root: gathered arrays of the whole sequence
};
// The shard functions read world and rank only: a caller without a device may pass these two ints (sfmgpu/sched.py does).
static_assert(offsetof(sfmgpu_sched, world) == 0 && offsetof(sfmgpu_sched, rank) == sizeof(int), "sfmgpu_sched head");

#define SFM_NCCL(ctx, api, expr)                                                                                  \
  do {                                                                                                            \
    ncclResult_t r__ = (expr);                                                                                    \
    if (r__ != ncclSuccess)                                                                                       \
      return sfm_fail(ctx, SFMGPU_E_CUDA, "%s failed: %s (%s:%d)", #expr, (api)->GetErrorString(r__), __FILE__, __LINE__); \
  } while (0)

extern "C" {

int sfmgpu_sched_shard(int n_items, int world, int rank, int* begin, int* end) {
  if (world < 1 || rank < 0 || rank >= world || !begin || !end) return SFMGPU_E_ARG;
  shard(n_items, world, rank, begin, end);
  return 0;
}

int sfmgpu_sched_unique_id(void* id128) {
  if (!id128) return SFMGPU_E_ARG;
  NcclApi* api = nccl_api();
  if (!api->lib) return SFMGPU_E_CUDA;
  static_assert(sizeof(ncclUniqueId) == SFMGPU_SCHED_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  if (api->GetUniqueId(&id) != ncclSuccess) return SFMGPU_E_CUDA;
  memcpy(id128, &id, sizeof id);
  return 0;
}

int sfmgpu_sched_create(sfmgpu_ctx* ctx, int world, int rank, const void* id128, void* nccl_comm, sfmgpu_sched** out) {
  SFM_ENTER(ctx);
  if (!ctx || !out || world < 1 || rank < 0 || rank >= world) return sfm_fail(ctx, SFMGPU_E_ARG, "sched_create: bad world / rank");
  sfmgpu_sched* s = new sfmgpu_sched();
  s->world = world;
  s->rank = rank;
  if (nccl_comm) {
    s->comm = (ncclComm_t)nccl_comm;  // the caller's communicator (ncclComm_t), not destroyed here
  } else if (world > 1) {
    if (!id128) {
      delete s;
      return sfm_fail(ctx, SFMGPU_E_ARG, "sched_create: %d ranks need a unique id (sfmgpu_sched_unique_id on rank 0) or a communicator", world);
    }
    NcclApi* api = nccl_api();
    if (!api->lib) {
      delete s;
      return sfm_fail(ctx, SFMGPU_E_CUDA, "sched_create: %s", api->err.c_str());
    }
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    ncclResult_t r = api->CommInitRank(&s->comm, world, id, rank);
    if (r != ncclSuccess) {
      delete s;
      return sfm_fail(ctx, SFMGPU_E_CUDA, "sched_create: ncclCommInitRank failed: %s", api->GetErrorString(r));
    }
    s->own_comm = true;
  }
  *out = s;
  return 0;
}

void sfmgpu_sched_destroy(sfmgpu_ctx* ctx, sfmgpu_sched* s) {
  SFM_ENTER_VOID(ctx);
  if (!s) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  if (s->own_comm && s->comm) nccl_api()->CommDestroy(s->comm);
  if (s->stage.p) cudaFree(s->stage.p);
  delete s;
}

int sfmgpu_sched_pair_shard(const sfmgpu_sched* s, int n_frames, int* pair_begin, int* pair_end, int* frame_begin, int* frame_end) {
  if (!s) return SFMGPU_E_ARG;
  int a = 0, b = 0;
  shard(n_frames > 0 ? n_frames - 1 : 0, s->world, s->rank, &a, &b);
  if (pair_begin) *pair_begin = a;
  if (pair_end) *pair_end = b;
  if (frame_begin) *frame_begin = a;
  if (frame_end) *frame_end = b > a ? b + 1 : a;  // one halo frame: the second frame of the block's last pair
  return 0;
}

// Segment mode (SURVEY.md §8e): G segments of L = ceil((T-1)/G) steps each, spread evenly over the T-1 frame pairs.  Segment j
// starts on frame floor(j * (T-1-L) / (G-1)) (G = 1: 0), so the first starts on frame 0, the last ends on frame T-1, neighbouring
// starts are at most L apart (every pair of the sequence is a step of some segment) and G*L - (T-1) < G steps are done twice.
int sfmgpu_sched_segment_shard(const sfmgpu_sched* s, int n_frames, int n_segments, int* steps, int* seg_begin, int* seg_end,
                               int32_t* seg_first, int* frame_begin, int* frame_end) {
  if (!s || s->world < 1 || s->rank < 0 || s->rank >= s->world) return SFMGPU_E_ARG;
  const long long T = n_frames, G = n_segments;
  if (T < 2 || G < 1 || G > T - 1) return SFMGPU_E_ARG;
  const long long L = (T - 1 + G - 1) / G;
  auto first = [&](long long j) { return G == 1 ? 0 : j * (T - 1 - L) / (G - 1); };
  int a = 0, b = 0;
  shard((int)G, s->world, s->rank, &a, &b);
  if (steps) *steps = (int)L;
  if (seg_begin) *seg_begin = a;
  if (seg_end) *seg_end = b;
  if (seg_first)
    for (long long j = 0; j < G; j++) seg_first[j] = (int32_t)first(j);
  if (frame_begin) *frame_begin = b > a ? (int)first(a) : 0;
  if (frame_end) *frame_end = b > a ? (int)(first(b - 1) + L + 1) : 0;
  return 0;
}

namespace {

struct GatherArr {
  size_t per_pair;  // bytes per pair
  const void* src;  // this rank's device array
  void* host;       // root: destination of the whole sequence (may be null)
};

// Collective of the gathers: this rank's block of n_pairs_total (sfmgpu_sched_shard's rule) must be the last batch of p.
// Non-root ranks send and return after the sends have completed (*base = null).  The root receives every block into its
// staging area (array k at *base + off[k]), queues the D2H copies of the arrays with a host pointer, and returns with them in
// flight: the caller adds its own copies and synchronises.
int gather_rows(sfmgpu_ctx* ctx, sfmgpu_sched* s, sfmgpu_pairs* p, int n_pairs_total, int root, const GatherArr* arr, int narr,
                const char* who, char** base, size_t* off) {
  *base = nullptr;
  if (root < 0 || root >= s->world || n_pairs_total < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: bad root / size", who);
  int a = 0, b = 0;
  shard(n_pairs_total, s->world, s->rank, &a, &b);
  if (b - a != p->last_npairs)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: rank %d holds %d pairs, its block [%d,%d) has %d", who, s->rank, p->last_npairs, a, b, b - a);
  NcclApi* api = s->world > 1 ? nccl_api() : nullptr;
  if (s->world > 1 && (!api->lib || !s->comm)) return sfm_fail(ctx, SFMGPU_E_STATE, "%s: no communicator", who);
  if (s->rank != root) {
    SFM_NCCL(ctx, api, api->GroupStart());
    for (int k = 0; k < narr; k++)
      if (b > a) SFM_NCCL(ctx, api, api->Send(arr[k].src, arr[k].per_pair * (size_t)(b - a), ncclUint8, root, s->comm, ctx->stream));
    SFM_NCCL(ctx, api, api->GroupEnd());
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
  }
  // root: staging area for the whole sequence
  off[0] = 0;
  for (int k = 0; k < narr; k++) off[k + 1] = off[k] + ((arr[k].per_pair * (size_t)n_pairs_total + 255) & ~(size_t)255);
  SFM_TRY(sfm_reserve(ctx, s->stage, off[narr] + 256));
  char* stage = (char*)s->stage.p;
  if (s->world > 1) SFM_NCCL(ctx, api, api->GroupStart());
  for (int r = 0; r < s->world; r++) {
    int ra = 0, rb = 0;
    shard(n_pairs_total, s->world, r, &ra, &rb);
    if (rb <= ra) continue;
    for (int k = 0; k < narr; k++) {
      void* dst = stage + off[k] + arr[k].per_pair * (size_t)ra;
      const size_t bytes = arr[k].per_pair * (size_t)(rb - ra);
      if (r == root)
        SFM_CUDA(ctx, cudaMemcpyAsync(dst, arr[k].src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
      else
        SFM_NCCL(ctx, api, api->Recv(dst, bytes, ncclUint8, r, s->comm, ctx->stream));
    }
  }
  if (s->world > 1) SFM_NCCL(ctx, api, api->GroupEnd());
  for (int k = 0; k < narr; k++)
    if (arr[k].host && n_pairs_total > 0)
      SFM_CUDA(ctx, cudaMemcpyAsync(arr[k].host, stage + off[k], arr[k].per_pair * (size_t)n_pairs_total, cudaMemcpyDeviceToHost, ctx->stream));
  *base = stage;
  return 0;
}

}  // namespace

// Gather.  Every rank calls it with its pairs object (last batch = its block of pairs, in order); on `root` the host
// arrays receive the whole sequence: li / lj [n_pairs_total][max_corners][2], n_kept / n_corners [n_pairs_total] and -
// when with_ransac - status / best_n [n_pairs_total], inliers [n_pairs_total][max_corners], R [..][9], t [..][3].
// Host pointers are ignored on the other ranks; any may be NULL on the root.
int sfmgpu_sched_gather_pairs(sfmgpu_ctx* ctx, sfmgpu_sched* s, sfmgpu_pairs* p, int n_pairs_total, int root, int with_ransac,
                              double* li_xy, double* lj_xy, int32_t* n_kept, int32_t* n_corners, int32_t* status, int32_t* best_n,
                              int32_t* inliers, double* R, double* t) {
  SFM_ENTER(ctx);
  if (!ctx || !s || !p) return SFMGPU_E_ARG;
  if (root < 0 || root >= s->world || n_pairs_total < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "sched_gather_pairs: bad root / size");
  int a = 0, b = 0;
  shard(n_pairs_total, s->world, s->rank, &a, &b);
  if (b - a != p->last_npairs)
    return sfm_fail(ctx, SFMGPU_E_ARG, "sched_gather_pairs: rank %d holds %d pairs, its block [%d,%d) has %d", s->rank, p->last_npairs, a, b, b - a);
  void *d_st = nullptr, *d_best = nullptr, *d_inl = nullptr, *d_R = nullptr, *d_t = nullptr;
  if (with_ransac && sfmgpu_pairs_ransac_device_ptrs(p, &d_st, &d_best, &d_inl, &d_R, &d_t) != 0)
    return sfm_fail(ctx, SFMGPU_E_STATE, "sched_gather_pairs: the RANSAC stage has not run on this rank");
  const size_t cap = (size_t)p->cap;
  const GatherArr arr[9] = {{cap * 16, p->li, li_xy}, {cap * 16, p->lj, lj_xy}, {4, p->nkept, n_kept}, {4, p->ncorn, n_corners},
                            {4, d_st, status},        {8, d_best, nullptr},     {cap * 4, d_inl, inliers}, {72, d_R, R},
                            {24, d_t, t}};
  char* base = nullptr;
  size_t off[10];
  SFM_TRY(gather_rows(ctx, s, p, n_pairs_total, root, arr, with_ransac ? 9 : 4, "sched_gather_pairs", &base, off));
  if (!base) return 0;  // not the root: the sends have completed
  if (with_ransac && best_n && n_pairs_total > 0)  // best is (winner, count) per pair: the count column
    SFM_CUDA(ctx, cudaMemcpy2DAsync(best_n, 4, base + off[5] + 4, 8, 4, (size_t)n_pairs_total, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

// The track ids of a segment call ([n_pairs_total][max_corners] on the root), gathered as sfmgpu_sched_gather_pairs gathers the
// rows they belong to.
int sfmgpu_sched_gather_pair_ids(sfmgpu_ctx* ctx, sfmgpu_sched* s, sfmgpu_pairs* p, int n_pairs_total, int root, int32_t* ids) {
  SFM_ENTER(ctx);
  if (!ctx || !s || !p) return SFMGPU_E_ARG;
  void* d_ids = nullptr;
  if (sfmgpu_pairs_ids_device_ptr(p, &d_ids) != 0)
    return sfm_fail(ctx, SFMGPU_E_STATE, "sched_gather_pair_ids: the last batch of rank %d carries no track ids (not a segment call)", s->rank);
  const GatherArr arr[1] = {{(size_t)p->cap * 4, d_ids, ids}};
  char* base = nullptr;
  size_t off[2];
  SFM_TRY(gather_rows(ctx, s, p, n_pairs_total, root, arr, 1, "sched_gather_pair_ids", &base, off));
  if (base) SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

}  // extern "C"
