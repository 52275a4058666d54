// segments_test.cpp — C++ test of segment mode across GPUs (include/sfmgpu.h: sfmgpu_sched_segment_shard,
// sfmgpu_pair_frontend_segments, sfmgpu_sched_gather_pairs / _gather_pair_ids), no Python, no torch.
// One host thread per rank (= per GPU; world = min(requested, visible GPUs)).  G = world * per_rank segments of one synthetic
// sequence: every rank generates only the frames its block of segments reads, runs its segments with the RANSAC stage on and
// takes part in the gathers; the root compares rows, track ids and stage results with a single-GPU run of all G segments, byte
// for byte.  usage: segments_test [world=2] [frames=40] [per_rank=8] [w=320] [h=240] [max_tracks=300]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "../../include/sfmgpu.h"

#define CK(ctx, expr)                                                                         \
  do {                                                                                        \
    int rc__ = (expr);                                                                        \
    if (rc__ != 0) {                                                                          \
      fprintf(stderr, "FAILED %s -> %d: %s\n", #expr, rc__, sfmgpu_last_error(ctx));          \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

struct Results {
  std::vector<double> li, lj, R, t;
  std::vector<int32_t> nk, nc, st, bn, inl, ids;
  void size(int P, int cap) {
    li.assign((size_t)P * cap * 2, -1.0);
    lj.assign((size_t)P * cap * 2, -1.0);
    R.assign((size_t)P * 9, -1.0);
    t.assign((size_t)P * 3, -1.0);
    nk.assign(P, -1);
    nc.assign(P, -1);
    st.assign(P, -1);
    bn.assign(P, -1);
    inl.assign((size_t)P * cap, -1);
    ids.assign((size_t)P * cap, -1);
  }
};

static const double K[9] = {1520.4, 0, 302.32, 0, 1525.9, 246.87, 0, 0, 1.0};
static const uint32_t SEED = 20261124u;

static int run_rank(int world, int rank, int device, const void* id, int frames, int G, int w, int h, int max_tracks, Results* out) {
  sfmgpu_ctx* ctx = nullptr;
  if (sfmgpu_create(device, &ctx) != 0) {
    fprintf(stderr, "rank %d: no CUDA device %d\n", rank, device);
    return 1;
  }
  // a byte comparison between different batch sizes pins the KLT kernel family and the RANSAC solver (both are otherwise
  // chosen by the size of a launch; the alternatives agree to ~1e-13, not bit for bit)
  CK(ctx, sfmgpu_klt_set_mode(ctx, 2));
  CK(ctx, sfmgpu_solver_set_mode(ctx, 0));
  sfmgpu_sched* s = nullptr;
  CK(ctx, sfmgpu_sched_create(ctx, world, rank, id, nullptr, &s));
  int L = 0, a = 0, b = 0, f0 = 0, f1 = 0;
  std::vector<int32_t> first(G);
  CK(ctx, sfmgpu_sched_segment_shard(s, frames, G, &L, &a, &b, first.data(), &f0, &f1));
  const int nf = f1 - f0, nseg = b - a;
  std::vector<int32_t> local(nseg > 0 ? nseg : 1);
  for (int j = 0; j < nseg; j++) local[j] = first[a + j] - f0;
  sfmgpu_lkcfg cfg;
  sfmgpu_lkcfg_default(&cfg);
  cfg.max_tracks = max_tracks;
  cfg.min_tracks = max_tracks - max_tracks / 20;  // replenishment in most steps
  const int cap = max_tracks + 1;                 // max(max_tracks, min_tracks, 1) + 1
  sfmgpu_ransac_cfg rc = {2500, 1e-3, 60, 1};     // :1739
  sfmgpu_frames* fr = nullptr;
  sfmgpu_pairs* pr = nullptr;
  CK(ctx, sfmgpu_frames_create(ctx, w, h, nf > 2 ? nf : 2, cfg.pyr_levels, &fr));
  CK(ctx, sfmgpu_pairs_create(ctx, nseg > 0 ? nseg * L : 1, cap, &pr));
  CK(ctx, sfmgpu_pairs_set_ransac(ctx, pr, K, &rc));
  if (nf > 0) {
    CK(ctx, sfmgpu_frames_synth(ctx, fr, 0, nf, SEED, f0));  // this rank's frames of THE sequence
    CK(ctx, sfmgpu_pyramid_build(ctx, fr, 0, nf));
  }
  CK(ctx, sfmgpu_pair_frontend_segments(ctx, fr, local.data(), nseg, L, &cfg, pr));
  const int P = G * L;
  const bool root = rank == 0;
  if (root) out->size(P, cap);
  CK(ctx, sfmgpu_sched_gather_pairs(ctx, s, pr, P, 0, 1, root ? out->li.data() : nullptr, root ? out->lj.data() : nullptr,
                                    root ? out->nk.data() : nullptr, root ? out->nc.data() : nullptr, root ? out->st.data() : nullptr,
                                    root ? out->bn.data() : nullptr, root ? out->inl.data() : nullptr, root ? out->R.data() : nullptr,
                                    root ? out->t.data() : nullptr));
  CK(ctx, sfmgpu_sched_gather_pair_ids(ctx, s, pr, P, 0, root ? out->ids.data() : nullptr));
  sfmgpu_sched_destroy(ctx, s);
  sfmgpu_pairs_destroy(ctx, pr);
  sfmgpu_frames_destroy(ctx, fr);
  sfmgpu_destroy(ctx);
  return 0;
}

int main(int argc, char** argv) {
  const int want = argc > 1 ? atoi(argv[1]) : 2, frames = argc > 2 ? atoi(argv[2]) : 40, per_rank = argc > 3 ? atoi(argv[3]) : 8;
  const int w = argc > 4 ? atoi(argv[4]) : 320, h = argc > 5 ? atoi(argv[5]) : 240, max_tracks = argc > 6 ? atoi(argv[6]) : 300;
  int ndev = 0;
  for (; ndev < 16; ndev++) {
    sfmgpu_ctx* c = nullptr;
    if (sfmgpu_create(ndev, &c) != 0) break;
    sfmgpu_destroy(c);
  }
  if (ndev == 0) {
    fprintf(stderr, "no CUDA device: the library has no CPU fallback\n");
    return 2;
  }
  const int world = want < ndev ? want : ndev;
  const int G = world * per_rank;  // the gathers' block rule over rows equals the segment blocks when world divides G
  unsigned char id[SFMGPU_SCHED_ID_BYTES] = {0};
  if (world > 1 && sfmgpu_sched_unique_id(id) != 0) {
    fprintf(stderr, "sfmgpu_sched_unique_id failed (NCCL library not found?)\n");
    return 1;
  }
  Results got, ref;
  std::vector<int> rcs(world, 0);
  std::vector<std::thread> pool;
  for (int r = 0; r < world; r++)
    pool.emplace_back([&, r]() { rcs[r] = run_rank(world, r, r, id, frames, G, w, h, max_tracks, &got); });
  for (auto& th : pool) th.join();
  for (int r = 0; r < world; r++)
    if (rcs[r] != 0) return 1;
  // all segments on ONE GPU through the same entry points (world = 1: no communicator, the gathers are local copies)
  if (run_rank(1, 0, 0, nullptr, frames, G, w, h, max_tracks, &ref) != 0) return 1;
  const int P = (int)ref.nk.size(), cap = max_tracks + 1;
  bool ok = got.nk == ref.nk && got.nc == ref.nc && got.st == ref.st && got.bn == ref.bn;
  long tracks = 0, poses = 0;
  for (int p = 0; p < P && ok; p++) {
    const size_t o = (size_t)p * cap, n = (size_t)ref.nk[p];
    tracks += ref.nc[p];
    ok = ok && memcmp(&got.li[2 * o], &ref.li[2 * o], n * 16) == 0 && memcmp(&got.lj[2 * o], &ref.lj[2 * o], n * 16) == 0 &&
         memcmp(&got.ids[o], &ref.ids[o], n * 4) == 0;
    if (ref.st[p] == 2) {
      poses++;
      ok = ok && memcmp(&got.inl[o], &ref.inl[o], (size_t)ref.bn[p] * 4) == 0 && memcmp(&got.R[9 * p], &ref.R[9 * p], 72) == 0 &&
           memcmp(&got.t[3 * p], &ref.t[3 * p], 24) == 0;
    }
  }
  ok = ok && poses > 0;
  printf("segments_test: world %d (of %d GPUs), %d segments, %d rows, %ld feature-tracks, %ld poses: %s\n", world, ndev,
         world * per_rank, P, tracks, poses, ok ? "gathered == single-GPU, OK" : "MISMATCH");
  return ok ? 0 : 1;
}
