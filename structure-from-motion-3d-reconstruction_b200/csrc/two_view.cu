// two_view.cu — the RANSAC stage of the two-view unit, batched over the pairs of a batch.
//
// Replaces (reference cpp/src/templering_sfm.cpp) what the loop-closure block does after the fb filter, :1855-1857:
//     if (li.size() >= 120) { auto lopt = find_E_ransac(K, li, lj, 4000, 2e-3, 80); ... }
// i.e. find_E_ransac :640-761 for every pair of a batch in ONE launch set per stage:
//   norm_point :498-501 / :649-655    tv_normalize_kernel   (K^-1 from the host, invert_K :471-486; FP64, no contraction)
//   seeded sampling :657-665          tv_sample_kernel      std::mt19937(12345) raw stream (generated once on the host, the
//                                                           generator is sequential) mapped to [0, n) exactly as libstdc++'s
//                                                           uniform_int_distribution does (Lemire multiply-shift WITH its
//                                                           rejection loop, bits/uniform_int_dist.h:257-279): a rejected raw
//                                                           value is skipped, so the octets are an ordered compaction of the
//                                                           accepted values - bit-exact index octets for every n
//   eight_point_E :609-627            eight_point_kernel    (solver.cu; device solver, hypotheses equal to ~1e-9) - or the
//                                                           caller's own hypotheses (bit-identical path, E_host)
//   scoring loop :667-676             ransac_count/argmax/mask kernels (ransac.cu; counts, winner, inlier list bit-exact
//                                                           for the hypotheses given)
//   min_inliers test :678, tail :680-760   tv_finalize_kernel, pose_kernel (solver.cu)
// Everything stays on the device; per pair the stage leaves status, winner, count, inlier indices, E, R, t.
#include <random>
#include <vector>

#include "common.cuh"

struct TwoViewState {
  bool enabled = false;  // run the stage inside sfmgpu_pair_frontend(_host)
  sfmgpu_ransac_cfg rc{};
  double Kinv[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  double2 *xi = nullptr, *xj = nullptr;  // [max_pairs][cap] normalised survivors
  int *neff = nullptr;                   // [max_pairs] points entering RANSAC (0: skipped by min_points)
  int *status = nullptr, *best = nullptr, *inl = nullptr;  // [max_pairs], [max_pairs][2], [max_pairs][cap]
  double *bestE = nullptr, *R = nullptr, *t = nullptr;     // [max_pairs][9], [9], [3]
  int* flags = nullptr;                  // [1] != 0: the raw stream was too short for some pair (cannot happen, checked)
  DevBuf idx8, E, counts;                // chunk scratch: [chunk][H][8], [chunk][H][9], [chunk][H]
  DevBuf neff2;                          // chunk scratch [chunk]: neff, or 0 for pairs whose scoring stopped early
  DevBuf raw;                            // mt19937(12345) outputs
  int raw_n = 0;
  // host outputs of the streaming front end (any may be null)
  int32_t *h_status = nullptr, *h_best_n = nullptr, *h_inl = nullptr;
  double *h_R = nullptr, *h_t = nullptr;
};

namespace {

constexpr int TV_CHUNK = 1024;  // pairs per launch set: bounds the scratch (1024 x 4000 hypotheses: 295 MB of E, 131 MB of octets).
                                // The small kernels of a set (sampler, repeated-index and winner solves, argmax, mask, pose) are
                                // latency-bound, ~0.6 ms per set: 256 pairs per set cost C3 (1999 pairs) 8 x that, C2 4 x

__global__ void __launch_bounds__(256) tv_normalize_kernel(const double2* __restrict__ li, const double2* __restrict__ lj,
                                                          const int* __restrict__ nkept, int cap, int min_points, double k0, double k1,
                                                          double k2, double k3, double k4, double k5, double k6, double k7, double k8,
                                                          double2* __restrict__ xi, double2* __restrict__ xj, int* __restrict__ neff) {
  const int pair = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = nkept[pair];
  n = n < 0 ? 0 : (n > cap ? cap : n);
  if (n < min_points) n = 0;
  if (i == 0) neff[pair] = n;
  if (i >= n) return;
  const size_t o = (size_t)pair * cap + i;
  // Kinv * (u, v, 1) then divide by z (:498-501; Mat33 * Vec3 of linalg.hpp:70-76: left-to-right sums, no contraction)
  const double2 p = li[o], q = lj[o];
  const double pa = k0 * p.x + k1 * p.y + k2 * 1.0, pb = k3 * p.x + k4 * p.y + k5 * 1.0, pc = k6 * p.x + k7 * p.y + k8 * 1.0;
  const double qa = k0 * q.x + k1 * q.y + k2 * 1.0, qb = k3 * q.x + k4 * q.y + k5 * 1.0, qc = k6 * q.x + k7 * q.y + k8 * 1.0;
  xi[o] = make_double2(pa / pc, pb / pc);
  xj[o] = make_double2(qa / qc, qb / qc);
}

// `want` draws of uniform_int_distribution<int>(0, n-1) from the raw 32-bit stream: raw value g is accepted iff
// low32(g * n) >= (2^32 - n) % n, its draw is high32(g * n); accepted values keep their order.  One block per set.
__global__ void __launch_bounds__(1024) tv_sample_kernel(const unsigned* __restrict__ raw, int raw_n, const int* __restrict__ npts,
                                                        int n_single, int want, int* __restrict__ idx, int* __restrict__ flags) {
  __shared__ int wcnt[32], wpre[32];
  __shared__ int base, total;
  const int pair = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = npts ? npts[pair] : n_single;
  if (n < 1 || (npts && n < 8)) return;
  idx += (size_t)pair * want;
  const unsigned range = (unsigned)n, threshold = (0u - range) % range;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int s = 0; s < raw_n; s += 1024) {
    const int i = s + tid;
    unsigned long long prod = 0;
    bool ok = false;
    if (i < raw_n) {
      prod = (unsigned long long)raw[i] * range;
      ok = (unsigned)prod >= threshold;
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
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
    if (ok) {
      const int r = base + wpre[warp] + __popc(m & ((1u << lane) - 1u));
      if (r < want) idx[r] = (int)(prod >> 32);
    }
    __syncthreads();
    if (tid == 0) base += total;
    __syncthreads();
    if (base >= want) return;
  }
  if (tid == 0 && base < want) atomicOr(flags, 1);
}

// Early stop (exact).  The scoring loop keeps the FIRST hypothesis with the largest count (:673, strict >) and a count cannot
// exceed the number of points, so once some hypothesis h explains ALL n points of a pair no later hypothesis can replace the
// winner: the winner is the lowest such h, and nothing after it has to be solved or scored.  With the reference's thresholds
// (2e-3 / 1e-3 on the Sampson error in normalised coordinates: tens of pixels) that is the common case.  The stage therefore
// scores the first TV_EARLY_H hypotheses of every pair, and this kernel takes the pairs that already hold a full count out
// of the rest of the launch set (n2 = 0: the solver and count kernels skip sets with fewer than 8 points); their remaining
// counts stay 0, so the arg-max finds the same winner, and the inlier list, count and pose come from it as before.
constexpr int TV_EARLY_H = 128;  // = one hypothesis chunk of the batched count kernel

__global__ void __launch_bounds__(128) tv_early_kernel(const int* __restrict__ counts, int H, int h1, const int* __restrict__ neff,
                                                      int* __restrict__ neff2, int* __restrict__ n_early) {
  const int pair = blockIdx.x, n = neff[pair];
  bool full = false;
  if (n >= 8)
    for (int h = threadIdx.x; h < h1; h += blockDim.x) full |= counts[(size_t)pair * H + h] == n;
  const int any = __syncthreads_or(full ? 1 : 0);
  if (threadIdx.x == 0) {
    neff2[pair] = any ? 0 : n;
    if (any) atomicAdd(n_early, 1);
  }
}

// status (0 skipped by min_points, 1 no pose: n < 8 or best < min_inliers, 2 pose wanted) and the winner's hypothesis
__global__ void tv_finalize_kernel(const int* __restrict__ nkept, const int* __restrict__ neff, const int* __restrict__ best,
                                   const double* __restrict__ E, int H, int npairs, int min_points, int min_inliers,
                                   int* __restrict__ status, double* __restrict__ bestE) {
  const int pair = blockIdx.x * blockDim.x + threadIdx.x;
  if (pair >= npairs) return;
  const int n = neff[pair], bh = best[2 * pair], bn = best[2 * pair + 1];
  int st;
  if (nkept[pair] < min_points) st = 0;
  else if (n < 8 || bn < min_inliers) st = 1;
  else st = 2;
  status[pair] = st;
  for (int i = 0; i < 9; i++) bestE[(size_t)pair * 9 + i] = (n >= 8 && bh >= 0) ? E[((size_t)pair * H + bh) * 9 + i] : 0.0;  // bestE starts as Mat33{}
}

bool invert_K_host(const double* K, double* o) {
  const double d = K[0] * (K[4] * K[8] - K[5] * K[7]) - K[1] * (K[3] * K[8] - K[5] * K[6]) + K[2] * (K[3] * K[7] - K[4] * K[6]);
  if (fabs(d) < 1e-12) return false;
  o[0] = (K[4] * K[8] - K[5] * K[7]) / d;
  o[1] = -(K[1] * K[8] - K[2] * K[7]) / d;
  o[2] = (K[1] * K[5] - K[2] * K[4]) / d;
  o[3] = -(K[3] * K[8] - K[5] * K[6]) / d;
  o[4] = (K[0] * K[8] - K[2] * K[6]) / d;
  o[5] = -(K[0] * K[5] - K[2] * K[3]) / d;
  o[6] = (K[3] * K[7] - K[4] * K[6]) / d;
  o[7] = -(K[0] * K[7] - K[1] * K[6]) / d;
  o[8] = (K[0] * K[4] - K[1] * K[3]) / d;
  return true;
}

// mt19937(12345) raw outputs, resident: enough for `draws` accepted values when at most `rej_frac` of the raw values are
// rejected (rejection probability of range n is (2^32 mod n) / 2^32 < n / 2^32).
int raw_stream(sfmgpu_ctx* ctx, DevBuf& buf, int& have, long long draws, double rej_frac) {
  const long long need = (long long)((double)draws / (1.0 - rej_frac) * 1.02) + 2048;
  if (need <= have) return 0;
  if (need > (1ll << 30)) return sfm_fail(ctx, SFMGPU_E_ARG, "ransac: %lld random draws are more than the sampler supports", draws);
  std::vector<unsigned> h((size_t)need);
  std::mt19937 rng(12345);  // :657
  for (auto& v : h) v = (unsigned)rng();
  SFM_TRY(sfm_reserve(ctx, buf, (size_t)need * 4));
  SFM_CUDA(ctx, cudaMemcpyAsync(buf.p, h.data(), (size_t)need * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // h goes out of scope
  have = (int)need;
  return 0;
}

// Result sets that did not go through the stage (a tracker step that reset the sequence instead of tracking it): status
// SKIPPED and winner / count (-1, 0), what the stage leaves for a set below min_points.  n_in: only sets with n_in[s] == 0
// (nullptr: every set).
__global__ void tv_skip_kernel(const int* __restrict__ n_in, int nsets, int* __restrict__ status, int* __restrict__ best) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nsets || (n_in && n_in[s] != 0)) return;
  status[s] = SFMGPU_TV_SKIPPED;
  best[2 * s] = -1;
  best[2 * s + 1] = 0;
}

// The stage's state for max_sets result sets of cap rows each (no-op when *tvp exists).
int tv_alloc(sfmgpu_ctx* ctx, TwoViewState** tvp, int max_sets, int cap) {
  if (*tvp) return 0;
  TwoViewState* tv = new TwoViewState();
  const size_t n = (size_t)max_sets * cap, P = (size_t)max_sets;
  cudaError_t e = cudaSuccess;
  auto al = [&](void** q, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(q, bytes + 256);
  };
  al((void**)&tv->xi, n * 16);
  al((void**)&tv->xj, n * 16);
  al((void**)&tv->inl, n * 4);
  al((void**)&tv->neff, P * 4);
  al((void**)&tv->status, P * 4);
  al((void**)&tv->best, P * 8);
  al((void**)&tv->bestE, P * 72);
  al((void**)&tv->R, P * 72);
  al((void**)&tv->t, P * 24);
  al((void**)&tv->flags, 64);
  if (e == cudaSuccess) e = cudaMemsetAsync(tv->flags, 0, 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(tv->status, 0, P * 4, ctx->stream);
  *tvp = tv;
  if (e != cudaSuccess) {
    sfm_two_view_free(ctx, tvp);
    return sfm_fail(ctx, SFMGPU_E_CUDA, "ransac stage: cudaMalloc failed: %s", cudaGetErrorString(e));
  }
  return 0;
}

}  // namespace

void sfm_two_view_free(sfmgpu_ctx* ctx, TwoViewState** tvp) {
  (void)ctx;
  TwoViewState* tv = *tvp;
  if (!tv) return;
  void* ptrs[] = {tv->xi, tv->xj, tv->inl, tv->neff, tv->status, tv->best, tv->bestE, tv->R, tv->t, tv->flags, tv->idx8.p, tv->E.p, tv->counts.p, tv->neff2.p, tv->raw.p};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  delete tv;
  *tvp = nullptr;
}

// The stage for result sets [pair_off, pair_off + npairs) on the context's CURRENT stream (the KLT stream of the chunk
// pipeline: the scratch is used by one chunk at a time).  Set k's correspondences are li/lj [k][cap], the first nkept[k]
// valid (a pairs batch: its survivors per pair; the lock-step tracker: the survivors of every sequence in track order).
// E_host: optional caller hypotheses [npairs][iters][9].
int sfm_two_view_stage(sfmgpu_ctx* ctx, TwoViewState* tv, const double2* li, const double2* lj, const int* nkept, int cap, int pair_off,
                       int npairs, const double* E_host) {
  if (!tv || npairs <= 0) return 0;
  const sfmgpu_ransac_cfg& rc = tv->rc;
  const int H = rc.iters > 0 ? rc.iters : 0;
  const int Hs = H > 0 ? H : 1;
  const int chunk = npairs < TV_CHUNK ? npairs : TV_CHUNK;
  SFM_TRY(sfm_reserve(ctx, tv->E, (size_t)chunk * Hs * 72));
  SFM_TRY(sfm_reserve(ctx, tv->counts, (size_t)chunk * Hs * 4));
  if (!E_host) {
    SFM_TRY(sfm_reserve(ctx, tv->idx8, (size_t)chunk * Hs * 32));
    SFM_TRY(raw_stream(ctx, tv->raw, tv->raw_n, (long long)H * 8, (double)cap / 4294967296.0));
  }
  const int mp = rc.min_points > 0 ? rc.min_points : 0;
  const int screen = (!E_host && H > 0 && sfm_solver_screens(ctx, chunk, H)) ? 1 : 0;  // see solver.cu: eight_point_qr_kernel
  // early stop: the device solver's own hypotheses, more than one probe's worth of them, not the whole-set test solver
  const bool early = ctx->rs_early && !E_host && H > 2 * TV_EARLY_H && ctx->solver_mode != 2;
  if (early) SFM_TRY(sfm_reserve(ctx, tv->neff2, (size_t)chunk * sizeof(int)));
  const double* k = tv->Kinv;
  for (int c0 = 0; c0 < npairs; c0 += chunk) {
    const int pc = npairs - c0 < chunk ? npairs - c0 : chunk, po = pair_off + c0;
    const size_t so = (size_t)po * cap;
    SFM_LAUNCH(ctx, tv_normalize_kernel, dim3(sfm_cdiv(cap, 256), pc), 256, 0, li + so, lj + so, nkept + po, cap, mp, k[0], k[1], k[2],
               k[3], k[4], k[5], k[6], k[7], k[8], tv->xi + so, tv->xj + so, tv->neff + po);
    if (H > 0) {
      if (E_host) {
        SFM_CUDA(ctx, cudaMemcpyAsync(tv->E.p, E_host + (size_t)c0 * H * 9, (size_t)pc * H * 72, cudaMemcpyHostToDevice, ctx->stream));
      } else {
        SFM_LAUNCH(ctx, tv_sample_kernel, pc, 1024, 0, (const unsigned*)tv->raw.p, tv->raw_n, (const int*)(tv->neff + po), 0, H * 8,
                   (int*)tv->idx8.p, tv->flags);
        if (!early)
          SFM_TRY(sfm_eight_point_batched(ctx, tv->xi + so, tv->xj + so, (size_t)cap, tv->neff + po, 0, pc, (const int*)tv->idx8.p, H,
                                          (double*)tv->E.p, screen));
      }
    }
    if (early) {
      // (the octets above are sampled for all H hypotheses: cheap, and the winner's octet is needed either way)
      const int scr = screen && sfm_solver_screens(ctx, pc, H);  // one decision for both parts of the set
      const double2 *cxi = tv->xi + so, *cxj = tv->xj + so;
      int* n2 = (int*)tv->neff2.p;
      SFM_CUDA(ctx, cudaMemsetAsync(tv->counts.p, 0, (size_t)pc * H * sizeof(int), ctx->stream));
      SFM_TRY(sfm_eight_point_range(ctx, cxi, cxj, (size_t)cap, tv->neff + po, 0, pc, (const int*)tv->idx8.p, H, 0, TV_EARLY_H, (double*)tv->E.p, scr));
      SFM_TRY(sfm_ransac_count_range(ctx, cxi, cxj, (size_t)cap, tv->neff + po, cap, pc, (const double*)tv->E.p, H, 0, TV_EARLY_H, rc.thr,
                                     (int*)tv->counts.p));
      SFM_LAUNCH(ctx, tv_early_kernel, pc, 128, 0, (const int*)tv->counts.p, H, TV_EARLY_H, (const int*)(tv->neff + po), n2, tv->flags + 1);
      SFM_TRY(sfm_eight_point_range(ctx, cxi, cxj, (size_t)cap, (const int*)n2, 0, pc, (const int*)tv->idx8.p, H, TV_EARLY_H, H, (double*)tv->E.p, scr));
      SFM_TRY(sfm_ransac_count_range(ctx, cxi, cxj, (size_t)cap, (const int*)n2, cap, pc, (const double*)tv->E.p, H, TV_EARLY_H, H, rc.thr,
                                     (int*)tv->counts.p));
      SFM_TRY(sfm_ransac_finish(ctx, cxi, cxj, (size_t)cap, tv->neff + po, cap, pc, (double*)tv->E.p, H, rc.thr, (const int*)tv->counts.p,
                                tv->best + 2 * po, tv->inl + so, screen ? (const int*)tv->idx8.p : nullptr));
    } else {
      SFM_TRY(sfm_ransac_score_batched(ctx, tv->xi + so, tv->xj + so, (size_t)cap, tv->neff + po, cap, pc, (double*)tv->E.p, H, rc.thr,
                                       (int*)tv->counts.p, tv->best + 2 * po, tv->inl + so, screen ? (const int*)tv->idx8.p : nullptr));
    }
    SFM_LAUNCH(ctx, tv_finalize_kernel, sfm_cdiv(pc, 128), 128, 0, nkept + po, (const int*)(tv->neff + po),
               (const int*)(tv->best + 2 * po), (const double*)tv->E.p, Hs, pc, mp, rc.min_inliers, tv->status + po, tv->bestE + 9 * (size_t)po);
    SFM_TRY(sfm_pose_batched(ctx, tv->xi + so, tv->xj + so, (size_t)cap, pc, tv->status + po, tv->best + 2 * po, tv->inl + so,
                             tv->bestE + 9 * (size_t)po, tv->R + 9 * (size_t)po, tv->t + 3 * (size_t)po));
  }
  return 0;
}

bool sfm_two_view_enabled(const TwoViewState* tv) { return tv && tv->enabled; }

int sfm_two_view_skip(sfmgpu_ctx* ctx, TwoViewState* tv, const int* n_in, int nsets) {
  if (!tv || nsets <= 0) return 0;
  SFM_LAUNCH(ctx, tv_skip_kernel, sfm_cdiv(nsets, 128), 128, 0, n_in, nsets, tv->status, tv->best);
  return 0;
}

// H index octets of find_E_ransac's seeded sampling (:657-665) for ONE set of n correspondences into d_idx8 [H][8], from the
// context's resident mt19937(12345) stream; *d_flag (device, 4 bytes, zeroed here) becomes non-zero if the stream was too
// short (it is sized with a margin: cannot happen, the caller checks).
int sfm_sample_octets(sfmgpu_ctx* ctx, int n, int H, int* d_idx8, int* d_flag) {
  if (H <= 0) return 0;
  const double rej = (double)(4294967296ull % (unsigned long long)n) / 4294967296.0;
  SFM_TRY(raw_stream(ctx, ctx->rs_raw, ctx->rs_raw_n, (long long)H * 8, rej));
  SFM_CUDA(ctx, cudaMemsetAsync(d_flag, 0, 4, ctx->stream));
  SFM_LAUNCH(ctx, tv_sample_kernel, 1, 1024, 0, (const unsigned*)ctx->rs_raw.p, ctx->rs_raw_n, (const int*)nullptr, n, H * 8, d_idx8, d_flag);
  return 0;
}

// D2H of the stage's per-set results for sets [pair_off, pair_off + npairs) (cap inlier rows each) into the registered host
// outputs, on `s`.
int sfm_two_view_download(sfmgpu_ctx* ctx, TwoViewState* tv, int cap_rows, int pair_off, int npairs, cudaStream_t s) {
  if (!tv || npairs <= 0) return 0;
  const size_t o = (size_t)pair_off, np_ = (size_t)npairs, cap = (size_t)cap_rows;
  if (tv->h_status) SFM_CUDA(ctx, cudaMemcpyAsync(tv->h_status + o, tv->status + o, np_ * 4, cudaMemcpyDeviceToHost, s));
  if (tv->h_best_n)
    SFM_CUDA(ctx, cudaMemcpy2DAsync(tv->h_best_n + o, 4, tv->best + 2 * o + 1, 8, 4, np_, cudaMemcpyDeviceToHost, s));
  if (tv->h_inl) SFM_CUDA(ctx, cudaMemcpyAsync(tv->h_inl + o * cap, tv->inl + o * cap, np_ * cap * 4, cudaMemcpyDeviceToHost, s));
  if (tv->h_R) SFM_CUDA(ctx, cudaMemcpyAsync(tv->h_R + 9 * o, tv->R + 9 * o, np_ * 72, cudaMemcpyDeviceToHost, s));
  if (tv->h_t) SFM_CUDA(ctx, cudaMemcpyAsync(tv->h_t + 3 * o, tv->t + 3 * o, np_ * 24, cudaMemcpyDeviceToHost, s));
  return 0;
}

// Checks K and the configuration, allocates *tvp for max_sets sets of cap rows on first use, stores both and switches the
// stage on (rc == nullptr: off again).  `who` names the entry point in error messages.
int sfm_two_view_configure(sfmgpu_ctx* ctx, TwoViewState** tvp, int max_sets, int cap, const double* K, const sfmgpu_ransac_cfg* rc,
                           const char* who) {
  if (!rc) {
    if (*tvp) (*tvp)->enabled = false;
    return 0;
  }
  if (!K) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null K", who);
  if (rc->iters < 0 || rc->iters > (1 << 24)) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: bad iteration count", who);
  double Ki[9];
  if (!invert_K_host(K, Ki)) return sfm_fail(ctx, SFMGPU_E_ARG, "Singular K");  // the reference throws "Singular K" (:474)
  SFM_TRY(tv_alloc(ctx, tvp, max_sets, cap));
  TwoViewState* tv = *tvp;
  tv->rc = *rc;
  for (int i = 0; i < 9; i++) tv->Kinv[i] = Ki[i];
  tv->enabled = true;
  return 0;
}

// Sets stopped early since the last call (reads and resets the counter; synchronises).
int sfm_two_view_early(sfmgpu_ctx* ctx, TwoViewState* tv, long long* stopped) {
  *stopped = 0;
  if (!tv) return 0;
  int v = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&v, tv->flags + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemsetAsync(tv->flags + 1, 0, 4, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *stopped = v;
  return 0;
}

// Results of sets [0, nsets) into the given host arrays (any may be null; layout of sfmgpu_pairs_ransac_host_outputs with
// cap inlier rows per set); synchronises.
int sfm_two_view_download_all(sfmgpu_ctx* ctx, TwoViewState* tv, int cap, int nsets, int32_t* status, int32_t* best_n, int32_t* inliers,
                              double* R, double* t, const char* who) {
  TwoViewState saved = *tv;
  tv->h_status = status;
  tv->h_best_n = best_n;
  tv->h_inl = inliers;
  tv->h_R = R;
  tv->h_t = t;
  int rcode = sfm_two_view_download(ctx, tv, cap, 0, nsets, ctx->stream);
  tv->h_status = saved.h_status;
  tv->h_best_n = saved.h_best_n;
  tv->h_inl = saved.h_inl;
  tv->h_R = saved.h_R;
  tv->h_t = saved.h_t;
  SFM_TRY(rcode);
  int flag = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&flag, tv->flags, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (flag) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "%s: the random stream was too short (internal)", who);
  return 0;
}

extern "C" {

int sfmgpu_pairs_set_ransac(sfmgpu_ctx* ctx, sfmgpu_pairs* p, const double* K, const sfmgpu_ransac_cfg* rc) {
  SFM_ENTER(ctx);
  if (!ctx || !p) return SFMGPU_E_ARG;
  return sfm_two_view_configure(ctx, &p->tv, p->max_pairs, p->cap, K, rc, "pairs_set_ransac");
}

int sfmgpu_ransac_set_early_stop(sfmgpu_ctx* ctx, int on) {
  if (!ctx) return SFMGPU_E_ARG;
  ctx->rs_early = on ? 1 : 0;
  return 0;
}

int sfmgpu_pairs_ransac_early(sfmgpu_ctx* ctx, sfmgpu_pairs* p, long long* pairs_stopped) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !pairs_stopped) return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_ransac_early: null pointer");
  return sfm_two_view_early(ctx, p->tv, pairs_stopped);
}

int sfmgpu_pairs_ransac_host_outputs(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int32_t* status, int32_t* best_n, int32_t* inliers, double* R,
                                     double* t) {
  SFM_ENTER(ctx);
  if (!ctx || !p) return SFMGPU_E_ARG;
  SFM_TRY(tv_alloc(ctx, &p->tv, p->max_pairs, p->cap));
  p->tv->h_status = status;
  p->tv->h_best_n = best_n;
  p->tv->h_inl = inliers;
  p->tv->h_R = R;
  p->tv->h_t = t;
  return 0;
}

int sfmgpu_pairs_ransac(sfmgpu_ctx* ctx, sfmgpu_pairs* p, const double* K, const sfmgpu_ransac_cfg* rc, const double* E_host) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !rc) return SFMGPU_E_ARG;
  const bool was_enabled = p->tv && p->tv->enabled;
  SFM_TRY(sfmgpu_pairs_set_ransac(ctx, p, K, rc));
  p->tv->enabled = was_enabled;  // an explicit call does not change what the front end does
  SFM_TRY(sfm_two_view_stage(ctx, p->tv, p->li, p->lj, p->nkept, p->cap, 0, p->last_npairs, E_host));
  if (E_host) SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the caller's hypotheses were read asynchronously
  return 0;
}

int sfmgpu_pairs_ransac_download(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int pair, int* status, int* best_h, int* best_n, int32_t* inliers,
                                 int cap, double* E9, double* R9, double* t3) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !p->tv) return sfm_fail(ctx, SFMGPU_E_STATE, "pairs_ransac_download: the RANSAC stage has not run");
  if (pair < 0 || pair >= p->last_npairs) return sfm_fail(ctx, SFMGPU_E_ARG, "pairs_ransac_download: bad pair index");
  TwoViewState* tv = p->tv;
  int st = 0, b[2] = {-1, 0}, flag = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&st, tv->status + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(b, tv->best + 2 * pair, 8, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(&flag, tv->flags, 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (E9) SFM_CUDA(ctx, cudaMemcpyAsync(E9, tv->bestE + 9 * (size_t)pair, 72, cudaMemcpyDeviceToHost, ctx->stream));
  if (R9) SFM_CUDA(ctx, cudaMemcpyAsync(R9, tv->R + 9 * (size_t)pair, 72, cudaMemcpyDeviceToHost, ctx->stream));
  if (t3) SFM_CUDA(ctx, cudaMemcpyAsync(t3, tv->t + 3 * (size_t)pair, 24, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (flag) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pairs_ransac: the random stream was too short (internal)");
  if (status) *status = st;
  if (best_h) *best_h = b[0];
  if (best_n) *best_n = b[1];
  if (inliers && st != 0 && b[0] >= 0 && b[1] > 0) {
    if (b[1] > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "pairs_ransac_download: %d inliers, room for %d", b[1], cap);
    SFM_CUDA(ctx, cudaMemcpyAsync(inliers, tv->inl + (size_t)pair * p->cap, (size_t)b[1] * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

int sfmgpu_pairs_ransac_download_all(sfmgpu_ctx* ctx, sfmgpu_pairs* p, int32_t* status, int32_t* best_n, int32_t* inliers, double* R,
                                     double* t) {
  SFM_ENTER(ctx);
  if (!ctx || !p || !p->tv) return sfm_fail(ctx, SFMGPU_E_STATE, "pairs_ransac_download_all: the RANSAC stage has not run");
  return sfm_two_view_download_all(ctx, p->tv, p->cap, p->last_npairs, status, best_n, inliers, R, t, "pairs_ransac");
}

int sfmgpu_pairs_ransac_device_ptrs(sfmgpu_pairs* p, void** status, void** best, void** inliers, void** R, void** t) {
  if (!p || !p->tv) return SFMGPU_E_STATE;
  if (status) *status = p->tv->status;
  if (best) *best = p->tv->best;
  if (inliers) *inliers = p->tv->inl;
  if (R) *R = p->tv->R;
  if (t) *t = p->tv->t;
  return 0;
}

// `count` draws of std::uniform_int_distribution<int>(0, n-1) on std::mt19937(12345), computed on the device (:657-665).
int sfmgpu_ransac_sample(sfmgpu_ctx* ctx, int n, int count, int32_t* out) {
  SFM_ENTER(ctx);
  if (!ctx || n < 1 || count < 0 || (count > 0 && !out)) return sfm_fail(ctx, SFMGPU_E_ARG, "ransac_sample: bad arguments");
  if (count == 0) return 0;
  const double rej = (double)(4294967296ull % (unsigned long long)n) / 4294967296.0;
  DevBuf raw;
  int have = 0;
  SFM_TRY(raw_stream(ctx, raw, have, count, rej));
  SFM_TRY(sfm_reserve(ctx, ctx->rs_idx8, (size_t)count * 4 + 64));
  int* flag = (int*)((char*)ctx->rs_idx8.p + (((size_t)count * 4 + 15) & ~(size_t)15));
  cudaError_t e = cudaMemsetAsync(flag, 0, 4, ctx->stream);
  if (e == cudaSuccess) {
    tv_sample_kernel<<<1, 1024, 0, ctx->stream>>>((const unsigned*)raw.p, have, nullptr, n, count, (int*)ctx->rs_idx8.p, flag);
    ctx->launches++;
    e = cudaGetLastError();
  }
  int hflag = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, ctx->rs_idx8.p, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(raw.p);
  if (e != cudaSuccess) return sfm_fail(ctx, SFMGPU_E_CUDA, "ransac_sample: %s", cudaGetErrorString(e));
  if (hflag) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "ransac_sample: the random stream was too short (internal)");
  return 0;
}

}  // extern "C"
