// multitracker_sizes_shim.cpp — flat C wrappers around the drop-in shim (host/sfmgpu_shim.hpp) for
// tests/test_gpu_multitracker_sizes.py: a MultiKLTTracker over sequences of their own sizes with one camera per sequence, and the
// per-sequence alternative it replaces, a KLTTracker plus find_E_ransac.  Test plumbing.
#define SFMGPU_SHIM_STANDALONE
#include "sfmgpu_shim.hpp"

#include <string>
#include <utility>
#include <vector>

namespace {
thread_local std::string g_err;
template <class F>
int guarded(F&& f) {
  try {
    return f();
  } catch (const std::exception& e) {
    g_err = e.what();
    return -1000;
  }
}

// points [n][2] of a step's output
void put_pts(const std::vector<Vec2>& p, double* xy, int cap) {
  for (int i = 0; i < (int)p.size() && i < cap; i++) {
    xy[2 * i] = p[i].x;
    xy[2 * i + 1] = p[i].y;
  }
}

// has = 1 and R [9], t [3], inliers (n_inl) for a pose; 0 for std::nullopt
int put_pose(const std::optional<RelPose>& r, double* R, double* t, int* inl, int* n_inl, int cap) {
  *n_inl = 0;
  if (!r) return 0;
  for (int i = 0; i < 9; i++) R[i] = r->R_ji.a[i];
  t[0] = r->t_ji.x;
  t[1] = r->t_ji.y;
  t[2] = r->t_ji.z;
  *n_inl = (int)r->inliers.size();
  for (int i = 0; i < *n_inl && i < cap; i++) inl[i] = r->inliers[i];
  return 1;
}
}  // namespace

extern "C" {

const char* msz_last_error() { return g_err.c_str(); }

// Sequence s has images of w[s] x h[s].
void* msz_create(int n_sequences, const int* w, const int* h, int max_tracks, int min_tracks) {
  try {
    LKConfig c;
    c.max_tracks = max_tracks;
    c.min_tracks = min_tracks;
    std::vector<std::pair<int, int>> sizes;
    for (int s = 0; s < n_sequences; s++) sizes.push_back({w[s], h[s]});
    return new MultiKLTTracker(c, sizes);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
void msz_destroy(void* t) { delete (MultiKLTTracker*)t; }

// K [n_sequences][9]: the camera of every sequence.
int msz_set_two_view(void* t, int n_sequences, const double* K, int iters, double thr, int min_inliers) {
  return guarded([&] {
    std::vector<Mat33> Ks((size_t)n_sequences);
    for (int s = 0; s < n_sequences; s++)
      for (int i = 0; i < 9; i++) Ks[s].a[i] = K[9 * (size_t)s + i];
    ((MultiKLTTracker*)t)->set_two_view(Ks, iters, thr, min_inliers);
    return 0;
  });
}

// One step on frames given one by one (pix[s], w[s] x h[s]): per sequence s its survivors in rows s * cap of ids / prev / cur
// (count n_out[s]), then two_view_results: has[s], R [S][9], t [S][3], inliers [S][cap] (first n_inl[s]).
int msz_step(void* t, int n_sequences, const uint8_t* const* pix, const int* w, const int* h, int* ids, double* prev, double* cur,
             int* n_out, int cap, int* has, double* R, double* tv, int* inliers, int* n_inl) {
  return guarded([&] {
    std::vector<GrayImage> imgs((size_t)n_sequences);
    std::vector<const GrayImage*> ptrs;
    for (int s = 0; s < n_sequences; s++) {
      imgs[s].w = w[s];
      imgs[s].h = h[s];
      imgs[s].pix.assign(pix[s], pix[s] + (size_t)w[s] * h[s]);
      ptrs.push_back(&imgs[s]);
    }
    auto* mt = (MultiKLTTracker*)t;
    const auto out = mt->step(ptrs);
    const auto res = two_view_results(*mt);
    for (int s = 0; s < n_sequences; s++) {
      const size_t o = (size_t)s * cap;
      n_out[s] = (int)out[s].ids.size();
      for (int i = 0; i < n_out[s] && i < cap; i++) ids[o + i] = out[s].ids[i];
      put_pts(out[s].prev_pts, prev + 2 * o, cap);
      put_pts(out[s].cur_pts, cur + 2 * o, cap);
      has[s] = put_pose(res[s], R + 9 * (size_t)s, tv + 3 * (size_t)s, inliers + o, n_inl + s, cap);
    }
    return 0;
  });
}

void* msz_single_create(int max_tracks, int min_tracks) {
  try {
    LKConfig c;
    c.max_tracks = max_tracks;
    c.min_tracks = min_tracks;
    return new KLTTracker(c);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
void msz_single_destroy(void* t) { delete (KLTTracker*)t; }

// KLTTracker::step, then find_E_ransac(K, prev_pts, cur_pts, ...) where it has survivors (:1715): has = 1 with R, t, inliers.
int msz_single_step(void* t, const uint8_t* pix, int w, int h, const double* K, int iters, double thr, int min_inliers, int* ids,
                    double* prev, double* cur, int* n_out, int cap, int* has, double* R, double* tv, int* inliers, int* n_inl) {
  return guarded([&] {
    GrayImage g;
    g.w = w;
    g.h = h;
    g.pix.assign(pix, pix + (size_t)w * h);
    const auto o = ((KLTTracker*)t)->step(g);
    *n_out = (int)o.ids.size();
    for (int i = 0; i < *n_out && i < cap; i++) ids[i] = o.ids[i];
    put_pts(o.prev_pts, prev, cap);
    put_pts(o.cur_pts, cur, cap);
    *has = 0;
    *n_inl = 0;
    if (o.prev_pts.empty()) return 0;
    Mat33 Km;
    for (int i = 0; i < 9; i++) Km.a[i] = K[i];
    *has = put_pose(find_E_ransac(Km, o.prev_pts, o.cur_pts, iters, thr, min_inliers), R, tv, inliers, n_inl, cap);
    return 0;
  });
}
}
