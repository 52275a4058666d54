// shim_two_view_capi.cpp — flat C wrappers around MultiKLTTracker::set_two_view and two_view_results (host/sfmgpu_shim.hpp,
// host/sfmgpu_two_view.hpp) so that the tests can drive the lock-step tracker's find_E_ransac stage through the C++ shim
// with ctypes.  Test plumbing, built into libsfmshim_tv.so.
#define SFMGPU_SHIM_STANDALONE
#include "sfmgpu_shim.hpp"

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
}  // namespace

extern "C" {

const char* shim_tv_last_error() { return g_err.c_str(); }

void* shim_tv_create(int n_sequences, int w, int h, int max_tracks, int min_tracks) {
  try {
    LKConfig c;
    c.max_tracks = max_tracks;
    c.min_tracks = min_tracks;
    return new MultiKLTTracker(c, n_sequences, w, h);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}

void shim_tv_destroy(void* t) { delete (MultiKLTTracker*)t; }

int shim_tv_set_two_view(void* t, const double* K, int iters, double thr, int min_inliers) {
  return guarded([&] {
    Mat33 Km;
    for (int i = 0; i < 9; i++) Km.a[i] = K[i];
    ((MultiKLTTracker*)t)->set_two_view(Km, iters, thr, min_inliers);
    return 0;
  });
}

// One step on pix = [n_sequences][h][w]: survivor ids [n_sequences][cap] and counts n_out; then per sequence the
// std::optional<RelPose> of two_view_results: has[s] = 1 (RelPose) or 0 (std::nullopt), R [S][9], t [S][3], inliers
// [S][cap] (first n_inl[s] valid).
int shim_tv_step(void* t, const uint8_t* pix, int n_sequences, int w, int h, int* ids, int* n_out, int cap, int* has, double* R,
                 double* tv, int* inliers, int* n_inl) {
  return guarded([&] {
    std::vector<GrayImage> imgs((size_t)n_sequences);
    std::vector<const GrayImage*> ptrs;
    for (int s = 0; s < n_sequences; s++) {
      imgs[s].w = w;
      imgs[s].h = h;
      imgs[s].pix.assign(pix + (size_t)s * w * h, pix + (size_t)(s + 1) * w * h);
      ptrs.push_back(&imgs[s]);
    }
    auto* mt = (MultiKLTTracker*)t;
    const auto out = mt->step(ptrs);
    const auto res = two_view_results(*mt);
    for (int s = 0; s < n_sequences; s++) {
      n_out[s] = (int)out[s].ids.size();
      for (int i = 0; i < n_out[s] && i < cap; i++) ids[(size_t)s * cap + i] = out[s].ids[i];
      has[s] = res[s] ? 1 : 0;
      n_inl[s] = 0;
      if (!res[s]) continue;
      for (int i = 0; i < 9; i++) R[9 * (size_t)s + i] = res[s]->R_ji.a[i];
      tv[3 * (size_t)s] = res[s]->t_ji.x;
      tv[3 * (size_t)s + 1] = res[s]->t_ji.y;
      tv[3 * (size_t)s + 2] = res[s]->t_ji.z;
      n_inl[s] = (int)res[s]->inliers.size();
      for (int i = 0; i < n_inl[s] && i < cap; i++) inliers[(size_t)s * cap + i] = res[s]->inliers[i];
    }
    return 0;
  });
}
}
