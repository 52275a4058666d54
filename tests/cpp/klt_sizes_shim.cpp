// klt_sizes_shim.cpp — flat C wrappers around the drop-in shim (host/sfmgpu_shim.hpp) for tests/test_gpu_klt_sizes.py:
// KLTTracker reset / step / tracks at any image size, and track_one_public between live Pyramids.  Test plumbing.
#define SFMGPU_SHIM_STANDALONE
#include "sfmgpu_shim.hpp"

#include <cstring>
#include <string>

namespace {
GrayImage wrap(const uint8_t* pix, int w, int h) {
  GrayImage g;
  g.w = w;
  g.h = h;
  g.pix.assign(pix, pix + (size_t)w * h);
  return g;
}
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

const char* sz_last_error() { return g_err.c_str(); }

void* sz_tracker_create(int max_tracks, int min_tracks, int levels) {
  try {
    LKConfig lc;
    lc.max_tracks = max_tracks;
    lc.min_tracks = min_tracks;
    lc.pyr_levels = levels;
    return new KLTTracker(lc);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
void sz_tracker_destroy(void* t) { delete (KLTTracker*)t; }

int sz_tracker_reset(void* t, const uint8_t* pix, int w, int h) {
  return guarded([&] {
    ((KLTTracker*)t)->reset(wrap(pix, w, h));
    return 0;
  });
}

int sz_tracker_step(void* t, const uint8_t* pix, int w, int h, double* prev_xy, double* cur_xy, int* ids, int cap) {
  return guarded([&] {
    auto o = ((KLTTracker*)t)->step(wrap(pix, w, h));
    const int n = (int)o.ids.size();
    for (int i = 0; i < n && i < cap; i++) {
      prev_xy[2 * i] = o.prev_pts[i].x;
      prev_xy[2 * i + 1] = o.prev_pts[i].y;
      cur_xy[2 * i] = o.cur_pts[i].x;
      cur_xy[2 * i + 1] = o.cur_pts[i].y;
      ids[i] = o.ids[i];
    }
    return n;
  });
}

int sz_tracker_tracks(void* t, double* xy, int* ids, int cap) {
  const auto& tr = ((KLTTracker*)t)->tracks();
  const int n = (int)tr.size();
  for (int i = 0; i < n && i < cap; i++) {
    xy[2 * i] = tr[i].p.x;
    xy[2 * i + 1] = tr[i].p.y;
    ids[i] = tr[i].id;
  }
  return n;
}

void* sz_pyr_build(const uint8_t* pix, int w, int h, int levels) {
  try {
    return new Pyramid(build_pyr(wrap(pix, w, h), levels));
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
void sz_pyr_free(void* p) { delete (Pyramid*)p; }
int sz_same_pool(void* a, void* b) { return ((Pyramid*)a)->dev->pool == ((Pyramid*)b)->dev->pool ? 1 : 0; }

// out[2i..2i+1] = tracker.track_one_public(a, b, p[i]) for n points, one call each (:396-398)
int sz_track_one(void* t, void* a, void* b, const double* p, int n, double* out) {
  return guarded([&] {
    for (int i = 0; i < n; i++) {
      const Vec2 r = ((KLTTracker*)t)->track_one_public(*(Pyramid*)a, *(Pyramid*)b, Vec2{p[2 * i], p[2 * i + 1]});
      out[2 * i] = r.x;
      out[2 * i + 1] = r.y;
    }
    return 0;
  });
}

}  // extern "C"
