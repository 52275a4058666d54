// sfmgpu_shim.hpp — C++ source-compatible drop-in for the reference's front-end entry points, on top of the C ABI
// (include/sfmgpu.h).  Same names, parameter lists, return types, ordering guarantees and error behaviour as
// cpp/src/templering_sfm.cpp:
//     Pyramid build_pyr(const GrayImage&, int levels)                                   :220-232
//     std::vector<Vec2> shi_tomasi(const GrayImage&, int max_corners, double q, int d)  :237-302
//     struct LKConfig / struct Track / class KLTTracker {reset, step, tracks,
//                                                        track_one_public}             :307-466
//     struct RelPose; std::optional<RelPose> find_E_ransac(K, pi, pj, iters, thr, mi)   :640-761   (sfmgpu_two_view.hpp)
// plus one batched extra, track_pairs(), for callers that loop over track_one_public (:1845-1849).
//
// Two ways to use it (INTEGRATION.md):
//   * inside the reference TU: include this header after the reference's own headers (its sfm::GrayImage / Vec2 / Vec3 /
//     Mat33 are used as they are) in place of the reference's front-end definitions, and sfmgpu_two_view.hpp where the
//     reference defines RelPose / find_E_ransac (:640-761) - there the TU's OWN invert_K, norm_point, eight_point_E, svd3,
//     AtA_from_A and sfm::jacobi_eig_sym are in scope and are what find_E_ransac calls (nothing of them is restated);
//   * stand-alone: define SFMGPU_SHIM_STANDALONE first: the minimal PODs below are provided, two_view_host.hpp supplies
//     the host-side linear algebra, and sfmgpu_two_view.hpp is included at the end of this header.
//
// Errors: CUDA / library failures throw std::runtime_error (the reference's main catches std::exception at
// :1913); two-view failure is std::nullopt; step() on the first frame returns empty vectors.  There is no CPU
// fallback: without libsfmgpu.so and a GPU every call throws.
// Threading: like the reference, one calling thread and one process-wide context (device SFMGPU_DEVICE, default 0);
// find_E_ransac spreads its independent 8-point solves over a few host threads (link with -pthread).
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <optional>
#include <random>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/sfmgpu.h"
#ifdef SFMGPU_SHIM_STANDALONE
#include "two_view_host.hpp"  // stand-alone builds have no reference TU to take invert_K / eight_point_E / svd3 from
#endif

#ifdef SFMGPU_SHIM_STANDALONE
// Layout-compatible stand-ins for cpp/include/pgm_io.hpp:10-15 and cpp/include/linalg.hpp:15-35.
namespace sfm {
struct GrayImage {
  int w = 0, h = 0;
  std::vector<std::uint8_t> pix;
  std::uint8_t at(int x, int y) const { return pix[(size_t)y * w + x]; }
};
struct Vec2 {
  double x{}, y{};
};
struct Vec3 {
  double x{}, y{}, z{};
};
struct Mat33 {
  std::array<double, 9> a{};
  double& operator()(int r, int c) { return a[3 * r + c]; }
  double operator()(int r, int c) const { return a[3 * r + c]; }
};
}  // namespace sfm
using sfm::GrayImage;
using sfm::Mat33;
using sfm::Vec2;
using sfm::Vec3;
#endif

namespace sfmgpu_shim {

inline void check(sfmgpu_ctx* ctx, int rc, const char* what) {
  if (rc != 0) throw std::runtime_error(std::string("sfmgpu: ") + what + ": " + sfmgpu_last_error(ctx));
}

// Opt-in: minimal solver on the device (SURVEY.md §8f-1).  Default off: hypotheses come from the host solver and are
// bit-identical to the reference's.
inline bool& device_solver_flag() {
  static bool on = [] {
    const char* e = std::getenv("SFMGPU_DEVICE_SOLVER");
    return e && *e && *e != '0';
  }();
  return on;
}
inline bool device_solver() { return device_solver_flag(); }
// Host threads for the 8-point solves of find_E_ransac (SFMGPU_SOLVER_THREADS, default: the hardware's, at most 16).
inline int solver_threads() {
  static int n = [] {
    const char* e = std::getenv("SFMGPU_SOLVER_THREADS");
    int v = e && *e ? std::atoi(e) : (int)std::thread::hardware_concurrency();
    return v < 1 ? 1 : (v > 16 ? 16 : v);
  }();
  return n;
}
inline void set_device_solver(bool on) { device_solver_flag() = on; }

// Rows of a track list / of the per-sequence output arrays: max(max_tracks, min_tracks, 1) + 1 (see sfmgpu.h, tracker).
inline int track_rows(int max_tracks, int min_tracks) {
  int m = max_tracks < 1 ? 1 : max_tracks;
  if (min_tracks > m) m = min_tracks;
  return m + 1;
}

// Process-wide context.
inline sfmgpu_ctx* context() {
  static sfmgpu_ctx* ctx = [] {
    sfmgpu_ctx* c = nullptr;
    const char* dev = std::getenv("SFMGPU_DEVICE");
    if (sfmgpu_create(dev ? std::atoi(dev) : 0, &c) != 0)
      throw std::runtime_error("sfmgpu: no usable CUDA device (the GPU front end has no CPU fallback)");
    return c;
  }();
  return ctx;
}

// Device twin of one Pyramid: a slot in a small pool of equally sized frames, so that two pyramids of the same
// size (the only case the reference ever tracks between) live in one batch.
struct Pool {
  sfmgpu_frames* frames = nullptr;
  int w = 0, h = 0, levels = 0;
  std::vector<char> used;
  ~Pool() {
    if (frames) sfmgpu_frames_destroy(context(), frames);
  }
};
struct DevicePyr {
  std::shared_ptr<Pool> pool;
  int slot = -1;
  unsigned long long serial = 0;  // unique per build_pyr call (slots are reused, serials are not)
  unsigned long long imgkey = 0;  // content key of the level-0 image (image_key)
  ~DevicePyr() {
    if (pool && slot >= 0) pool->used[slot] = 0;
  }
};

// Content key of an image: size + a multiplicative hash over its 8-byte words (~0.05 ms per 640x480 image).
inline unsigned long long image_key(const GrayImage& im) {
  unsigned long long h = 0x9E3779B97F4A7C15ull ^ ((unsigned long long)(unsigned)im.w << 32) ^ (unsigned)im.h;
  const size_t n = im.pix.size(), nw = n / 8;
  const unsigned char* p = im.pix.data();
  for (size_t i = 0; i < nw; i++) {
    unsigned long long w;
    std::memcpy(&w, p + 8 * i, 8);
    h = (h ^ w) * 0xFF51AFD7ED558CCDull;
    h ^= h >> 29;
  }
  for (size_t i = nw * 8; i < n; i++) h = (h ^ p[i]) * 0x100000001B3ull;
  return h ? h : 1;
}

// ---- speculation behind track_one_public --------------------------------------------------------------------------------------
// The reference's loop-closure block (:1841-1852) detects corners on an image, builds two pyramids and then calls
// track_one_public twice per corner (forward, then backward from the result): 2 x 1200 launches + synchronisations, ~60 ms.
// The shim remembers the corners shi_tomasi last returned per image; the first track_one_public(a, b, p) whose point is one
// of the corners of a's image tracks ALL of them forward and backward in one batch (the kernel a single call runs, so
// every value is bit-identical to what the single calls would return) and answers this and the following calls - the
// forward ones by (a, b, corner), the backward ones by (b, a, forward result) - from that table.  Anything else (other
// points, other parameters) takes the single-call path.  SFMGPU_SPECULATE=0 turns it off.
struct CornerMemo {
  unsigned long long imgkey = 0;
  std::vector<Vec2> corners;
};
inline CornerMemo* corner_memos() {
  static CornerMemo m[2];
  return m;
}
inline void remember_corners(const GrayImage& im, const std::vector<Vec2>& c) {
  CornerMemo* m = corner_memos();
  m[1] = std::move(m[0]);
  m[0].imgkey = image_key(im);
  m[0].corners = c;
}
struct TrackKey {
  unsigned long long a, b, x, y;
  bool operator==(const TrackKey& o) const { return a == o.a && b == o.b && x == o.x && y == o.y; }
};
struct TrackKeyHash {
  size_t operator()(const TrackKey& k) const {
    unsigned long long h = k.a * 0x9E3779B97F4A7C15ull ^ k.b * 0xC2B2AE3D27D4EB4Full ^ k.x * 0xFF51AFD7ED558CCDull ^ (k.y + (k.y << 31));
    return (size_t)(h ^ (h >> 32));
  }
};
struct TrackMemo {
  unsigned long long a = 0, b = 0;  // pyramid serials of the speculated pair
  int radius = 0, iters = 0;
  std::unordered_map<TrackKey, Vec2, TrackKeyHash> table;
};
inline TrackMemo& track_memo() {
  static TrackMemo m;
  return m;
}
inline bool& speculate_flag() {
  static bool on = [] {
    const char* e = std::getenv("SFMGPU_SPECULATE");
    return !(e && e[0] == '0');
  }();
  return on;
}
inline bool speculate() { return speculate_flag(); }
inline void set_speculate(bool on) { speculate_flag() = on; }
inline unsigned long long dbits(double v) {
  unsigned long long u;
  std::memcpy(&u, &v, 8);
  return u;
}
inline std::shared_ptr<DevicePyr> acquire_slot(int w, int h, int levels) {
  static std::vector<std::shared_ptr<Pool>> pools;
  constexpr int SLOTS = 8;
  for (auto& p : pools)
    if (p->w == w && p->h == h && p->levels == levels)
      for (int s = 0; s < SLOTS; s++)
        if (!p->used[s]) {
          p->used[s] = 1;
          auto d = std::make_shared<DevicePyr>();
          d->pool = p;
          d->slot = s;
          return d;
        }
  auto p = std::make_shared<Pool>();
  p->w = w;
  p->h = h;
  p->levels = levels;
  p->used.assign(SLOTS, 0);
  check(context(), sfmgpu_frames_create(context(), w, h, SLOTS, levels, &p->frames), "frames_create");
  pools.push_back(p);
  p->used[0] = 1;
  auto d = std::make_shared<DevicePyr>();
  d->pool = p;
  d->slot = 0;
  return d;
}

}  // namespace sfmgpu_shim

// ---- Pyramid / build_pyr (:220-232) -----------------------------------------------------------------------------
struct Pyramid {
  std::vector<GrayImage> lvl;                    // host copies, exactly what the reference exposes
  std::shared_ptr<sfmgpu_shim::DevicePyr> dev;   // the same pyramid resident on the GPU
};

static Pyramid build_pyr(const GrayImage& im, int levels) {
  using namespace sfmgpu_shim;
  if (levels < 1 || levels > 8 || im.w <= 0 || im.h <= 0) throw std::runtime_error("sfmgpu: build_pyr: unsupported image / levels");
  sfmgpu_ctx* ctx = context();
  Pyramid p;
  p.dev = acquire_slot(im.w, im.h, levels);
  static unsigned long long next_serial = 1;
  p.dev->serial = next_serial++;
  p.dev->imgkey = speculate() ? image_key(im) : 0;
  sfmgpu_frames* f = p.dev->pool->frames;
  check(ctx, sfmgpu_frames_upload(ctx, f, p.dev->slot, 1, im.pix.data()), "frames_upload");
  check(ctx, sfmgpu_pyramid_build(ctx, f, p.dev->slot, 1), "pyramid_build");
  p.lvl.reserve((size_t)levels);
  p.lvl.push_back(im);  // level 0 is a copy of the input (:227)
  for (int l = 1; l < levels; l++) {
    GrayImage g;
    sfmgpu_frames_level_size(f, l, &g.w, &g.h);
    g.pix.resize((size_t)g.w * g.h);
    check(ctx, sfmgpu_frames_download(ctx, f, p.dev->slot, l, g.pix.data()), "frames_download");
    p.lvl.push_back(std::move(g));
  }
  return p;
}

// ---- shi_tomasi (:237-302) ------------------------------------------------------------------------------------------
static std::vector<Vec2> shi_tomasi(const GrayImage& im, int max_corners, double quality, int min_dist) {
  using namespace sfmgpu_shim;
  sfmgpu_ctx* ctx = context();
  auto slot = acquire_slot(im.w, im.h, 1);
  sfmgpu_frames* f = slot->pool->frames;
  check(ctx, sfmgpu_frames_upload(ctx, f, slot->slot, 1, im.pix.data()), "frames_upload");
  std::vector<double> xy(2 * (size_t)(max_corners < 1 ? 1 : max_corners));
  int n = 0;
  check(ctx, sfmgpu_corners(ctx, f, slot->slot, max_corners, quality, min_dist, xy.data(), &n), "corners");
  std::vector<Vec2> out((size_t)n);
  for (int i = 0; i < n; i++) out[i] = Vec2{xy[2 * i], xy[2 * i + 1]};
  if (speculate()) remember_corners(im, out);
  return out;
}

// ---- KLT (:307-466) -----------------------------------------------------------------------------------------------
struct LKConfig {
  int max_tracks = 2200;
  int min_tracks = 900;
  double quality = 0.01;
  int min_distance = 8;
  int pyr_levels = 3;
  int win_radius = 5;
  int iters = 10;
  double fb_thresh = 1.0;
};

struct Track {
  int id;
  Vec2 p;
};

// Batched form of the loop at :1845-1849: forward a->b and backward b->a for all points in one launch.
static void track_pairs(const Pyramid& a, const Pyramid& b, const std::vector<Vec2>& p0, int win_radius, int iters,
                        std::vector<Vec2>& p1, std::vector<Vec2>* p0_back) {
  using namespace sfmgpu_shim;
  if (!a.dev || !b.dev || a.dev->pool != b.dev->pool)
    throw std::runtime_error("sfmgpu: track: pyramids must come from build_pyr and have the same size / levels");
  sfmgpu_ctx* ctx = context();
  const int n = (int)p0.size();
  p1.resize(p0.size());
  if (p0_back) p0_back->resize(p0.size());
  if (n == 0) return;
  static_assert(sizeof(Vec2) == 2 * sizeof(double), "Vec2 must be two packed doubles");
  check(ctx,
        sfmgpu_klt_track(ctx, a.dev->pool->frames, a.dev->slot, b.dev->slot, reinterpret_cast<const double*>(p0.data()), n,
                         win_radius, iters, reinterpret_cast<double*>(p1.data()),
                         p0_back ? reinterpret_cast<double*>(p0_back->data()) : nullptr, nullptr),
        "klt_track");
}

class KLTTracker {
 public:
  explicit KLTTracker(LKConfig cfg) : cfg_(cfg) {
    sfmgpu_lkcfg c;
    c.max_tracks = cfg.max_tracks;
    c.min_tracks = cfg.min_tracks;
    c.quality = cfg.quality;
    c.min_distance = cfg.min_distance;
    c.pyr_levels = cfg.pyr_levels;
    c.win_radius = cfg.win_radius;
    c.iters = cfg.iters;
    c.fb_thresh = cfg.fb_thresh;
    sfmgpu_tracker* t = nullptr;
    sfmgpu_shim::check(sfmgpu_shim::context(), sfmgpu_tracker_create(sfmgpu_shim::context(), &c, &t), "tracker_create");
    trk_ = std::shared_ptr<sfmgpu_tracker>(t, [](sfmgpu_tracker* p) { sfmgpu_tracker_destroy(sfmgpu_shim::context(), p); });
    cap_ = sfmgpu_shim::track_rows(cfg.max_tracks, cfg.min_tracks);
  }
  // The device state is owned, not shared: a copy would alias one tracker (stepping the copy would advance the
  // original).  The reference class is copyable but never copied (:1688, :1841); the drop-in is move-only.
  KLTTracker(const KLTTracker&) = delete;
  KLTTracker& operator=(const KLTTracker&) = delete;
  KLTTracker(KLTTracker&&) = default;
  KLTTracker& operator=(KLTTracker&&) = default;

  void reset(const GrayImage& gray) {
    auto* ctx = sfmgpu_shim::context();
    sfmgpu_shim::check(ctx, sfmgpu_tracker_reset(ctx, trk_.get(), gray.pix.data(), gray.w, gray.h), "tracker_reset");
    fetch_tracks();
  }

  struct StepOut {
    std::vector<Vec2> prev_pts;
    std::vector<Vec2> cur_pts;
    std::vector<int> ids;
  };

  StepOut step(const GrayImage& gray) {
    auto* ctx = sfmgpu_shim::context();
    StepOut out;
    out.prev_pts.resize((size_t)cap_);
    out.cur_pts.resize((size_t)cap_);
    out.ids.resize((size_t)cap_);
    int n = 0;
    sfmgpu_shim::check(ctx,
                       sfmgpu_tracker_step(ctx, trk_.get(), gray.pix.data(), gray.w, gray.h,
                                           reinterpret_cast<double*>(out.prev_pts.data()),
                                           reinterpret_cast<double*>(out.cur_pts.data()), out.ids.data(), cap_, &n),
                       "tracker_step");
    out.prev_pts.resize((size_t)n);
    out.cur_pts.resize((size_t)n);
    out.ids.resize((size_t)n);
    fetch_tracks();
    return out;
  }

  const std::vector<Track>& tracks() const { return tracks_; }

  // Single-direction, single-point track (:396-398).  A loop over the corners of a's image (:1845-1849) is answered from
  // ONE batched forward + backward track of all of them (see "speculation" above); any other call is one launch.
  Vec2 track_one_public(const Pyramid& a, const Pyramid& b, Vec2 p0) const {
    using namespace sfmgpu_shim;
    if (speculate() && a.dev && b.dev && a.dev->pool == b.dev->pool) {
      TrackMemo& tm = track_memo();
      const bool same_cfg = tm.radius == cfg_.win_radius && tm.iters == cfg_.iters;
      if (same_cfg && ((tm.a == a.dev->serial && tm.b == b.dev->serial) || (tm.a == b.dev->serial && tm.b == a.dev->serial))) {
        auto it = tm.table.find(TrackKey{a.dev->serial, b.dev->serial, dbits(p0.x), dbits(p0.y)});
        if (it != tm.table.end()) return it->second;
      }
      for (int m = 0; m < 2; m++) {
        const CornerMemo& cm = corner_memos()[m];
        if (cm.imgkey == 0 || cm.imgkey != a.dev->imgkey || cm.corners.size() < 2) continue;
        bool member = false;
        for (const Vec2& c : cm.corners)
          if (dbits(c.x) == dbits(p0.x) && dbits(c.y) == dbits(p0.y)) {
            member = true;
            break;
          }
        if (!member) continue;
        // all corners of a's image, forward and backward, through the kernel a single call runs (warp per feature)
        std::vector<Vec2> p1, pb;
        sfmgpu_ctx* ctx = context();
        check(ctx, sfmgpu_klt_set_mode(ctx, 1), "klt_set_mode");
        try {
          track_pairs(a, b, cm.corners, cfg_.win_radius, cfg_.iters, p1, &pb);
        } catch (...) {
          sfmgpu_klt_set_mode(ctx, 0);
          throw;
        }
        check(ctx, sfmgpu_klt_set_mode(ctx, 0), "klt_set_mode");
        tm.a = a.dev->serial;
        tm.b = b.dev->serial;
        tm.radius = cfg_.win_radius;
        tm.iters = cfg_.iters;
        tm.table.clear();
        tm.table.reserve(2 * cm.corners.size());
        Vec2 answer = p0;
        for (size_t k = 0; k < cm.corners.size(); k++) {
          const Vec2& c = cm.corners[k];
          tm.table[TrackKey{tm.a, tm.b, dbits(c.x), dbits(c.y)}] = p1[k];
          tm.table[TrackKey{tm.b, tm.a, dbits(p1[k].x), dbits(p1[k].y)}] = pb[k];
          if (dbits(c.x) == dbits(p0.x) && dbits(c.y) == dbits(p0.y)) answer = p1[k];
        }
        return answer;
      }
    }
    std::vector<Vec2> in{p0}, out;
    track_pairs(a, b, in, cfg_.win_radius, cfg_.iters, out, nullptr);
    return out[0];
  }

 private:
  void fetch_tracks() {
    auto* ctx = sfmgpu_shim::context();
    std::vector<double> xy(2 * (size_t)cap_);
    std::vector<int> ids((size_t)cap_);
    int n = 0;
    sfmgpu_shim::check(ctx, sfmgpu_tracker_tracks(ctx, trk_.get(), xy.data(), ids.data(), cap_, &n), "tracker_tracks");
    tracks_.resize((size_t)n);
    for (int i = 0; i < n; i++) tracks_[i] = Track{ids[i], Vec2{xy[2 * i], xy[2 * i + 1]}};
  }
  LKConfig cfg_;
  std::shared_ptr<sfmgpu_tracker> trk_;
  std::vector<Track> tracks_;
  int cap_ = 0;
};

// S KLTTrackers advanced in lock step (no counterpart in the reference, which tracks one sequence: this is the C++ face of
// sfmgpu_multitracker for callers with several independent sequences per GPU).  Per sequence the results equal a
// KLTTracker's; all images must be w x h.
class MultiKLTTracker {
 public:
  MultiKLTTracker(const MultiKLTTracker&) = delete;
  MultiKLTTracker& operator=(const MultiKLTTracker&) = delete;
  MultiKLTTracker(LKConfig cfg, int n_sequences, int w, int h) : S_(n_sequences), w_(w), h_(h) {
    sfmgpu_lkcfg c;
    c.max_tracks = cfg.max_tracks;
    c.min_tracks = cfg.min_tracks;
    c.quality = cfg.quality;
    c.min_distance = cfg.min_distance;
    c.pyr_levels = cfg.pyr_levels;
    c.win_radius = cfg.win_radius;
    c.iters = cfg.iters;
    c.fb_thresh = cfg.fb_thresh;
    sfmgpu_multitracker* t = nullptr;
    auto* ctx = sfmgpu_shim::context();
    sfmgpu_shim::check(ctx, sfmgpu_multitracker_create(ctx, &c, n_sequences, w, h, &t), "multitracker_create");
    trk_ = std::shared_ptr<sfmgpu_multitracker>(t, [](sfmgpu_multitracker* p) { sfmgpu_multitracker_destroy(sfmgpu_shim::context(), p); });
    cap_ = sfmgpu_shim::track_rows(cfg.max_tracks, cfg.min_tracks);
    void* pin = nullptr;  // page-locked staging for the S frames of a step
    sfmgpu_shim::check(ctx, sfmgpu_host_alloc(ctx, (size_t)S_ * w * h, &pin), "host_alloc");
    stage_ = std::shared_ptr<uint8_t>((uint8_t*)pin, [](uint8_t* p) { sfmgpu_host_free(sfmgpu_shim::context(), p); });
  }

  // frames[s] = the next frame of sequence s; returns one StepOut per sequence (empty on the first call)
  std::vector<KLTTracker::StepOut> step(const std::vector<const GrayImage*>& frames) {
    auto* ctx = sfmgpu_shim::context();
    if ((int)frames.size() != S_) throw std::runtime_error("sfmgpu: MultiKLTTracker::step: one frame per sequence expected");
    const size_t px = (size_t)w_ * h_;
    for (int s = 0; s < S_; s++) {
      if (!frames[s] || frames[s]->w != w_ || frames[s]->h != h_) throw std::runtime_error("sfmgpu: MultiKLTTracker::step: frame size differs");
      std::copy(frames[s]->pix.begin(), frames[s]->pix.begin() + px, stage_.get() + (size_t)s * px);
    }
    std::vector<double> prev(2 * (size_t)S_ * cap_), cur(2 * (size_t)S_ * cap_);
    std::vector<std::int32_t> ids((size_t)S_ * cap_), n((size_t)S_);
    sfmgpu_shim::check(ctx, sfmgpu_multitracker_step(ctx, trk_.get(), stage_.get(), prev.data(), cur.data(), ids.data(), n.data()),
                       "multitracker_step");
    std::vector<KLTTracker::StepOut> out((size_t)S_);
    for (int s = 0; s < S_; s++) {
      const size_t o = (size_t)s * cap_;
      out[s].prev_pts.resize((size_t)n[s]);
      out[s].cur_pts.resize((size_t)n[s]);
      out[s].ids.assign(ids.begin() + o, ids.begin() + o + n[s]);
      for (int i = 0; i < n[s]; i++) {
        out[s].prev_pts[i] = Vec2{prev[2 * (o + i)], prev[2 * (o + i) + 1]};
        out[s].cur_pts[i] = Vec2{cur[2 * (o + i)], cur[2 * (o + i) + 1]};
      }
    }
    return out;
  }

  std::vector<Track> tracks(int sequence) const {
    auto* ctx = sfmgpu_shim::context();
    std::vector<double> xy(2 * (size_t)cap_);
    std::vector<std::int32_t> ids((size_t)cap_);
    int n = 0;
    sfmgpu_shim::check(ctx, sfmgpu_multitracker_tracks(ctx, trk_.get(), sequence, xy.data(), ids.data(), cap_, &n), "multitracker_tracks");
    std::vector<Track> out((size_t)n);
    for (int i = 0; i < n; i++) out[i] = Track{ids[i], Vec2{xy[2 * i], xy[2 * i + 1]}};
    return out;
  }

  // find_E_ransac(K, step.prev_pts, step.cur_pts, iters, thr, min_inliers) (:1739) on every sequence's survivors inside every
  // later step, skipped where a sequence has none (:1715); the results of a step: two_view_results(*this), sfmgpu_two_view.hpp
  void set_two_view(const Mat33& K, int iters, double thr, int min_inliers) {
    auto* ctx = sfmgpu_shim::context();
    const sfmgpu_ransac_cfg rc{iters, thr, min_inliers, 1};
    sfmgpu_shim::check(ctx, sfmgpu_multitracker_set_ransac(ctx, trk_.get(), K.a.data(), &rc), "multitracker_set_ransac");
  }

  sfmgpu_multitracker* handle() const { return trk_.get(); }
  int n_sequences() const { return S_; }
  int rows() const { return cap_; }

 private:
  int S_, w_, h_, cap_ = 0;
  std::shared_ptr<sfmgpu_multitracker> trk_;
  std::shared_ptr<uint8_t> stage_;
};

// ---- loop-closure descriptor (:1100-1129) -------------------------------------------------------------------------------
static std::vector<float> global_desc_32(const GrayImage& im) {
  using namespace sfmgpu_shim;
  if (im.w <= 0 || im.h <= 0) throw std::runtime_error("sfmgpu: global_desc_32: empty image");
  sfmgpu_ctx* ctx = context();
  auto dev = acquire_slot(im.w, im.h, 1);
  sfmgpu_frames* f = dev->pool->frames;
  check(ctx, sfmgpu_frames_upload(ctx, f, dev->slot, 1, im.pix.data()), "frames_upload");
  std::vector<float> v(1024);
  check(ctx, sfmgpu_global_desc32(ctx, f, dev->slot, 1, v.data()), "global_desc32");
  return v;
}

// dot_desc :1124-1129 is a 1024-term loop: it stays a host inline (same float arithmetic, no contraction on x86-64);
// the search over all stored keyframes (:1823-1831) has the batched device twin loop_candidate().
static float dot_desc(const std::vector<float>& a, const std::vector<float>& b) {
  float s = 0.0f;
  const size_t n = std::min(a.size(), b.size());
  for (size_t i = 0; i < n; i++) s += a[i] * b[i];
  return s;
}

// best_id / best_score of the loop at :1823-1831 over kf_desc[0 .. n_search)
static int loop_candidate(const std::vector<std::vector<float>>& kf_desc, int n_search, const std::vector<float>& query,
                          float* best_score) {
  using namespace sfmgpu_shim;
  if (n_search <= 0) {
    if (best_score) *best_score = 0.0f;
    return -1;
  }
  std::vector<float> flat((size_t)n_search * 1024);
  for (int k = 0; k < n_search; k++) std::copy(kf_desc[k].begin(), kf_desc[k].begin() + 1024, flat.begin() + (size_t)k * 1024);
  int bid = -1;
  float bs = 0.0f;
  check(context(), sfmgpu_desc_search(context(), flat.data(), n_search, query.data(), nullptr, &bid, &bs), "desc_search");
  if (best_score) *best_score = bs;
  return bid;
}

// ---- triangulate_dlt (:1477-1516) -------------------------------------------------------------------------------------------
// PoseCW is defined inside the reference TU (:157-168), after the point where this header is included, so the shim
// takes the pose as (R camera->world, camera centre).  The single-track form runs on the host and is bit-identical;
// triangulate_tracks() is the batched device twin (opt-in, ~1e-10 relative).
#ifdef SFMGPU_SHIM_STANDALONE
static Vec3 triangulate_dlt_rt(const Mat33& K, const Mat33& Ri, const Vec3& Ci, const Mat33& Rj, const Vec3& Cj, Vec2 ui, Vec2 uj) {
  double ki[9];
  if (!sfmgpu_host::invert_K(K.a.data(), ki)) throw std::runtime_error("Singular K");
  const double ci[3] = {Ci.x, Ci.y, Ci.z}, cj[3] = {Cj.x, Cj.y, Cj.z}, a[2] = {ui.x, ui.y}, b[2] = {uj.x, uj.y};
  double X[3];
  sfmgpu_host::triangulate_dlt(K.a.data(), Ri.a.data(), ci, Rj.a.data(), cj, a, b, X);
  return Vec3{X[0], X[1], X[2]};
}
#endif  // inside the reference TU its own triangulate_dlt (:1477-1516) stays in place

static std::vector<Vec3> triangulate_tracks(const Mat33& K, const std::vector<std::array<double, 12>>& poses, const std::vector<int>& ia,
                                            const std::vector<int>& ib, const std::vector<Vec2>& ui, const std::vector<Vec2>& uj) {
  using namespace sfmgpu_shim;
  const int n = (int)ui.size();
  std::vector<Vec3> out((size_t)n);
  if (n == 0) return out;
  static_assert(sizeof(Vec2) == 16 && sizeof(Vec3) == 24, "layout");
  check(context(), sfmgpu_triangulate_dlt(context(), K.a.data(), poses[0].data(), (int)poses.size(), ia.data(), ib.data(), &ui[0].x, &uj[0].x,
                                          n, &out[0].x), "triangulate_dlt");
  return out;
}

#ifdef SFMGPU_SHIM_STANDALONE
#include "sfmgpu_two_view.hpp"
#endif
