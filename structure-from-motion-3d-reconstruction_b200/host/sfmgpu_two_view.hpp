// sfmgpu_two_view.hpp — RelPose + find_E_ransac (cpp/src/templering_sfm.cpp:640-761) of the C++ drop-in, on top of the C ABI.
//
// Include it where the reference defines RelPose / find_E_ransac (after sfmgpu_shim.hpp, INTEGRATION.md §2).  What runs
// where:
//   K^-1 normalisation, seeded octets (:649-665)      host, the reference's own arithmetic
//   eight_point_E per octet (:666)                    INSIDE THE REFERENCE TU: the TU's own eight_point_E (bit-identical
//                                                     hypotheses by construction), spread over a few host threads;
//                                                     stand-alone builds use the restatement in two_view_host.hpp;
//                                                     opt-in: the device solver (sfmgpu_ransac_hypotheses)
//   Sampson scoring, winner, inlier list (:667-676)   GPU (sfmgpu_ransac_score): bit-exact counts for the hypotheses given
//   min_inliers test, E -> (R, t) (:678-760)          host: inside the TU with its own svd3 / AtA_from_A / jacobi_eig_sym /
//                                                     Mat33 operators, stand-alone with two_view_host.hpp
// The pose tail is part of find_E_ransac's body in the reference, so it cannot be called there; it is written here against
// the TU's own linear algebra (same calls in the same order, hence the same R and t bit for bit).
#pragma once
#include <optional>
#include <random>
#include <thread>
#include <vector>

struct RelPose {
  Mat33 R_ji;
  Vec3 t_ji;
  std::vector<int> inliers;
};

namespace sfmgpu_shim {

#ifdef SFMGPU_SHIM_STANDALONE
// ---- stand-alone: plain-array linear algebra of two_view_host.hpp -------------------------------------------------------------
struct TwoViewLA {
  double Ki[9];
  std::vector<double> xi, xj;
  explicit TwoViewLA(const Mat33& K) {
    if (!sfmgpu_host::invert_K(K.a.data(), Ki)) throw std::runtime_error("Singular K");
  }
  void normalise(const std::vector<Vec2>& pi, const std::vector<Vec2>& pj) {
    const size_t n = pi.size();
    xi.resize(2 * n);
    xj.resize(2 * n);
    for (size_t i = 0; i < n; i++) {
      sfmgpu_host::norm_point(Ki, pi[i].x, pi[i].y, &xi[2 * i]);
      sfmgpu_host::norm_point(Ki, pj[i].x, pj[i].y, &xj[2 * i]);
    }
  }
  const double* xi_ptr() const { return xi.data(); }
  const double* xj_ptr() const { return xj.data(); }
  void solve(const int* idx8, double* E9) const { sfmgpu_host::eight_point_E(xi.data(), xj.data(), idx8, E9); }
  void pose(const double* E9, const int* inl, int n_inl, RelPose& rp) const {
    double R[9], t[3];
    sfmgpu_host::recover_pose(E9, xi.data(), xj.data(), inl, n_inl, R, t);
    for (int k = 0; k < 9; k++) rp.R_ji.a[k] = R[k];
    rp.t_ji = Vec3{t[0], t[1], t[2]};
  }
};
#else
// ---- inside the reference TU: its own functions (defined above the include point, :471-627, linalg.hpp) -------------------------
struct TwoViewLA {
  Mat33 Kinv;
  std::vector<Vec2> xi, xj;
  explicit TwoViewLA(const Mat33& K) : Kinv(invert_K(K)) {}  // throws "Singular K" itself (:474)
  void normalise(const std::vector<Vec2>& pi, const std::vector<Vec2>& pj) {
    xi.resize(pi.size());
    xj.resize(pj.size());
    for (size_t i = 0; i < pi.size(); ++i) {
      xi[i] = norm_point(Kinv, pi[i]);
      xj[i] = norm_point(Kinv, pj[i]);
    }
  }
  static_assert(sizeof(Vec2) == 2 * sizeof(double), "Vec2 must be two packed doubles");
  const double* xi_ptr() const { return reinterpret_cast<const double*>(xi.data()); }
  const double* xj_ptr() const { return reinterpret_cast<const double*>(xj.data()); }
  void solve(const int* idx8, double* E9) const {
    const std::vector<int> idx(idx8, idx8 + 8);
    const Mat33 E = eight_point_E(xi, xj, idx);
    for (int k = 0; k < 9; k++) E9[k] = E.a[k];
  }
  // :680-760 with the TU's svd3 / AtA_from_A / sfm::jacobi_eig_sym / Mat33 operators
  void pose(const double* E9, const int* inl, int n_inl, RelPose& rp) const {
    Mat33 bestE{};
    for (int k = 0; k < 9; k++) bestE.a[k] = E9[k];
    const auto svd = svd3(bestE);
    Mat33 W{};
    W(0, 1) = -1;
    W(1, 0) = 1;
    W(2, 2) = 1;
    const Mat33 Vt = sfm::transpose(svd.V);
    Mat33 R1 = svd.U * W * Vt, R2 = svd.U * sfm::transpose(W) * Vt;
    if (sfm::det(R1) < 0)
      for (double& v : R1.a) v = -v;
    if (sfm::det(R2) < 0)
      for (double& v : R2.a) v = -v;
    const Vec3 t = sfm::unit(Vec3{svd.U(0, 2), svd.U(1, 2), svd.U(2, 2)});
    auto depth_ok = [&](const Mat33& R, const Vec3& tt, const Vec2& x, const Vec2& xp) {
      std::vector<double> A = {-1, 0, x.x, 0,
                               0, -1, x.y, 0,
                               xp.x * R(2, 0) - R(0, 0), xp.x * R(2, 1) - R(0, 1), xp.x * R(2, 2) - R(0, 2), xp.x * tt.z - tt.x,
                               xp.y * R(2, 0) - R(1, 0), xp.y * R(2, 1) - R(1, 1), xp.y * R(2, 2) - R(1, 2), xp.y * tt.z - tt.y};
      const auto eig = sfm::jacobi_eig_sym(AtA_from_A(A, 4, 4), 4, 80);
      const double w = eig.V[12];
      const Vec3 X{eig.V[0] / w, eig.V[4] / w, eig.V[8] / w};
      const Vec3 X2 = (R * X) + tt;
      return X.z > 0 && X2.z > 0;
    };
    const Mat33* Rs[4] = {&R1, &R1, &R2, &R2};
    const Vec3 ts[4] = {t, Vec3{-t.x, -t.y, -t.z}, t, Vec3{-t.x, -t.y, -t.z}};
    int best = 0, bestok = -1;
    const int M = n_inl < 20 ? n_inl : 20;
    for (int c = 0; c < 4; c++) {
      int ok = 0;
      for (int k = 0; k < M; k++)
        if (depth_ok(*Rs[c], ts[c], xi[inl[k]], xj[inl[k]])) ok++;
      if (ok > bestok) {
        bestok = ok;
        best = c;
      }
    }
    rp.R_ji = *Rs[best];
    rp.t_ji = ts[best];
  }
};
#endif

}  // namespace sfmgpu_shim

static std::optional<RelPose> find_E_ransac(const Mat33& K, const std::vector<Vec2>& pi, const std::vector<Vec2>& pj, int iters = 2000,
                                            double thr = 1e-4, int min_inliers = 80) {
  using namespace sfmgpu_shim;
  if (pi.size() < 8) return std::nullopt;  // before any RNG use (:648)
  const int n = (int)pi.size();
  TwoViewLA la(K);
  la.normalise(pi, pj);
  const int H = iters > 0 ? iters : 0;
  // the reference's seeded sampling (:657-665), one continuing stream, re-seeded on every call (host solver; the device
  // solver path samples on the device: the same octets, sfmgpu_ransac_solve_score with idx8 == NULL)
  std::vector<int> idx;
  if (!device_solver()) {
    std::mt19937 rng(12345);
    std::uniform_int_distribution<int> uni(0, n - 1);
    idx.resize((size_t)8 * H);
    for (size_t k = 0; k < idx.size(); k++) idx[k] = uni(rng);
  }
  std::vector<double> E(9 * (size_t)H);
  sfmgpu_ctx* ctx = context();
  std::vector<int> inl((size_t)n);
  int best_h = -1, best_n = 0;
  if (!device_solver()) {
    // every solve is a pure function of its octet: solving them on several host threads leaves every hypothesis
    // bit-identical to the reference's
    const int nthr = H >= 64 ? solver_threads() : 1;
    auto solve = [&](int h0, int h1) {
      for (int it = h0; it < h1; it++) la.solve(&idx[8 * (size_t)it], &E[9 * (size_t)it]);
    };
    if (nthr <= 1) {
      solve(0, H);
    } else {
      std::vector<std::thread> pool;
      const int per = (H + nthr - 1) / nthr;
      for (int t = 1; t < nthr; t++)
        if (t * per < H) pool.emplace_back(solve, t * per, std::min(H, (t + 1) * per));
      solve(0, std::min(H, per));
      for (auto& th : pool) th.join();
    }
    // scoring loop (:667-676) on the GPU: exact counts, first hypothesis with the strictly largest count
    check(ctx, sfmgpu_ransac_score(ctx, la.xi_ptr(), la.xj_ptr(), n, E.data(), H, thr, nullptr, &best_h, inl.data(), &best_n),
          "ransac_score");
  } else {
    // opt-in (SFMGPU_DEVICE_SOLVER=1 or set_device_solver(true)): the same octets, hypotheses solved on the device.  The
    // counts come from the screening solver, the winner is solved again by the Jacobi emulation (equal to the host
    // solver's hypothesis to ~1e-9, not bit for bit): its E, count and inlier list come back
    static_assert(sizeof(int) == sizeof(std::int32_t), "int32 octets");
    double bestE[9];
    check(ctx, sfmgpu_ransac_solve_score(ctx, la.xi_ptr(), la.xj_ptr(), n, nullptr, H, thr, &best_h, &best_n, bestE, inl.data()),
          "ransac_solve_score");
    if (best_h >= 0)
      for (int i = 0; i < 9; i++) E[9 * (size_t)best_h + i] = bestE[i];
  }
  if (best_n < min_inliers) return std::nullopt;
  RelPose rp;
  // best_h < 0 means "no hypothesis won": the reference then decomposes the zero matrix
  const double zeroE[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  la.pose(best_h >= 0 ? &E[9 * (size_t)best_h] : zeroE, inl.data(), best_n, rp);
  rp.inliers.assign(inl.begin(), inl.begin() + best_n);
  return rp;
}

// find_E_ransac's answer for every sequence of the last MultiKLTTracker::step (set_two_view on), computed inside the step on
// the device: std::nullopt where the reference has none (no survivors, :1715; fewer than 8 points or min_inliers, :648 /
// :678), else R_ji, t_ji and the inlier indices into that sequence's step.prev_pts / cur_pts.
static std::vector<std::optional<RelPose>> two_view_results(const MultiKLTTracker& mt) {
  using namespace sfmgpu_shim;
  const int S = mt.n_sequences(), rows = mt.rows();
  std::vector<std::int32_t> st((size_t)S), bn((size_t)S), inl((size_t)S * rows);
  std::vector<double> R(9 * (size_t)S), t(3 * (size_t)S);
  sfmgpu_ctx* ctx = context();
  check(ctx, sfmgpu_multitracker_ransac_download_all(ctx, mt.handle(), st.data(), bn.data(), inl.data(), R.data(), t.data()),
        "multitracker_ransac_download_all");
  std::vector<std::optional<RelPose>> out((size_t)S);
  for (int s = 0; s < S; s++) {
    if (st[s] != SFMGPU_TV_OK) continue;
    RelPose rp;
    for (int k = 0; k < 9; k++) rp.R_ji.a[k] = R[9 * (size_t)s + k];
    rp.t_ji = Vec3{t[3 * (size_t)s], t[3 * (size_t)s + 1], t[3 * (size_t)s + 2]};
    rp.inliers.assign(inl.begin() + (size_t)s * rows, inl.begin() + (size_t)s * rows + bn[s]);
    out[s] = std::move(rp);
  }
  return out;
}
