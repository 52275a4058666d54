// klt_sizes_oracle.cpp — the restatement's KLT between two pyramids of any sizes, for tests/test_gpu_klt_sizes.py.
// Test plumbing: oracle/sfm_oracle.cpp compiled as it is, plus one flat export over its track(const Pyr& A, const Pyr& B, ...),
// which walks `levels` levels of both pyramids and samples each image against its own level size (:183-198, :402-460).
#include "../../oracle/sfm_oracle.cpp"

extern "C" int orc_klt_track2(const uint8_t* im0, int w0, int h0, const uint8_t* im1, int w1, int h1, int levels, int radius,
                              int iters, const double* p0, int n, double* p1, double* p0b) {
  Pyr A = make_pyr(im0, w0, h0, levels), B = make_pyr(im1, w1, h1, levels);
  LK c{levels, radius, iters};
  for (int i = 0; i < n; i++) {
    track(A, B, c, p0[2 * i], p0[2 * i + 1], p1[2 * i], p1[2 * i + 1]);
    track(B, A, c, p1[2 * i], p1[2 * i + 1], p0b[2 * i], p0b[2 * i + 1]);
  }
  return 0;
}
