// klt.cu — pyramidal Lucas-Kanade, one warp per feature, FP64, forward + backward in one launch.
//
// Replaces (reference cpp/src/templering_sfm.cpp): sample_bilinear :183-198, KLTTracker::track_one :402-422,
// lk_step :424-460, and the per-track fwd/bwd + fb test of step() :356-362 / the two-view loop :1845-1849.
//
// Behaviour kept bug-for-bug (SURVEY.md facts 5, §7.3-3):
//   * both images are sampled at the SAME moving location (err = I0(p+d) - I1(p+d)), so the update does not
//     converge; every iteration adds about the local flow;
//   * any bilinear tap outside the image zeroes the whole sample; |det| < 1e-9 gives a zero step;
//   * the early exit tests the step that was just added (hypot(step) < 1e-3);
//   * p is rescaled from the running full-resolution position at every level.
//
// Arithmetic: positions, bilinear weights, accumulators and the 2x2 solve are FP64.  The file is compiled with
// -fmad=false; fused multiply-adds appear only where written explicitly (__fma_rn).  Deliberate, measured
// deviations from the reference's operation ORDER / rounding (never from its formulas or its discontinuities):
//   (1) the window's six samples per pixel come from one shared grid of bilinear samples whose column / row
//       coordinates are fl(x+i), fl(y+j) (the reference reaches the +-1 neighbours as fl(fl(x+i)+-1));
//   (2) lerps are evaluated as a + (b-a)*t with one FMA; the normal equations are accumulated with FMAs,
//       lane-strided and then butterfly-reduced instead of sequentially in raster order;
//   (3) the 0.5 factors of the central differences are folded into the solve (exact power-of-two scaling).
//   Measured against the exact order: max deviation ~1e-13 px on smooth, checker and pure-noise images
//   (tests/test_gpu_parity.py prints it), 10 orders of magnitude inside the 1e-3 px parity budget; the
//   reference's update is non-contractive but not chaotic (perturbations of 1e-13 stay below 1e-10 after the
//   60 iterations of a fwd+bwd track).
//
// Roofline: FP64 CUDA-core pipe, not HBM (algorithmic traffic is 2,092 B per track-step, SURVEY.md §8d).
#include "common.cuh"

namespace {

constexpr int KLT_MARGIN = 4;

template <int R>
struct KltSmem {
  static constexpr int NC = 2 * R + 3;                         // sample-grid columns / rows (window + 1 each side)
  static constexpr int TH = 2 * KLT_MARGIN + 2 * R + 6;        // cached tile rows (24 for R = 5)
  static constexpr int TW = ((2 * R + 17 + 3) / 4) * 4;        // cached tile row bytes, origin 4-aligned (28 for R = 5)
  static constexpr int WPR = TW / 4;
  double cfy[NC + 3];      // per grid row: fractional weight of the lower tap row
  int cvy[NC + 3];         // per grid row: both tap rows inside the image (two geometries: bit 0 image A, bit 1 image B)
  uint32_t t0[TH * WPR];   // cached u8 tile of image A around the window (rows of TW bytes)
  uint32_t t1[TH * WPR];   // same for image B
};

// Sum five per-lane partials over the warp by recursive halving (8 exchanges instead of 25), then broadcast.
__device__ __forceinline__ void reduce5(double& a00, double& a01, double& a11, double& b0, double& b1, int lane) {
  const unsigned FULL = 0xffffffffu;
  const bool up16 = lane & 16, up8 = lane & 8, up4 = lane & 4;
  // xor 16: lower half keeps (a00,a01,a11), upper half keeps (b0,b1)
  const double x0 = __shfl_xor_sync(FULL, up16 ? a00 : b0, 16);
  const double x1 = __shfl_xor_sync(FULL, up16 ? a01 : b1, 16);
  const double x2 = __shfl_xor_sync(FULL, up16 ? a11 : 0.0, 16);
  double u0 = (up16 ? b0 : a00) + x0, u1 = (up16 ? b1 : a01) + x1, u2 = up16 ? 0.0 : a11 + x2;
  // xor 8: bit3 == 0 keeps (u0,u1), bit3 == 1 keeps u2
  const double y0 = __shfl_xor_sync(FULL, up8 ? u0 : u2, 8);
  const double y1 = __shfl_xor_sync(FULL, up8 ? u1 : 0.0, 8);
  double v0 = up8 ? u2 + y0 : u0 + y0, v1 = up8 ? 0.0 : u1 + y1;
  // xor 4: bit2 == 0 keeps v0, bit2 == 1 keeps v1
  const double z0 = __shfl_xor_sync(FULL, up4 ? v0 : v1, 4);
  double z = (up4 ? v1 : v0) + z0;
  z = z + __shfl_xor_sync(FULL, z, 2);
  z = z + __shfl_xor_sync(FULL, z, 1);
  a00 = __shfl_sync(FULL, z, 0);
  a01 = __shfl_sync(FULL, z, 4);
  a11 = __shfl_sync(FULL, z, 8);
  b0 = __shfl_sync(FULL, z, 16);
  b1 = __shfl_sync(FULL, z, 20);
}

// Stage TH rows of TW bytes starting at (tx0 [multiple of 4], ty0) with aligned 32-bit loads.  Coordinates are
// clamped to the allocation; bytes outside the image are garbage that only ever feeds samples the bounds test zeroes.
template <int R>
__device__ __forceinline__ void stage_tile(uint32_t* tile, const uint8_t* __restrict__ img, int h, int pitch, int tx0, int ty0,
                                           int lane) {
  constexpr int TH = KltSmem<R>::TH, WPR = KltSmem<R>::WPR;
  const int wmax = (pitch >> 2) - 1, wx0 = tx0 >> 2;
#pragma unroll 2
  for (int idx = lane; idx < TH * WPR; idx += 32) {
    const int r = idx / WPR, c = idx - r * WPR;
    int gw = wx0 + c, gy = ty0 + r;
    gw = gw < 0 ? 0 : (gw > wmax ? wmax : gw);
    gy = gy < 0 ? 0 : (gy > h - 1 ? h - 1 : gy);
    tile[idx] = __ldg(reinterpret_cast<const uint32_t*>(img + (size_t)gy * pitch) + gw);
  }
}

// The window walk of one LK iteration for this lane (see track_one).  INTERIOR: every tap is inside the image, so
// the per-sample bounds logic (:188) is compiled out.  TWO: images A and B have their own bounds; vx / bit 1 of cvy test
// B's, vx0 / bit 0 of cvy test A's.
template <int R, bool FIXED, bool INTERIOR, bool TWO = false>
__device__ __forceinline__ void walk_rows(const KltSmem<R>& sm, int NK, int nc, int rowbase, int col, int p0, int p1, bool pix_col,
                                          bool vx, double fx, double& a00, double& a01, double& a11, double& b0, double& b1,
                                          bool vx0 = false) {
  constexpr int TW = KltSmem<R>::TW;
  const uint8_t* q1 = reinterpret_cast<const uint8_t*>(sm.t1) + rowbase * TW + col;
  const uint8_t* q0 = reinterpret_cast<const uint8_t*>(sm.t0) + rowbase * TW + col;
  double h1p = 0, h0p = 0, s1a = 0, s1b = 0, s0b = 0;
#pragma unroll
  for (int k = 0; k < (FIXED ? (2 * R + 1 + 32 / (2 * R + 3) - 1) / (32 / (2 * R + 3)) + 3 : NK); k++) {
    const int a1 = q1[k * TW], c1 = q1[k * TW + 1], a0 = q0[k * TW], c0 = q0[k * TW + 1];
    // horizontal lerp v00 + (v10 - v00)*dx  (== v00*(1-dx) + v10*dx up to one rounding)
    const double h1 = __fma_rn(fx, (double)(c1 - a1), (double)a1);
    const double h0 = __fma_rn(fx, (double)(c0 - a0), (double)a0);
    if (k >= 1) {
      int j = p0 + k - 1;  // grid row just completed
      j = j > nc - 1 ? nc - 1 : j;
      const double fy = sm.cfy[j];
      double s1c = __fma_rn(fy, h1 - h1p, h1p);
      double s0c = __fma_rn(fy, h0 - h0p, h0p);
      if (!INTERIOR && TWO) {
        const int cy = sm.cvy[j];
        s1c = (vx && (cy & 2)) ? s1c : 0.0;  // a sample of B is zeroed by B's bounds, a sample of A by A's
        s0c = (vx0 && (cy & 1)) ? s0c : 0.0;
      } else if (!INTERIOR) {
        const bool ok = vx && sm.cvy[j];
        s1c = ok ? s1c : 0.0;  // any out-of-range tap zeroes the whole sample (:188)
        s0c = ok ? s0c : 0.0;
      }
      if (k >= 3) {
        // pixel row p0+k-3: centre sample s1b, vertical neighbours s1a / s1c, horizontal from lanes +-1
        const double left = __shfl_up_sync(0xffffffffu, s1b, 1);
        const double right = __shfl_down_sync(0xffffffffu, s1b, 1);
        if (pix_col && p0 + k - 3 < p1) {
          const double gx2 = right - left;  // 2*Ix: the reference's 0.5 factors are folded into the solve
          const double gy2 = s1c - s1a;     // 2*Iy
          const double e = s0b - s1b;
          a00 = __fma_rn(gx2, gx2, a00);
          a01 = __fma_rn(gx2, gy2, a01);
          a11 = __fma_rn(gy2, gy2, a11);
          b0 = __fma_rn(gx2, e, b0);
          b1 = __fma_rn(gy2, e, b1);
        }
      }
      s1a = s1b;
      s1b = s1c;
      s0b = s0c;
    }
    h1p = h1;
    h0p = h0;
  }
}

// One pyramidal track (:402-422) of point (px,py) from pyramid A to pyramid B.  All lanes hold identical
// scalars; shared memory `sm` is private to the warp.
//
// Lane layout ("column lanes"): lane = g*nc + i owns grid column i (x offset i-r-1) for the g-th contiguous
// chunk of window rows; G = 32/nc groups (2 for r = 5: 26 of 32 lanes busy).  A lane walks down its rows keeping
// the horizontal lerps, the last three I1 samples and the last two I0 samples in REGISTERS; the only exchanges
// are two shuffles per pixel row (left / right neighbour sample) and the final 5-value warp reduction.
// Shared memory holds just the cached u8 tiles and the tiny per-row weight table.
//
// Weights: column i uses the REGULAR tap pair (FX+i-r-1, +1) with f = fl(x+i') - (FX+i') in [0,1].  In the rare
// case where fl(x+i') rounds up to the next integer the reference's own floor moves by one and its fraction is
// 0; f == 1 on the regular pair selects exactly the same tap (weights 0 and 1), so no special case is needed
// for the value, only for the bounds test, which uses the reference's floor.
//
// TWO: image A (frame fa of pva) and image B (frame fb of pv) have their own level sizes, as the reference's
// track(Pyr A, Pyr B) allows: each tile is staged from its own image and each sample is zeroed by its own image's
// bounds (:188).  The step is zero whenever B has fewer than 2 columns or rows (no gradient); an A that small only
// zeroes its own samples.  Without TWO, pva is pv.
//
// GEO: the list's own geometry table `geo` (one size for both images) replaces pv's sizes and the frame indices; back = true
// tracks from its image B to its image A.
template <int R, bool FIXED, bool TWO = false, bool GEO = false>
__device__ void track_one(KltSmem<R>& sm, const PyrView& pv, int fa, int fb, int radius_rt, int iters, double& px, double& py,
                          int& n_it, int lane, const PyrView& pva, const KltGeoLevel* geo = nullptr, bool back = false) {
  constexpr int TH = KltSmem<R>::TH, TW = KltSmem<R>::TW;
  const int radius = FIXED ? R : radius_rt;  // compile-time window for the default radius
  const int nc = 2 * radius + 3;
  const int nw = 2 * radius + 1;
  const int G = 32 / nc;                     // >= 1 for r <= 14
  const int chunk = (nw + G - 1) / G;        // pixel rows per group
  const int NK = chunk + 3;                  // tap rows a group walks
  const int gi = lane / nc, i = lane - gi * nc;
  const bool col_active = gi < G;
  const bool pix_col = col_active && i >= 1 && i <= nc - 2;
  const int p0 = (col_active ? gi : 0) * chunk;          // first pixel row of this lane's group
  const int p1 = p0 + chunk < nw ? p0 + chunk : nw;      // one past the last
  const double off_i = (double)(i - radius - 1);

  for (int l = pv.levels - 1; l >= 0; --l) {
    int w, h, pitch;
    const uint8_t *I0, *I1;
    if constexpr (GEO) {
      const KltGeoLevel g = geo[l];
      w = g.w;
      h = g.h;
      pitch = g.pitch;
      I0 = back ? g.b : g.a;
      I1 = back ? g.a : g.b;
    } else {
      w = pv.w[l];
      h = pv.h[l];
      pitch = pv.pitch[l];
      const PyrView& va = TWO ? pva : pv;
      I0 = va.base[l] + (size_t)fa * va.fstride[l];
      I1 = pv.base[l] + (size_t)fb * pv.fstride[l];
    }
    const int w0 = TWO ? pva.w[l] : w, h0 = TWO ? pva.h[l] : h;
    const bool a_ok = !TWO || (w0 >= 2 && h0 >= 2);  // otherwise no sample of A is inside A: its tile is not staged
    const double scale = 1.0 / (double)(1 << l);
    const double plx = px * scale, ply = py * scale;
    double dlx = 0.0, dly = 0.0;
    int tx0 = 0, ty0 = 0;
    bool have_tile = false;

    for (int it = 0; it < iters; ++it) {
      const double x = plx + dlx, y = ply + dly;
      const double fxx = floor(x), fyy = floor(y);
      // Window entirely unusable (non-finite or far outside): every sample is 0 -> A = 0 -> zero step.
      const bool finite_ok = (fabs(fxx) < 1.0e9) && (fabs(fyy) < 1.0e9);
      double sx = 0.0, sy = 0.0;
      if (finite_ok && w >= 2 && h >= 2) {
        const int FX = (int)fxx, FY = (int)fyy;
        // cached tile must cover columns [FX-r-1, FX+r+3] and rows [FY-r-1, FY+r+3]
        if (!have_tile || FX - radius - 1 < tx0 || FX + radius + 3 > tx0 + TW - 1 || FY - radius - 1 < ty0 ||
            FY + radius + 3 > ty0 + TH - 1) {
          tx0 = (FX - radius - 1 - KLT_MARGIN) & ~3;
          ty0 = FY - radius - 1 - KLT_MARGIN;
          __syncwarp();
          if (a_ok) stage_tile<R>(sm.t0, I0, h0, TWO ? pva.pitch[l] : pitch, tx0, ty0, lane);
          stage_tile<R>(sm.t1, I1, h, pitch, tx0, ty0, lane);
          have_tile = true;
        }
        bool interior = FX - radius - 1 >= 0 && FX + radius + 3 <= w - 1 && FY - radius - 1 >= 0 && FY + radius + 3 <= h - 1;
        if (TWO) interior = interior && FX + radius + 3 <= w0 - 1 && FY + radius + 3 <= h0 - 1;
        // per-row weight table (lanes 0..nc-1), per-column weights in registers
        if (lane < nc) {
          const double reg = fyy + off_i;            // off_i == lane - r - 1 here
          const double f = (y + off_i) - reg;        // == x - x0 of :189-190, or exactly 1 after a round-up
          sm.cfy[lane] = f;
          if (!interior) {
            const double tf = f == 1.0 ? reg + 1.0 : reg;
            if (TWO)
              sm.cvy[lane] = ((tf >= 0.0 && tf <= (double)(h0 - 2)) ? 1 : 0) | ((tf >= 0.0 && tf <= (double)(h - 2)) ? 2 : 0);
            else
              sm.cvy[lane] = (tf >= 0.0 && tf <= (double)(h - 2)) ? 1 : 0;
          }
        }
        const double regx = fxx + off_i;
        const double fx = (x + off_i) - regx;
        const int col = FX - radius - 1 - tx0 + i;
        const int rowbase = FY - radius - 1 - ty0 + p0;
        __syncwarp();

        double a00 = 0, a01 = 0, a11 = 0, b0 = 0, b1 = 0;
        if (interior) {
          walk_rows<R, FIXED, true>(sm, NK, nc, rowbase, col, p0, p1, pix_col, true, fx, a00, a01, a11, b0, b1);
        } else {
          const double tfx = fx == 1.0 ? regx + 1.0 : regx;
          const bool vx = col_active && tfx >= 0.0 && tfx <= (double)(w - 2);
          if (TWO) {
            const bool vx0 = col_active && tfx >= 0.0 && tfx <= (double)(w0 - 2);
            walk_rows<R, FIXED, false, true>(sm, NK, nc, rowbase, col, p0, p1, pix_col, vx, fx, a00, a01, a11, b0, b1, vx0);
          } else {
            walk_rows<R, FIXED, false>(sm, NK, nc, rowbase, col, p0, p1, pix_col, vx, fx, a00, a01, a11, b0, b1);
          }
        }
        reduce5(a00, a01, a11, b0, b1, lane);
        // a** = 4*A, b* = 2*b of :444-448 (exact power-of-two scalings): det' = 16 det, step = 2 * A'^-1 b'
        const double det = a00 * a11 - a01 * a01;
        if (!(fabs(det) < 16.0 * 1e-9)) {  // |det| < 1e-9 of :452, scaled exactly
          const double rd = 2.0 / det;
          sx = (a11 * b0 - a01 * b1) * rd;
          sy = (a00 * b1 - a01 * b0) * rd;
        }
      }
      n_it++;
      dlx += sx;
      dly += sy;
      if (sfm_lk_step_small(sx, sy)) break;  // hypot(step) < 1e-3 (:416)
    }
    const double up = (double)(1 << l);
    px = (plx + dlx) * up;
    py = (ply + dly) * up;
  }
}

// list == nullptr: one warp per slot of the launch (grid covers them all).  list != nullptr: the warps of a
// fixed-size grid walk the deferred-feature list written by klt_lane_kernel (count read from device memory).
// TWO: image A from k.pv, image B from k.pvb (two batches, any sizes); the backward track swaps the two views.
// GEO: both images of pair k from k.geo[k].
template <int R, bool FIXED, bool TWO, bool GEO = false>
__global__ void __launch_bounds__(128, (R <= 5 ? 6 : 3)) klt_kernel(KltLaunch k, const int* __restrict__ list,
                                                                    const int* __restrict__ list_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  KltSmem<R>& sm = reinterpret_cast<KltSmem<R>*>(smem_raw)[warp];
  const long long nwork = list ? (long long)*list_count : (long long)k.npairs * k.cap;
  for (long long idx = (long long)blockIdx.x * (blockDim.x >> 5) + warp; idx < nwork; idx += (long long)gridDim.x * (blockDim.x >> 5)) {
    const long long g = list ? (long long)list[idx] : idx;
    const int pair = (int)(g / k.cap), slot = (int)(g - (long long)pair * k.cap);
    if (k.counts && slot >= k.counts[pair]) continue;
    const int fa = k.fa0 + pair * k.fa_step, fb = k.fb0 + pair * k.fb_step;
    const double2 p0 = k.p0[g];
    int n_it = 0;
    double x = p0.x, y = p0.y;
    __syncwarp();
    if constexpr (GEO) {
      const KltGeoLevel* geo = k.geo[pair].lv;
      track_one<R, FIXED, false, true>(sm, k.pv, 0, 0, k.radius, k.iters, x, y, n_it, lane, k.pv, geo, false);
    } else {
      track_one<R, FIXED, TWO>(sm, TWO ? k.pvb : k.pv, fa, fb, k.radius, k.iters, x, y, n_it, lane, k.pv);
    }
    const double x1 = x, y1 = y;
    __syncwarp();
    if (k.pb) {  // pb == null: forward only
      if constexpr (GEO)
        track_one<R, FIXED, false, true>(sm, k.pv, 0, 0, k.radius, k.iters, x, y, n_it, lane, k.pv, k.geo[pair].lv, true);
      else
        track_one<R, FIXED, TWO>(sm, k.pv, fb, fa, k.radius, k.iters, x, y, n_it, lane, TWO ? k.pvb : k.pv);
    }
    if (lane == 0) {
      k.p1[g] = make_double2(x1, y1);
      if (k.pb) k.pb[g] = make_double2(x, y);
      if (k.nit) k.nit[g] = n_it;
      if (k.keep) {
        const double fbd = hypot(x - p0.x, y - p0.y);
        k.keep[g] = (fbd >= k.fb_thresh) ? 0 : 1;  // NaN is kept (:362)
      }
    }
  }
}

template <int R, bool FIXED, bool TWO = false, bool GEO = false>
int launch_r(sfmgpu_ctx* ctx, const KltLaunch& k, const int* list, const int* list_count) {
  const int warps_per_block = 4;
  // Without FIXED, the last row group of a window of radius 1..3 walks up to two tap rows past the rows its pixels need
  // (G * chunk exceeds 2r + 2), which can lie past the tile; those samples are never accumulated, and the pad keeps the
  // last warp's reads inside the block's shared memory.
  const size_t smem = sizeof(KltSmem<R>) * warps_per_block + (FIXED ? 0 : 2 * KltSmem<R>::TW);
  static const int cfg_id = sfm_next_cfg_id();  // one per template instantiation
  SFM_SMEM_OPTIN(ctx, cfg_id, (klt_kernel<R, FIXED, TWO, GEO>), smem);
  const long long total = (long long)k.npairs * k.cap;
  if (total == 0) return 0;
  unsigned grid = sfm_cdiv(total, warps_per_block);
  if (list) {
    const unsigned cap = (unsigned)ctx->n_sm * 24;  // deferred features are a few % of the batch: a resident grid walks the list
    grid = grid < cap ? grid : cap;
  }
  SFM_LAUNCH(ctx, (klt_kernel<R, FIXED, TWO, GEO>), grid, warps_per_block * 32, smem, k, list, list_count);
  return 0;
}

}  // namespace

// klt_lane.cu
int sfm_klt_lane_launch(sfmgpu_ctx* ctx, const KltLaunch& k, int* defer_count, int* defer_list, int variant);
int sfm_klt_lane_masked_launch(sfmgpu_ctx* ctx, const KltLaunch& k, const int* in_list, const int* in_count, int* defer_count,
                               int* defer_list);

// Batches of at least this many feature slots go to the lane-per-feature kernel (32 features per warp need many
// features to fill 148 SMs); smaller ones (a single tracker step) keep one warp per feature.
static const long long KLT_LANE_MIN = 6000;

static bool same_view(const PyrView& a, const PyrView& b) {
  if (a.levels != b.levels) return false;
  for (int l = 0; l < a.levels; l++)
    if (a.base[l] != b.base[l] || a.w[l] != b.w[l] || a.h[l] != b.h[l] || a.pitch[l] != b.pitch[l] || a.fstride[l] != b.fstride[l])
      return false;
  return true;
}

int sfm_klt_launch(sfmgpu_ctx* ctx, const KltLaunch& k) {
  if (k.radius < 1 || k.radius > 10)
    return sfm_fail(ctx, SFMGPU_E_ARG, "klt: win_radius %d outside the supported range [1,10]", k.radius);
  if (k.iters < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "klt: negative iteration count");
  if (!k.geo && !same_view(k.pv, k.pvb)) {  // two batches: the lane kernels assume one geometry, so the mode does not apply
    if (k.pv.levels != k.pvb.levels) return sfm_fail(ctx, SFMGPU_E_ARG, "klt: pyramid level counts differ (%d, %d)", k.pv.levels, k.pvb.levels);
    if (k.radius == 5) return launch_r<5, true, true>(ctx, k, nullptr, nullptr);
    if (k.radius < 5) return launch_r<5, false, true>(ctx, k, nullptr, nullptr);
    if (k.radius == 10) return launch_r<10, true, true>(ctx, k, nullptr, nullptr);
    return launch_r<10, false, true>(ctx, k, nullptr, nullptr);
  }
  const long long total = (long long)k.npairs * k.cap;
  const int* list = nullptr;
  const int* list_count = nullptr;
  const int mode = ctx->klt_mode;  // 0 auto, 1 warp-per-feature only, 2 lane-per-feature (+ deferred) always, 10+v tuning variant v
  if (k.radius == 5 && total < (1ll << 31) && (mode >= 2 || (mode == 0 && total >= KLT_LANE_MIN))) {
    // chain: interior windows (lane kernel) -> border windows (masked lane kernel) -> the rest (warp-per-feature)
    SFM_TRY(sfm_reserve(ctx, ctx->klt_defer, 2 * (size_t)(total + 2) * sizeof(int)));
    int* dcount = (int*)ctx->klt_defer.p;  // [0] first list, [1] second list
    int* dlist1 = dcount + 2;
    int* dlist2 = dlist1 + total;
    SFM_CUDA(ctx, cudaMemsetAsync(dcount, 0, 2 * sizeof(int), ctx->stream));
    SFM_TRY(sfm_klt_lane_launch(ctx, k, dcount, dlist1, mode >= 10 ? mode - 10 : 0));
    if (mode == 19) {  // tuning: skip the masked kernel
      list = dlist1;
      list_count = dcount;
    } else {
      SFM_TRY(sfm_klt_lane_masked_launch(ctx, k, dlist1, dcount, dcount + 1, dlist2));
      list = dlist2;
      list_count = dcount + 1;
    }
  }
  if (k.geo) {  // per-list geometry: the same chain through the table instantiations
    if (k.radius == 5) return launch_r<5, true, false, true>(ctx, k, list, list_count);
    if (k.radius < 5) return launch_r<5, false, false, true>(ctx, k, list, list_count);
    if (k.radius == 10) return launch_r<10, true, false, true>(ctx, k, list, list_count);
    return launch_r<10, false, false, true>(ctx, k, list, list_count);
  }
  if (k.radius == 5) return launch_r<5, true>(ctx, k, list, list_count);
  if (k.radius < 5) return launch_r<5, false>(ctx, k, list, list_count);
  if (k.radius == 10) return launch_r<10, true>(ctx, k, list, list_count);
  return launch_r<10, false>(ctx, k, list, list_count);
}

extern "C" int sfmgpu_klt_set_mode(sfmgpu_ctx* ctx, int mode) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  if (mode < 0 || (mode > 2 && (mode < 10 || mode > 19)))
    return sfm_fail(ctx, SFMGPU_E_ARG, "klt_set_mode: mode %d not in {0,1,2} (10..19: tuning variants)", mode);
  ctx->klt_mode = mode;
  return 0;
}

// Host points in, host results out: frame_a of view a -> frame_b of view b and back.
static int klt_track_host(sfmgpu_ctx* ctx, const PyrView& va, int frame_a, const PyrView& vb, int frame_b, const double* p0_xy, int n,
                          int win_radius, int iters, double* p1_xy, double* p0_back_xy, int32_t* n_iters) {
  const size_t pb = (size_t)n * sizeof(double2);
  SFM_TRY(sfm_reserve(ctx, ctx->klt_in, pb));
  SFM_TRY(sfm_reserve(ctx, ctx->klt_p1, pb));
  SFM_TRY(sfm_reserve(ctx, ctx->klt_pb, pb));
  SFM_TRY(sfm_reserve(ctx, ctx->klt_nit, (size_t)n * sizeof(int)));
  SFM_CUDA(ctx, cudaMemcpyAsync(ctx->klt_in.p, p0_xy, pb, cudaMemcpyHostToDevice, ctx->stream));
  KltLaunch k;
  k.pv = va;
  k.pvb = vb;
  k.p0 = (const double2*)ctx->klt_in.p;
  k.counts = nullptr;
  k.npairs = 1;
  k.cap = n;
  k.fa0 = frame_a;
  k.fa_step = 0;
  k.fb0 = frame_b;
  k.fb_step = 0;
  k.radius = win_radius;
  k.iters = iters;
  k.fb_thresh = 0.0;
  k.p1 = (double2*)ctx->klt_p1.p;
  k.pb = p0_back_xy ? (double2*)ctx->klt_pb.p : nullptr;  // forward only when the caller does not want the way back
  k.nit = (int*)ctx->klt_nit.p;
  k.keep = nullptr;
  SFM_TRY(sfm_klt_launch(ctx, k));
  SFM_CUDA(ctx, cudaMemcpyAsync(p1_xy, ctx->klt_p1.p, pb, cudaMemcpyDeviceToHost, ctx->stream));
  if (p0_back_xy) SFM_CUDA(ctx, cudaMemcpyAsync(p0_back_xy, ctx->klt_pb.p, pb, cudaMemcpyDeviceToHost, ctx->stream));
  if (n_iters)
    SFM_CUDA(ctx, cudaMemcpyAsync(n_iters, ctx->klt_nit.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int sfmgpu_klt_track(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame_a, int frame_b, const double* p0_xy, int n,
                                int win_radius, int iters, double* p1_xy, double* p0_back_xy, int32_t* n_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !f) return SFMGPU_E_ARG;
  if (frame_a < 0 || frame_a >= f->n || frame_b < 0 || frame_b >= f->n || n < 0)
    return sfm_fail(ctx, SFMGPU_E_ARG, "klt_track: bad frame index or count");
  if (n == 0) return 0;
  if (!p0_xy || !p1_xy) return sfm_fail(ctx, SFMGPU_E_ARG, "klt_track: null pointer");
  const PyrView v = f->view();
  return klt_track_host(ctx, v, frame_a, v, frame_b, p0_xy, n, win_radius, iters, p1_xy, p0_back_xy, n_iters);
}

extern "C" int sfmgpu_klt_track_between(sfmgpu_ctx* ctx, sfmgpu_frames* fa, int frame_a, sfmgpu_frames* fb, int frame_b,
                                        const double* p0_xy, int n, int win_radius, int iters, double* p1_xy, double* p0_back_xy,
                                        int32_t* n_iters) {
  SFM_ENTER(ctx);
  if (!ctx || !fa || !fb) return SFMGPU_E_ARG;
  if (fa == fb) return sfmgpu_klt_track(ctx, fa, frame_a, frame_b, p0_xy, n, win_radius, iters, p1_xy, p0_back_xy, n_iters);
  if (frame_a < 0 || frame_a >= fa->n || frame_b < 0 || frame_b >= fb->n || n < 0)
    return sfm_fail(ctx, SFMGPU_E_ARG, "klt_track_between: bad frame index or count");
  if (fa->levels != fb->levels)
    return sfm_fail(ctx, SFMGPU_E_ARG, "klt_track_between: pyramid level counts differ (%d, %d)", fa->levels, fb->levels);
  if (n == 0) return 0;
  if (!p0_xy || !p1_xy) return sfm_fail(ctx, SFMGPU_E_ARG, "klt_track_between: null pointer");
  return klt_track_host(ctx, fa->view(), frame_a, fb->view(), frame_b, p0_xy, n, win_radius, iters, p1_xy, p0_back_xy, n_iters);
}
