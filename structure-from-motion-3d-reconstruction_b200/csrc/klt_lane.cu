// klt_lane.cu — pyramidal Lucas-Kanade for LARGE batches: one LANE per feature (32 features per warp).
//
// Same reference functions as klt.cu (cpp/src/templering_sfm.cpp: sample_bilinear :183-198, track_one :402-422,
// lk_step :424-460, fwd/bwd + fb test :356-362 / :1845-1849) and the same bug-for-bug behaviour; what changes is
// the mapping.  Measured on B200 (scripts/ubench_pipes.cu): a DFMA/DADD holds the issue port of its
// sub-partition for ~2.3 cycles and does NOT overlap with ALU/LSU issue, so the cost of an LK iteration is
// (2.3 x FP64 instructions + 1 x everything else).  The warp-per-feature kernel of klt.cu spends 77 % of its issue
// slots on "everything else" (byte loads, conversions, shuffles, predication, the warp reduction).  Here a lane
// owns a whole window, so there are no shuffles and no reduction, each tile byte is loaded and converted once, and
// the FP64 instructions are ~75 % of the issue slots.
//
//   * Tile: the 14 x 14 u8 taps of both images around the window, 16-byte rows, private to the lane in shared
//     memory (464 B per lane, lane stride chosen so that the per-row LDS.128 is bank-conflict free).  The tile is
//     re-staged only when the INTEGER window position changes; staging is cooperative (28 lanes fetch the 28 rows
//     of one feature with 16-byte loads and realign them), so global traffic stays sector-efficient.
//   * u8 -> double: one PRMT (byte extract) + one I2F.F64 per tile byte.  The conversion pipe runs beside the
//     FP64 pipe (measured: a DFMA + I2F.F64 pair costs what the I2F alone costs), so conversions only cost their
//     issue slot.  (Dropping the byte into the mantissa of a constant needs a second ALU instruction to zero the low
//     word of every register pair and would move the lerp roundings to ulp(4096).)
//   * One fractional offset (fx, fy) = position - floor(position) is shared by the whole window (the reference
//     re-rounds x + dx per tap, which jitters each sample position by <= ulp(x)/2 ~ 1e-13 px).
//   * Only INTERIOR windows are handled (every tap of the 14 x 14 region, plus the reference's round-up tap, inside
//     the image).  A feature whose window touches the border, or whose position is not finite, is appended to a
//     "deferred" list and recomputed from scratch by the exact warp-per-feature kernel of klt.cu (which implements
//     the out-of-bounds rule :188 tap by tap).
#include <type_traits>

#include "common.cuh"

namespace {

constexpr int LR = 5;                        // window radius handled here (the reference default, LKConfig :313)
constexpr int LN = 2 * LR + 4;               // 14 tap rows / columns
constexpr int LNC = 2 * LR + 3;              // 13 grid rows / columns (window + 1 each side)
constexpr int LIMG = LN * 16;                // bytes of one staged image tile
constexpr int LSTRIDE = 2 * LIMG + 16;       // bytes per lane: 116 words, == 20 (mod 32) -> LDS.128 conflict free
constexpr int LWARPS = 1;                    // warps per block (no block-level cooperation)

__device__ __forceinline__ double byte_f64(uint32_t w, int k) {
  // PRMT extracts the byte, the conversion pipe (I2F.F64, overlaps with FP64 issue) widens it.  Inline PTX keeps
  // the compiler from rewriting (double)c - (double)a as a second conversion of the integer difference.
  const uint32_t b = __byte_perm(w, 0, 0x4440 | k);
  double d;
  asm("cvt.rn.f64.u32 %0, %1;" : "=d"(d) : "r"(b));
  return d;
}

// 14 consecutive tap bytes of one tile row as doubles
__device__ __forceinline__ void row_bytes(const uint4 q, double (&v)[LN]) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < LN; i++) v[i] = byte_f64(w[i >> 2], i & 3);
}

// Horizontal lerps a + (b - a) * fx of one tile row (grid columns I0..I1-1 use taps i, i+1)
template <int I0, int I1>
__device__ __forceinline__ void hlerp_row(const unsigned char* rowp, double fx, double (&h)[LNC]) {
  double px[LN];
  row_bytes(*reinterpret_cast<const uint4*>(rowp), px);
#pragma unroll
  for (int i = I0; i < I1; i++) h[i] = __fma_rn(fx, px[i + 1] - px[i], px[i]);
}

// One tap row of the main window walk, straight-line.  v = tap row (3..13, warp-uniform, runtime).  Computes the
// horizontal lerps of I1 row v, completes grid row v-1 of I1 into `snew`, and accumulates pixel row g = v-2 from
// sold = S1[g-1], smid = S1[g], snew = S1[g+1] and S0[g] (I0 tap rows g = h0p and g+1 = tap row v-1).
// ACC: accumulator sets (2 = even / odd columns: shorter dependent DFMA chains).
// MASKED: out-of-bounds rule of sample_bilinear (:188) - a sample whose tap pair leaves the image in x (bit i of cm
// clear) or in y (bit of rm clear) is 0.0; cm / rm are per-lane masks over grid columns / rows.
template <int ACC, bool MASKED>
__device__ __forceinline__ void walk_row(const unsigned char* tile, int v, double fx, double fy, unsigned cm, unsigned rm,
                                         double (&h1p)[LNC], double (&h0p)[LNC], const double (&sold)[LNC], const double (&smid)[LNC],
                                         double (&snew)[LNC], double (&acc)[ACC][5]) {
  double px[LN];
  row_bytes(*reinterpret_cast<const uint4*>(tile + v * 16), px);
  const unsigned cnew = MASKED ? (((rm >> (v - 1)) & 1u) ? cm : 0u) : 0u;  // grid row v-1
  const unsigned cpix = MASKED ? (((rm >> (v - 2)) & 1u) ? cm : 0u) : 0u;  // grid row v-2 (the pixel row)
#pragma unroll
  for (int i = 0; i < LNC; i++) {
    const double h = __fma_rn(fx, px[i + 1] - px[i], px[i]);
    double sn = __fma_rn(fy, h - h1p[i], h1p[i]);  // grid row v-1 of I1
    if (MASKED) sn = ((cnew >> i) & 1u) ? sn : 0.0;
    snew[i] = sn;
    h1p[i] = h;
  }
  row_bytes(*reinterpret_cast<const uint4*>(tile + LIMG + (v - 1) * 16), px);
#pragma unroll
  for (int i = 1; i <= LNC - 2; i++) {
    const double h = __fma_rn(fx, px[i + 1] - px[i], px[i]);
    double s0 = __fma_rn(fy, h - h0p[i], h0p[i]);
    if (MASKED) s0 = ((cpix >> i) & 1u) ? s0 : 0.0;
    h0p[i] = h;
    const double gx2 = smid[i + 1] - smid[i - 1];  // 2*Ix (:439)
    const double gy2 = snew[i] - sold[i];          // 2*Iy (:440)
    const double e = s0 - smid[i];                 // I0 - I1 at the same location (:441-442)
    double(&a)[5] = acc[i % ACC];
    a[0] = __fma_rn(gx2, gx2, a[0]);
    a[1] = __fma_rn(gx2, gy2, a[1]);
    a[2] = __fma_rn(gy2, gy2, a[2]);
    a[3] = __fma_rn(gx2, e, a[3]);
    a[4] = __fma_rn(gy2, e, a[4]);
  }
}

// The five sums of lk_step (:431-448) for one interior window.  tile: this lane's staged taps (image B = I1 first,
// then image A = I0).  Returns 4*A and 2*b like klt.cu (the 0.5 factors are folded into the solve).
//
// Tap rows 0..2 only feed lerps (no pixel row is complete yet) and are peeled.  Rows 3..13 are a ROLLED loop over
// groups of three rows (the three S1 row buffers rotate by argument order), so the hot code is ~16 KB and stays in
// the 32 KB instruction cache.  Fully unrolled, the 14 rows are 53 KB and the kernel stalls on instruction fetch
// (measured: 'no_instruction' was the top stall reason).  The 15th row of the last group does not exist and is skipped.
template <int ACC, bool MASKED>
__device__ __forceinline__ void window_sums(const unsigned char* tile, double fx, double fy, unsigned cm, unsigned rm, double& a00,
                                            double& a01, double& a11, double& b0, double& b1) {
  double h1p[LNC], h0p[LNC], s0[LNC], s1[LNC], s2[LNC], t[LNC];
  double acc[ACC][5];
#pragma unroll
  for (int j = 0; j < ACC; j++)
#pragma unroll
    for (int q = 0; q < 5; q++) acc[j][q] = 0.0;
  hlerp_row<0, LNC>(tile, fx, h1p);  // I1 tap row 0
  hlerp_row<0, LNC>(tile + 16, fx, t);  // I1 tap row 1 -> grid row 0
  const unsigned c0 = MASKED ? ((rm & 1u) ? cm : 0u) : 0u, c1 = MASKED ? ((rm & 2u) ? cm : 0u) : 0u;
#pragma unroll
  for (int i = 0; i < LNC; i++) {
    s0[i] = __fma_rn(fy, t[i] - h1p[i], h1p[i]);
    if (MASKED) s0[i] = ((c0 >> i) & 1u) ? s0[i] : 0.0;
    h1p[i] = t[i];
  }
  hlerp_row<0, LNC>(tile + 32, fx, t);  // I1 tap row 2 -> grid row 1
#pragma unroll
  for (int i = 0; i < LNC; i++) {
    s1[i] = __fma_rn(fy, t[i] - h1p[i], h1p[i]);
    if (MASKED) s1[i] = ((c1 >> i) & 1u) ? s1[i] : 0.0;
    h1p[i] = t[i];
  }
  hlerp_row<1, LNC - 1>(tile + LIMG + 16, fx, h0p);  // I0 tap row 1
  // step v writes grid row v-1 into buffer (v-1) % 3 and reads grid rows v-3, v-2 from the other two
#pragma unroll 1
  for (int v = 3; v < LN; v += 3) {
    walk_row<ACC, MASKED>(tile, v, fx, fy, cm, rm, h1p, h0p, s0, s1, s2, acc);      // writes s2
    walk_row<ACC, MASKED>(tile, v + 1, fx, fy, cm, rm, h1p, h0p, s1, s2, s0, acc);  // writes s0
    if (v + 2 < LN) walk_row<ACC, MASKED>(tile, v + 2, fx, fy, cm, rm, h1p, h0p, s2, s0, s1, acc);  // writes s1
  }
  a00 = acc[0][0]; a01 = acc[0][1]; a11 = acc[0][2]; b0 = acc[0][3]; b1 = acc[0][4];
#pragma unroll
  for (int j = 1; j < ACC; j++) {
    a00 += acc[j][0]; a01 += acc[j][1]; a11 += acc[j][2]; b0 += acc[j][3]; b1 += acc[j][4];
  }
}

// Cooperative staging of one feature's tiles, split in two halves so that the loads of several features are in
// flight together: lanes 0..27 each fetch one 14-byte row segment (image = t / 14, row = t % 14) starting at byte
// column x0 with two aligned 16-byte loads (stage_load), then realign and store one 16-byte smem row (stage_store).
struct StageRegs {
  uint4 lo, hi;
};

// CLAMP (border windows): rows are clamped to the image and each 16-byte chunk to the row's allocation; a chunk that
// had to move only ever held taps outside the image, whose samples the masks zero (pitch is a multiple of 16, so a
// chunk lies either entirely inside [0, pitch) or entirely outside).
template <bool CLAMP>
__device__ __forceinline__ void stage_load(StageRegs& r, const uint8_t* __restrict__ imgA, const uint8_t* __restrict__ imgB, int pitch,
                                           int h, int x0, int y0, int lane) {
  const int img = lane >= LN ? 1 : 0, row = lane - img * LN;
  int y = y0 + row;
  if (CLAMP) y = y < 0 ? 0 : (y > h - 1 ? h - 1 : y);
  const uint8_t* rowp = (img ? imgA : imgB) + (size_t)y * pitch;  // tile order: I1 (= image B) first
  const int xa = x0 & ~15, o = x0 & 15;
  int c0 = xa, c1 = xa + 16;
  if (CLAMP) {
    c0 = c0 < 0 ? 0 : (c0 > pitch - 16 ? pitch - 16 : c0);
    c1 = c1 < 0 ? 0 : (c1 > pitch - 16 ? pitch - 16 : c1);
  }
  r.lo = __ldg(reinterpret_cast<const uint4*>(rowp + c0));
  r.hi = make_uint4(0, 0, 0, 0);
  if (o > 2) r.hi = __ldg(reinterpret_cast<const uint4*>(rowp + c1));  // needed bytes reach the next chunk
}

// Bytes 14 and 15 of a staged row are zero: the Gram build of klt_quad_kernel masks a pixel by selecting byte 15.
__device__ __forceinline__ void stage_store(const StageRegs& r, unsigned char* tile_s, int x0, int lane) {
  const int img = lane >= LN ? 1 : 0, row = lane - img * LN;
  const int o = x0 & 15, q = o >> 2, sh = (o & 3) * 8;
  uint32_t W[8] = {r.lo.x, r.lo.y, r.lo.z, r.lo.w, r.hi.x, r.hi.y, r.hi.z, r.hi.w};
  if (q & 2) { W[0] = W[2]; W[1] = W[3]; W[2] = W[4]; W[3] = W[5]; W[4] = W[6]; W[5] = W[7]; }
  if (q & 1) { W[0] = W[1]; W[1] = W[2]; W[2] = W[3]; W[3] = W[4]; W[4] = W[5]; }
  uint4 out;
  out.x = __funnelshift_r(W[0], W[1], sh);
  out.y = __funnelshift_r(W[1], W[2], sh);
  out.z = __funnelshift_r(W[2], W[3], sh);
  out.w = __funnelshift_r(W[3], W[4], sh) & 0xFFFFu;
  *reinterpret_cast<uint4*>(tile_s + img * LIMG + row * 16) = out;
}

// MASKED = false: slots of the launch, interior windows only; everything else goes to defer_list.
// MASKED = true : walks in_list (the first kernel's deferred features) with the out-of-bounds rule applied through
//                 masks; what it still cannot do exactly (non-finite positions, a fractional part so close to 1 that
//                 the reference's own floor(fl(x + dx)) may land on the next integer, degenerate level sizes) is
//                 deferred once more, to the warp-per-feature kernel of klt.cu.
template <int ACC, int MINB, int LSTAGE, bool MASKED>
__global__ void __launch_bounds__(32 * LWARPS, MINB) klt_lane_kernel(KltLaunch k, const int* __restrict__ in_list,
                                                                     const int* __restrict__ in_count, int* __restrict__ defer_count,
                                                                     int* __restrict__ defer_list) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned FULL = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* wtile = smem_raw + (size_t)warp * 32 * LSTRIDE;
  unsigned char* tile = wtile + lane * LSTRIDE;
  const long long total = (long long)k.npairs * k.cap;
  const long long nwork = MASKED ? (long long)*in_count : total;
  for (long long wbase = ((long long)blockIdx.x * LWARPS + warp) * 32; wbase < nwork; wbase += (long long)gridDim.x * LWARPS * 32) {
  const long long widx = wbase + lane;
  long long g = widx;
  if (MASKED) g = widx < nwork ? (long long)in_list[widx] : total;
  const int pair = g < total ? (int)(g / k.cap) : 0;
  const int slot = (int)(g - (long long)pair * k.cap);
  const bool valid = g < total && (!k.counts || slot < k.counts[pair]);

  double2 p0 = make_double2(0.0, 0.0);
  if (valid) p0 = k.p0[g];
  double px = p0.x, py = p0.y, x1 = 0.0, y1 = 0.0;
  int n_it = 0;
  bool alive = valid;
  const int ndir = k.pb ? 2 : 1;

  for (int dir = 0; dir < ndir; dir++) {
    for (int l = k.pv.levels - 1; l >= 0; --l) {
      const int w = k.pv.w[l], h = k.pv.h[l], pitch = k.pv.pitch[l];
      const uint8_t* lbase = k.pv.base[l];
      const size_t fstride = k.pv.fstride[l];
      const double scale = 1.0 / (double)(1 << l);
      const double plx = px * scale, ply = py * scale;
      double dlx = 0.0, dly = 0.0;
      bool done = !alive;
      int tFX = INT_MIN, tFY = INT_MIN;
      for (int it = 0; it < k.iters; ++it) {
        if (!__any_sync(FULL, !done)) break;
        const double x = plx + dlx, y = ply + dly;
        const double fxx = floor(x), fyy = floor(y);
        int FX = 0, FY = 0;
        unsigned cm = 0, rm = 0;
        bool act = !done;
        if (act) {
          const bool finite_ok = (fabs(fxx) < 1.0e9) && (fabs(fyy) < 1.0e9);
          FX = finite_ok ? (int)fxx : 0;
          FY = finite_ok ? (int)fyy : 0;
          bool ok;
          if (!MASKED) {
            ok = finite_ok && FX - LR - 1 >= 0 && FX + LR + 3 <= w - 1 && FY - LR - 1 >= 0 && FY + LR + 3 <= h - 1;
          } else {
            const double lim = 1.0 - 5.9604644775390625e-8;  // 1 - 2^-24 >> the ulp of any x + dx: the floors agree below it
            ok = finite_ok && w >= 16 && h >= 16 && (x - fxx) <= lim && (y - fyy) <= lim;
            if (ok) {
              // grid column i / row j uses taps FX + i - r - 1 (+1): inside iff 0 <= tap <= w - 2
#pragma unroll
              for (int i = 0; i < LNC; i++) {
                const int cx = FX + i - LR - 1, cy = FY + i - LR - 1;
                cm |= (cx >= 0 && cx <= w - 2) ? (1u << i) : 0u;
                rm |= (cy >= 0 && cy <= h - 2) ? (1u << i) : 0u;
              }
            }
          }
          if (!ok) {  // the next kernel in the chain redoes this feature from scratch
            alive = false;
            done = true;
            act = false;
          }
        }
        unsigned need = __ballot_sync(FULL, act && (FX != tFX || FY != tFY));
        if (need) {
          __syncwarp();
          while (need) {
            // up to LSTAGE features per round: all their loads are issued before the first realign / store
            int ss[LSTAGE], sx0[LSTAGE];
            StageRegs sr[LSTAGE];
#pragma unroll
            for (int j = 0; j < LSTAGE; j++) {
              ss[j] = need ? __ffs(need) - 1 : -1;
              need &= need - 1;
              const int src = ss[j] < 0 ? 0 : ss[j];
              const int sFX = __shfl_sync(FULL, FX, src), sFY = __shfl_sync(FULL, FY, src), spair = __shfl_sync(FULL, pair, src);
              const int sA = k.fa0 + spair * k.fa_step, sB = k.fb0 + spair * k.fb_step;
              sx0[j] = sFX - LR - 1;
              if (ss[j] >= 0 && lane < 2 * LN)
                stage_load<MASKED>(sr[j], lbase + (size_t)(dir ? sB : sA) * fstride, lbase + (size_t)(dir ? sA : sB) * fstride, pitch, h,
                                   sx0[j], sFY - LR - 1, lane);
            }
#pragma unroll
            for (int j = 0; j < LSTAGE; j++)
              if (ss[j] >= 0 && lane < 2 * LN) stage_store(sr[j], wtile + ss[j] * LSTRIDE, sx0[j], lane);
          }
          __syncwarp();
        }
        if (act) {
          tFX = FX;
          tFY = FY;
          double a00, a01, a11, b0, b1;
          window_sums<ACC, MASKED>(tile, x - fxx, y - fyy, cm, rm, a00, a01, a11, b0, b1);
          double sx = 0.0, sy = 0.0;
          const double det = a00 * a11 - a01 * a01;
          if (!(fabs(det) < 16.0 * 1e-9)) {  // |det| < 1e-9 of :452 on the 16x scaled determinant
            const double rd = 2.0 / det;
            sx = (a11 * b0 - a01 * b1) * rd;
            sy = (a00 * b1 - a01 * b0) * rd;
          }
          n_it++;
          dlx += sx;
          dly += sy;
          if (sfm_lk_step_small(sx, sy)) done = true;  // hypot(step) < 1e-3 (:416), tested on the step just added
        }
      }
      const double up = (double)(1 << l);
      px = (plx + dlx) * up;
      py = (ply + dly) * up;
    }
    if (dir == 0) {
      x1 = px;
      y1 = py;
    }
  }
  if (alive) {
    k.p1[g] = make_double2(x1, y1);
    if (k.pb) k.pb[g] = make_double2(px, py);
    if (k.nit) k.nit[g] = n_it;
    if (k.keep) {
      const double fbd = hypot(px - p0.x, py - p0.y);
      k.keep[g] = (fbd >= k.fb_thresh) ? 0 : 1;  // NaN is kept (:362)
    }
  }
  // deferred features: one atomic per warp, list order is irrelevant (results are written by slot)
  const unsigned dm = __ballot_sync(FULL, valid && !alive);
  if (dm) {
    int base = 0;
    if (lane == 0) base = atomicAdd(defer_count, __popc(dm));
    base = __shfl_sync(FULL, base, 0);
    if (valid && !alive) defer_list[base + __popc(dm & ((1u << lane) - 1u))] = (int)g;
  }
  __syncwarp();
  }
}


// ---- quadratic-form kernel (interior windows) ---------------------------------------------------------------------------
// Every sample of lk_step's window is taken at the SAME fractional offset (fx, fy), so a bilinear sample is the dot
// product w . n of the weight vector w = ((1-fx)(1-fy), fx(1-fy), (1-fx)fy, fx fy) with four INTEGER tap values, and
// 2*Ix, 2*Iy and the error I0 - I1 (:439-442) are w . vx, w . vy, w . ve with integer tap differences.  The five sums
// of :443-447 are therefore quadratic forms  w^T M w  with 4x4 INTEGER matrices M = sum over the window of v v'^T that
// depend only on the two images and the integer window position.  While the position stays inside one pixel - steps
// are a few hundredths of a pixel - an LK iteration costs ~90 FP64 instructions instead of ~2,500; the matrices are
// rebuilt (exact integer arithmetic: one Gram matrix of raw taps per feature on the tensor cores, below) only when
// floor(position) or the pyramid level changes.  The matrices
// are exact, so the sums differ from the reference's 121-term FP64 loops only by rounding (measured: DESIGN.md §4).
//
// Build: with D[r][c] the tap-difference images (DX[r][c] = T1[r][c+1] - T1[r][c-1], DY[r][c] = T1[r+1][c] - T1[r-1][c],
// DE[r][c] = T0[r][c] - T1[r][c]; r, c = 1..12 in tile coordinates), window pixel (r, c), r, c = 1..11, has
// v = (D[r][c], D[r][c+1], D[r+1][c], D[r+1][c+1]).  Entry (k, l) of M is a sum of products A[.]B[.] over a shifted
// 11 x 11 window of the 12 x 12 grid, so the ten entries of a family come from FIVE product sums over the grid (same
// position, right neighbour, lower neighbour, the two diagonals) minus boundary rows / columns.
//
// (Tried and dropped: the build in FP32 on integer-valued floats - FFMA issues on both FP32 pipes - needs two more
// accumulators per mixed family to stay below 2^24 and spills: 23.8 ms vs 16.1 ms; staging rounds of 8 / 16 features
// instead of 4: 27 / 57 ms, spills again.)
//
// (Also tried: a quadratic-form variant for BORDER windows.  The out-of-bounds rule zeroes whole samples, so the mask
// does not shift with the tap index and all 68 products per pixel must be accumulated directly: ~12 k instructions per
// build, no faster than the FP64 masked walk of klt_lane_kernel<..., true> - 15.05 vs 14.96 ms for the stage.)
//
// (Also tried, round 2: the build on packed FP32 - FFMA2 with (dx, dy) register pairs advances the xx and yy families, the two
// orders of the mixed family and (xe, ye) together: 216 FFMA2 per grid row instead of 414 FFMA, 521 instead of 805
// instructions per row, bit-identical matrices - and SLOWER: 15.7 vs 14.8 ms on C2, 24.4 vs 22.8 ms on 400 4K frames; with
// the row loops unrolled by two 19.0 / 30.0 ms.  An FFMA2 holds the FMA pipe for ~2.4 cycles, so a build that is bound by the
// FMA pipe gains nothing from the saved issue slots and pays for the register-pair moves.)
//
// Lanes of a warp advance independently (level, iteration): a lane iterates while its matrices are valid and waits when
// it needs new ones; when every unfinished lane waits, all of them stage their tiles and build together.
constexpr int QM = 50;                         // doubles per lane: XX, YY, XY, XE, YE x 10 upper-triangle entries
static_assert(QM * 8 <= 2 * LIMG, "the matrices alias the lane's tile");

// Scalar type of the build: int32 (IMAD) or FP32 on integer-valued floats (FFMA, exact below 2^24: the largest entry is a
// sum of 2 x 121 products of magnitude <= 65,025 = 15.7e6).
template <typename T>
struct QuadFam {
  T m[10];  // entries (0,0) (0,1) (0,2) (0,3) (1,1) (1,2) (1,3) (2,2) (2,3) (3,3)
};

__device__ __forceinline__ int qmad(int a, int b, int c) { return a * b + c; }
__device__ __forceinline__ float qmad(float a, float b, float c) { return __fmaf_rn(a, b, c); }

// Products inside grid row rr (a, b: that row's difference values, index c-1).  The row's "same position" sum feeds the
// diagonal entries (columns 1..11 for k = 0, 2; columns 2..12 for k = 1, 3; rows 1..11 for k = 0, 1; rows 2..12 for
// k = 2, 3), the "right neighbour" sum feeds (0,1) (rows 1..11) and (2,3) (rows 2..12).
template <bool SYM, typename T>
__device__ __forceinline__ void quad_same_row(QuadFam<T>& f, const T (&a)[12], const T (&b)[12], bool first, bool last) {
  const T p1 = a[0] * b[0], p12 = a[11] * b[11];
  T mid = a[1] * b[1];
#pragma unroll
  for (int c = 2; c < 11; c++) mid = qmad(a[c], b[c], mid);
  const T left = mid + p1, right = mid + p12;  // columns 1..11 / 2..12
  T rs01 = a[0] * b[1];
  if (!SYM) rs01 = qmad(b[0], a[1], rs01);
#pragma unroll
  for (int c = 1; c < 11; c++) {
    rs01 = qmad(a[c], b[c + 1], rs01);
    if (!SYM) rs01 = qmad(b[c], a[c + 1], rs01);
  }
  const T zero = (T)0;
  f.m[0] += last ? zero : left;
  f.m[4] += last ? zero : right;
  f.m[1] += last ? zero : rs01;
  f.m[7] += first ? zero : left;
  f.m[9] += first ? zero : right;
  f.m[8] += first ? zero : rs01;
}

// products between grid rows rr-1 (ap, bp) and rr (ac, bc): entries (0,2) (columns 1..11), (1,3) (columns 2..12), (0,3), (1,2)
template <bool SYM, typename T>
__device__ __forceinline__ void quad_cross_row(QuadFam<T>& f, const T (&ap)[12], const T (&bp)[12], const T (&ac)[12],
                                               const T (&bc)[12]) {
  T q1 = ap[0] * bc[0], q12 = ap[11] * bc[11], mid = ap[1] * bc[1];
  if (!SYM) {
    q1 = qmad(bp[0], ac[0], q1);
    q12 = qmad(bp[11], ac[11], q12);
    mid = qmad(bp[1], ac[1], mid);
  }
#pragma unroll
  for (int c = 2; c < 11; c++) {
    mid = qmad(ap[c], bc[c], mid);
    if (!SYM) mid = qmad(bp[c], ac[c], mid);
  }
  f.m[2] += mid + q1;
  f.m[6] += mid + q12;
  T m03 = f.m[3], m12 = f.m[5];
#pragma unroll
  for (int c = 0; c < 11; c++) {
    m03 = qmad(ap[c], bc[c + 1], m03);
    m12 = qmad(ap[c + 1], bc[c], m12);
    if (!SYM) {
      m03 = qmad(bp[c], ac[c + 1], m03);
      m12 = qmad(bp[c + 1], ac[c], m12);
    }
  }
  f.m[3] = m03;
  f.m[5] = m12;
}

// off-diagonal entries of a symmetric family count twice in the quadratic form
template <bool SYM, typename T>
__device__ __forceinline__ void quad_store(const QuadFam<T>& f, double* m) {
#pragma unroll
  for (int e = 0; e < 10; e++) {
    const bool diag = e == 0 || e == 4 || e == 7 || e == 9;
    const double v = (double)f.m[e];
    m[e] = (SYM && !diag) ? v + v : v;
  }
}

__device__ __forceinline__ void row_vals(const uint4 q, int (&v)[LN]) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < LN; i++) v[i] = (int)__byte_perm(w[i >> 2], 0, 0x4440 | (i & 3));
}
// floats 2^23 + byte (one PRMT each); the offset cancels in every difference
__device__ __forceinline__ void row_vals(const uint4 q, float (&v)[LN]) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < LN; i++) v[i] = __uint_as_float(__byte_perm(w[i >> 2], 0x4B000000u, 0x7650 | (i & 3)));
}

// One sweep over the 12 grid rows for a subset of the families (PASS 0: xx, yy, xy; 1: xe; 2: ye), taps re-read from the
// lane's tile every row: three short sweeps keep ~100 registers live instead of ~200 for a single one, which is what lets
// twice as many warps share an SM (the kernel is latency-bound: 2 warps per scheduler issue half of the time).
template <typename T, int PASS>
__device__ __forceinline__ void quad_sweep(const unsigned char* tile, QuadFam<T>& f0, QuadFam<T>& f1, QuadFam<T>& f2) {
  constexpr bool NX = PASS != 2, NY = PASS != 1, NE = PASS != 0;  // which difference images the pass needs
  T dxp[12], dyp[12], dep[12];
#pragma unroll
  for (int c = 0; c < 12; c++) dxp[c] = dyp[c] = dep[c] = (T)0;
#pragma unroll 1
  for (int rr = 1; rr <= 12; rr++) {
    T dxc[12], dyc[12], dec[12];
    {
      T t1c[LN];
      if (NX || NE) row_vals(*reinterpret_cast<const uint4*>(tile + rr * 16), t1c);
      if (NX) {
#pragma unroll
        for (int c = 1; c <= 12; c++) dxc[c - 1] = t1c[c + 1] - t1c[c - 1];
      }
      if (NE) {
        T t0[LN];
        row_vals(*reinterpret_cast<const uint4*>(tile + LIMG + rr * 16), t0);
#pragma unroll
        for (int c = 1; c <= 12; c++) dec[c - 1] = t0[c] - t1c[c];
      }
    }
    if (NY) {
      T t1m[LN], t1p[LN];
      row_vals(*reinterpret_cast<const uint4*>(tile + (rr - 1) * 16), t1m);
      row_vals(*reinterpret_cast<const uint4*>(tile + (rr + 1) * 16), t1p);
#pragma unroll
      for (int c = 1; c <= 12; c++) dyc[c - 1] = t1p[c] - t1m[c];
    }
    const bool first = rr == 1, last = rr == 12;
    if (PASS == 0) {
      quad_same_row<true>(f0, dxc, dxc, first, last);
      quad_same_row<true>(f1, dyc, dyc, first, last);
      quad_same_row<false>(f2, dxc, dyc, first, last);
      if (rr >= 2) {
        quad_cross_row<true>(f0, dxp, dxp, dxc, dxc);
        quad_cross_row<true>(f1, dyp, dyp, dyc, dyc);
        quad_cross_row<false>(f2, dxp, dyp, dxc, dyc);
      }
    } else if (PASS == 1) {
      quad_same_row<false>(f0, dxc, dec, first, last);
      if (rr >= 2) quad_cross_row<false>(f0, dxp, dep, dxc, dec);
    } else {
      quad_same_row<false>(f0, dyc, dec, first, last);
      if (rr >= 2) quad_cross_row<false>(f0, dyp, dep, dyc, dec);
    }
#pragma unroll
    for (int c = 0; c < 12; c++) {
      if (NX) dxp[c] = dxc[c];
      if (NY) dyp[c] = dyc[c];
      if (NE) dep[c] = dec[c];
    }
  }
}

// tile: this lane's staged taps (I1 rows, then I0 rows); m: where the lane's 50 doubles go.  m may alias the tile: the
// results are held in registers (as doubles) until the last sweep has read its taps.
template <typename T>
__device__ __forceinline__ void quad_build(const unsigned char* tile, double* m) {
  QuadFam<T> a, b, c, dummy;
#pragma unroll
  for (int e = 0; e < 10; e++) a.m[e] = b.m[e] = c.m[e] = (T)0;
  quad_sweep<T, 0>(tile, a, b, c);
  double r[30];
  quad_store<true>(a, r);
  quad_store<true>(b, r + 10);
  quad_store<false>(c, r + 20);
#pragma unroll
  for (int e = 0; e < 10; e++) a.m[e] = b.m[e] = (T)0;
  quad_sweep<T, 1>(tile, a, dummy, dummy);
  quad_sweep<T, 2>(tile, b, dummy, dummy);
#pragma unroll
  for (int e = 0; e < 30; e++) m[e] = r[e];
  quad_store<false>(a, m + 30);
  quad_store<false>(b, m + 40);
}

// ---- Gram build (the default) -------------------------------------------------------------------------------------------
// Every difference is a +-1 combination of raw taps, so every matrix entry is an integer combination of the entries of ONE
// 16 x 16 Gram matrix G = sum over the window of t(p) t(p)^T, where t(p) holds the 16 u8 taps that any component at window
// pixel p = (r, c) touches (tile coordinates; (dr, dc) = offset from p):
//   taps 0..7    I1, rows r, r+1 (dr = j >> 2), columns c-1 .. c+2 (dc = (j & 3) - 1)
//   taps 8..11   I1, rows r-1 (8, 9) and r+2 (10, 11), columns c, c+1
//   taps 12..15  I0, rows r, r+1, columns c, c+1
// A diagonal entry of a family is a_k' G b_k, an off-diagonal one a_k' G b_l + a_l' G b_k (a_k, b_l: the +-1 tap vectors of the
// two differences; for XX and YY that is 2 a_k' G a_l, the doubling of quad_store).  G <= 121 * 255^2 and an entry sums at most
// 8 of them, so s32 is exact: the entries are the integers the FFMA build computes, and the same doubles.
//
// G = R'R, R = one row per window pixel (K), one column per tap, is one warp-wide integer MMA per k-step and n8 half
// (mma.sync m16n8k32 u8 x u8 -> s32, IMMA.16832): 5 k-steps, 10 IMMA per feature.  K order: groups of 4 consecutive pixels of
// one window row, columns 1-4, 5-8, 9-12 (classes 0, 1, 2); column 12 is outside the window and its byte comes from the zeroed
// byte 15 of the tile row.  A 32-bit fragment word is one group of one tap: one PRMT of two words of one tile row, since the
// tap offset only shifts the bytes.  Slot u = 2 * kstep + half (16 K) holds class u / 3 (u < 9) and window row
// 1 + t + 4 (u % 3) for lane t of a quad; row 12 and slot 9 are zero (33 groups + 7 zero groups = 5 x 32 K).  The A words of
// taps g and g + 8 of lane (g, t) are also the B fragments of the two n8 halves.
// Cost: the FFMA build costs the same per round whatever the number of lanes that build; this one costs per building lane.
// In a fully packed round (32 lanes) it is 1.19x the FFMA build (scripts/klt_build_bench.py, DESIGN.md §9-1): its shared
// memory traffic (fragment loads of every lane from the same tile, G lookups with bank conflicts) and the per-feature chain
// bound it, not instruction issue.  It wins on the partly packed rounds: KLT stage 114.1 -> 107.4 ms on C3.
struct GramBuild {};                    // build tag of klt_quad_kernel
constexpr int GRAM_SCRATCH = 3 * 256;   // G as three 8 x 8 s32 blocks: G[0..7][0..7], G[0..7][8..15], G[8..15][8..15]
constexpr int ZROW = 2 * LIMG;          // the 16 bytes after a lane's tiles: zeroed once, never written

__device__ __forceinline__ void gram_tap(int j, int& dr, int& dc, int& img) {
  if (j < 8) { dr = j >> 2; dc = (j & 3) - 1; img = 0; }
  else if (j < 12) { dr = j < 10 ? -1 : 2; dc = j & 1; img = 0; }
  else { dr = (j - 12) >> 1; dc = j & 1; img = 1; }
}

// tap of the + / - term of difference component k (at offset (k >> 1, k & 1) from the pixel); side 0 = DX, 1 = DY, 2 = DE
__device__ __forceinline__ int gram_diff_tap(int side, int k, bool plus) {
  const int a = k >> 1, b = k & 1;
  if (side == 0) return a * 4 + b + (plus ? 2 : 0);
  if (side == 1) return plus ? (a ? 10 + b : 5 + b) : (a ? 1 + b : 8 + b);
  return plus ? 12 + 2 * a + b : a * 4 + b + 1;
}

// byte offset of G[i][j] in the scratch
__device__ __forceinline__ int gram_at(int i, int j) {
  if (i >= 8 && j < 8) { const int s = i; i = j; j = s; }
  return i < 8 ? (j < 8 ? (i * 8 + j) * 4 : 256 + (i * 8 + j - 8) * 4) : 512 + ((i - 8) * 8 + j - 8) * 4;
}

struct GramLane {
  int rb[2], r2[2];          // tile byte offsets of taps g, g + 8 at window row 1 + t (u % 3 == 0); row 9 + t or ZROW (u % 3 == 2)
  uint32_t sel[2], selm[2];  // PRMT selectors of the two taps; selm: class 2, the column-12 byte taken from byte 15
  int ga[2][8];              // scratch byte offsets of the G entries of matrix entries lane, lane + 32 (+ + - - pattern below)
};

// zero_off: scratch-relative offset of a zero word (the second half of a diagonal entry and lanes without a second entry)
__device__ __forceinline__ void gram_lane_init(GramLane& L, int lane, int zero_off) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int x = 0; x < 2; x++) {
    int dr, dc, img;
    gram_tap(g + 8 * x, dr, dc, img);
    L.rb[x] = img * LIMG + (dr + t + 1) * 16;
    L.r2[x] = t == 3 ? ZROW : L.rb[x] + 128;
    L.sel[x] = 0x3210u + 0x1111u * (uint32_t)(dc + 1);
    L.selm[x] = (L.sel[x] & 0x0FFFu) | 0x7000u;
  }
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int e = lane + 32 * h, f = e / 10, q = e % 10;
    const int k = q < 4 ? 0 : q < 7 ? 1 : q < 9 ? 2 : 3;
    const int l = k + q - (q < 4 ? 0 : q < 7 ? 4 : q < 9 ? 7 : 9);
    const int sa = (f == 1 || f == 4) ? 1 : 0, sb = f == 0 ? 0 : f <= 2 ? 1 : 2;  // XX, YY, XY, XE, YE
#pragma unroll
    for (int d = 0; d < 2; d++) {  // a_k' G b_l, then a_l' G b_k
      const int ka = d ? l : k, kb = d ? k : l;
      const int ap = gram_diff_tap(sa, ka, true), am = gram_diff_tap(sa, ka, false);
      const int bp = gram_diff_tap(sb, kb, true), bm = gram_diff_tap(sb, kb, false);
      const bool z = e >= QM || (d == 1 && k == l);
      L.ga[h][4 * d + 0] = z ? zero_off : gram_at(ap, bp);
      L.ga[h][4 * d + 1] = z ? zero_off : gram_at(ap, bm);
      L.ga[h][4 * d + 2] = z ? zero_off : gram_at(am, bp);
      L.ga[h][4 * d + 3] = z ? zero_off : gram_at(am, bm);
    }
  }
}

// fragment word of slot U for tap g + 8x of this lane
template <int U>
__device__ __forceinline__ uint32_t gram_word(const unsigned char* ftile, const GramLane& L, int x) {
  constexpr int CLS = U / 3, J = U % 3;
  if (U >= 9) return 0u;
  const unsigned char* rowp = ftile + (J == 2 ? L.r2[x] : L.rb[x] + 64 * J);
  const uint32_t sel = CLS == 2 ? L.selm[x] : L.sel[x];
  if (CLS == 1) {
    const uint4 q = *reinterpret_cast<const uint4*>(rowp);
    return __byte_perm(q.y, q.z, sel);
  }
  const uint2 q = *reinterpret_cast<const uint2*>(rowp + 4 * CLS);
  return __byte_perm(q.x, q.y, sel);
}

__device__ __forceinline__ void imma_16832(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Warp-cooperative: the 50 doubles of the feature whose staged tile is ftile, written over that tile.  Every lane calls it.
__device__ __forceinline__ void gram_build(unsigned char* ftile, unsigned char* scratch, const GramLane& L, int lane) {
  uint32_t w[2][10];
#pragma unroll
  for (int x = 0; x < 2; x++) {
    w[x][0] = gram_word<0>(ftile, L, x);
    w[x][1] = gram_word<1>(ftile, L, x);
    w[x][2] = gram_word<2>(ftile, L, x);
    w[x][3] = gram_word<3>(ftile, L, x);
    w[x][4] = gram_word<4>(ftile, L, x);
    w[x][5] = gram_word<5>(ftile, L, x);
    w[x][6] = gram_word<6>(ftile, L, x);
    w[x][7] = gram_word<7>(ftile, L, x);
    w[x][8] = gram_word<8>(ftile, L, x);
    w[x][9] = gram_word<9>(ftile, L, x);
  }
  int d0[4] = {0, 0, 0, 0}, d1[4] = {0, 0, 0, 0};  // n8 halves: taps 0..7, 8..15
#pragma unroll
  for (int s = 0; s < 5; s++) {
    const uint32_t a0 = w[0][2 * s], a1 = w[1][2 * s], a2 = w[0][2 * s + 1], a3 = w[1][2 * s + 1];
    imma_16832(d0, a0, a1, a2, a3, a0, a2);
    imma_16832(d1, a0, a1, a2, a3, a1, a3);
  }
  // accumulator (g, 2t..2t+1) of half 0 is G[g][2t..], of half 1 G[g][8+2t..]; rows g + 8 of half 1 are G[8+g][8+2t..]
  const int o = (lane >> 2) * 8 + 2 * (lane & 3);
  int* G = reinterpret_cast<int*>(scratch);
  *reinterpret_cast<int2*>(G + o) = make_int2(d0[0], d0[1]);
  *reinterpret_cast<int2*>(G + 64 + o) = make_int2(d1[0], d1[1]);
  *reinterpret_cast<int2*>(G + 128 + o) = make_int2(d1[2], d1[3]);
  __syncwarp();
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int e = lane + 32 * h;
    if (e < QM) {
      const int* a = L.ga[h];
#define GR(i) (*reinterpret_cast<const int*>(scratch + a[i]))
      const int v = (GR(0) - GR(1) - GR(2) + GR(3)) + (GR(4) - GR(5) - GR(6) + GR(7));
#undef GR
      reinterpret_cast<double*>(ftile)[e] = (double)v;
    }
  }
  __syncwarp();  // the scratch is rewritten by the next feature
}

// the five sums from the matrices: 4*Sxx, 4*Sxy, 4*Syy, 2*bx, 2*by in the conventions of window_sums
__device__ __forceinline__ void quad_eval(const double* m, double fx, double fy, double& a00, double& a01, double& a11, double& b0,
                                          double& b1) {
  const double gx = 1.0 - fx, gy = 1.0 - fy;
  const double w0 = gx * gy, w1 = fx * gy, w2 = gx * fy, w3 = fx * fy;
  const double ww[10] = {w0 * w0, w0 * w1, w0 * w2, w0 * w3, w1 * w1, w1 * w2, w1 * w3, w2 * w2, w2 * w3, w3 * w3};
  double s[5];
#pragma unroll
  for (int f = 0; f < 5; f++) {
    double mm[10];
#pragma unroll
    for (int q = 0; q < 5; q++) {
      const double2 t = *reinterpret_cast<const double2*>(m + f * 10 + 2 * q);
      mm[2 * q] = t.x;
      mm[2 * q + 1] = t.y;
    }
    double acc = mm[0] * ww[0];
#pragma unroll
    for (int q = 1; q < 10; q++) acc = __fma_rn(mm[q], ww[q], acc);
    s[f] = acc;
  }
  a00 = s[0];
  a11 = s[1];
  a01 = s[2];
  b0 = s[3];
  b1 = s[4];
}

#ifdef KLT_ROUND_STATS
__device__ unsigned long long klt_round_hist[2][33];  // [0]: build rounds by lanes building, [1]: iteration rounds by lanes iterating
#endif

template <int MINB, int LSTAGE, typename T>
__global__ void __launch_bounds__(32, MINB) klt_quad_kernel(KltLaunch k, int* __restrict__ defer_count, int* __restrict__ defer_list) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  unsigned char* wtile = smem_raw;
  unsigned char* tile = wtile + lane * LSTRIDE;
  double* mq = reinterpret_cast<double*>(tile);  // the matrices replace the taps they were built from (400 B <= 448 B)
  const long long total = (long long)k.npairs * k.cap;
  const int ndir = k.pb ? 2 : 1;
  constexpr bool GRAM = std::is_same<T, GramBuild>::value;
  unsigned char* scratch = smem_raw + 32 * LSTRIDE;
  GramLane gl;
  if (GRAM) {
    gram_lane_init(gl, lane, ZROW - 32 * LSTRIDE);  // lane 0's zero row
    *reinterpret_cast<uint4*>(tile + ZROW) = make_uint4(0u, 0u, 0u, 0u);
  }
  for (long long wbase = (long long)blockIdx.x * 32; wbase < total; wbase += (long long)gridDim.x * 32) {
    const long long g = wbase + lane;
    const int pair = g < total ? (int)(g / k.cap) : 0;
    const int slot = (int)(g - (long long)pair * k.cap);
    const bool valid = g < total && (!k.counts || slot < k.counts[pair]);
    double2 p0 = make_double2(0.0, 0.0);
    if (valid) p0 = k.p0[g];
    double px = p0.x, py = p0.y, x1 = 0.0, y1 = 0.0;
    int n_it = 0;
    bool alive = valid, finished = !valid;
    // per-lane progress
    int dir = 0, l = k.pv.levels - 1, it = 0;
    bool leveldone = false;
    double plx = px * (1.0 / (double)(1 << l)), ply = py * (1.0 / (double)(1 << l)), dlx = 0.0, dly = 0.0;
    int tFX = INT_MIN, tFY = INT_MIN, tkey = -1;  // position / (dir, level) the lane's matrices belong to

    while (true) {
      // a finished level hands its result to the next one (:404-420)
      if (!finished && (leveldone || it >= k.iters)) {
        const double up = (double)(1 << l);
        px = (plx + dlx) * up;
        py = (ply + dly) * up;
        if (l > 0) {
          l--;
        } else {
          if (dir == 0) {
            x1 = px;
            y1 = py;
          }
          dir++;
          l = k.pv.levels - 1;
          if (dir >= ndir) finished = true;
        }
        const double scale = 1.0 / (double)(1 << l);
        plx = px * scale;
        ply = py * scale;
        dlx = dly = 0.0;
        it = 0;
        leveldone = false;
      }
      if (!__any_sync(FULL, !finished)) break;
      const bool canwork = !finished && it < k.iters && !leveldone;
      const double x = plx + dlx, y = ply + dly;
      const double fxx = floor(x), fyy = floor(y);
      int FX = 0, FY = 0;
      bool act = canwork;
      if (act) {
        const int w = k.pv.w[l], h = k.pv.h[l];
        const bool finite_ok = (fabs(fxx) < 1.0e9) && (fabs(fyy) < 1.0e9);
        FX = finite_ok ? (int)fxx : 0;
        FY = finite_ok ? (int)fyy : 0;
        const bool ok = finite_ok && FX - LR - 1 >= 0 && FX + LR + 3 <= w - 1 && FY - LR - 1 >= 0 && FY + LR + 3 <= h - 1;
        if (!ok) {  // the next kernel in the chain redoes this feature from scratch
          alive = false;
          finished = true;
          act = false;
        }
      }
      const int key = dir * SFM_MAXL + l;
      const bool hit = act && FX == tFX && FY == tFY && key == tkey;
#ifdef KLT_ROUND_STATS
      {
        const unsigned hm = __ballot_sync(FULL, hit);
        if (hm && lane == 0) atomicAdd(&klt_round_hist[1][__popc(hm)], 1ull);
      }
#endif
      if (__any_sync(FULL, hit)) {
        if (hit) {
          double a00, a01, a11, b0, b1;
          quad_eval(mq, x - fxx, y - fyy, a00, a01, a11, b0, b1);
          double sx = 0.0, sy = 0.0;
          const double det = a00 * a11 - a01 * a01;
          if (!(fabs(det) < 16.0 * 1e-9)) {  // |det| < 1e-9 of :452 on the 16x scaled determinant
            const double rd = 2.0 / det;
            sx = (a11 * b0 - a01 * b1) * rd;
            sy = (a00 * b1 - a01 * b0) * rd;
          }
          n_it++;
          it++;
          dlx += sx;
          dly += sy;
          if (sfm_lk_step_small(sx, sy)) leveldone = true;  // hypot(step) < 1e-3 (:416), tested on the step just added
        }
        continue;
      }
      // nobody can iterate: every lane that still has work needs matrices for its position
      unsigned need = __ballot_sync(FULL, act);
      if (!need) continue;  // only level hand-overs are pending
#ifdef KLT_ROUND_STATS
      if (lane == 0) atomicAdd(&klt_round_hist[0][__popc(need)], 1ull);
#endif
      const unsigned build = need;
      __syncwarp();
      while (need) {
        int ss[LSTAGE], sx0[LSTAGE];
        StageRegs sr[LSTAGE];
#pragma unroll
        for (int j = 0; j < LSTAGE; j++) {
          ss[j] = need ? __ffs(need) - 1 : -1;
          need &= need - 1;
          const int src = ss[j] < 0 ? 0 : ss[j];
          const int sFX = __shfl_sync(FULL, FX, src), sFY = __shfl_sync(FULL, FY, src), spair = __shfl_sync(FULL, pair, src);
          const int sl = __shfl_sync(FULL, l, src), sdir = __shfl_sync(FULL, dir, src);
          const int sA = k.fa0 + spair * k.fa_step, sB = k.fb0 + spair * k.fb_step;
          const uint8_t* lbase = k.pv.base[sl];
          const size_t fstride = k.pv.fstride[sl];
          sx0[j] = sFX - LR - 1;
          if (ss[j] >= 0 && lane < 2 * LN)
            stage_load<false>(sr[j], lbase + (size_t)(sdir ? sB : sA) * fstride, lbase + (size_t)(sdir ? sA : sB) * fstride,
                              k.pv.pitch[sl], k.pv.h[sl], sx0[j], sFY - LR - 1, lane);
        }
#pragma unroll
        for (int j = 0; j < LSTAGE; j++)
          if (ss[j] >= 0 && lane < 2 * LN) stage_store(sr[j], wtile + ss[j] * LSTRIDE, sx0[j], lane);
      }
      __syncwarp();
      if constexpr (GRAM) {
        for (unsigned todo = build; todo; todo &= todo - 1) gram_build(wtile + (__ffs(todo) - 1) * LSTRIDE, scratch, gl, lane);
      } else if (act) {
        quad_build<T>(tile, mq);
      }
      if (act) {
        tFX = FX;
        tFY = FY;
        tkey = key;
      }
      __syncwarp();
    }
    if (alive) {
      k.p1[g] = make_double2(x1, y1);
      if (k.pb) k.pb[g] = make_double2(px, py);
      if (k.nit) k.nit[g] = n_it;
      if (k.keep) {
        const double fbd = hypot(px - p0.x, py - p0.y);
        k.keep[g] = (fbd >= k.fb_thresh) ? 0 : 1;  // NaN is kept (:362)
      }
    }
    const unsigned dm = __ballot_sync(FULL, valid && !alive);
    if (dm) {
      int base = 0;
      if (lane == 0) base = atomicAdd(defer_count, __popc(dm));
      base = __shfl_sync(FULL, base, 0);
      if (valid && !alive) defer_list[base + __popc(dm & ((1u << lane) - 1u))] = (int)g;
    }
    __syncwarp();
  }
}

}  // namespace

template <int ACC, int MINB, int LSTAGE, bool MASKED>
static int lane_launch(sfmgpu_ctx* ctx, const KltLaunch& k, const int* in_list, const int* in_count, int* defer_count, int* defer_list) {
  const size_t smem = (size_t)LWARPS * 32 * LSTRIDE;
  static const int cfg_id = sfm_next_cfg_id();  // one per template instantiation
  SFM_SMEM_OPTIN(ctx, cfg_id, (klt_lane_kernel<ACC, MINB, LSTAGE, MASKED>), smem);
  const long long total = (long long)k.npairs * k.cap;
  if (total == 0) return 0;
  unsigned grid = sfm_cdiv(total, 32 * LWARPS);
  if (MASKED) {  // a few % of the batch: a resident grid walks the list
    const unsigned cap = (unsigned)ctx->n_sm * 8;
    grid = grid < cap ? grid : cap;
  }
  SFM_LAUNCH(ctx, (klt_lane_kernel<ACC, MINB, LSTAGE, MASKED>), grid, 32 * LWARPS, smem, k, in_list, in_count, defer_count, defer_list);
  return 0;
}

// Interior windows of every slot; features it cannot handle are appended to defer_list (device), count in
// *defer_count (device, zeroed by the caller on the same stream).  variant: tuning builds (A/B runs).
template <int MINB, int LSTAGE, typename T>
static int quad_launch(sfmgpu_ctx* ctx, const KltLaunch& k, int* defer_count, int* defer_list) {
  const size_t smem = (size_t)32 * LSTRIDE + (std::is_same<T, GramBuild>::value ? GRAM_SCRATCH : 0);
  static const int cfg_id = sfm_next_cfg_id();  // one per template instantiation
  SFM_SMEM_OPTIN(ctx, cfg_id, (klt_quad_kernel<MINB, LSTAGE, T>), smem);
  const long long total = (long long)k.npairs * k.cap;
  if (total == 0) return 0;
  SFM_LAUNCH(ctx, (klt_quad_kernel<MINB, LSTAGE, T>), sfm_cdiv(total, 32), 32, smem, k, defer_count, defer_list);
  return 0;
}

int sfm_klt_lane_launch(sfmgpu_ctx* ctx, const KltLaunch& k, int* defer_count, int* defer_list, int variant) {
  // Measured on B200, C2 shape (scripts/klt_ab.py, KLT stage incl. the deferred pass, 238k tracks): <1,12,4> 4.43 ms
  // (168 registers, spills), <1,8,4> 3.57 ms, <2,8,4> 3.66 ms, <2,8,8> 3.97 ms: the schedule wants registers, not warps.
  switch (variant) {
    case 1: return lane_launch<1, 12, 4, false>(ctx, k, nullptr, nullptr, defer_count, defer_list);
    case 2: return lane_launch<2, 8, 4, false>(ctx, k, nullptr, nullptr, defer_count, defer_list);
    case 3: return lane_launch<1, 8, 4, false>(ctx, k, nullptr, nullptr, defer_count, defer_list);  // the FP64 window walk
    case 4: return quad_launch<8, 4, int>(ctx, k, defer_count, defer_list);
    case 5: return quad_launch<8, 4, float>(ctx, k, defer_count, defer_list);
    case 6: return quad_launch<12, 4, float>(ctx, k, defer_count, defer_list);
    // Measured on B200 (C2, KLT stage incl. the border pass): <8,4,int> 16.8 ms, <8,4,float> 16.6, <10,4,float> 15.6,
    // <12,4,float> 15.0, <12,2,float> 14.8 (no spills), <16,4,float> 24.2 (spills), staging rounds of 8: 20.2 (spills); a
    // single-sweep build (255 registers, 8 warps) 15.2 ms.
    // Gram build, measured on B200 (1000 W, C3 KLT stage incl. the border pass, 3 alternated runs): <14,2,Gram> 107.4 ms
    // (128 registers, 16 B spilled outside the build loop, 14 warps/SM), <12,2,Gram> 107.1 (156 registers, no spills),
    // the FFMA build <12,2,float> 114.1.
    case 7: return quad_launch<12, 2, float>(ctx, k, defer_count, defer_list);  // the FFMA build
    case 8: return quad_launch<12, 2, GramBuild>(ctx, k, defer_count, defer_list);
    default: return quad_launch<14, 2, GramBuild>(ctx, k, defer_count, defer_list);  // quadratic forms over integer matrices
  }
}

// Border windows: the features of in_list with the out-of-bounds rule as masks; the rest goes to defer_list.
int sfm_klt_lane_masked_launch(sfmgpu_ctx* ctx, const KltLaunch& k, const int* in_list, const int* in_count, int* defer_count,
                               int* defer_list) {
  return lane_launch<1, 8, 4, true>(ctx, k, in_list, in_count, defer_count, defer_list);
}

#ifdef KLT_ROUND_STATS
extern "C" int sfmgpu_debug_klt_round_hist(unsigned long long* out66) {
  return (int)cudaMemcpyFromSymbol(out66, klt_round_hist, sizeof(unsigned long long) * 66);
}
#endif
