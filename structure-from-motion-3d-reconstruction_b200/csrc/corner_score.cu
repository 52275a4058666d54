// corner_score.cu — Shi-Tomasi min-eigenvalue score, global maximum, and the raster-ordered candidate list.
//
// Replaces (reference cpp/src/templering_sfm.cpp) shi_tomasi :237-285: clamped central-difference gradients
// (:242-249), 5x5 structure tensor (:252-264), lmin = 0.5*(tr - sqrt(max(0, tr^2 - 4 det))) (:266-270), zero
// 2-px border (:253-254), thr = max*quality (:274-275), candidates s >= thr in raster order (:280-285).
//
// Exactness.  With Gx = I[x+1]-I[x-1], Gy likewise (integers in [-255,255]; the reference uses gx = Gx/2), let
// a = sum Gx^2, b = sum Gy^2, c = sum GxGy over the window (int32 <= 1.63e6).  Every intermediate of the
// reference up to disc is a dyadic rational below 2^53, hence exact in double, and
//        lmin = 0.125 * fl( (a+b) - fl(sqrt( (a-b)^2 + 4c^2 )) )
// bit for bit (scaling by powers of two commutes with rounding).  The kernels therefore keep integer sums and
// evaluate that single expression in FP64 (IEEE sqrt) — only for pixels that pass an exact INTEGER screen
// D <= (T - theta)^2 against the running threshold, so the FP64 pipe sees a few percent of the pixels.
//
// FP32 is exact here: Gx, Gy are integers of magnitude <= 255, every product is <= 65025 and every window sum is
// <= 25 * 65025 = 1,625,625 < 2^24, so the gradient products and both sliding 5-sums run as FFMA/FADD on
// integer-valued floats without a single rounding.  Bytes become floats with one PRMT (0x4B000000 | b = 2^23 + b);
// the offset cancels in the gradient differences.
//
// Which pixels see the FP64 expression: every pixel gets the FP32 ESTIMATE u~ = T - sqrt.approx(D) (error < 0.72: root <=
// T <= 3.25e6, D carries two roundings, sqrt.approx 2^-23 relative; tests/test_score_estimate_cpu.py).  A pixel can only matter if
// u~ >= bound - 2 (bound = the tile's / frame's running maximum in the max pass, 8*thr in the candidate pass); those
// few are queued and evaluated DENSELY with the exact FP64 expression afterwards, which alone decides.
//
// (Tried and dropped: persistent blocks with cp.async double-buffered taps: 5.13 ms vs 4.46 ms per 299 frames; 64 x 48
// tiles at 4 blocks per SM and 63 registers: 8.06 vs 8.11 ms per 998 frames - occupancy is not what limits it.)
// Kernels (tile = 64 x 60 output pixels, 256 threads, taps staged once in shared memory with clamping):
//   score_tile_kernel<0>  per-frame maximum of u = 8*lmin  (atomicMax on the double's bit pattern)
//   score_tile_kernel<1>  candidate bitmap (one word per 32 pixels) + unordered (pixel, score) list
//   bitmap_scan_kernel    exclusive prefix of the bitmap popcounts -> raster rank of every candidate
//   order_kernel          scatter the unordered list to raster order (the order std::sort starts from)
// Roofline: ~45 instructions per pixel and pass against 1 B/pixel of traffic: bound by instruction issue, not HBM
// (DESIGN.md §corner-score).
#include <type_traits>

#include "common.cuh"
#include "corner_work.cuh"

namespace {

constexpr int TW = 64, TH = 60;
constexpr int TAP_H = TH + 6, TAP_S = 76;   // tap rows; 19-word row stride: conflict-free when lanes walk rows
constexpr int HS_ROWS = TH + 4, HS_S = 65;  // horizontal sums: 64 rows, padded
constexpr int RUN = 16;                     // phase 1: outputs per thread (64 rows x 4 runs)
constexpr int VRUN = 15;                    // phase 2: outputs per thread (64 columns x 4 row groups)
constexpr float EST_MARGIN = 2.0f;          // > 2.7x the error bound of the FP32 estimate (0.72; observed worst case 0.58)

struct ScoreSmem {
  float hxx[HS_ROWS * HS_S], hxy[HS_ROWS * HS_S], hyy[HS_ROWS * HS_S];
  uint8_t taps[TAP_H * TAP_S];
  unsigned short queue[TW * TH];
  unsigned tile_bm[TH * 2];
  float wmaxf[8];
  int wcnt[8];
  double wmax[8];
  int qn;
};

__device__ __forceinline__ double i2d(int v) {
  // exact int32 -> double without the slow conversion pipe: (2^52 + 2^31 + v) - (2^52 + 2^31)
  return __hiloint2double(0x43300000, v ^ 0x80000000) - 4503601774854144.0;
}

// u = 8*lmin, bit-exact with the reference's lmin/0.125 (see header).
__device__ __forceinline__ double exact_u(int a, int b, int c) {
  const double dd = i2d(a - b), c2 = i2d(2 * c);
  const double D = dd * dd + c2 * c2;
  return i2d(a + b) - sqrt(D);
}

// byte k of w as the float 2^23 + byte (exact)
__device__ __forceinline__ float bytef(uint32_t w, int k) { return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7650 | k)); }

__device__ __forceinline__ float est_u(float a, float b, float c) {
  const float d = a - b, c2 = c + c;
  const float D = fmaf(c2, c2, d * d);
  float s;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(D));
  return (a + b) - s;
}

// One tile of one frame.  MODE 0: frame maximum only.  MODE 1: candidates against the FINAL threshold (maximum known).
template <int MODE>
__device__ __forceinline__ void score_tile(ScoreSmem& sm, const uint8_t* __restrict__ im, int w, int h, int pitch, int X0, int Y0,
                                           int fr, const CornerWorkView& wv, double quality) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < TH * 2) sm.tile_bm[tid] = 0;
  if (tid == 0) sm.qn = 0;

  // phase 0: taps of image(X0-3 .., Y0-3 ..) with clamped coordinates (= the reference's clamped gradient taps).
  // Shared rows start at image column X0-4 (4-aligned), so image column X0+c lives at byte c+4.  Tiles whose halo
  // lies inside the image are staged with aligned 32-bit loads (all loads issued before the stores); border tiles
  // take the byte path, which implements the clamp.
  if (X0 >= 4 && X0 + 68 <= w) {
    // columns inside the image: aligned 32-bit loads, rows clamped (top / bottom tiles)
    constexpr int WPT = (TAP_H * 18 + 255) / 256;
    uint32_t v[WPT];
    const uint8_t* src = im + (X0 - 4);
#pragma unroll
    for (int k = 0; k < WPT; k++) {
      const int idx = tid + 256 * k, r = idx / 18, c = idx - r * 18;
      int gy = Y0 - 3 + r;
      gy = gy < 0 ? 0 : (gy > h - 1 ? h - 1 : gy);
      if (idx < TAP_H * 18) v[k] = __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)gy * pitch) + c);
    }
#pragma unroll
    for (int k = 0; k < WPT; k++) {
      const int idx = tid + 256 * k, r = idx / 18, c = idx - r * 18;
      if (idx < TAP_H * 18) reinterpret_cast<uint32_t*>(sm.taps)[r * (TAP_S / 4) + c] = v[k];
    }
  } else {
    for (int idx = tid; idx < TAP_H * 72; idx += 256) {
      const int ty = idx / 72, tb = idx - ty * 72;
      int gx = X0 - 4 + tb, gy = Y0 - 3 + ty;
      gx = gx < 0 ? 0 : (gx > w - 1 ? w - 1 : gx);
      gy = gy < 0 ? 0 : (gy > h - 1 ? h - 1 : gy);
      sm.taps[ty * TAP_S + tb] = __ldg(im + (size_t)gy * pitch + gx);
    }
  }
  __syncthreads();

  // phase 1: horizontal 5-sums of the gradient products.  lane = row (two row groups), warp pair = run of 16 columns.
  // Output column c needs products of columns c-2..c+2; column cc's gradients are C[cc+5] - C[cc+3] (centre row) and
  // P[cc+4] - M[cc+4] (rows below / above), byte offsets within the shared row.
  {
    const int r = (warp & 1) * 32 + lane, k0 = (warp >> 1) * RUN;  // h row r <-> image row Y0-2+r; tap rows r, r+1, r+2
    const uint32_t* wm = reinterpret_cast<const uint32_t*>(sm.taps + r * TAP_S + k0);
    const uint32_t* wc = reinterpret_cast<const uint32_t*>(sm.taps + (r + 1) * TAP_S + k0);
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(sm.taps + (r + 2) * TAP_S + k0);
    uint32_t cw[6], pw[6], mw[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
      cw[i] = wc[i];
      pw[i] = wp[i];
      mw[i] = wm[i];
    }
    float gx[RUN + 4], gy[RUN + 4];
#pragma unroll
    for (int j = 0; j < RUN + 4; j++) {  // column cc = k0 - 2 + j: bytes (relative to k0) j+3, j+1 / j+2
      gx[j] = bytef(cw[(j + 3) >> 2], (j + 3) & 3) - bytef(cw[(j + 1) >> 2], (j + 1) & 3);
      gy[j] = bytef(pw[(j + 2) >> 2], (j + 2) & 3) - bytef(mw[(j + 2) >> 2], (j + 2) & 3);
    }
    float sxx = 0.f, sxy = 0.f, syy = 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      sxx = fmaf(gx[j], gx[j], sxx);
      sxy = fmaf(gx[j], gy[j], sxy);
      syy = fmaf(gy[j], gy[j], syy);
    }
    float* oxx = sm.hxx + r * HS_S + k0;
    float* oxy = sm.hxy + r * HS_S + k0;
    float* oyy = sm.hyy + r * HS_S + k0;
#pragma unroll
    for (int t = 0; t < RUN; t++) {
      sxx = fmaf(gx[t + 4], gx[t + 4], sxx);
      sxy = fmaf(gx[t + 4], gy[t + 4], sxy);
      syy = fmaf(gy[t + 4], gy[t + 4], syy);
      oxx[t] = sxx;
      oxy[t] = sxy;
      oyy[t] = syy;
      sxx = fmaf(-gx[t], gx[t], sxx);
      sxy = fmaf(-gx[t], gy[t], sxy);
      syy = fmaf(-gy[t], gy[t], syy);
    }
  }
  __syncthreads();

  // phase 2: vertical 5-sums and the FP32 estimate.  thread = column, VRUN consecutive rows.
  const int oc = tid & 63, q = tid >> 6;
  const int x = X0 + oc;
  const float* cxx = sm.hxx + (q * VRUN) * HS_S + oc;
  const float* cxy = sm.hxy + (q * VRUN) * HS_S + oc;
  const float* cyy = sm.hyy + (q * VRUN) * HS_S + oc;
  unsigned long long* maxbits = wv.maxbits + fr;
  double thr8 = 0.0;
  float bound;
  if (MODE == 0) {
    bound = __double2float_rd(__longlong_as_double(*(volatile unsigned long long*)maxbits));  // what earlier blocks found
  } else {
    const double maxv = 0.125 * __longlong_as_double(*maxbits);
    const double thr = maxv * quality;  // (:275)
    thr8 = 8.0 * thr;                   // s >= thr  <=>  u >= 8*thr
    bound = __double2float_rd(thr8);
  }
  const bool col_in = x < w, col_interior = x >= 2 && x < w - 2;
  const bool tile_inner = X0 >= 2 && X0 + TW <= w - 2 && Y0 >= 2 && Y0 + TH <= h - 2;  // no border pixel in this tile
  float ra[4], rb[4], rc[4];  // ring of the last four row sums; the fifth enters in the loop
#pragma unroll
  for (int i = 0; i < 4; i++) {
    ra[i] = cxx[i * HS_S];
    rc[i] = cxy[i * HS_S];
    rb[i] = cyy[i * HS_S];
  }
  float a = (ra[0] + ra[1]) + (ra[2] + ra[3]), c = (rc[0] + rc[1]) + (rc[2] + rc[3]), b = (rb[0] + rb[1]) + (rb[2] + rb[3]);
  float uf[VRUN];
  float tmax = 0.f;
  unsigned pmask = 0;  // MODE 1: rows of this thread that go to the queue (bit 15: as border pixels)
  // the walk exists twice: tiles without border pixels (the vast majority) skip every per-pixel position test
  auto walk = [&](auto inner_tag) {
    constexpr bool INNER = decltype(inner_tag)::value;
#pragma unroll
    for (int j = 0; j < VRUN; j++) {
      const float na = cxx[(j + 4) * HS_S], nc = cxy[(j + 4) * HS_S], nb = cyy[(j + 4) * HS_S];
      a += na;
      c += nc;
      b += nb;
      const int y = Y0 + q * VRUN + j;
      const bool interior = INNER || (col_interior && y >= 2 && y < h - 2);
      const float u = est_u(a, b, c);
      if (MODE == 0) {
        uf[j] = interior ? u : -1.0e30f;
        tmax = fmaxf(tmax, uf[j]);
      } else {
        if (INNER || (col_in && y < h)) {
          if (interior) {
            if (u >= bound - EST_MARGIN) pmask |= 1u << j;
          } else if (0.0 >= thr8) {
            pmask |= (1u << j) | (1u << (16 + j));  // border score is exactly 0 (:240, :253-254)
          }
        }
      }
      a -= ra[j & 3];
      c -= rc[j & 3];
      b -= rb[j & 3];
      ra[j & 3] = na;
      rc[j & 3] = nc;
      rb[j & 3] = nb;
    }
  };
  if (tile_inner)
    walk(std::true_type{});
  else
    walk(std::false_type{});

  if (MODE == 0) {
    // tile maximum of the estimates
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    if (lane == 0) sm.wmaxf[warp] = tmax;
    __syncthreads();
    float bm = sm.wmaxf[0];
#pragma unroll
    for (int k = 1; k < 8; k++) bm = fmaxf(bm, sm.wmaxf[k]);
    bound = fmaxf(bound, bm) - EST_MARGIN;  // a pixel below this cannot be the frame maximum
    // queue every pixel that can still be the frame maximum
#pragma unroll
    for (int j = 0; j < VRUN; j++)
      if (uf[j] >= bound) sm.queue[atomicAdd(&sm.qn, 1)] = (unsigned short)((q * VRUN + j) * TW + oc);
  } else {
    // ordered block compaction of the per-thread row masks (no atomics: ~5 % of the pixels get here)
    const int cnt = __popc(pmask & 0x7fffu);
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) sm.wcnt[warp] = inc;
    __syncthreads();
    int base = inc - cnt;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int wc = sm.wcnt[k];
      if (k < warp) base += wc;
    }
    if (tid == 255) sm.qn = base + cnt;
    unsigned m = pmask & 0x7fffu;
    while (m) {
      const int j = __ffs(m) - 1;
      m &= m - 1;
      sm.queue[base++] = (unsigned short)(((q * VRUN + j) * TW + oc) | (((pmask >> (16 + j)) & 1u) << 15));
    }
  }
  __syncthreads();

  // dense exact evaluation of the queued pixels
  const int nq = sm.qn;
  double best = 0.0;
  for (int e0 = 0; e0 < nq; e0 += 256) {  // uniform trip count: the ballots below are warp-complete
    const int e = e0 + tid;
    bool cand = false;
    double u = 0.0;
    int row = 0, col = 0;
    if (e < nq) {
      const int id = sm.queue[e], loc = id & 0x7fff;
      row = loc / TW;
      col = loc - row * TW;
      cand = true;
      if (!(id & 0x8000)) {
        const float* pxx = sm.hxx + row * HS_S + col;
        const float* pxy = sm.hxy + row * HS_S + col;
        const float* pyy = sm.hyy + row * HS_S + col;
        const int ia = __float2int_rn((pxx[0] + pxx[HS_S]) + (pxx[2 * HS_S] + pxx[3 * HS_S]) + pxx[4 * HS_S]);
        const int ic = __float2int_rn((pxy[0] + pxy[HS_S]) + (pxy[2 * HS_S] + pxy[3 * HS_S]) + pxy[4 * HS_S]);
        const int ib = __float2int_rn((pyy[0] + pyy[HS_S]) + (pyy[2 * HS_S] + pyy[3 * HS_S]) + pyy[4 * HS_S]);
        u = exact_u(ia, ib, ic);
        cand = u >= thr8;
      }
    }
    if (MODE == 0) best = fmax(best, u);
    if (MODE == 1) {
      const unsigned m = __ballot_sync(0xffffffffu, cand);
      if (m) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(wv.nfinal + fr, (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (cand) {
          atomicOr(&sm.tile_bm[row * 2 + (col >> 5)], 1u << (col & 31));
          const unsigned slot = base + __popc(m & ((1u << lane) - 1u));
          if (slot < (unsigned)wv.cand_cap) {
            wv.tmp_idx[(size_t)fr * wv.cand_cap + slot] = ((unsigned)(Y0 + row) << 16) | (unsigned)(X0 + col);
            wv.tmp_key[(size_t)fr * wv.cand_cap + slot] = (unsigned long long)__double_as_longlong(0.125 * u);
          }
        }
      }
    }
  }
  if (MODE == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (lane == 0) sm.wmax[warp] = best;
    __syncthreads();
    if (tid == 0) {
      double m = sm.wmax[0];
      for (int k = 1; k < 8; k++) m = fmax(m, sm.wmax[k]);
      const unsigned long long mb = (unsigned long long)__double_as_longlong(m);
      if (mb > *(volatile unsigned long long*)maxbits) atomicMax(maxbits, mb);  // u >= 0: bit order == value order
    }
  }
  if (MODE == 1) {
    __syncthreads();
    if (tid < TH * 2) {
      const int y = Y0 + (tid >> 1), xw = X0 + 32 * (tid & 1);
      if (y < h && xw < w) wv.bitmap[(size_t)fr * wv.words_per_frame + (size_t)y * wv.wpr + (xw >> 5)] = sm.tile_bm[tid];
    }
  }
}

// Full grid: tile (blockIdx.x, blockIdx.y) of frame blockIdx.z.  Probe (tmul > 1): every tmul-th tile in x and y only, to
// seed the running maximum before the fused pass.
template <int MODE>
__global__ void __launch_bounds__(256, 3) score_tile_kernel(const uint8_t* __restrict__ img, int w, int h, int pitch, size_t fstride,
                                                           int frame0, CornerWorkView wv, double quality, int tmul) {
  extern __shared__ __align__(16) unsigned char score_raw[];
  ScoreSmem& sm = *reinterpret_cast<ScoreSmem*>(score_raw);
  const int fr = blockIdx.z;
  int tx = blockIdx.x, ty = blockIdx.y;
  if (tmul > 1) {
    const int ntx = (w + TW - 1) / TW, nty = (h + TH - 1) / TH;
    tx = min(tx * tmul + tmul / 2, ntx - 1);
    ty = min(ty * tmul + tmul / 2, nty - 1);
  }
  score_tile<MODE>(sm, img + (size_t)(frame0 + fr) * fstride, w, h, pitch, tx * TW, ty * TH, fr, wv, quality);
}

// ---- fused pass, walk-down form ---------------------------------------------------------------------------------------------
// One WARP owns a strip of 256 columns (8 per lane) and walks down a segment of rows; a block is 4 horizontally adjacent
// strips of the same segment.  Per tap row a lane reads its 8 bytes with ONE 64-bit load (a warp reads 256 contiguous
// bytes, a block 2 KB; two rows are in flight ahead of the arithmetic), takes the 3 + 3 halo bytes from its neighbours'
// words by shuffle, and keeps the last three rows as integer-valued floats in registers: the gradients of the middle
// row, their products and the horizontal 5-sums (sliding FFMA in / out, all exact) never leave the register file.  The
// vertical 5-sum is a running sum per column: add the new row of horizontal sums, subtract the one five rows back,
// which comes from a per-warp ring in shared memory (lane-contiguous float4: conflict-free, no block barrier anywhere
// in the kernel).  ~31 instructions per pixel against ~82 of the tile kernel (3 rows converted per thread and row
// there, two shared-memory round trips, three block barriers per tile).
// Candidates: FP32 estimate for every pixel, the exact FP64 score for pixels within the estimate's error of the
// provisional threshold quality * L, L = max(frame maximum so far, this warp's own exact maximum) <= final maximum:
// multiplication by quality > 0 is monotone, so the provisional threshold never exceeds the final one and the list is a
// superset of the candidates (the selection drops the surplus once the maximum is final).  The screened pixels are
// queued per warp and evaluated densely (see drain below).
constexpr int WK_COLS = 8, WK_WARPS = 4, WK_MINB = 3, WK_STRIP = 32 * WK_COLS;  // 12 warps per SM: 222 KB of rings + queues, <= 170 registers
constexpr int WK_RING = 5 * 6 * 32;  // float4 per warp: 5 rows x (24 sums = 6 float4) x 32 lanes
constexpr int WK_QUEUE = 224;        // screened pixels queued per warp before they are evaluated densely
constexpr size_t WK_SMEM_WARP = WK_RING * sizeof(float4) + WK_QUEUE * sizeof(uint4);

__device__ __forceinline__ uint2 ldg_pinned(const uint8_t* p) {
  uint2 v;
  asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}

// Dense evaluation of a warp's queue of screened pixels (called every ~15 rows: kept out of line, the row loop should stay small).
__device__ __noinline__ void walk_drain(uint4* queue, int& qn, double& wmax, double thr8, int fr, const CornerWorkView& wv, int lane) {
  const size_t lb_off = (size_t)fr * wv.cand_cap;
  __syncwarp();
  // pass 1: exact scores (kept in registers: WK_QUEUE / 32 entries per lane), candidate count
  constexpr int PER = WK_QUEUE / 32;
  double u[PER];
  unsigned pos[PER], cm[PER];
  int ncand = 0;
#pragma unroll
  for (int k = 0; k < PER; k++) {
    const int e = k * 32 + lane;
    bool c = false;
    u[k] = 0.0;
    pos[k] = 0;
    if (e < qn) {
      const uint4 q = queue[e];
      pos[k] = q.x & 0x7FFFFFFFu;
      if (!(q.x >> 31)) {
        u[k] = exact_u(__float2int_rn(__uint_as_float(q.y)), __float2int_rn(__uint_as_float(q.z)), __float2int_rn(__uint_as_float(q.w)));
        wmax = fmax(wmax, u[k]);
        c = u[k] >= thr8;
      } else {
        c = true;  // border pixel: queued only while 0 >= thr8
      }
    }
    cm[k] = __ballot_sync(0xffffffffu, c);
    ncand += __popc(cm[k]);
  }
  if (ncand > 0) {
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(wv.ncand + fr, (unsigned)ncand);
    base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
    for (int k = 0; k < PER; k++) {
      if (cm[k] & (1u << lane)) {
        const unsigned slot = base + __popc(cm[k] & ((1u << lane) - 1u));
        if (slot < (unsigned)wv.cand_cap) {
          wv.tmp_idx[lb_off + slot] = pos[k];
          wv.tmp_key[lb_off + slot] = (unsigned long long)__double_as_longlong(0.125 * u[k]);
        }
      }
      base += __popc(cm[k]);
    }
  }
  qn = 0;
  __syncwarp();
}

__global__ void __launch_bounds__(WK_WARPS * 32, WK_MINB) score_walk_kernel(const uint8_t* __restrict__ img, int w, int h, int pitch,
                                                                      size_t fstride, int frame0, CornerWorkView wv, double quality,
                                                                      int seg_rows) {
  extern __shared__ __align__(16) unsigned char score_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int strip = blockIdx.x * WK_WARPS + warp;
  const int xs = strip * WK_STRIP;  // first column of the strip
  if (xs >= w) return;               // no block barrier below: a warp may leave
  const int x0 = xs + lane * WK_COLS;
  const int fr = blockIdx.z;
  const int y_begin = blockIdx.y * seg_rows, y_end = min(h, y_begin + seg_rows);
  const uint8_t* im = img + (size_t)(frame0 + fr) * fstride;
  unsigned char* wbase = score_raw + (size_t)warp * WK_SMEM_WARP;
  float4* ring = reinterpret_cast<float4*>(wbase) + lane;  // [row % 5][k] at ring[(row5 * 6 + k) * 32]
  // Screened pixels (FP32 estimate within its error of the provisional threshold: a few percent) are not evaluated where
  // they are found - one lane with a hit would drag the whole warp through the FP64 expression - but queued with their
  // exact (integer-valued) sums and evaluated DENSELY, 32 at a time; survivors get their list slots with one global atomic
  // per drain.  (The candidate bitmap is not written here: only the raster-order paths need it and build it from the list.)
  uint4* queue = reinterpret_cast<uint4*>(wbase + WK_RING * sizeof(float4));  // (y << 16 | x | border << 31, a, b, c as float bits)
  int qn = 0;
  double wmax = 0.0;      // this warp's exact maximum so far (lane-local until published)
  double lb = 0.0;        // lower bound of the frame maximum the threshold was derived from
  double thr8 = 0.0;      // provisional 8 * thr
  float boundf = -EST_MARGIN;
  bool border_on = true;  // 0 >= thr8: border pixels (score exactly 0, :240, :253-254) are candidates
  auto drain = [&]() { walk_drain(queue, qn, wmax, thr8, fr, wv, lane); };
  unsigned long long* maxbits = wv.maxbits + fr;
  const int wm1 = w - 1;
  // Warp-uniform: does any of the strip's tap columns xs-3 .. xs+258 fall outside the image?  Only such strips run the
  // per-byte clamp (the reference clamps its gradient taps into the image, :242-249).
  const bool edge_strip = xs == 0 || xs + WK_STRIP + 2 > wm1;
  // per-lane column masks (bit t = column x0 + t)
  unsigned in_img = 0, interior_cols = 0;
#pragma unroll
  for (int t = 0; t < 8; t++) {
    if (x0 + t < w) in_img |= 1u << t;
    if (x0 + t >= 2 && x0 + t < w - 2) interior_cols |= 1u << t;
  }

  // Raw taps of one row: the 8 bytes before the lane's columns, its own 8, the 8 after (three 64-bit loads; the
  // neighbours' lines are in L1 already).  Addresses stay inside the frame batch: a row's over-read ends in the next row.
  struct Raw {
    uint2 l, m, r;
  };
  const int xl = (x0 >= 8) ? x0 - 8 : x0, xr = (x0 + 16 <= pitch) ? x0 + 8 : x0;  // rows are pitch bytes: stay inside them
  auto load_row = [&](int t) {
    Raw q;
    t = t < 0 ? 0 : (t > h - 1 ? h - 1 : t);  // clamped tap rows
    const uint8_t* row = im + (size_t)t * pitch;
    // volatile asm: the loads are issued HERE, three rows before their conversion (the compiler would sink them to their use)
    q.m = ldg_pinned(row + (x0 + 8 <= pitch ? x0 : 0));
    q.l = ldg_pinned(row + (x0 + 8 <= pitch ? xl : 0));
    q.r = ldg_pinned(row + (x0 + 8 <= pitch ? xr : 0));
    return q;
  };
  // 14 integer-valued floats (2^23 + byte) of tap columns x0-3 .. x0+10
  auto convert = [&](const Raw& q, float* F) {
    uint32_t left = q.l.y, lo = q.m.x, hi = q.m.y, right = q.r.x;
    if (edge_strip) {  // clamp every tap column into [0, w-1]: replicate the border byte
      if (x0 < 3) left = 0x01010101u * (lo & 0xffu);  // x0 == 0: columns < 0 take column 0
      if (x0 + 10 > wm1) {                             // columns > w-1 take column w-1
        const int last = wm1 - x0;                     // position of the last valid byte (own bytes 0..7, right 8..11)
        uint32_t b;
        if (last < 0) b = 0;  // whole lane beyond the image: its values are never used
        else if (last < 4) b = (lo >> (8 * last)) & 0xffu;
        else if (last < 8) b = (hi >> (8 * (last - 4))) & 0xffu;
        else b = (right >> (8 * (last - 8))) & 0xffu;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (k > last) lo = (lo & ~(0xffu << (8 * k))) | (b << (8 * k));
          if (4 + k > last) hi = (hi & ~(0xffu << (8 * k))) | (b << (8 * k));
          if (8 + k > last) right = (right & ~(0xffu << (8 * k))) | (b << (8 * k));
        }
      }
    }
    F[0] = bytef(left, 1);
    F[1] = bytef(left, 2);
    F[2] = bytef(left, 3);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      F[3 + k] = bytef(lo, k);
      F[7 + k] = bytef(hi, k);
    }
    F[11] = bytef(right, 0);
    F[12] = bytef(right, 1);
    F[13] = bytef(right, 2);
  };

  float V[24];  // vertical running sums: xx[0..7], xy[0..7], yy[0..7]
#pragma unroll
  for (int k = 0; k < 24; k++) V[k] = 0.f;
  {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 30; k++) ring[k * 32] = z;
  }
  __syncwarp();
  unsigned long long gmax_bits = *(volatile unsigned long long*)maxbits;
  const int T0 = y_begin - 3;  // first tap row
  const int n_iter = (y_end - y_begin) + 4;

  // One row: tap rows G-1 (Fm), G (Fc), G+1 (Fp) are in registers; i counts rows from the segment's first gradient row
  // G = y_begin - 2; once five rows of horizontal sums are in (i >= 4) the output row y = G - 2 is complete.
  auto row_step = [&](const float* Fm, const float* Fc, const float* Fp, int i) {
    const int y = y_begin + i - 4;
    // running lower bound of the frame maximum -> provisional threshold (re-read every 8 rows; the load is issued four
    // rows before its value is used)
    if ((i & 7) == 4) gmax_bits = *(volatile unsigned long long*)maxbits;
    if ((i & 7) == 0) {
      const double g = __longlong_as_double(gmax_bits);
      const double nl = fmax(g, wmax);
      if (nl > lb || i == 0) {
        lb = nl;
        thr8 = 8.0 * ((0.125 * lb) * quality);
        boundf = __double2float_rd(thr8) - EST_MARGIN;
        border_on = 0.0 >= thr8;
      }
    }
    // gradients of row G at columns x0-2 .. x0+9, horizontal 5-sums of their products at x0 .. x0+7
    float gx[12], gy[12];
#pragma unroll
    for (int c = 0; c < 12; c++) {
      gx[c] = Fc[c + 2] - Fc[c];
      gy[c] = Fp[c + 1] - Fm[c + 1];
    }
    float hx[8], hxy[8], hy[8];
    {
      float sxx = 0.f, sxy = 0.f, syy = 0.f;
#pragma unroll
      for (int c = 0; c < 4; c++) {
        sxx = fmaf(gx[c], gx[c], sxx);
        sxy = fmaf(gx[c], gy[c], sxy);
        syy = fmaf(gy[c], gy[c], syy);
      }
#pragma unroll
      for (int t = 0; t < 8; t++) {
        sxx = fmaf(gx[t + 4], gx[t + 4], sxx);
        sxy = fmaf(gx[t + 4], gy[t + 4], sxy);
        syy = fmaf(gy[t + 4], gy[t + 4], syy);
        hx[t] = sxx;
        hxy[t] = sxy;
        hy[t] = syy;
        sxx = fmaf(-gx[t], gx[t], sxx);
        sxy = fmaf(-gx[t], gy[t], sxy);
        syy = fmaf(-gy[t], gy[t], syy);
      }
    }
    // vertical: V += h[G] - h[G-5]; the ring slot of row G-5 is the one row G takes
    {
      const int slot = (i % 5) * 6 * 32;
      float4 o[6];
#pragma unroll
      for (int k = 0; k < 6; k++) o[k] = ring[slot + k * 32];
      ring[slot + 0 * 32] = make_float4(hx[0], hx[1], hx[2], hx[3]);
      ring[slot + 1 * 32] = make_float4(hx[4], hx[5], hx[6], hx[7]);
      ring[slot + 2 * 32] = make_float4(hxy[0], hxy[1], hxy[2], hxy[3]);
      ring[slot + 3 * 32] = make_float4(hxy[4], hxy[5], hxy[6], hxy[7]);
      ring[slot + 4 * 32] = make_float4(hy[0], hy[1], hy[2], hy[3]);
      ring[slot + 5 * 32] = make_float4(hy[4], hy[5], hy[6], hy[7]);
      const float* of = reinterpret_cast<const float*>(o);
#pragma unroll
      for (int t = 0; t < 8; t++) {
        V[t] += hx[t] - of[t];
        V[8 + t] += hxy[t] - of[8 + t];
        V[16 + t] += hy[t] - of[16 + t];
      }
    }
    if (i < 4) return;  // warm-up rows (warp-uniform)
    // FP32 estimates against the screen
    unsigned pass = 0;
#pragma unroll
    for (int t = 0; t < 8; t++) {
      const float u = est_u(V[t], V[16 + t], V[8 + t]);
      if (u >= boundf) pass |= 1u << t;
    }
    const bool row_interior = y >= 2 && y < h - 2;
    const unsigned flags = row_interior ? (pass & interior_cols) : 0u;
    const unsigned border = border_on ? (in_img & ~(row_interior ? interior_cols : 0u)) : 0u;
    const unsigned want = flags | border;
    if (__any_sync(0xffffffffu, want != 0)) {
      auto push = [&](unsigned m) {
        const int cnt = __popc(m);
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += v;
        }
        const int total = __shfl_sync(0xffffffffu, inc, 31);
        if (qn + total > WK_QUEUE) drain();
        int e = qn + inc - cnt;
#pragma unroll
        for (int t = 0; t < 8; t++)
          if (m & (1u << t)) {
            const unsigned bd = (border >> t) & 1u;
            queue[e] = make_uint4(((unsigned)y << 16) | (unsigned)(x0 + t) | (bd << 31), __float_as_uint(V[t]), __float_as_uint(V[16 + t]),
                                  __float_as_uint(V[8 + t]));
            e++;
          }
        qn += total;
      };
      // more screened pixels in one row than the queue holds (flat / weak frames): two halves
      const int parts = __reduce_add_sync(0xffffffffu, __popc(want)) <= WK_QUEUE ? 1 : 2;
#pragma unroll 1
      for (int part = 0; part < parts; part++) push(parts == 1 ? want : (part == 0 ? want & 0x0Fu : want & 0xF0u));
    }
    // publish a new maximum as soon as it is known (other warps' thresholds follow it)
    if ((i & 7) == 7) {
      double m = wmax;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
      wmax = m;
      if (lane == 0) {
        const unsigned long long mb = (unsigned long long)__double_as_longlong(m);
        if (mb > *(volatile unsigned long long*)maxbits) atomicMax(maxbits, mb);  // u >= 0: bit order == value order
      }
    }
  };

  // two raw rows are in flight ahead of the row being converted; the three float rows shift by register moves (an
  // unrolled-by-three rotation tripled the code and cost more in instruction fetch than the 28 moves)
  float Fm[14], Fc[14], Fp[14];
  Raw r0 = load_row(T0), r1 = load_row(T0 + 1), r2 = load_row(T0 + 2);
  convert(r0, Fm);
  convert(r1, Fc);
  r0 = load_row(T0 + 3);
  r1 = load_row(T0 + 4);
#pragma unroll 1
  for (int i = 0; i < n_iter; i++) {
    convert(r2, Fp);
    r2 = r0;
    r0 = r1;
    r1 = load_row(T0 + 5 + i);
    row_step(Fm, Fc, Fp, i);
#pragma unroll
    for (int c = 0; c < 14; c++) {
      Fm[c] = Fc[c];
      Fc[c] = Fp[c];
    }
  }
  drain();
  // the maximum of the last rows and the last drain
  {
    double m = wmax;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) {
      const unsigned long long mb = (unsigned long long)__double_as_longlong(m);
      if (mb > *(volatile unsigned long long*)maxbits) atomicMax(maxbits, mb);
    }
  }
}

// Frames whose PROVISIONAL list overflowed the capacity are redone against the final threshold (their exact list may
// still fit): a small persistent grid walks the rescue list.
__global__ void __launch_bounds__(256, 3) score_rescue_kernel(const uint8_t* __restrict__ img, int w, int h, int pitch, size_t fstride,
                                                             int frame0, CornerWorkView wv, double quality) {
  extern __shared__ __align__(16) unsigned char score_raw[];
  ScoreSmem& sm = *reinterpret_cast<ScoreSmem*>(score_raw);
  const int nres = *wv.rescue_count;
  for (int k = blockIdx.z; k < nres; k += gridDim.z) {
    const int fr = wv.rescue_list[k];
    score_tile<1>(sm, img + (size_t)(frame0 + fr) * fstride, w, h, pitch, blockIdx.x * TW, blockIdx.y * TH, fr, wv, quality);
    __syncthreads();
  }
}

// After the fused pass: frames whose provisional list overflowed go on the rescue list (one thread per frame).
__global__ void rescue_mark_kernel(CornerWorkView wv, int count) {
  const int fr = blockIdx.x * blockDim.x + threadIdx.x;
  if (fr >= count || wv.ncand[fr] <= (unsigned)wv.cand_cap) return;
  wv.nfinal[fr] = 0;
  wv.exact_list[fr] = 1;
  wv.rescue_list[atomicAdd(wv.rescue_count, 1)] = fr;
}

// The raster-order paths (exact emulation of a flagged frame, candidate-list API, select mode 1) need the candidate bitmap.
// Frames with an exact list got it from the tile kernel; for a provisional list (walk-down pass, which writes no bitmap) it
// is built here from the list entries that reach the FINAL threshold: cleared by bitmap_clear_kernel, set below.
// flagged_only: only frames the selection flagged (status 3).
__global__ void __launch_bounds__(256) bitmap_clear_kernel(CornerWorkView wv, int flagged_only) {
  const int fr = blockIdx.y;
  if (wv.exact_list[fr]) return;
  if (flagged_only && wv.status[fr] != 3) return;
  unsigned* bm = wv.bitmap + (size_t)fr * wv.words_per_frame;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < wv.words_per_frame; i += (size_t)gridDim.x * blockDim.x) bm[i] = 0u;
}

// Provisional list -> candidate bitmap: sets the bit of every entry that reaches the final threshold.
__global__ void __launch_bounds__(256) candidate_finalize_kernel(CornerWorkView wv, double quality, int flagged_only) {
  const int fr = blockIdx.y;
  if (wv.exact_list[fr]) return;
  if (flagged_only && wv.status[fr] != 3) return;
  const unsigned nprov = wv.ncand[fr];
  const size_t cb = (size_t)fr * wv.cand_cap, wb = (size_t)fr * wv.words_per_frame;
  const double thr = (0.125 * __longlong_as_double(wv.maxbits[fr])) * quality;
  for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < nprov; e += gridDim.x * blockDim.x) {
    if (!(__longlong_as_double((long long)wv.tmp_key[cb + e]) >= thr)) continue;  // s >= thr (:282)
    const unsigned yx = wv.tmp_idx[cb + e], x = yx & 0xFFFFu, y = yx >> 16;
    atomicOr(wv.bitmap + wb + (size_t)y * wv.wpr + (x >> 5), 1u << (x & 31));
  }
}

// Exclusive prefix sum of popc(bitmap word) over one frame (one block per frame).
__global__ void __launch_bounds__(1024) bitmap_scan_kernel(CornerWorkView wv, int only_flagged) {
  __shared__ unsigned wsum[32];
  const int fr = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (only_flagged && wv.status[fr] != 3) return;
  const size_t nwords = wv.words_per_frame;
  const unsigned* bm = wv.bitmap + (size_t)fr * nwords;
  unsigned* off = wv.wordoff + (size_t)fr * nwords;
  const size_t chunk = (nwords + 1023) / 1024;
  const size_t beg = (size_t)tid * chunk, end = beg + chunk < nwords ? beg + chunk : nwords;
  unsigned s = 0;
  for (size_t i = beg; i < end; i++) s += __popc(bm[i]);
  // block exclusive scan of s
  unsigned v = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) wsum[warp] = v;
  __syncthreads();
  if (warp == 0) {
    unsigned t = wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned u = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += u;
    }
    wsum[lane] = t;
  }
  __syncthreads();
  unsigned run = v - s + (warp ? wsum[warp - 1] : 0u);
  for (size_t i = beg; i < end; i++) {
    off[i] = run;
    run += __popc(bm[i]);
  }
  if (tid == 1023) wv.ntotal[fr] = run;  // chunk boundaries are monotone: the last thread ends at the total
}

// Scatter the candidate list into raster order (the order std::sort starts from).  A provisional list (fused pass) still
// holds the entries below the final threshold: they are skipped, their bitmap bits are already cleared.
__global__ void __launch_bounds__(256) order_kernel(CornerWorkView wv, double quality, int only_flagged) {
  const int fr = blockIdx.y;
  if (only_flagged && wv.status[fr] != 3) return;
  const bool exact = wv.exact_list[fr] != 0;
  const unsigned n = min(exact ? wv.nfinal[fr] : wv.ncand[fr], (unsigned)wv.cand_cap);
  const double thr = (0.125 * __longlong_as_double(wv.maxbits[fr])) * quality;
  const size_t cb = (size_t)fr * wv.cand_cap, wb = (size_t)fr * wv.words_per_frame;
  for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const unsigned long long k = wv.tmp_key[cb + e];
    if (!exact && !(__longlong_as_double((long long)k) >= thr)) continue;
    const unsigned yx = wv.tmp_idx[cb + e];
    const unsigned y = yx >> 16, x = yx & 0xFFFFu;
    const size_t word = wb + (size_t)y * wv.wpr + (x >> 5);
    const unsigned rank = wv.wordoff[word] + __popc(wv.bitmap[word] & ((1u << (x & 31)) - 1u));
    if (rank < (unsigned)wv.cand_cap) {
      wv.key[cb + rank] = k;
      wv.idx[cb + rank] = yx;
    }
  }
}

}  // namespace

// Raster order for the frames of the batch (all of them, or only those the selection flagged with status 3): ntotal,
// key[], idx[].  Needed by the introsort emulation and the candidate-list API; bucket_select_kernel works on the
// unordered list.
int sfm_corner_raster_order(sfmgpu_ctx* ctx, int count, const CornerWorkView& wv, double quality, int only_flagged) {
  // provisional lists (walk-down score pass): build the candidate bitmap from the entries that reach the final threshold
  SFM_LAUNCH(ctx, bitmap_clear_kernel, dim3(32, count), 256, 0, wv, only_flagged);
  SFM_LAUNCH(ctx, candidate_finalize_kernel, dim3(32, count), 256, 0, wv, quality, only_flagged);
  SFM_LAUNCH(ctx, bitmap_scan_kernel, count, 1024, 0, wv, only_flagged);
  SFM_LAUNCH(ctx, order_kernel, dim3(16, count), 256, 0, wv, quality, only_flagged);
  return 0;
}

// Maximum and candidates for frames [first, first+count); leaves the unordered (pixel, score) list in the work area.
// quality in (0, 1]: sparse probe pass + ONE walk-down pass against a provisional threshold (a superset of the candidates,
// ncand entries, no candidate bitmap) + the rescue of frames whose list overflowed; otherwise (the provisional-threshold
// argument needs quality > 0) the two full tile passes, which leave the exact list (nfinal entries) and its bitmap.
int sfm_corner_candidates_batch(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, double quality,
                                const CornerWorkView& wv) {
  SFM_CUDA(ctx, cudaMemsetAsync(wv.maxbits, 0, sizeof(unsigned long long) * count, ctx->stream));
  SFM_CUDA(ctx, cudaMemsetAsync(wv.ncand, 0, sizeof(unsigned) * count, ctx->stream));
  SFM_CUDA(ctx, cudaMemsetAsync(wv.nfinal, 0, sizeof(unsigned) * count, ctx->stream));
  SFM_CUDA(ctx, cudaMemsetAsync(wv.rescue_count, 0, sizeof(int), ctx->stream));
  const int ntx = sfm_cdiv(f->w, TW), nty = sfm_cdiv(f->h, TH);
  dim3 grid(ntx, nty, count);
  static const int cfg_id[3] = {sfm_next_cfg_id(), sfm_next_cfg_id(), sfm_next_cfg_id()};
  SFM_SMEM_OPTIN(ctx, cfg_id[0], score_tile_kernel<0>, sizeof(ScoreSmem));
  SFM_SMEM_OPTIN(ctx, cfg_id[1], score_tile_kernel<1>, sizeof(ScoreSmem));
  SFM_SMEM_OPTIN(ctx, cfg_id[2], score_rescue_kernel, sizeof(ScoreSmem));
  if (quality > 0.0 && quality <= 1.0) {  // (quality > 1: a pixel between the maximum and the threshold would be skipped)
    // every 6th tile in x and y seeds the running maximum (1/36 of a pass; measured per 999 1080p frames: every 4th tile 6.78 ms
    // for the stage, every 6th or 8th 6.45 ms)
    constexpr int PROBE = 6;
    SFM_CUDA(ctx, cudaMemsetAsync(wv.exact_list, 0, sizeof(int) * count, ctx->stream));
    SFM_LAUNCH(ctx, score_tile_kernel<0>, dim3(sfm_cdiv(ntx, PROBE), sfm_cdiv(nty, PROBE), count), 256, sizeof(ScoreSmem), f->lvl[0], f->w,
               f->h, f->pitch[0], f->fstride[0], first, wv, quality, PROBE);
    // segments of ~270 rows (6 warm-up rows each: 2 %), 4 strips of 256 columns per block
    const int nseg = f->h > 400 ? (f->h + 269) / 270 : 1, seg_rows = (f->h + nseg - 1) / nseg;
    static const int walk_id = sfm_next_cfg_id();
    const size_t wsm = (size_t)WK_WARPS * WK_SMEM_WARP;
    SFM_SMEM_OPTIN(ctx, walk_id, score_walk_kernel, wsm);
    SFM_LAUNCH(ctx, score_walk_kernel, dim3(sfm_cdiv(f->w, WK_WARPS * WK_STRIP), sfm_cdiv(f->h, seg_rows), count), WK_WARPS * 32, wsm,
               f->lvl[0], f->w, f->h, f->pitch[0], f->fstride[0], first, wv, quality, seg_rows);
    SFM_LAUNCH(ctx, rescue_mark_kernel, sfm_cdiv(count, 256), 256, 0, wv, count);
    SFM_LAUNCH(ctx, score_rescue_kernel, dim3(ntx, nty, count < 2 ? count : 2), 256, sizeof(ScoreSmem), f->lvl[0], f->w, f->h,
               f->pitch[0], f->fstride[0], first, wv, quality);
    static const bool trace = getenv("SFMGPU_TRACE_RESCUE") != nullptr;  // diagnostics only (synchronises)
    if (trace) {
      int nres = 0;
      SFM_CUDA(ctx, cudaMemcpyAsync(&nres, wv.rescue_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      fprintf(stderr, "[score] %d of %d frames redone against the final threshold (provisional list overflow)\n", nres, count);
    }
  } else {
    SFM_CUDA(ctx, cudaMemsetAsync(wv.exact_list, 1, sizeof(int) * count, ctx->stream));
    SFM_LAUNCH(ctx, score_tile_kernel<0>, grid, 256, sizeof(ScoreSmem), f->lvl[0], f->w, f->h, f->pitch[0], f->fstride[0], first, wv,
               quality, 1);
    SFM_LAUNCH(ctx, score_tile_kernel<1>, grid, 256, sizeof(ScoreSmem), f->lvl[0], f->w, f->h, f->pitch[0], f->fstride[0], first, wv,
               quality, 1);
  }
  return 0;
}

int sfm_candidates_single(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int frame, double quality, int32_t* xy, double* score,
                          int cap, int* n_out, double* max_score) {
  if (f->w > 32767 || f->h > 32767) return sfm_fail(ctx, SFMGPU_E_ARG, "corner_candidates: image larger than 32767 px");
  const int cand_cap = f->w * f->h;
  const size_t bytes = sfm_corner_work_bytes_md(f->w, f->h, 1, cand_cap, 0);
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, bytes));
  CornerWorkView wv;
  corner_work_carve(wv, ctx->cs_work.p, f->w, f->h, 1, cand_cap);
  SFM_TRY(sfm_corner_candidates_batch(ctx, f, frame, 1, quality, wv));
  SFM_TRY(sfm_corner_raster_order(ctx, 1, wv, quality, 0));
  unsigned long long mb = 0;
  unsigned n = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&mb, wv.maxbits, 8, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(&n, wv.ntotal, 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (max_score) {
    double u;
    memcpy(&u, &mb, 8);
    *max_score = 0.125 * u;
  }
  if (n_out) *n_out = (int)n;
  if ((int)n > cap) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "corner_candidates: %u candidates, room for %d", n, cap);
  if (n == 0) return 0;
  std::vector<unsigned> idx(n);
  SFM_CUDA(ctx, cudaMemcpyAsync(idx.data(), wv.idx, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (score) SFM_CUDA(ctx, cudaMemcpyAsync(score, wv.key, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (xy)
    for (unsigned i = 0; i < n; i++) {
      xy[2 * i] = (int32_t)(idx[i] & 0xFFFFu);  // idx holds y << 16 | x
      xy[2 * i + 1] = (int32_t)(idx[i] >> 16);
    }
  return 0;
}

extern "C" int sfmgpu_corner_candidates(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, double quality, int32_t* xy,
                                        double* score, int cap, int* n_out, double* max_score) {
  SFM_ENTER(ctx);
  if (!ctx || !f) return SFMGPU_E_ARG;
  if (frame < 0 || frame >= f->n || cap < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "corner_candidates: bad frame/cap");
  return sfm_candidates_single(ctx, f, frame, quality, xy, score, cap, n_out, max_score);
}
