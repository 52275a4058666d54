// corner_select.cu — the order std::sort gives the candidates + greedy min-distance selection, one thread block per frame.
//
// Replaces (reference cpp/src/templering_sfm.cpp) shi_tomasi :286-301: std::sort of the candidates by score
// descending (unstable: libstdc++ introsort decides the order of ties), then the sequential greedy loop that
// accepts a candidate iff no already accepted corner lies at squared distance < min_dist^2, capped at
// max_corners (tested after the push, so at least one corner comes back whenever a candidate exists).
//
// Default: bucket_select_kernel.  The order std::sort produces is unique wherever the scores are distinct, so the
// candidates are put into order-code buckets and only the still unblocked ones of the buckets the selection reaches are
// sorted (see the kernel).  Inside a group of IDENTICAL scores introsort's order is only observable if at least two
// members are still unblocked when the selection reaches them (DESIGN.md §4); the kernel detects that conservatively and
// such a frame (status 3) is redone by the exact emulation below (select_kernel mode 3).
//
// Exact emulation (select_kernel): runs for the frames flagged with status 3, for every frame under select_set_mode(1),
// and as the sort of sfmgpu_sort_perm_desc.  The introsort segment tree is walked LEFT-FIRST and LAZILY (sort_emul.h
// facts 1-4): only as much of the array is sorted as the selection consumes.  Segments larger than SMALL are partitioned
// by the whole block (two ordered compactions of the misfits + pairwise swaps); smaller ones are handed to warps, up to
// 32 at a time, each warp finishing its segment completely (warp partitions, then one leaf per lane with the stable
// insertion sort).  Depth-limit exhaustion takes the sequential heap-sort restatement.
//
// Selection (both kernels): greedy acceptance only ever depends on higher-priority candidates, so a chunk of the sorted
// prefix is decided in parallel: (1) kill candidates within min_dist of corners accepted in earlier chunks
// (bucket_select_kernel: one bit per pixel, accepted corners mark their disc; select_kernel: a min_dist-cell grid holding
// <= 2 corners per cell), (2) resolve conflicts inside the chunk by rounds (a candidate is accepted once every closer,
// higher-priority survivor is decided), (3) append the accepted ones in priority order.  Coordinates are integers: the
// arithmetic is exact.
#include "common.cuh"
#include "corner_work.cuh"
#include "sort_emul.h"

int sfm_corner_candidates_batch(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, double quality,
                                const CornerWorkView& wv);
int sfm_corner_raster_order(sfmgpu_ctx* ctx, int count, const CornerWorkView& wv, double quality, int only_flagged);

namespace {

constexpr int SEL_THREADS = 256;          // small blocks: several frames resident per SM hide the serial latencies
constexpr int SEL_WARPS = SEL_THREADS / 32;
constexpr int EPT = 4;                    // elements per thread / lane and pass
// Measured on B200 (C2, 999 frames, select stage): SMALL/WINDOW 2048/8192 15.4 ms, 1024/8192 14.8, 512/8192 15.0,
// 4096/8192 17.8, 2048/4096 17.1, 2048/16384 15.0.  (Also tried and dropped: 128-thread blocks x 8 per SM: 14.5 ms
// resident but slower per launch; 16 candidates per thread in the selection rounds: 17.8 ms; staging segments <= 256
// in shared memory with one-lane sequential finishing: 17.1 ms.)
constexpr int SMALL = 1024;               // segments up to this size are sorted by one warp
constexpr int WINDOW = 8192;              // the sorted prefix is extended in windows of about this many elements
constexpr int CHUNK = SEL_THREADS * EPT;  // candidates examined per selection round
constexpr int ALIVE_CAP = SEL_THREADS;    // survivors resolved per selection round
constexpr int BSTACK = 640;               // block stack entries (<= depth limit + WINDOW/17 in the worst case)
constexpr int MAXT = 256;                 // small segments sorted per window at most
constexpr int WSTACK = 64;                // per-warp stack entries (>= 2*lg(n))
constexpr unsigned EMPTY = 0xFFFFFFFFu;

struct Seg {
  int f, l, d;
};

struct SelSmem {
  Seg bstack[BSTACK];
  Seg wstack[SEL_WARPS][WSTACK];
  int2 leaf[SEL_WARPS][32];
  int wcnt[SEL_WARPS], wpre[SEL_WARPS];
  int tot;
  int bsp, big_at, ntask, next_task, sorted_upto, consumed, accepted, flag, cut, error;
  int red[SEL_WARPS];
  // selection chunk
  unsigned short ax[ALIVE_CAP], ay[ALIVE_CAP];
  unsigned char st[ALIVE_CAP];
};

enum { ST_UNDEC = 0, ST_ACC = 1, ST_DEAD = 2 };

// Leaf (<= 16 elements): stable insertion sort done in registers/local memory instead of on L2-resident data.
__device__ __forceinline__ void leaf_sort_local(sfm_key_t* key, uint32_t* idx, int f, int l) {
  sfm_key_t k[SFM_SORT_THRESHOLD];
  uint32_t v[SFM_SORT_THRESHOLD];
  const int n = l - f;
#pragma unroll
  for (int i = 0; i < SFM_SORT_THRESHOLD; i++)
    if (i < n) {
      k[i] = key[f + i];
      v[i] = idx[f + i];
    }
  for (int i = 1; i < n; i++) {
    const sfm_key_t vk = k[i];
    const uint32_t vi = v[i];
    int j = i;
    while (j > 0 && vk > k[j - 1]) {
      k[j] = k[j - 1];
      v[j] = v[j - 1];
      j--;
    }
    k[j] = vk;
    v[j] = vi;
  }
#pragma unroll
  for (int i = 0; i < SFM_SORT_THRESHOLD; i++)
    if (i < n) {
      key[f + i] = k[i];
      idx[f + i] = v[i];
    }
}

// ---- warp-level partition of [f, l) (l - f > 16); returns cut (identical in all lanes) --------------------
// Each lane owns EPT consecutive positions per pass (from the left for the "left misfit" scan, from the right
// for the "right misfit" scan), so ranks are lane-prefix + in-lane order: two ordered compactions.
__device__ int warp_partition(sfm_key_t* key, uint32_t* idx, int f, int l, uint32_t* lpos, uint32_t* rpos, int lane) {
  if (lane == 0) sfm_median_to_first(key, idx, f, l);
  __syncwarp();
  const sfm_key_t p = key[f];
  const int mR = l - f - 1;
  int nl = 0, nr = 0;
  for (int t0 = 0; t0 < mR; t0 += 32 * EPT) {
    const int tb = t0 + lane * EPT;
    sfm_key_t kl[EPT], kr[EPT];
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      const bool v = tb + e < mR;
      kl[e] = v ? key[f + 1 + tb + e] : 0;
      kr[e] = v ? key[l - 1 - tb - e] : 0;
    }
    unsigned ml = 0, mr = 0;
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      const bool v = tb + e < mR;
      if (v && !(kl[e] > p)) ml |= 1u << e;
      if (v && !(p > kr[e])) mr |= 1u << e;
    }
    const int c = __popc(ml) | (__popc(mr) << 16);
    int inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += u;
    }
    const int tot = __shfl_sync(0xffffffffu, inc, 31);
    const int exc = inc - c;
    int ol = f + nl + (exc & 0xFFFF), orr = f + nr + (exc >> 16);
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      if (ml & (1u << e)) lpos[ol++] = (uint32_t)(f + 1 + tb + e);
      if (mr & (1u << e)) rpos[orr++] = (uint32_t)(l - 1 - tb - e);
    }
    nl += tot & 0xFFFF;
    nr += tot >> 16;
  }
  __syncwarp();
  const int lim = nl < nr ? nl : nr;
  int m = 0;
  for (int k0 = 0; k0 < lim; k0 += 32) {
    const int k = k0 + lane;
    const bool ok = k < lim && lpos[f + k] < rpos[f + k];
    const unsigned b = __ballot_sync(0xffffffffu, ok);
    m += __popc(b);
    if (b != 0xffffffffu) break;  // the predicate is a prefix (monotone), uniform exit
  }
  for (int k = lane; k < m; k += 32) sfm_swap_elem(key, idx, (int)lpos[f + k], (int)rpos[f + k]);
  uint32_t cut = EMPTY;
  if (m < nl) cut = lpos[f + m];
  if (m > 0) {
    const uint32_t r = rpos[f + m - 1];
    cut = r < cut ? r : cut;
  }
  __syncwarp();
  return (int)cut;
}

// ---- one warp sorts [f, l) completely ------------------------------------------------------------------------
__device__ void warp_sort_segment(SelSmem& sm, sfm_key_t* key, uint32_t* idx, uint32_t* lpos, uint32_t* rpos, Seg s0,
                                  int warp, int lane) {
  Seg* stk = sm.wstack[warp];
  int2* leaf = sm.leaf[warp];
  int sp = 0, nleaf = 0;
  if (lane == 0) stk[0] = s0;
  sp = 1;
  __syncwarp();
  while (sp > 0) {
    const Seg s = stk[sp - 1];
    sp--;
    __syncwarp();
    if (s.l - s.f <= SFM_SORT_THRESHOLD) {
      if (lane == 0) leaf[nleaf] = make_int2(s.f, s.l);
      nleaf++;
      if (nleaf == 32) {
        __syncwarp();
        leaf_sort_local(key, idx, leaf[lane].x, leaf[lane].y);
        nleaf = 0;
        __syncwarp();
      }
      continue;
    }
    if (s.d == 0 || sp + 2 > WSTACK) {
      // depth limit reached (libstdc++: __partial_sort); the stack guard cannot trigger while WSTACK >= 2*lg(n)
      if (lane == 0) sfm_heap_sort(key, idx, s.f, s.l);
      __syncwarp();
      continue;
    }
    const int cut = warp_partition(key, idx, s.f, s.l, lpos, rpos, lane);
    if (lane == 0) {
      stk[sp] = Seg{cut, s.l, s.d - 1};
      stk[sp + 1] = Seg{s.f, cut, s.d - 1};
    }
    sp += 2;
    __syncwarp();
  }
  __syncwarp();
  if (lane < nleaf) leaf_sort_local(key, idx, leaf[lane].x, leaf[lane].y);
  __syncwarp();
}

// Block-wide exclusive scan of a packed pair of 16-bit counts (value < 2^16 in total per field).
__device__ __forceinline__ int block_scan_packed(SelSmem& sm, int c, int& total) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) sm.wcnt[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int a = lane < SEL_WARPS ? sm.wcnt[lane] : 0;
    int ia = a;
#pragma unroll
    for (int o = 1; o < SEL_WARPS; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, ia, o);
      if (lane >= o) ia += u;
    }
    if (lane < SEL_WARPS) sm.wpre[lane] = ia - a;
    if (lane == SEL_WARPS - 1) sm.tot = ia;
  }
  __syncthreads();
  total = sm.tot;
  return inc - c + sm.wpre[warp];
}

// ---- block-level partition of [f, l); returns cut (identical in all threads) ------------------------------------
__device__ int block_partition(SelSmem& sm, sfm_key_t* key, uint32_t* idx, int f, int l, uint32_t* lpos, uint32_t* rpos) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) sfm_median_to_first(key, idx, f, l);
  __syncthreads();
  const sfm_key_t p = key[f];
  const int mR = l - f - 1;
  int nl = 0, nr = 0;
  for (int t0 = 0; t0 < mR; t0 += SEL_THREADS * EPT) {
    const int tb = t0 + tid * EPT;
    sfm_key_t kl[EPT], kr[EPT];
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      const bool v = tb + e < mR;
      kl[e] = v ? key[f + 1 + tb + e] : 0;
      kr[e] = v ? key[l - 1 - tb - e] : 0;
    }
    unsigned ml = 0, mr = 0;
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      const bool v = tb + e < mR;
      if (v && !(kl[e] > p)) ml |= 1u << e;
      if (v && !(p > kr[e])) mr |= 1u << e;
    }
    int tot;
    const int exc = block_scan_packed(sm, __popc(ml) | (__popc(mr) << 16), tot);
    int ol = f + nl + (exc & 0xFFFF), orr = f + nr + (exc >> 16);
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      if (ml & (1u << e)) lpos[ol++] = (uint32_t)(f + 1 + tb + e);
      if (mr & (1u << e)) rpos[orr++] = (uint32_t)(l - 1 - tb - e);
    }
    nl += tot & 0xFFFF;
    nr += tot >> 16;
    __syncthreads();  // sm.tot / wpre are reused by the next pass
  }
  const int lim = nl < nr ? nl : nr;
  int cnt = 0;
  for (int k = tid; k < lim; k += SEL_THREADS) cnt += (lpos[f + k] < rpos[f + k]) ? 1 : 0;
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) sm.red[warp] = cnt;
  __syncthreads();
  int m = 0;
#pragma unroll
  for (int k = 0; k < SEL_WARPS; k++) m += sm.red[k];
  for (int k = tid; k < m; k += SEL_THREADS) sfm_swap_elem(key, idx, (int)lpos[f + k], (int)rpos[f + k]);
  uint32_t cut = EMPTY;
  if (m < nl) cut = lpos[f + m];
  if (m > 0) {
    const uint32_t r = rpos[f + m - 1];
    cut = r < cut ? r : cut;
  }
  __syncthreads();
  return (int)cut;
}

// Extend the sorted prefix until at least `want` sorted-but-unconsumed elements exist or everything is sorted.
// The block stack holds the pending introsort segments left to right (top = leftmost).  Within a window past
// the sorted prefix every segment larger than SMALL is first split by the whole block; the small segments of
// the window are then sorted concurrently, one warp each (dynamic assignment).
__device__ void produce_sorted(SelSmem& sm, sfm_key_t* key, uint32_t* idx, uint32_t* lpos, uint32_t* rpos, int want) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  while (true) {
    __syncthreads();
    if (sm.bsp == 0 || sm.sorted_upto - sm.consumed >= want) break;
    if (tid == 0) {
      // scan the window from the top of the stack: first unsorted big segment, or the number of small ones
      const long long target = (long long)sm.sorted_upto + WINDOW;
      int e = sm.bsp - 1, nt = 0, big = -1;
      while (e >= 0 && sm.bstack[e].f < target && nt < MAXT) {
        if (sm.bstack[e].l - sm.bstack[e].f > SMALL && sm.bstack[e].d >= 0) {
          big = e;
          break;
        }
        nt++;
        e--;
      }
      sm.big_at = big;
      sm.ntask = nt;
      sm.next_task = 0;
    }
    __syncthreads();
    const int big = sm.big_at;
    if (big >= 0) {
      const Seg s = sm.bstack[big];
      __syncthreads();
      if (sm.bsp + 1 > BSTACK) {
        // Unreachable: at most 2*lg(n) pending right siblings + MAXT small segments are ever stacked.  Never
        // degrade silently: flag the frame and stop.
        if (tid == 0) sm.error = 1;
        __syncthreads();
        return;
      }
      if (s.d == 0) {
        // depth limit reached (libstdc++: __partial_sort): sequential heap sort, then the segment only waits
        // to be retired (d = -1 marks "sorted")
        if (tid == 0) {
          sfm_heap_sort(key, idx, s.f, s.l);
          sm.bstack[big].d = -1;
        }
        continue;
      }
      const int cut = block_partition(sm, key, idx, s.f, s.l, lpos, rpos);
      if (tid == 0) {
        for (int e = sm.bsp; e > big + 1; e--) sm.bstack[e] = sm.bstack[e - 1];  // make room above `big`
        sm.bstack[big] = Seg{cut, s.l, s.d - 1};
        sm.bstack[big + 1] = Seg{s.f, cut, s.d - 1};
        sm.bsp++;
      }
      continue;
    }
    // every segment of the window is small: sort them concurrently, one warp per segment
    const int nt = sm.ntask, top = sm.bsp - 1;
    while (true) {
      int t = 0;
      if (lane == 0) t = atomicAdd(&sm.next_task, 1);
      t = __shfl_sync(0xffffffffu, t, 0);
      if (t >= nt) break;
      const Seg s = sm.bstack[top - t];
      if (s.d >= 0) warp_sort_segment(sm, key, idx, lpos, rpos, s, warp, lane);
    }
    __syncthreads();
    if (tid == 0) {
      sm.sorted_upto = sm.bstack[top - (nt - 1)].l;
      sm.bsp -= nt;
    }
  }
}

// ---- bucket selection (default path) ------------------------------------------------------------------------------------------
// The greedy loop only ever accepts candidates that no accepted corner blocks, and a candidate that is blocked once stays
// blocked.  With ~50 candidates per accepted corner almost every candidate is blocked by the time its turn comes, so the
// list is NOT sorted as a whole: one block per frame
//   (1) sweeps the unordered list once: entries that reach the final threshold become words (order code << 30 | y << 15 | x,
//       order code = up to 34 leading bits of the score's distance below the frame maximum: ascending word = descending
//       score) and are counted per MSD bucket (top 7 bits of the code);
//   (2) scatters the words into bucket order (one pass, unordered inside a bucket);
//   (3) walks the buckets from the best score down in gathers of <= 4096 words: a word whose pixel is already blocked is
//       dropped at once (order-independent, exact); the SURVIVORS of the gather - all of them early on, a few per cent
//       later - are sorted in shared memory (bitonic, 64-bit words) and go through the greedy rounds (conflict bit rows);
//       accepted corners mark their discs; the walk stops when max_corners are accepted.
// Buckets the selection never reaches are never sorted, blocked candidates are never sorted, and nothing is gathered
// through a slot index: the word carries the pixel.
// (Tried and dropped: the blocked-pixel map in 8 x 4 pixel tiles, a 32-byte sector = 16 x 16 pixels, so that a disc touches
// ~4 sectors instead of one per row: 3.37 vs 3.41 ms per 999 1080p frames, 7.04 vs 6.80 ms per 399 4K frames.)
// Equal order codes among the survivors of a gather (rare with 34 bits): the members' exact scores are recomputed from
// the image (same expression as the score kernels) and the run is ordered by them; IDENTICAL scores are flagged and
// handled by the observable-tie rule (DESIGN.md §4): if two members of a tie are still unblocked when the rounds reach
// them, or a run is longer than 64, or a single SUB-bucket's survivors (2^-15 of the score range) do not fit, the frame gets
// status 3 and is redone by the exact emulation (select_kernel mode 3).
constexpr int BK_THREADS = 256, BK_WARPS = BK_THREADS / 32;
#ifndef BK_NB_BITS_V
#define BK_NB_BITS_V 7
#endif
constexpr int BK_NB_BITS = BK_NB_BITS_V, BK_NB = 1 << BK_NB_BITS;
constexpr int BK_CODE_BITS = 34;
#ifndef BK_T_V
#define BK_T_V 4096
#endif
constexpr int BK_T = BK_T_V;                    // survivors held per gather
constexpr int BK_EPT = 8, BK_PIECE = BK_THREADS * BK_EPT;
constexpr int BK_ALIVE = BK_THREADS;            // survivors resolved per greedy round, one per thread
constexpr int BK_MAXRUN = 64;
constexpr unsigned BK_YX = 0x3FFFFFFFu;
static_assert((BK_T & (BK_T - 1)) == 0 && BK_T >= BK_PIECE, "the bitonic sort pads a gather to a power of two inside sv[]");
static_assert(BK_NB % BK_THREADS == 0 || BK_NB < BK_THREADS, "bucket starts: BK_NB / BK_THREADS counters per thread");
// Measured (select stage, ms per 999 1080p frames / per 399 4K frames, T = 4096): buckets 2048: 3.39 / 6.71, 1024: 3.08 / 6.41,
// 512: 2.65 / 6.09, 256: 2.57 / 5.75, 128: 2.37 / 5.53, 64: 2.26 / 5.34, 32: 2.21 / 39, 16: 2.55 / 40 (T = 2048: 64 buckets
// 2.19 / 5.43).  Fewer buckets: the scatter's writes coalesce better and the walk has fewer steps; a bucket is then often larger
// than a gather, which is fine while its UNBLOCKED words fit (the dense buckets lie near the threshold, where almost everything
// is blocked); a bucket whose unblocked words do not fit is walked in runs of its 256 sub-buckets, re-read once per run - cheap
// for the occasional bucket, quadratic when most buckets need it (32 buckets on 4K frames).  128 buckets keep a factor of four
// of bucket size between the default and that regime.

struct BucketSmem {
  __align__(16) unsigned long long sv[BK_T];
  unsigned cur[BK_NB];
  __align__(16) unsigned pxy[BK_ALIVE];
  unsigned accm[BK_ALIVE / 32], deadm[BK_ALIVE / 32];
  unsigned short accl[BK_ALIVE];
  unsigned char tf[BK_T];  // bit 0: identical score as the predecessor, bit 1: member of a group of >= 3
  int wcnt[BK_WARPS];
  unsigned subh[256];  // unblocked words per sub-bucket (next 8 code bits) of a bucket whose unblocked words exceed a gather
  unsigned nkeep, tgt;
  int accepted, cut, tiehit, eqrun, bi, sub_lo, sub_hi;
};

__device__ __forceinline__ int bk_block_scan(BucketSmem& sm, int c, int& total) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) sm.wcnt[warp] = inc;
  __syncthreads();
  int pre = 0, tot = 0;
#pragma unroll
  for (int k = 0; k < BK_WARPS; k++) {
    const int v = sm.wcnt[k];
    if (k < warp) pre += v;
    tot += v;
  }
  __syncthreads();  // wcnt is reused by the next scan
  total = tot;
  return inc - c + pre;
}

// shi_tomasi's score of one pixel (:252-270) from the image: integer window sums, then the single FP64 expression the score
// kernels evaluate (corner_score.cu: exact_u) - bit-identical to the list's value.
__device__ double bk_exact_score(const uint8_t* __restrict__ im, int pitch, int w, int h, int x, int y) {
  if (x < 2 || y < 2 || x >= w - 2 || y >= h - 2) return 0.0;
  int a = 0, b = 0, c = 0;
  for (int yy = y - 2; yy <= y + 2; yy++) {
    const uint8_t* r0 = im + (size_t)yy * pitch;
    const uint8_t* rm = im + (size_t)max(yy - 1, 0) * pitch;
    const uint8_t* rp = im + (size_t)min(yy + 1, h - 1) * pitch;
    for (int xx = x - 2; xx <= x + 2; xx++) {
      const int gx = (int)r0[min(xx + 1, w - 1)] - (int)r0[max(xx - 1, 0)];
      const int gy = (int)rp[xx] - (int)rm[xx];
      a += gx * gx;
      b += gy * gy;
      c += gx * gy;
    }
  }
  const double dd = (double)(a - b), c2 = (double)(2 * c);
  const double D = dd * dd + c2 * c2;
  return 0.125 * ((double)(a + b) - sqrt(D));
}

__global__ void __launch_bounds__(BK_THREADS, 4) bucket_select_kernel(CornerWorkView wv, const uint8_t* __restrict__ img, int pitch,
                                                                      size_t fstride, int first, int w, int h, int max_corners,
                                                                      int min_dist, double quality, int code_bits, int gather_cap,
                                                                      double2* __restrict__ out_xy, int* __restrict__ out_n) {
  extern __shared__ __align__(16) unsigned char bk_raw[];
  BucketSmem& sm = *reinterpret_cast<BucketSmem*>(bk_raw);
  const int fr = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t cb = (size_t)fr * wv.cand_cap;
  unsigned long long* B = wv.words + cb;
  const bool exact = wv.exact_list[fr] != 0;
  const unsigned nlist = exact ? wv.nfinal[fr] : wv.ncand[fr];
  if (nlist > (unsigned)wv.cand_cap) {  // capacity exceeded: report, never truncate silently
    if (tid == 0) {
      wv.status[fr] = 1;
      if (out_n) out_n[fr] = -1;
    }
    return;
  }
  for (int i = tid; i < BK_NB; i += BK_THREADS) sm.cur[i] = 0;
  if (tid == 0) {
    sm.nkeep = 0;
    sm.accepted = 0;
    sm.tiehit = 0;
  }
  __syncthreads();

  // (1) list -> words + bucket counts.  The frame maximum is final: entries of a provisional list below the final threshold
  // are dropped here (s >= thr, :282).
  const double maxv = 0.125 * __longlong_as_double(wv.maxbits[fr]);
  const double thr = maxv * quality;
  const unsigned long long maxkey = (unsigned long long)__double_as_longlong(maxv);
  const unsigned long long thrkey = thr > 0.0 ? (unsigned long long)__double_as_longlong(thr) : 0ull;
  const unsigned long long range = maxkey > thrkey ? maxkey - thrkey : 0ull;
  const int bits = 64 - __clzll((long long)range);
  const int shift = bits > code_bits ? bits - code_bits : 0;
  const int used_bits = bits < code_bits ? bits : code_bits;
  const int bshift = used_bits > BK_NB_BITS ? used_bits - BK_NB_BITS : 0;
  const unsigned long long* lkey = wv.tmp_key + cb;
  const unsigned* lidx = wv.tmp_idx + cb;
  // sweep 1: bucket counts (keys only); the loads of the next round are in flight while this one is counted
  {
    unsigned long long k[4], kn[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const unsigned e = q * BK_THREADS + tid;
      kn[q] = e < nlist ? __ldcg(lkey + e) : 0ull;
    }
    unsigned cnt = 0;
    for (unsigned i0 = 0; i0 < nlist; i0 += BK_THREADS * 4) {  // block-uniform trip count
#pragma unroll
      for (int q = 0; q < 4; q++) {
        k[q] = kn[q];
        const unsigned e = i0 + BK_THREADS * 4 + q * BK_THREADS + tid;
        kn[q] = e < nlist ? __ldcg(lkey + e) : 0ull;
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const unsigned e = i0 + q * BK_THREADS + tid;
        if (e < nlist && __longlong_as_double((long long)k[q]) >= thr) {
          atomicAdd(&sm.cur[(unsigned)(((maxkey - k[q]) >> shift) >> bshift)], 1u);
          cnt++;
        }
      }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0 && cnt) atomicAdd(&sm.nkeep, cnt);
  }
  __syncthreads();
  const unsigned n = sm.nkeep;
  if (tid == 0) wv.nfinal[fr] = n;
  const int cap_out = max_corners < 1 ? 1 : max_corners;  // the cap is tested after the push (:298-299)
  if (n == 0) {
    if (tid == 0) {
      wv.status[fr] = 0;
      if (out_n) out_n[fr] = 0;
    }
    return;
  }
  // bucket starts
  {
    constexpr int PER = BK_NB >= BK_THREADS ? BK_NB / BK_THREADS : 1;
    unsigned c[PER];
    int s = 0;
#pragma unroll
    for (int j = 0; j < PER; j++) {
      c[j] = tid * PER + j < BK_NB ? sm.cur[tid * PER + j] : 0u;
      s += (int)c[j];
    }
    int tot;
    unsigned run = (unsigned)bk_block_scan(sm, s, tot);
#pragma unroll
    for (int j = 0; j < PER; j++) {
      if (tid * PER + j < BK_NB) sm.cur[tid * PER + j] = run;
      run += c[j];
    }
  }
  __syncthreads();
  // sweep 2: words into bucket order (unordered inside a bucket); cur[b] ends up as the END of bucket b
  {
    unsigned long long k[4], kn[4];
    unsigned yx[4], yxn[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const unsigned e = q * BK_THREADS + tid;
      kn[q] = e < nlist ? __ldcg(lkey + e) : 0ull;
      yxn[q] = e < nlist ? __ldcg(lidx + e) : 0u;
    }
    for (unsigned i0 = 0; i0 < nlist; i0 += BK_THREADS * 4) {
#pragma unroll
      for (int q = 0; q < 4; q++) {
        k[q] = kn[q];
        yx[q] = yxn[q];
        const unsigned e = i0 + BK_THREADS * 4 + q * BK_THREADS + tid;
        kn[q] = e < nlist ? __ldcg(lkey + e) : 0ull;
        yxn[q] = e < nlist ? __ldcg(lidx + e) : 0u;
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const unsigned e = i0 + q * BK_THREADS + tid;
        const bool in = e < nlist && __longlong_as_double((long long)k[q]) >= thr;
        const unsigned long long code = (maxkey - k[q]) >> shift;
        const unsigned b = in ? (unsigned)(code >> bshift) : 0xFFFFFFFFu;
        const unsigned pm = __match_any_sync(0xffffffffu, b);
        const int leader = __ffs(pm) - 1;
        unsigned old = 0;
        if (in && lane == leader) old = atomicAdd(&sm.cur[b], (unsigned)__popc(pm));
        old = __shfl_sync(0xffffffffu, old, leader);
        if (in)
          B[old + __popc(pm & ((1u << lane) - 1u))] = (code << 30) | (unsigned long long)(((yx[q] >> 16) << 15) | (yx[q] & 0x7FFFu));
      }
    }
  }
  __threadfence_block();
  __syncthreads();

  // (3) the walk
  unsigned* blocked = wv.wordoff + (size_t)fr * wv.words_per_frame;  // free until a fallback frame needs raster ranks
  const uint8_t* im = img + (size_t)(first + fr) * fstride;
  double2* out = out_xy + (size_t)fr * cap_out;
  const int d = min_dist, d2 = min_dist * min_dist, rows = 2 * d - 1;
  const bool suppress = wv.cell > 0;
  unsigned pos = 0;  // words [0, pos) are done (block-uniform)
  int bi = 0;        // first bucket that is not done
  // A bucket whose UNBLOCKED words exceed a gather is walked in runs of its sub-buckets (the next 8 bits of the order code):
  // sub_next >= 0 while that is going on; [pos, tgt) is then that bucket, re-read once per run.
  const int sbits = bshift < 8 ? bshift : 8, sshift = bshift - sbits;
  const unsigned smask = (1u << sbits) - 1u;
  int sub_next = -1;
  unsigned tgt = 0;
  while (pos < n && sm.accepted < cap_out && !sm.tiehit) {
    unsigned s_lo = 0, s_hi = smask;
    if (sub_next < 0) {
      // as many whole buckets as certainly fit; a bucket that does not fit by itself is filtered anyway (see below)
      if (warp == 0) {  // 32 buckets per step
        int b2 = bi;
        while (b2 < BK_NB) {
          const bool fits = b2 + lane < BK_NB && sm.cur[b2 + lane] - pos <= (unsigned)gather_cap;
          const int run = __ffs(~__ballot_sync(0xffffffffu, fits)) - 1;  // leading buckets that fit (32: all of them)
          b2 += run < 0 ? 32 : run;
          if (run >= 0 && run < 32) break;
        }
        if (b2 > BK_NB) b2 = BK_NB;
        if (b2 == bi) b2++;  // the next bucket does not fit by itself
        if (lane == 0) {
          sm.bi = b2;
          sm.tgt = sm.cur[b2 - 1];
        }
      }
      __syncthreads();
      bi = sm.bi;
      tgt = sm.tgt;
    } else {
      // the next run of sub-buckets whose (earlier counted, since then only shrunk) unblocked words fit
      if (tid == 0) {
        int hi = sub_next;
        unsigned sum = sm.subh[hi];
        while (hi + 1 <= (int)smask && sum + sm.subh[hi + 1] <= (unsigned)gather_cap) sum += sm.subh[++hi];
        sm.sub_lo = sub_next;
        sm.sub_hi = hi;
        if (sm.subh[sub_next] > (unsigned)gather_cap) sm.tiehit = 1;  // more unblocked words than a gather within 2^-15 of the score range
      }
      __syncthreads();
      if (sm.tiehit) break;
      s_lo = (unsigned)sm.sub_lo;
      s_hi = (unsigned)sm.sub_hi;
    }
    int nsv = 0;
    bool overflow = false;
    for (unsigned p0 = pos; p0 < tgt; p0 += BK_PIECE) {
      unsigned long long v[BK_EPT];
      unsigned bw[BK_EPT];
#pragma unroll
      for (int e = 0; e < BK_EPT; e++) {
        const unsigned i = p0 + tid * BK_EPT + e;
        v[e] = i < tgt ? __ldcg(B + i) : ~0ull;
      }
#pragma unroll
      for (int e = 0; e < BK_EPT; e++) {
        const unsigned x = (unsigned)v[e] & 0x7FFFu, y = ((unsigned)v[e] >> 15) & 0x7FFFu;
        bw[e] = (suppress && p0 + tid * BK_EPT + e < tgt) ? __ldcg(blocked + (size_t)y * wv.wpr + (x >> 5)) : 0u;
      }
      unsigned am = 0;
#pragma unroll
      for (int e = 0; e < BK_EPT; e++) {
        const unsigned sub = (unsigned)(v[e] >> (30 + sshift)) & smask;
        if (p0 + tid * BK_EPT + e < tgt && !((bw[e] >> ((unsigned)v[e] & 31u)) & 1u) && sub >= s_lo && sub <= s_hi) am |= 1u << e;
      }
      int tot;
      int r = nsv + bk_block_scan(sm, __popc(am), tot);
      if (nsv + tot > gather_cap) {  // block-uniform
        overflow = true;
        break;
      }
#pragma unroll
      for (int e = 0; e < BK_EPT; e++)
        if (am & (1u << e)) sm.sv[r++] = v[e];
      nsv += tot;
    }
    if (overflow) {
      // only a single bucket can overflow (several are gathered only if all their words fit): count its unblocked words per
      // sub-bucket and walk it in runs of sub-buckets.  No sub-bits left, or already in that mode (the counts bound every
      // run): the exact emulation takes the frame.
      if (sub_next >= 0 || sbits == 0) {
        if (tid == 0) sm.tiehit = 1;
        __syncthreads();
        break;
      }
      for (int i = tid; i < 256; i += BK_THREADS) sm.subh[i] = 0;
      __syncthreads();
      for (unsigned p0 = pos; p0 < tgt; p0 += BK_THREADS) {
        const unsigned i = p0 + tid;
        if (i < tgt) {
          const unsigned long long v = __ldcg(B + i);
          const unsigned x = (unsigned)v & 0x7FFFu, y = ((unsigned)v >> 15) & 0x7FFFu;
          const unsigned bwd = suppress ? __ldcg(blocked + (size_t)y * wv.wpr + (x >> 5)) : 0u;
          if (!((bwd >> (x & 31u)) & 1u)) atomicAdd(&sm.subh[(unsigned)(v >> (30 + sshift)) & smask], 1u);
        }
      }
      __syncthreads();
      sub_next = 0;
      continue;
    }
    if (sub_next >= 0) {
      sub_next = (int)s_hi + 1;
      if (sub_next > (int)smask) {  // the bucket is done
        sub_next = -1;
        pos = tgt;
      }
    } else {
      pos = tgt;
    }
    if (nsv == 0) {
      __syncthreads();
      continue;
    }
    // sort the survivors (ascending word = descending score); pad to a power of two
    int N2 = 32;
    while (N2 < nsv) N2 <<= 1;
    for (int i = nsv + tid; i < N2; i += BK_THREADS) sm.sv[i] = ~0ull;
    for (int i = tid; i < nsv; i += BK_THREADS) sm.tf[i] = 0;
    if (tid == 0) sm.eqrun = 0;
    __syncthreads();
    for (int k = 2; k <= N2; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = tid; t < (N2 >> 1); t += BK_THREADS) {
          const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), p = i | j;  // the pair (i, i + j) of this step
          const unsigned long long a = sm.sv[i], b = sm.sv[p];
          const bool up = (i & k) == 0;
          if ((a > b) == up) {
            sm.sv[i] = b;
            sm.sv[p] = a;
          }
        }
        __syncthreads();
      }
    // equal order codes among the survivors: order by the exact score, flag identical scores (rare)
    for (int i = tid; i + 1 < nsv; i += BK_THREADS)
      if ((sm.sv[i] >> 30) == (sm.sv[i + 1] >> 30)) sm.eqrun = 1;
    __syncthreads();
    if (sm.eqrun) {
      for (int i = tid; i + 1 < nsv; i += BK_THREADS) {
        const unsigned long long code = sm.sv[i] >> 30;
        if ((sm.sv[i + 1] >> 30) != code || (i > 0 && (sm.sv[i - 1] >> 30) == code)) continue;  // not the start of a run
        int j = i + 2;
        while (j < nsv && j - i < BK_MAXRUN && (sm.sv[j] >> 30) == code) j++;
        if (j < nsv && (sm.sv[j] >> 30) == code) {  // pathological pile-up: let the exact path decide
          sm.tiehit = 1;
          continue;
        }
        // insertion sort of [i, j) by the exact score, descending (scores recomputed on every comparison: the runs are pairs)
        for (int p = i + 1; p < j; p++) {
          const unsigned long long e = sm.sv[p];
          const double se = bk_exact_score(im, pitch, w, h, (int)((unsigned)e & 0x7FFFu), (int)(((unsigned)e >> 15) & 0x7FFFu));
          int q = p;
          while (q > i) {
            const unsigned long long f = sm.sv[q - 1];
            const double sf = bk_exact_score(im, pitch, w, h, (int)((unsigned)f & 0x7FFFu), (int)(((unsigned)f >> 15) & 0x7FFFu));
            if (!(sf < se)) break;
            sm.sv[q] = f;
            q--;
          }
          sm.sv[q] = e;
        }
        double sprev = 0.0;
        for (int p = i; p < j; p++) {
          const unsigned long long e = sm.sv[p];
          const double s = bk_exact_score(im, pitch, w, h, (int)((unsigned)e & 0x7FFFu), (int)(((unsigned)e >> 15) & 0x7FFFu));
          if (p > i && s == sprev) {
            sm.tf[p] |= 1;
            if (p > i + 1 && (sm.tf[p - 1] & 1)) {
              sm.tf[p - 2] |= 2;
              sm.tf[p - 1] |= 2;
              sm.tf[p] |= 2;
            }
          }
          sprev = s;
        }
      }
      __syncthreads();
    }
    // greedy rounds over the sorted survivors
    // A round resolves at most BK_ALIVE unblocked survivors: where most survivors are still unblocked (the first gathers)
    // a short chunk holds that many, and whatever a round does not consume is tested again by the next one
    int t0 = 0, want = 2 * BK_ALIVE;
    while (t0 < nsv) {
      const int acc0 = sm.accepted;
      if (acc0 >= cap_out) break;
      const int cnt = min(want, nsv - t0);
      unsigned yx[BK_EPT], bw[BK_EPT];
      unsigned tie = 0, big = 0;
#pragma unroll
      for (int e = 0; e < BK_EPT; e++) {
        const int t = tid * BK_EPT + e;
        yx[e] = t < cnt ? (unsigned)sm.sv[t0 + t] & BK_YX : 0u;
        const unsigned f = t < cnt ? sm.tf[t0 + t] : 0u;
        tie |= (f & 1u) << e;
        big |= ((f >> 1) & 1u) << e;
      }
#pragma unroll
      for (int e = 0; e < BK_EPT; e++) {
        const int t = tid * BK_EPT + e;
        const unsigned x = yx[e] & 0x7FFFu, y = yx[e] >> 15;
        // (the first round of a gather follows its filter directly: nothing has been marked since)
        bw[e] = (suppress && t < cnt && t0 > 0) ? __ldcg(blocked + (size_t)y * wv.wpr + (x >> 5)) : 0u;
      }
      unsigned am = 0;
#pragma unroll
      for (int e = 0; e < BK_EPT; e++)
        if (tid * BK_EPT + e < cnt && !((bw[e] >> (yx[e] & 31u)) & 1u)) am |= 1u << e;
      {
        // std::sort's order inside a group of identical scores is only observable if at least two of its members are still
        // unblocked (DESIGN.md §4).  Conservative test on the survivors of the bitmap check (predecessors outside the warp /
        // chunk count as unblocked).
        const unsigned up = __shfl_up_sync(0xffffffffu, am, 1);
        const unsigned prev_alive = (am << 1) | (lane > 0 ? (up >> (BK_EPT - 1)) & 1u : 1u);
        if (am & (big | (tie & prev_alive))) sm.tiehit = 1;
      }
      int na;
      const int exc = bk_block_scan(sm, __popc(am), na);
      if (sm.tiehit) break;  // block-uniform: written before the scan's barriers, not again before the next ones
      if (tid == 0) sm.cut = cnt;
      __syncthreads();
      {
        int r = exc;
#pragma unroll
        for (int e = 0; e < BK_EPT; e++)
          if (am & (1u << e)) {
            if (r < BK_ALIVE) sm.pxy[r] = yx[e];
            if (r == BK_ALIVE) sm.cut = tid * BK_EPT + e;  // first candidate that does not fit: it starts the next round
            r++;
          }
      }
      if (tid < BK_ALIVE / 32) sm.accm[tid] = sm.deadm[tid] = 0;
      na = na < BK_ALIVE ? na : BK_ALIVE;
      __syncthreads();
      const int used = sm.cut;
      // conflicts inside the round: thread i collects the higher-priority survivors closer than min_dist as a bit row, then
      // rounds of pure bit logic: dead if the row meets an accepted survivor, accepted once every member of it is dead
      const unsigned me = sm.pxy[tid];
      const int mx = (int)(me & 0x7FFFu), my = (int)(me >> 15);
      unsigned C[BK_ALIVE / 32];
#pragma unroll
      for (int wd = 0; wd < BK_ALIVE / 32; wd++) {
        C[wd] = 0;
        if (suppress && wd <= warp && wd * 32 < na) {
          unsigned bitsw = 0;
#pragma unroll
          for (int q = 0; q < 8; q++) {
            const uint4 o = *reinterpret_cast<const uint4*>(&sm.pxy[wd * 32 + q * 4]);
            const unsigned ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int kk = 0; kk < 4; kk++) {
              const int dx = (int)(ov[kk] & 0x7FFFu) - mx, dy = (int)(ov[kk] >> 15) - my;
              if (dx * dx + dy * dy < d2) bitsw |= 1u << (q * 4 + kk);
            }
          }
          if (wd == warp) bitsw &= (1u << lane) - 1u;  // strictly higher priority only
          C[wd] = bitsw;
        }
      }
      int state = tid < na ? ST_UNDEC : ST_DEAD;
      if (!suppress && tid < na) state = ST_ACC;
      while (true) {
        if (state == ST_UNDEC) {
          unsigned hit = 0, und = 0;
#pragma unroll
          for (int wd = 0; wd < BK_ALIVE / 32; wd++) {
            const unsigned a = sm.accm[wd], dd = sm.deadm[wd];
            hit |= C[wd] & a;
            und |= C[wd] & ~(a | dd);
          }
          state = hit ? ST_DEAD : (und ? ST_UNDEC : ST_ACC);
        }
        __syncthreads();  // everybody has read the masks of the previous round
        const unsigned ba = __ballot_sync(0xffffffffu, state == ST_ACC), bd = __ballot_sync(0xffffffffu, state == ST_DEAD);
        if (lane == 0) {
          sm.accm[warp] = ba;
          sm.deadm[warp] = bd;
        }
        if (__syncthreads_or(state == ST_UNDEC) == 0) break;
      }
      // append accepted survivors in priority order, stop at the cap; mark their discs
      const bool acc = state == ST_ACC;
      int nacc;
      const int rank = bk_block_scan(sm, acc ? 1 : 0, nacc);
      if (acc && acc0 + rank < cap_out) {
        out[acc0 + rank] = make_double2((double)mx, (double)my);
        sm.accl[rank] = (unsigned short)tid;
      }
      __syncthreads();
      const int nnew = min(nacc, cap_out - acc0);
      if (suppress && acc0 + nnew < cap_out) {  // nothing is looked up once the cap is reached
        for (int i = tid; i < nnew * rows; i += BK_THREADS) {
          const int c = i / rows, dy = i - c * rows - (d - 1);
          const unsigned sp = sm.pxy[sm.accl[c]];
          const int px = (int)(sp & 0x7FFFu), py = (int)(sp >> 15) + dy;
          if (py < 0 || py >= h) continue;
          const int r2 = d2 - 1 - dy * dy;  // dx^2 <= r2  <=>  dx^2 + dy^2 < d^2
          int r = (int)sqrtf((float)r2);
          while (r * r > r2) r--;
          while ((r + 1) * (r + 1) <= r2) r++;
          const int xa = max(px - r, 0), xb = min(px + r, w - 1);
          unsigned* rowp = blocked + (size_t)py * wv.wpr;
          for (int wd = xa >> 5; wd <= (xb >> 5); wd++) {
            const int lo = max(xa - wd * 32, 0), hi = min(xb - wd * 32, 31);
            atomicOr(rowp + wd, (0xFFFFFFFFu >> (31 - hi)) & (0xFFFFFFFFu << lo));
          }
        }
        __threadfence_block();
      }
      __syncthreads();
      if (tid == 0) sm.accepted = acc0 + nnew;
      t0 += used;
      want = used < cnt ? 2 * used : 2 * want;  // the chunk was cut (enough unblocked survivors) / was used up
      want = want < 2 * BK_ALIVE ? 2 * BK_ALIVE : (want > BK_PIECE ? BK_PIECE : want);
      __syncthreads();
    }
  }
  __syncthreads();
  if (tid == 0) {
    // an observable tie, an unresolved pile-up of equal order codes or a bucket whose survivors do not fit: the frame is
    // redone by select_kernel mode 3
    wv.status[fr] = sm.tiehit ? 3 : 0;
    if (out_n) out_n[fr] = sm.accepted;
  }
}

// mode 0: full shi_tomasi selection; mode 1: sort only (sfmgpu_sort_perm_desc).
// mode 3: redo exactly the frames bucket_select_kernel marked with status 3 (a consumed score tie) through the emulation.
__global__ void __launch_bounds__(SEL_THREADS, 4) select_kernel(CornerWorkView wv, int w, int max_corners, int min_dist, int mode,
                                                               double2* __restrict__ out_xy, int* __restrict__ out_n) {
  extern __shared__ __align__(16) unsigned char sel_raw[];
  SelSmem& sm = *reinterpret_cast<SelSmem*>(sel_raw);
  const int fr = blockIdx.x, tid = threadIdx.x;
  const size_t cb = (size_t)fr * wv.cand_cap;
  sfm_key_t* key = wv.key + cb;
  uint32_t* idx = wv.idx + cb;
  uint32_t* lpos = wv.lpos + cb;
  uint32_t* rpos = wv.rpos + cb;
  if (mode == 3) {  // every thread reads the status before thread 0 resets it below
    const bool redo = wv.status[fr] == 3;
    __syncthreads();
    if (!redo) return;
  }
  const unsigned ntot = wv.ntotal[fr];
  if (ntot > (unsigned)wv.cand_cap) {  // capacity exceeded: report, never truncate silently
    if (tid == 0) {
      wv.status[fr] = 1;
      if (out_n) out_n[fr] = -1;
    }
    return;
  }
  const int n = (int)ntot;
  const int cap_out = max_corners < 1 ? 1 : max_corners;  // the cap is tested after the push (:298-299)
  if (tid == 0) {
    wv.status[fr] = 0;
    sm.bsp = 0;
    if (n > 0) sm.bstack[sm.bsp++] = Seg{0, n, 2 * sfm_lg2((unsigned)n)};
    sm.sorted_upto = 0;
    sm.consumed = 0;
    sm.accepted = 0;
    sm.error = 0;
  }
  __syncthreads();
  if (mode == 1) {
    produce_sorted(sm, key, idx, lpos, rpos, 0x7fffffff);
    if (tid == 0 && sm.error) wv.status[fr] = 2;
    return;
  }
  const uint2* grid = reinterpret_cast<const uint2*>(wv.grid + (size_t)fr * wv.grid_per_frame);
  unsigned* gridw = wv.grid + (size_t)fr * wv.grid_per_frame;
  double2* out = out_xy + (size_t)fr * cap_out;
  const int d = min_dist, d2 = min_dist * min_dist;
  const bool suppress = wv.cell > 0;
  if (mode == 3) {  // the fast path skips the host-side grid reset
    for (size_t i = tid; i < wv.grid_per_frame; i += SEL_THREADS) gridw[i] = EMPTY;
    __threadfence_block();
    __syncthreads();
  }

  while (true) {
    produce_sorted(sm, key, idx, lpos, rpos, CHUNK);
    if (sm.error) {
      if (tid == 0) {
        wv.status[fr] = 2;
        if (out_n) out_n[fr] = -1;
      }
      return;
    }
    const int consumed = sm.consumed, upto = sm.sorted_upto, acc0 = sm.accepted;
    if (consumed >= upto || acc0 >= cap_out) break;
    const int cnt = min(CHUNK, upto - consumed);
    __syncthreads();
    // (1) candidates of this chunk vs corners accepted in earlier chunks; EPT consecutive candidates per thread
    int cx_[EPT], cy_[EPT];
    unsigned am = 0;
#pragma unroll
    for (int e = 0; e < EPT; e++) {
      const int t = tid * EPT + e;
      cx_[e] = cy_[e] = 0;
      if (t < cnt) {
        const unsigned pix = idx[consumed + t];  // y << 16 | x
        const int y = (int)(pix >> 16), x = (int)(pix & 0xFFFFu);
        cx_[e] = x;
        cy_[e] = y;
        bool alive = true;
        if (suppress) {
          const int gx0 = max(x / d - 1, 0), gx1 = min(x / d + 1, wv.gw - 1);
          const int gy0 = max(y / d - 1, 0), gy1 = min(y / d + 1, wv.gh - 1);
          for (int gy = gy0; gy <= gy1; gy++)
            for (int gx = gx0; gx <= gx1; gx++) {
              const uint2 v = __ldcg(grid + (size_t)gy * wv.gw + gx);
              if (v.x != EMPTY) {
                const int dx = (int)(v.x & 0xFFFFu) - x, dy = (int)(v.x >> 16) - y;
                if (dx * dx + dy * dy < d2) alive = false;
              }
              if (v.y != EMPTY) {
                const int dx = (int)(v.y & 0xFFFFu) - x, dy = (int)(v.y >> 16) - y;
                if (dx * dx + dy * dy < d2) alive = false;
              }
            }
        }
        if (alive) am |= 1u << e;
      }
    }
    // ordered compaction of the survivors; at most ALIVE_CAP are resolved now, the chunk is cut after the last one
    int na;
    const int exc = block_scan_packed(sm, __popc(am), na);
    if (tid == 0) sm.cut = cnt;
    __syncthreads();
    {
      int r = exc;
#pragma unroll
      for (int e = 0; e < EPT; e++)
        if (am & (1u << e)) {
          if (r < ALIVE_CAP) {
            sm.ax[r] = (unsigned short)cx_[e];
            sm.ay[r] = (unsigned short)cy_[e];
            sm.st[r] = ST_UNDEC;
          }
          if (r == ALIVE_CAP) sm.cut = tid * EPT + e;  // first candidate that does not fit: it starts the next chunk
          r++;
        }
    }
    na = na < ALIVE_CAP ? na : ALIVE_CAP;
    __syncthreads();
    const int used = sm.cut;
    // (2) conflicts inside the chunk, by rounds
    if (suppress) {
      while (true) {
        int ns = ST_DEAD + 1;  // "no change"
        if (tid < na && sm.st[tid] == ST_UNDEC) {
          const int mx = sm.ax[tid], my = sm.ay[tid];
          bool dead = false, blocked = false;
          for (int j = 0; j < tid; j++) {
            const int sj = sm.st[j];
            if (sj == ST_DEAD) continue;
            const int dx = (int)sm.ax[j] - mx, dy = (int)sm.ay[j] - my;
            if (dx * dx + dy * dy < d2) {
              if (sj == ST_ACC) {
                dead = true;
                break;
              }
              blocked = true;
            }
          }
          ns = dead ? ST_DEAD : (blocked ? ST_UNDEC : ST_ACC);
        }
        __syncthreads();
        if (tid == 0) sm.flag = 0;
        if (ns <= ST_DEAD) sm.st[tid] = (unsigned char)ns;
        __syncthreads();
        if (ns == ST_UNDEC) sm.flag = 1;
        __syncthreads();
        if (!sm.flag) break;
        __syncthreads();
      }
    } else {
      if (tid < na) sm.st[tid] = ST_ACC;
      __syncthreads();
    }
    // (3) append accepted survivors in priority order, stop at the cap
    const bool acc = tid < na && sm.st[tid] == ST_ACC;
    int nacc;
    const int rank = block_scan_packed(sm, acc ? 1 : 0, nacc);
    if (acc) {
      const int k = acc0 + rank;
      if (k < cap_out) {
        const int px = sm.ax[tid], py = sm.ay[tid];
        out[k] = make_double2((double)px, (double)py);
        if (suppress) {
          unsigned* cell = gridw + ((size_t)(py / d) * wv.gw + (px / d)) * 2;
          const unsigned v = ((unsigned)py << 16) | (unsigned)px;
          if (atomicCAS(cell, EMPTY, v) != EMPTY) atomicCAS(cell + 1, EMPTY, v);
        }
      }
    }
    __syncthreads();
    if (tid == 0) {
      sm.accepted = min(cap_out, acc0 + nacc);
      sm.consumed = consumed + used;
    }
    __syncthreads();
  }
  if (tid == 0 && out_n) out_n[fr] = sm.accepted;
}

int select_smem_config(sfmgpu_ctx* ctx) {
  static const int sel_id = sfm_next_cfg_id();
  SFM_SMEM_OPTIN(ctx, sel_id, select_kernel, sizeof(SelSmem));
  static const int bk_id = sfm_next_cfg_id();
  SFM_SMEM_OPTIN(ctx, bk_id, bucket_select_kernel, sizeof(BucketSmem));
  return 0;
}

}  // namespace

// Detect corners for frames [first, first+count): out_xy [count][max(1,max_corners)], out_n[count] (device).
// Two stages so that a caller can put them on different streams: score (max, candidates, raster order) and select
// (std::sort permutation + greedy NMS); both use the work area carved for (count, cand_cap, min_dist).
static int corners_args(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int count, int& min_dist, int cand_cap, void* work, size_t work_bytes,
                        CornerWorkView& wv) {
  if (f->w > 32767 || f->h > 32767)  // packed 16-bit coordinates; squared distances stay below 2^31
    return sfm_fail(ctx, SFMGPU_E_ARG, "corners: image larger than 32767 px");
  if (min_dist < 0) min_dist = -min_dist;  // the reference compares against (double)min_dist*min_dist (:295)
  if (min_dist > 30000) return sfm_fail(ctx, SFMGPU_E_ARG, "corners: min_dist too large");
  const size_t need = corner_work_carve(wv, work, f->w, f->h, count, cand_cap, min_dist);
  if (need > work_bytes) return sfm_fail(ctx, SFMGPU_E_ARG, "corners: work area too small (%zu < %zu)", work_bytes, need);
  return 0;
}

int sfm_corners_score_stage(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, double quality, int min_dist, int cand_cap,
                            void* work, size_t work_bytes) {
  CornerWorkView wv;
  SFM_TRY(corners_args(ctx, f, count, min_dist, cand_cap, work, work_bytes, wv));
  StageTimer st(ctx, 0);
  return sfm_corner_candidates_batch(ctx, f, first, count, quality, wv);
}

int sfm_corners_select_stage(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, int max_corners, double quality, int min_dist,
                             int cand_cap, void* work, size_t work_bytes, double2* out_xy, int* out_n) {
  CornerWorkView wv;
  SFM_TRY(corners_args(ctx, f, count, min_dist, cand_cap, work, work_bytes, wv));
  SFM_TRY(select_smem_config(ctx));
  StageTimer st(ctx, 1);
  if (ctx->select_mode == 1) {  // exact introsort emulation for every frame (tests / A-B timing)
    SFM_TRY(sfm_corner_raster_order(ctx, count, wv, quality, 0));
    if (wv.grid_per_frame)
      SFM_CUDA(ctx, cudaMemsetAsync(wv.grid, 0xFF, sizeof(unsigned) * wv.grid_per_frame * count, ctx->stream));
    SFM_LAUNCH(ctx, select_kernel, count, SEL_THREADS, sizeof(SelSmem), wv, f->w, max_corners, min_dist, 0, out_xy, out_n);
    return 0;
  }
  SFM_CUDA(ctx, cudaMemsetAsync(wv.wordoff, 0, sizeof(unsigned) * wv.words_per_frame * count, ctx->stream));  // the blocked-pixel map
  // tests: short codes make equal codes common (modes 12..34); small gathers make the sub-bucket walk common (modes 1000 + g)
  const int code_bits = (ctx->select_mode >= 12 && ctx->select_mode <= BK_CODE_BITS) ? ctx->select_mode : BK_CODE_BITS;
  const int gather_cap = ctx->select_mode >= 1000 ? ctx->select_mode - 1000 : BK_T;
  SFM_LAUNCH(ctx, bucket_select_kernel, count, BK_THREADS, sizeof(BucketSmem), wv, f->lvl[0], f->pitch[0], f->fstride[0], first, f->w, f->h,
             max_corners, min_dist, quality, code_bits, gather_cap, out_xy, out_n);
  // frames where a score tie was consumed (status 3): raster order, then the exact emulation.  Blocks of all other
  // frames return at once.
  SFM_TRY(sfm_corner_raster_order(ctx, count, wv, quality, 1));
  SFM_LAUNCH(ctx, select_kernel, count, SEL_THREADS, sizeof(SelSmem), wv, f->w, max_corners, min_dist, 3, out_xy, out_n);
  return 0;
}

int sfm_corners_batch(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, int max_corners, double quality,
                      int min_dist, int cand_cap, void* work, size_t work_bytes, double2* out_xy, int* out_n) {
  SFM_TRY(sfm_corners_score_stage(ctx, f, first, count, quality, min_dist, cand_cap, work, work_bytes));
  return sfm_corners_select_stage(ctx, f, first, count, max_corners, quality, min_dist, cand_cap, work, work_bytes, out_xy, out_n);
}

size_t sfm_corner_work_bytes_md(int w, int h, int nframes, int cand_cap, int min_dist) {
  CornerWorkView v;
  return corner_work_carve(v, nullptr, w, h, nframes, cand_cap, min_dist);
}

extern "C" int sfmgpu_select_set_mode(sfmgpu_ctx* ctx, int mode) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  if (mode != 0 && mode != 1 && !(mode >= 12 && mode <= BK_CODE_BITS) && !(mode >= 1000 + 64 && mode <= 1000 + BK_T))
    return sfm_fail(ctx, SFMGPU_E_ARG, "select_set_mode: mode %d not in {0, 1, 12..%d, %d..%d}", mode, BK_CODE_BITS, 1000 + 64, 1000 + BK_T);
  ctx->select_mode = mode;
  return 0;
}

extern "C" int sfmgpu_corners(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, int max_corners, double quality, int min_dist,
                              double* xy_out, int* n_out) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !xy_out || !n_out) return SFMGPU_E_ARG;
  if (frame < 0 || frame >= f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "corners: bad frame index");
  const int cap_out = max_corners < 1 ? 1 : max_corners;
  const int cand_cap = f->w * f->h;  // worst case (flat image: every pixel is a candidate)
  const size_t wb = sfm_corner_work_bytes_md(f->w, f->h, 1, cand_cap, min_dist < 0 ? -min_dist : min_dist);
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, wb));
  SFM_TRY(sfm_reserve(ctx, ctx->sel_work, (size_t)cap_out * sizeof(double2) + 256));
  double2* d_xy = (double2*)ctx->sel_work.p;
  int* d_n = (int*)((char*)ctx->sel_work.p + (size_t)cap_out * sizeof(double2));
  SFM_TRY(sfm_corners_batch(ctx, f, frame, 1, max_corners, quality, min_dist, cand_cap, ctx->cs_work.p, ctx->cs_work.cap, d_xy,
                            d_n));
  int n = 0;
  SFM_CUDA(ctx, cudaMemcpyAsync(&n, d_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n < 0) return sfm_fail(ctx, SFMGPU_E_CAPACITY, "corners: candidate capacity exceeded");
  *n_out = n;
  if (n > 0) {
    SFM_CUDA(ctx, cudaMemcpyAsync(xy_out, d_xy, (size_t)n * sizeof(double2), cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

// Device std::sort permutation of arbitrary non-negative keys (test / parity entry point).
int sfm_sort_perm(sfmgpu_ctx* ctx, const double* keys, int n, int32_t* perm) {
  if (n < 0) return sfm_fail(ctx, SFMGPU_E_ARG, "sort_perm: negative n");
  if (n == 0) return 0;
  for (int i = 0; i < n; i++)
    if (!(keys[i] >= 0.0)) return sfm_fail(ctx, SFMGPU_E_ARG, "sort_perm: keys must be non-negative, non-NaN (scores are)");
  CornerWorkView wv;
  const size_t wb = corner_work_carve(wv, nullptr, 32, 1, 1, n, 0);
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, wb));
  corner_work_carve(wv, ctx->cs_work.p, 32, 1, 1, n, 0);
  SFM_TRY(select_smem_config(ctx));
  std::vector<unsigned> iota(n);
  for (int i = 0; i < n; i++) iota[i] = (unsigned)i;
  const unsigned un = (unsigned)n;
  SFM_CUDA(ctx, cudaMemcpyAsync(wv.key, keys, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(wv.idx, iota.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(wv.ntotal, &un, 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_LAUNCH(ctx, select_kernel, 1, SEL_THREADS, sizeof(SelSmem), wv, 32, 0, 0, 1, (double2*)nullptr, (int*)nullptr);
  SFM_CUDA(ctx, cudaMemcpyAsync(perm, wv.idx, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int sfmgpu_sort_perm_desc(sfmgpu_ctx* ctx, const double* keys, int n, int32_t* perm) {
  SFM_ENTER(ctx);
  if (!ctx || (n > 0 && (!keys || !perm))) return SFMGPU_E_ARG;
  return sfm_sort_perm(ctx, keys, n, perm);
}
