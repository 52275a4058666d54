// codec.cu — packed frame input: the lossless tile codec of include/sfmgpu.h (format: DESIGN.md §2, numpy reference:
// tests/frame_codec.py), encoded and decoded on the device.
//
// A tile is TILE x TILE pixels of level 0 (edge tiles partial).  Its planar residuals (left + up - upleft, pixels outside the
// tile = 0, mod 256, zig-zagged) are Rice coded in runs of 32 with a k per run, as two streams: the remainders (k bits each,
// so every remainder's position follows from a scan over the runs' k) and the unary quotients (the q_j follow from the
// positions of the zero bits: popc + a block scan).  Decoding is therefore data parallel: no bit parser walks the record.
// The inverse predictor is a 2D inclusive prefix sum mod 256 (row scans, then column scans, by warp shuffles).
#include <string.h>

#include <vector>

#include "common.cuh"

namespace {

constexpr uint32_t PK_MAGIC = 0x504B4653u;  // "SFKP"
constexpr uint32_t PK_VERSION = 1;
constexpr int TILE = 64, RUN = 32, NT = 256;
constexpr int MAXV = TILE * TILE;             // values of a full tile
constexpr int MAXRUNS = MAXV / RUN;           // 128
constexpr int VPT = MAXV / NT;                // encoder: consecutive values per thread (16)
constexpr int RAW_MAX_WORDS = 1 + MAXV / 4;   // the longest record: a raw full tile
constexpr size_t HDR_BYTES = 32;
constexpr size_t STAGE_LIMIT = 256u << 20;    // bytes of blob staged per decode / encode batch (one frame at least)

struct PkHeader {
  uint32_t magic, version, w, h, n, tile, r0, r1;
};

__host__ __device__ inline int raw_words(int n) { return 1 + (n + 3) / 4; }

struct TileGeo {
  int x0, y0, tw, th, n, nruns, kw;
};
__device__ inline TileGeo tile_geo(int t, int w, int h, int tiles_x) {
  TileGeo g;
  g.x0 = (t % tiles_x) * TILE;
  g.y0 = (t / tiles_x) * TILE;
  g.tw = min(TILE, w - g.x0);
  g.th = min(TILE, h - g.y0);
  g.n = g.tw * g.th;
  g.nruns = (g.n + RUN - 1) / RUN;
  g.kw = (g.nruns + 7) / 8;
  return g;
}

// Exclusive block scan (NT threads); *total = the sum of all v.  sw: NT / 32 + 1 slots of shared memory.
template <typename T>
__device__ T block_exscan(T v, T* sw, T* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  T x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(~0u, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sw[wid] = x;
  __syncthreads();
  if (threadIdx.x == 0) {
    T s = 0;
    for (int i = 0; i < NT / 32; i++) {
      const T t = sw[i];
      sw[i] = s;
      s += t;
    }
    sw[NT / 32] = s;
  }
  __syncthreads();
  const T r = sw[wid] + x - v;
  *total = sw[NT / 32];
  __syncthreads();
  return r;
}

__device__ __forceinline__ uint32_t zigzag(int d) {  // d: residual mod 256 read as int8
  const int s = (int)(int8_t)(uint8_t)d;
  return s >= 0 ? 2u * s : (uint32_t)(-2 * s - 1);
}
__device__ __forceinline__ uint32_t unzigzag(uint32_t u) { return (u & 1) ? (uint32_t)(-(int)((u + 1) >> 1)) : u >> 1; }

// ---- encoder --------------------------------------------------------------------------------------------------------
// What both encoder passes know about a tile after tile_analyse: values u (padded to whole runs), k per run and its exclusive
// prefix, unary bits, record length in words and whether the record is raw.
struct EncSmem {
  uint8_t px[MAXV];
  uint8_t u[MAXV];
  uint8_t k[MAXRUNS];
  int kpre[MAXRUNS];
  int sw[NT / 32 + 1];
  uint32_t rec[RAW_MAX_WORDS + 1];
};
struct TileSize {
  int sumk, U, words, raw;
};

__device__ TileSize tile_analyse(EncSmem& s, const TileGeo& g, const uint8_t* __restrict__ src, int pitch) {
  for (int i = threadIdx.x; i < g.n; i += NT) {
    const int y = i / g.tw, x = i - y * g.tw;
    s.px[y * TILE + x] = src[(size_t)y * pitch + x];
  }
  __syncthreads();
  for (int j = threadIdx.x; j < g.nruns * RUN; j += NT) {
    uint32_t u = 0;
    if (j < g.n) {
      const int y = j / g.tw, x = j - y * g.tw;
      const int p = s.px[y * TILE + x];
      const int l = x > 0 ? s.px[y * TILE + x - 1] : 0;
      const int up = y > 0 ? s.px[(y - 1) * TILE + x] : 0;
      const int ul = (x > 0 && y > 0) ? s.px[(y - 1) * TILE + x - 1] : 0;
      u = zigzag((p - l - up + ul) & 255);
    }
    s.u[j] = (uint8_t)u;
  }
  __syncthreads();
  int k = 0, ub = 0;
  if ((int)threadIdx.x < g.nruns) {
    int q[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < RUN; i++) {
      const int v = s.u[threadIdx.x * RUN + i];
#pragma unroll
      for (int b = 0; b < 9; b++) q[b] += v >> b;
    }
    int best = q[0] + RUN;
#pragma unroll
    for (int b = 1; b < 9; b++)
      if (q[b] + RUN * (1 + b) < best) {  // strict: the smallest k wins a tie
        best = q[b] + RUN * (1 + b);
        k = b;
      }
    ub = best - RUN * k;  // q_sum + RUN terminators
    s.k[threadIdx.x] = (uint8_t)k;
  }
  TileSize ts;
  const int kp = block_exscan(k, s.sw, &ts.sumk);
  if ((int)threadIdx.x < g.nruns) s.kpre[threadIdx.x] = kp;
  block_exscan(ub, s.sw, &ts.U);
  const int coded = 1 + g.kw + ts.sumk + (ts.U + 31) / 32;
  ts.raw = coded >= raw_words(g.n);
  ts.words = ts.raw ? raw_words(g.n) : coded;
  return ts;
}

// Pass 1: record length (words) of every tile.  grid (ntiles, frames).
__global__ void __launch_bounds__(NT) pk_size_kernel(const uint8_t* __restrict__ lvl0, int pitch, size_t fstride, int first, int w, int h,
                                                     int tiles_x, int ntiles, int* __restrict__ words) {
  __shared__ EncSmem s;
  const TileGeo g = tile_geo(blockIdx.x, w, h, tiles_x);
  const uint8_t* src = lvl0 + (size_t)(first + blockIdx.y) * fstride + (size_t)g.y0 * pitch + g.x0;
  const TileSize ts = tile_analyse(s, g, src, pitch);
  if (threadIdx.x == 0) words[(size_t)blockIdx.y * ntiles + blockIdx.x] = ts.words;
}

// Per frame: tile table (byte offsets from the frame start) and frame size.  grid (frames).
__global__ void __launch_bounds__(NT) pk_tile_scan_kernel(const int* __restrict__ words, int ntiles, uint32_t* __restrict__ toff,
                                                          unsigned long long* __restrict__ fsize) {
  __shared__ uint32_t sw[NT / 32 + 1];
  const int* wd = words + (size_t)blockIdx.x * ntiles;
  uint32_t* to = toff + (size_t)blockIdx.x * (ntiles + 1);
  uint32_t carry = 4u * (ntiles + 1);
  for (int t0 = 0; t0 < ntiles; t0 += NT) {
    const int t = t0 + threadIdx.x;
    const uint32_t b = t < ntiles ? 4u * wd[t] : 0u;
    uint32_t tot;
    const uint32_t ex = block_exscan(b, sw, &tot);
    if (t < ntiles) to[t] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) {
    to[ntiles] = carry;
    fsize[blockIdx.x] = carry;
  }
}

// Frame offset table: fo[0] = the header and table bytes, fo[k+1] = fo[k] + size of frame k.  One block.
__global__ void __launch_bounds__(NT) pk_frame_scan_kernel(const unsigned long long* __restrict__ fsize, int n,
                                                           unsigned long long* __restrict__ fo) {
  __shared__ unsigned long long sw[NT / 32 + 1];
  unsigned long long carry = HDR_BYTES + 8ull * (n + 1);
  if (threadIdx.x == 0) fo[0] = carry;
  for (int k0 = 0; k0 < n; k0 += NT) {
    const int k = k0 + threadIdx.x;
    unsigned long long tot;
    const unsigned long long ex = block_exscan(k < n ? fsize[k] : 0ull, sw, &tot);
    if (k < n) fo[k + 1] = carry + ex + fsize[k];
    carry += tot;
  }
}

__device__ __forceinline__ void or_bits(uint32_t* rec, int bp, uint32_t v, int nb) {  // v < 2^nb, nb <= 8
  if (nb == 0) return;
  atomicOr(&rec[bp >> 5], v << (bp & 31));
  if ((bp & 31) + nb > 32) atomicOr(&rec[(bp >> 5) + 1], v >> (32 - (bp & 31)));
}

// Pass 2: write the tile records and tile tables of frames [first, first + gridDim.y) into out (frame k at fo[k] - base).
__global__ void __launch_bounds__(NT) pk_write_kernel(const uint8_t* __restrict__ lvl0, int pitch, size_t fstride, int first, int w, int h,
                                                      int tiles_x, int ntiles, const uint32_t* __restrict__ toff,
                                                      const unsigned long long* __restrict__ fo, unsigned long long base,
                                                      uint8_t* __restrict__ out) {
  __shared__ EncSmem s;
  const int t = blockIdx.x, fk = blockIdx.y;
  const TileGeo g = tile_geo(t, w, h, tiles_x);
  const uint8_t* src = lvl0 + (size_t)(first + fk) * fstride + (size_t)g.y0 * pitch + g.x0;
  const TileSize ts = tile_analyse(s, g, src, pitch);
  for (int i = threadIdx.x; i < ts.words; i += NT) s.rec[i] = 0;
  __syncthreads();
  if (ts.raw) {
    if (threadIdx.x == 0) s.rec[0] = 1;
    uint8_t* rb = reinterpret_cast<uint8_t*>(s.rec + 1);
    for (int i = threadIdx.x; i < g.n; i += NT) {
      const int y = i / g.tw, x = i - y * g.tw;
      rb[i] = s.px[y * TILE + x];
    }
  } else {
    if (threadIdx.x == 0) s.rec[0] = (uint32_t)ts.U << 1;
    if ((int)threadIdx.x < g.nruns) atomicOr(&s.rec[1 + threadIdx.x / 8], (uint32_t)s.k[threadIdx.x] << (4 * (threadIdx.x % 8)));
    const int rem0 = 32 * (1 + g.kw), una0 = 32 * (1 + g.kw + ts.sumk);
    const int j0 = threadIdx.x * VPT, nc = g.nruns * RUN;
    int qs = 0;
    for (int j = j0; j < j0 + VPT && j < nc; j++) qs += (s.u[j] >> s.k[j / RUN]) + 1;
    int tot;
    int pos = una0 + block_exscan(qs, s.sw, &tot);
    for (int j = j0; j < j0 + VPT && j < nc; j++) {
      const int r = j / RUN, k = s.k[r];
      const uint32_t u = s.u[j];
      or_bits(s.rec, rem0 + 32 * s.kpre[r] + (j - r * RUN) * k, u & ((1u << k) - 1u), k);
      int a = pos, b = pos + (int)(u >> k);  // q one-bits, then the terminating zero
      while (a < b) {
        const int sh = a & 31, cnt = min(32 - sh, b - a);
        atomicOr(&s.rec[a >> 5], (cnt == 32 ? ~0u : ((1u << cnt) - 1u)) << sh);
        a += cnt;
      }
      pos = b + 1;
    }
  }
  __syncthreads();
  uint8_t* fr = out + (fo[fk] - base);
  const uint32_t* to = toff + (size_t)fk * (ntiles + 1);
  uint32_t* dst = reinterpret_cast<uint32_t*>(fr + to[t]);
  for (int i = threadIdx.x; i < ts.words; i += NT) dst[i] = s.rec[i];
  if (threadIdx.x == 0) reinterpret_cast<uint32_t*>(fr)[t] = to[t];
  if (threadIdx.x == 0 && t == ntiles - 1) reinterpret_cast<uint32_t*>(fr)[ntiles] = to[ntiles];
}

// ---- decoder: one block per tile --------------------------------------------------------------------------------------
// stage holds blob bytes from absolute offset `base` on; fo[k] = absolute offset of frame k of the launch (the host has checked
// fo against the blob, and that every frame holds its tile table).  A tile whose record does not decode sets *bad and writes
// nothing.  TABLE = false: frames [first, first + gridDim.y) of one batch, grid (ntiles, frames).  TABLE = true: frames of any
// sizes, frame k of the launch into frames[k] (lvl0 ... ntiles are taken from there, fstride and first are 0); grid (the largest
// tile count, frames), and blocks past their frame's tile count return at once.
template <bool TABLE>
__global__ void __launch_bounds__(NT) pk_decode_kernel(const uint8_t* __restrict__ stage, const unsigned long long* __restrict__ fo,
                                                       unsigned long long base, uint8_t* __restrict__ lvl0, int pitch, size_t fstride,
                                                       int first, int w, int h, int tiles_x, int ntiles, int* __restrict__ bad,
                                                       const PkDst* __restrict__ frames) {
  if constexpr (TABLE) {
    const PkDst d = frames[blockIdx.y];
    if ((int)blockIdx.x >= d.ntiles) return;
    lvl0 = d.lvl0;
    pitch = d.pitch;
    w = d.w;
    h = d.h;
    tiles_x = d.tiles_x;
    ntiles = d.ntiles;
  }
  __shared__ uint32_t rec[RAW_MAX_WORDS + 1];
  __shared__ uint32_t tile[TILE][TILE + 1];
  __shared__ uint16_t zpos[MAXV];
  __shared__ int kpre[MAXRUNS];
  __shared__ uint8_t ks[MAXRUNS];
  __shared__ int sw[NT / 32 + 1];
  __shared__ uint32_t s_start, s_len;
  const int t = blockIdx.x, fk = blockIdx.y, tid = threadIdx.x;
  const TileGeo g = tile_geo(t, w, h, tiles_x);
  const uint8_t* fr = stage + (fo[fk] - base);
  int err = 0;
  if (tid == 0) {
    const unsigned long long fbytes = fo[fk + 1] - fo[fk];
    const uint32_t* to = reinterpret_cast<const uint32_t*>(fr);
    const uint32_t a = to[t], b = to[t + 1];
    const bool ok = a >= 4u * (ntiles + 1) && a <= b && b <= fbytes && ((a | b) & 3u) == 0 && b - a >= 4 &&
                    (b - a) / 4 <= (uint32_t)raw_words(g.n);
    s_start = a / 4;
    s_len = ok ? (b - a) / 4 : 0;
  }
  __syncthreads();
  const int len = (int)s_len;
  if (len == 0) {
    if (tid == 0) atomicOr(bad, 1);
    return;
  }
  const uint32_t* rsrc = reinterpret_cast<const uint32_t*>(fr) + s_start;
  for (int i = tid; i < len; i += NT) rec[i] = rsrc[i];
  __syncthreads();
  const uint32_t hdr = rec[0];
  if (hdr == 1) {  // raw tile
    err = len != raw_words(g.n);
    const uint8_t* rb = reinterpret_cast<const uint8_t*>(rec + 1);
    if (!err)
      for (int i = tid; i < g.n; i += NT) {
        const int y = i / g.tw;
        tile[y][i - y * g.tw] = rb[i];
      }
    if (__syncthreads_or(err)) {
      if (tid == 0) atomicOr(bad, 1);
      return;
    }
  } else {
    const uint32_t U = hdr >> 1;
    int k = 0;
    if (tid < g.nruns) {
      k = (rec[1 + tid / 8] >> (4 * (tid % 8))) & 15;
      ks[tid] = (uint8_t)k;
      err |= k > 8;
    }
    int sumk;
    const int kp = block_exscan(k, sw, &sumk);
    if (tid < g.nruns) kpre[tid] = kp;
    const int una0 = 1 + g.kw + sumk;
    const long long nuw = ((long long)U + 31) / 32;
    err |= (hdr & 1) || U == 0 || (long long)una0 + nuw != len;
    if (__syncthreads_or(err)) {
      if (tid == 0) atomicOr(bad, 1);
      return;
    }
    // zero bits of the unary stream: word tid + NT * p of page p per thread (nw <= len - 2 < 4 * NT), per-page block scans of
    // the counts, then the position of every zero
    const int nw = (int)nuw, nc = g.nruns * RUN, npage = (nw + NT - 1) / NT;
    int ztot = 0;
    for (int pg = 0; pg < npage; pg++) {
      const int wi = pg * NT + tid;
      uint32_t z = 0;
      if (wi < nw) {
        z = ~rec[una0 + wi];
        if (wi == nw - 1 && (U & 31)) z &= (1u << (U & 31)) - 1u;
      }
      int tot;
      int rank = ztot + block_exscan(__popc(z), sw, &tot);
      ztot += tot;
      if (ztot > nc) z = 0;  // more terminators than values: reported below, nothing written past zpos
      while (z) {
        const int bit = __ffs(z) - 1;
        z &= z - 1;
        zpos[rank++] = (uint16_t)(wi * 32 + bit);
      }
    }
    const int last_bit = (int)((U - 1) & 31);
    err = ztot != nc || ((rec[una0 + (int)((U - 1) >> 5)] >> last_bit) & 1u);
    if (__syncthreads_or(err)) {
      if (tid == 0) atomicOr(bad, 1);
      return;
    }
    // values j = tid + NT * i: a warp takes one run at a time (uniform k), neighbouring lanes read neighbouring words; q from
    // the zero positions, the remainder from its run's slot, then the residual
    for (int j = tid; j < nc; j += NT) {
      const int q = (int)zpos[j] - (j > 0 ? (int)zpos[j - 1] : -1) - 1;
      const int r = j / RUN, kk = ks[r];
      uint32_t rem = 0;
      if (kk) {
        const int bp = 32 * (1 + g.kw + kpre[r]) + (j - r * RUN) * kk;
        uint64_t two = rec[bp >> 5];
        if ((bp & 31) + kk > 32) two |= (uint64_t)rec[(bp >> 5) + 1] << 32;
        rem = (uint32_t)(two >> (bp & 31)) & ((1u << kk) - 1u);
      }
      const uint32_t u = ((uint32_t)q << kk) | rem;
      err |= q > (255 >> kk);
      if (j < g.n) {
        const int y = j / g.tw;
        tile[y][j - y * g.tw] = unzigzag(u) & 255u;
      }
    }
    if (__syncthreads_or(err)) {
      if (tid == 0) atomicOr(bad, 1);
      return;
    }
    // 2D inclusive prefix sum mod 256: rows, then columns; lane l holds entries 2l and 2l+1 (entries beyond the tile's width /
    // height only feed entries after them, which are not written)
    const int lane = tid & 31, wid = tid >> 5;
    for (int y = wid; y < g.th; y += NT / 32) {
      const uint32_t a = tile[y][2 * lane], b = tile[y][2 * lane + 1];
      uint32_t x = a + b;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(~0u, x, o);
        if (lane >= o) x += v;
      }
      tile[y][2 * lane] = x - b;
      tile[y][2 * lane + 1] = x;
    }
    __syncthreads();
    for (int xc = wid; xc < g.tw; xc += NT / 32) {
      const uint32_t a = tile[2 * lane][xc], b = tile[2 * lane + 1][xc];
      uint32_t x = a + b;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(~0u, x, o);
        if (lane >= o) x += v;
      }
      tile[2 * lane][xc] = x - b;
      tile[2 * lane + 1][xc] = x;
    }
    __syncthreads();
  }
  // exactly the w bytes per row that a raw upload writes: the tile's columns, 4 at a time where they fit
  uint8_t* dst = lvl0 + (size_t)(first + fk) * fstride + (size_t)g.y0 * pitch + g.x0;
  const int gw = (g.tw + 3) / 4;
  for (int i = tid; i < g.th * gw; i += NT) {
    const int y = i / gw, x = 4 * (i - y * gw);
    uint8_t* d = dst + (size_t)y * pitch + x;
    if (x + 4 <= g.tw) {
      *reinterpret_cast<uint32_t*>(d) = (tile[y][x] & 255u) | (tile[y][x + 1] & 255u) << 8 | (tile[y][x + 2] & 255u) << 16 |
                                        (tile[y][x + 3] & 255u) << 24;
    } else {
      for (int c = x; c < g.tw; c++) d[c - x] = (uint8_t)tile[y][c];
    }
  }
}

int tiles_x_of(int w) { return (w + TILE - 1) / TILE; }
int ntiles_of(int w, int h) { return tiles_x_of(w) * ((h + TILE - 1) / TILE); }

size_t frame_bound(int w, int h) {
  size_t b = 4 * ((size_t)ntiles_of(w, h) + 1);
  for (int y = 0; y < h; y += TILE)
    for (int x = 0; x < w; x += TILE) b += 4 * (size_t)raw_words((w - x < TILE ? w - x : TILE) * (h - y < TILE ? h - y : TILE));
  return b;
}

// Frames of fo (count + 1 offsets) cut into batches [cut[i], cut[i+1]) of at most STAGE_LIMIT bytes (one frame at least);
// *most = the largest batch.
std::vector<int> stage_batches(const std::vector<uint64_t>& fo, size_t* most) {
  const int count = (int)fo.size() - 1;
  std::vector<int> cut{0};
  for (int k = 1; k <= count; k++)
    if (k == count || fo[k + 1] - fo[cut.back()] > STAGE_LIMIT) {
      if (fo[k] - fo[cut.back()] > *most) *most = fo[k] - fo[cut.back()];
      cut.push_back(k);
    }
  return cut;
}

uint64_t rd64(const uint8_t* p) {
  uint64_t v;
  memcpy(&v, p, 8);
  return v;
}

}  // namespace

// Host-side checks of a blob against f and the frame range [blob_first, blob_first + count); fo receives the absolute offsets
// of frames blob_first .. blob_first + count.
int sfm_pk_check(sfmgpu_ctx* ctx, const sfmgpu_frames* f, const uint8_t* blob, size_t blob_bytes, int blob_first, int count,
                 std::vector<uint64_t>& fo, const char* who) {
  if (!blob) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: null blob", who);
  if (blob_bytes < HDR_BYTES) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: blob of %zu bytes has no header", who, blob_bytes);
  PkHeader hd;
  memcpy(&hd, blob, sizeof hd);
  if (hd.magic != PK_MAGIC) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: bad magic 0x%08x (not a packed frame blob)", who, hd.magic);
  if (hd.version != PK_VERSION) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: blob version %u, this library reads %u", who, hd.version, PK_VERSION);
  if (hd.tile != (uint32_t)TILE) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: tile size %u, this library reads %d", who, hd.tile, TILE);
  if (hd.w != (uint32_t)f->w || hd.h != (uint32_t)f->h)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: blob frames are %ux%u, the batch holds %dx%d", who, hd.w, hd.h, f->w, f->h);
  const uint64_t table_end = HDR_BYTES + 8ull * ((uint64_t)hd.n + 1);
  if (table_end > blob_bytes) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: blob truncated inside its frame table", who);
  if (blob_first < 0 || count < 0 || (uint64_t)blob_first + (uint64_t)count > hd.n)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: frames [%d,%lld) outside the blob's %u", who, blob_first, (long long)blob_first + count, hd.n);
  const uint64_t tbl = 4ull * ((uint64_t)ntiles_of(f->w, f->h) + 1);
  fo.resize((size_t)count + 1);
  for (int k = 0; k <= count; k++) fo[k] = rd64(blob + HDR_BYTES + 8 * ((size_t)blob_first + k));
  if (rd64(blob + HDR_BYTES) != table_end) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: first frame offset is not the table end", who);
  for (int k = 0; k < count; k++)
    if (fo[k] < table_end || (fo[k] & 3) || fo[k + 1] < fo[k] || fo[k + 1] - fo[k] < tbl || ((fo[k + 1] - fo[k]) & 3))
      return sfm_fail(ctx, SFMGPU_E_ARG, "%s: frame offsets of blob frame %d are not monotonic / aligned / large enough", who,
                      blob_first + k);
  if (fo[count] > blob_bytes)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: blob truncated: frame data ends at %llu, the blob has %zu bytes", who,
                    (unsigned long long)fo[count], blob_bytes);
  return 0;
}

// Queue the decode of `count` frames into frames [first, first + count) of f on ctx->stream.  stage holds blob bytes from
// absolute offset base on; d_fo the count + 1 absolute frame offsets.
int sfm_pk_decode(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* stage, const unsigned long long* d_fo,
                  unsigned long long base, int* d_bad) {
  StageTimer st(ctx, 6);
  const int nt = ntiles_of(f->w, f->h);
  for (int k = 0; k < count; k += 65535) {
    const int c = count - k < 65535 ? count - k : 65535;
    SFM_LAUNCH(ctx, pk_decode_kernel<false>, dim3(nt, c), NT, 0, stage, d_fo + k, base, f->lvl[0], f->pitch[0], f->fstride[0], first + k,
               f->w, f->h, tiles_x_of(f->w), nt, d_bad, (const PkDst*)nullptr);
  }
  return 0;
}

// Decode of `count` frames of any sizes on ctx->stream: frame k (records staged from offset 0 on, d_fo its count + 1 offsets)
// into d_dst[k]; max_tiles = the largest tile count of the entries.
int sfm_pk_decode_table(sfmgpu_ctx* ctx, const PkDst* d_dst, int count, int max_tiles, const uint8_t* stage,
                        const unsigned long long* d_fo, int* d_bad) {
  StageTimer st(ctx, 6);
  if (count > 0)
    SFM_LAUNCH(ctx, pk_decode_kernel<true>, dim3(max_tiles, count), NT, 0, stage, d_fo, 0ull, (uint8_t*)nullptr, 0, (size_t)0, 0, 0, 0, 0,
               0, d_bad, d_dst);
  return 0;
}

PkDst sfm_pk_dst(const sfmgpu_frames* f, int frame) {
  return {f->lvl[0] + (size_t)frame * f->fstride[0], f->pitch[0], f->w, f->h, tiles_x_of(f->w), ntiles_of(f->w, f->h)};
}

// The largest frame record a blob of w x h frames can hold (every tile raw).
size_t sfm_pk_frame_bound(int w, int h) { return frame_bound(w, h); }

// Largest staged byte range of frames [a, b) chunks: frames of fo (relative indices) split at `chunk` frames.
size_t sfm_pk_max_chunk_bytes(const std::vector<uint64_t>& fo, int chunk) {
  size_t m = 0;
  const int n = (int)fo.size() - 1;
  for (int a = 0; a < n; a += chunk) {
    const int b = a + chunk < n ? a + chunk : n;
    if (fo[b] - fo[a] > m) m = fo[b] - fo[a];
  }
  return m;
}

// Before the first chunk of a packed call (sized before any work is queued): nstage staging buffers of stage_bytes, the device
// copy of the frame offsets fo (blob frames blob_first ..), the decode flag cleared; on ctx->stream.
int sfm_pk_prepare(sfmgpu_ctx* ctx, const uint8_t* blob, int blob_first, const std::vector<uint64_t>& fo, size_t stage_bytes, int nstage) {
  for (int s = 0; s < nstage; s++) SFM_TRY(sfm_reserve(ctx, ctx->pk_stage[s], stage_bytes));
  SFM_TRY(sfm_reserve(ctx, ctx->pk_fo, 8 * fo.size()));
  SFM_TRY(sfm_reserve(ctx, ctx->pk_flag, sizeof(int)));
  SFM_CUDA(ctx, cudaMemsetAsync(ctx->pk_flag.p, 0, sizeof(int), ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(ctx->pk_fo.p, blob + HDR_BYTES + 8 * (size_t)blob_first, 8 * fo.size(), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int sfm_pk_read_flag(sfmgpu_ctx* ctx, const char* who) {
  SFM_TRY(sfm_pinned(ctx, sizeof(int)));
  SFM_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, ctx->pk_flag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (*(int*)ctx->pinned) return sfm_fail(ctx, SFMGPU_E_ARG, "%s: a tile record of the blob does not decode (its tile was not written)", who);
  return 0;
}

extern "C" {

int sfmgpu_pack_bound(int w, int h, int nframes, size_t* bytes) {
  if (w <= 0 || h <= 0 || nframes < 0 || !bytes) return SFMGPU_E_ARG;
  *bytes = HDR_BYTES + 8 * ((size_t)nframes + 1) + (size_t)nframes * frame_bound(w, h);
  return 0;
}

int sfmgpu_frames_pack(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, uint8_t* out, size_t cap, size_t* bytes) {
  SFM_ENTER(ctx);
  if (!ctx || !f || !bytes) return SFMGPU_E_ARG;
  if (first < 0 || count < 0 || first + count > f->n)
    return sfm_fail(ctx, SFMGPU_E_ARG, "frames_pack: frame range [%d,%d) outside [0,%d)", first, first + count, f->n);
  const int nt = ntiles_of(f->w, f->h), tx = tiles_x_of(f->w);
  const size_t n = (size_t)count;
  // scratch: record words [n][nt], tile tables [n][nt+1], frame sizes [n], frame offsets [n+1]
  const size_t o_toff = (n * nt * 4 + 15) & ~(size_t)15, o_fs = (o_toff + n * (nt + 1) * 4 + 15) & ~(size_t)15, o_fo = o_fs + n * 8;
  SFM_TRY(sfm_reserve(ctx, ctx->pk_tmp, o_fo + (n + 1) * 8));
  int* d_words = (int*)ctx->pk_tmp.p;
  uint32_t* d_toff = (uint32_t*)((uint8_t*)ctx->pk_tmp.p + o_toff);
  unsigned long long* d_fs = (unsigned long long*)((uint8_t*)ctx->pk_tmp.p + o_fs);
  unsigned long long* d_fo = (unsigned long long*)((uint8_t*)ctx->pk_tmp.p + o_fo);
  for (int k = 0; k < count; k += 65535) {
    const int c = count - k < 65535 ? count - k : 65535;
    SFM_LAUNCH(ctx, pk_size_kernel, dim3(nt, c), NT, 0, f->lvl[0], f->pitch[0], f->fstride[0], first + k, f->w, f->h, tx, nt,
               d_words + (size_t)k * nt);
  }
  if (count > 0) SFM_LAUNCH(ctx, pk_tile_scan_kernel, count, NT, 0, d_words, nt, d_toff, d_fs);
  SFM_LAUNCH(ctx, pk_frame_scan_kernel, 1, NT, 0, d_fs, count, d_fo);
  std::vector<uint64_t> fo(n + 1);
  SFM_CUDA(ctx, cudaMemcpyAsync(fo.data(), d_fo, (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *bytes = fo[n];
  if (!out || cap < fo[n])
    return sfm_fail(ctx, SFMGPU_E_CAPACITY, "frames_pack: the blob needs %llu bytes, the buffer has %zu", (unsigned long long)fo[n], cap);
  const PkHeader hd = {PK_MAGIC, PK_VERSION, (uint32_t)f->w, (uint32_t)f->h, (uint32_t)count, (uint32_t)TILE, 0, 0};
  memcpy(out, &hd, sizeof hd);
  memcpy(out + HDR_BYTES, fo.data(), (n + 1) * 8);
  // records in batches of at most STAGE_LIMIT bytes (one frame at least), each written to device scratch and copied out
  size_t most = 0;
  const std::vector<int> cut = stage_batches(fo, &most);
  if (count > 0) SFM_TRY(sfm_reserve(ctx, ctx->pk_enc, most));
  for (size_t i = 0; i + 1 < cut.size(); i++) {
    const int a = cut[i], b = cut[i + 1];
    for (int k = a; k < b; k += 65535) {
      const int c = b - k < 65535 ? b - k : 65535;
      SFM_LAUNCH(ctx, pk_write_kernel, dim3(nt, c), NT, 0, f->lvl[0], f->pitch[0], f->fstride[0], first + k, f->w, f->h, tx, nt,
                 d_toff + (size_t)k * (nt + 1), d_fo + k, (unsigned long long)fo[a], (uint8_t*)ctx->pk_enc.p);
    }
    SFM_CUDA(ctx, cudaMemcpyAsync(out + fo[a], ctx->pk_enc.p, fo[b] - fo[a], cudaMemcpyDeviceToHost, ctx->stream));
  }
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

int sfmgpu_frames_upload_packed(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, const uint8_t* blob, size_t blob_bytes, int blob_first,
                                int count) {
  SFM_ENTER(ctx);
  if (!ctx || !f) return SFMGPU_E_ARG;
  if (first < 0 || count < 0 || first + count > f->n)
    return sfm_fail(ctx, SFMGPU_E_ARG, "frames_upload_packed: frame range [%d,%d) outside [0,%d)", first, first + count, f->n);
  std::vector<uint64_t> fo;
  SFM_TRY(sfm_pk_check(ctx, f, blob, blob_bytes, blob_first, count, fo, "frames_upload_packed"));
  if (count == 0) return 0;
  size_t most = 0;
  const std::vector<int> cut = stage_batches(fo, &most);
  SFM_TRY(sfm_pk_prepare(ctx, blob, blob_first, fo, most, 1));
  const unsigned long long* d_fo = (const unsigned long long*)ctx->pk_fo.p;
  for (size_t i = 0; i + 1 < cut.size(); i++) {  // stream order: the next chunk's copy follows this chunk's decode
    const int a = cut[i], b = cut[i + 1];
    SFM_CUDA(ctx, cudaMemcpyAsync(ctx->pk_stage[0].p, blob + fo[a], fo[b] - fo[a], cudaMemcpyHostToDevice, ctx->stream));
    SFM_TRY(sfm_pk_decode(ctx, f, first + a, b - a, (const uint8_t*)ctx->pk_stage[0].p, d_fo + a, fo[a], (int*)ctx->pk_flag.p));
  }
  return sfm_pk_read_flag(ctx, "frames_upload_packed");
}

}  // extern "C"
