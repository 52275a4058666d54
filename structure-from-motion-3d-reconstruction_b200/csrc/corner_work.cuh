// corner_work.cuh — per-batch work area shared by corner_score.cu and corner_select.cu.
#pragma once
#include <stddef.h>
#include <stdint.h>

struct CornerWorkView {
  unsigned long long* maxbits;  // [nframes] bit pattern of max u = 8*lmin
  unsigned* ncand;              // [nframes] entries appended to the provisional list by the fused pass (may exceed cand_cap)
  unsigned* nfinal;             // [nframes] candidates that reach the final threshold (may exceed cand_cap: overflow)
  int* exact_list;              // [nframes] != 0: the unordered list holds exactly the nfinal candidates (two-pass / rescued)
  int* rescue_list;             // [nframes] frames whose provisional list overflowed
  int* rescue_count;            // [1]
  unsigned* ntotal;             // [nframes] candidates counted by the bitmap scan
  int* status;                  // [nframes] 0 ok, 1 candidate capacity exceeded
  unsigned* bitmap;             // [nframes][h][wpr] one bit per pixel
  unsigned* wordoff;            // [nframes][h][wpr] exclusive prefix of popcounts
  unsigned* tmp_idx;            // [nframes][cand_cap] unordered list: pixel as y << 16 | x
  unsigned long long* tmp_key;  // [nframes][cand_cap] unordered list: score bits
  unsigned long long* key;      // [nframes][cand_cap] raster order, then sorted in place
  unsigned* idx;                // [nframes][cand_cap] pixel as y << 16 | x
  unsigned* lpos;               // [nframes][cand_cap] partition scratch of the emulation (aliases words)
  unsigned* rpos;               // [nframes][cand_cap]
  unsigned* grid;               // [nframes][grid_cells][2] accepted corners per min_dist cell (packed y<<16|x)
  unsigned long long* words;    // [nframes][cand_cap] bucket_select_kernel: order code << 30 | y << 15 | x in bucket order
  int wpr;
  size_t words_per_frame;
  int cand_cap;
  int gw, gh, cell;             // NMS grid geometry (cell = min_dist), 0 cells when min_dist < 2
  size_t grid_per_frame;        // uints per frame
};

// Carves the view out of `base` (may be nullptr to only compute the size).  Returns the bytes needed.
static inline size_t corner_work_carve(CornerWorkView& v, void* base, int w, int h, int nframes, int cand_cap,
                                       int min_dist = 0) {
  size_t off = 0;
  char* b = (char*)base;
  auto take = [&](size_t bytes) {
    void* p = b ? (void*)(b + off) : nullptr;
    off += (bytes + 255) / 256 * 256;
    return p;
  };
  cand_cap = (cand_cap + 1) & ~1;  // per-frame strides of the 8-byte arrays stay 16-byte aligned
  v.wpr = (w + 31) / 32;
  v.words_per_frame = (size_t)v.wpr * h;
  v.cand_cap = cand_cap;
  v.cell = min_dist >= 2 ? min_dist : 0;
  v.gw = v.cell ? (w + v.cell - 1) / v.cell : 0;
  v.gh = v.cell ? (h + v.cell - 1) / v.cell : 0;
  v.grid_per_frame = (size_t)v.gw * v.gh * 2;
  v.maxbits = (unsigned long long*)take(sizeof(unsigned long long) * nframes);
  v.ncand = (unsigned*)take(sizeof(unsigned) * nframes);
  v.nfinal = (unsigned*)take(sizeof(unsigned) * nframes);
  v.exact_list = (int*)take(sizeof(int) * nframes);
  v.rescue_list = (int*)take(sizeof(int) * nframes);
  v.rescue_count = (int*)take(sizeof(int));
  v.ntotal = (unsigned*)take(sizeof(unsigned) * nframes);
  v.status = (int*)take(sizeof(int) * nframes);
  v.bitmap = (unsigned*)take(sizeof(unsigned) * v.words_per_frame * nframes);
  v.wordoff = (unsigned*)take(sizeof(unsigned) * v.words_per_frame * nframes);
  v.tmp_idx = (unsigned*)take(sizeof(unsigned) * (size_t)cand_cap * nframes);
  v.tmp_key = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)cand_cap * nframes);
  v.key = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)cand_cap * nframes);
  v.idx = (unsigned*)take(sizeof(unsigned) * (size_t)cand_cap * nframes);
  v.grid = (unsigned*)take(sizeof(unsigned) * (v.grid_per_frame ? v.grid_per_frame : 1) * nframes);
  v.words = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)cand_cap * nframes);
  v.lpos = (unsigned*)v.words;  // the emulation redoes a frame only after the bucket selection is done with every frame
  v.rpos = v.lpos ? v.lpos + (size_t)cand_cap * nframes : nullptr;
  return off + 256;
}
