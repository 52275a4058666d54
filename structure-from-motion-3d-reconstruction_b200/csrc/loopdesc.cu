// loopdesc.cu — loop-closure descriptor and candidate search (SURVEY.md §8f-3).
//
// Replaces (reference cpp/src/templering_sfm.cpp) global_desc_32 :1100-1122 (repeated downsample2 until both sides
// are <= 32, nearest sampling to 32x32, mean removal, L2 normalisation), dot_desc :1124-1129 and the candidate loop
// :1823-1831 (first strictly larger score wins, best_score starts at 0).
//
// Bit-exact: the box filter is integer; the mean is a sum of integers (exact in double in any order); the squared
// norm IS order dependent, so one thread accumulates it in raster order like the reference; the dot products are
// sequential float multiply-add pairs WITHOUT contraction, each in ascending i (desc_search_kernel below).
//
// Descriptors can stay on the device (sfmgpu_descs: a bank of slots filled by global_desc_32 or uploads) and be searched
// for many queries in one launch; the single-query host-array entry point runs through the same kernel.
#include <string.h>

#include "common.cuh"

struct sfmgpu_descs {
  int capacity = 0;
  float* d = nullptr;  // [capacity][1024]
  DevBuf work;         // query slots, windows, keys and scores of a search
};

namespace {

// dst(x, y) = (s00 + s10 + s01 + s11) / 4, floor(w/2) x floor(h/2), tight rows; grid.z = image
__global__ void __launch_bounds__(256) halve_kernel(const uint8_t* __restrict__ src, int sw, int sh, size_t spitch, size_t sstride,
                                                   uint8_t* __restrict__ dst, size_t dstride) {
  const int ow = sw / 2, oh = sh / 2;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= ow || y >= oh) return;
  const uint8_t* r0 = src + (size_t)blockIdx.z * sstride + (size_t)(2 * y) * spitch + 2 * x;
  const uint8_t* r1 = r0 + spitch;
  dst[(size_t)blockIdx.z * dstride + (size_t)y * ow + x] = (uint8_t)(((int)r0[0] + r0[1] + r1[0] + r1[1]) / 4);
}

// One block of 1024 threads per image: nearest sampling, mean, centring, norm, scaling.
__global__ void __launch_bounds__(1024) desc_finish_kernel(const uint8_t* __restrict__ src, int cw, int ch, size_t spitch, size_t sstride,
                                                          float* __restrict__ out) {
  __shared__ float v[1024];
  __shared__ double s_mean, s_invn;
  const int t = threadIdx.x, x = t & 31, y = t >> 5;
  const uint8_t* im = src + (size_t)blockIdx.x * sstride;
  int sx = (int)round((double)x * (double)(cw - 1) / 31.0), sy = (int)round((double)y * (double)(ch - 1) / 31.0);
  sx = sx < cw - 1 ? sx : cw - 1;
  sy = sy < ch - 1 ? sy : ch - 1;
  v[t] = (float)im[(size_t)sy * spitch + sx];
  __syncthreads();
  if (t == 0) {
    double m = 0.0;
    for (int i = 0; i < 1024; i++) m += v[i];  // integers: exact
    s_mean = m / (32.0 * 32.0);
  }
  __syncthreads();
  const float c = __fsub_rn(v[t], (float)s_mean);
  __syncthreads();
  v[t] = c;
  __syncthreads();
  if (t == 0) {
    double n2 = 0.0;
    for (int i = 0; i < 1024; i++) n2 = __dadd_rn(n2, __dmul_rn((double)v[i], (double)v[i]));  // raster order (:1118)
    s_invn = 1.0 / sqrt(n2 + 1e-12);
  }
  __syncthreads();
  out[(size_t)blockIdx.x * 1024 + t] = (float)__dmul_rn((double)c, s_invn);
}

// ---- batched candidate search: score[q][k] = dot_desc(bank[k], bank[query_slot[q]]) for k < n_search[q] ----------------
// Each score is the reference's sequential chain s = fadd_rn(s, fmul_rn(a[i], q[i])), i = 0..1023 (no contraction, no
// split over i), so the kernel is a register-tiled product WITHOUT split-K: a block owns 64 queries x 64 bank slots, stages
// 32-wide i-slices of both operands in shared memory (transposed: i-major) and every thread accumulates a 4 x 4 tile in
// ascending i.  Two outputs share one packed FP32 instruction: each half of __fmul2_rn / __ffma2_rn is the correctly rounded
// scalar operation.  The add is written s = ffma2(s, one, p) with `one` = 1.0f passed as a kernel argument: s * 1 is exact,
// so that is fadd_rn(s, p), and ptxas cannot fold it.  (ptxas contracts __fadd2_rn(s, __fmul2_rn(a, b)) into one FFMA2 even
// under -fmad=false, which rounds once instead of twice; the scalar __fadd_rn / __fmul_rn pair is left alone.)
// Candidate rule (:1827-1830, "first strictly larger score above 0"): every score s > 0 becomes the key
// (float_bits(s) << 32) | (0xFFFFFFFF - k); positive floats order like their bit patterns and equal scores order by the
// lowest slot, so the largest key IS the sequential scan's winner, whatever order the keys are combined in.  NaN, +-0 and
// negative scores never become keys (`s > bs` never accepts them either); key 0 = no candidate (-1, 0.0f).
constexpr int DS_T = 64, DS_KC = 32, DS_PAD = DS_T + 4;  // +4 floats: rows stay 16 B aligned for the float4 reads

__global__ void __launch_bounds__(256) desc_search_kernel(const float* __restrict__ bank, const int* __restrict__ qslot,
                                                         const int* __restrict__ nsearch, int nq, int ld,
                                                         unsigned long long* __restrict__ keys, float* __restrict__ scores, float one) {
  __shared__ __align__(16) float sa[DS_KC][DS_PAD], sb[DS_KC][DS_PAD];
  __shared__ int s_nmax;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int q0 = blockIdx.y * DS_T, k0 = blockIdx.x * DS_T;
  if (tid == 0) s_nmax = 0;
  __syncthreads();
  if (tid < DS_T && q0 + tid < nq) atomicMax(&s_nmax, nsearch[q0 + tid]);
  __syncthreads();
  if (k0 >= s_nmax) return;  // the tile lies beyond every query's window (e.g. the upper triangle)
  // staging: thread loads float4 column lc of rows lr and lr + 32 of both operands (128 B per row segment)
  const int lr = tid >> 3, lc = tid & 7;
  const float* ga[2];
  const float* gb[2];
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int q = min(q0 + lr + 32 * j, nq - 1), k = min(k0 + lr + 32 * j, ld - 1);
    ga[j] = bank + (size_t)qslot[q] * 1024 + lc * 4;
    gb[j] = bank + (size_t)k * 1024 + lc * 4;
  }
  const float2 one2 = make_float2(one, one);
  float2 acc[4][2];
#pragma unroll
  for (int m = 0; m < 4; m++) acc[m][0] = acc[m][1] = make_float2(0.0f, 0.0f);
  for (int i0 = 0; i0 < 1024; i0 += DS_KC) {
    float4 va[2], vb[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      va[j] = __ldg(reinterpret_cast<const float4*>(ga[j] + i0));
      vb[j] = __ldg(reinterpret_cast<const float4*>(gb[j] + i0));
    }
    __syncthreads();  // the previous slice has been consumed
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int r = lr + 32 * j, c = lc * 4;
      sa[c][r] = va[j].x, sa[c + 1][r] = va[j].y, sa[c + 2][r] = va[j].z, sa[c + 3][r] = va[j].w;
      sb[c][r] = vb[j].x, sb[c + 1][r] = vb[j].y, sb[c + 2][r] = vb[j].z, sb[c + 3][r] = vb[j].w;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < DS_KC; i++) {  // ascending i: every output keeps the reference's order
      const float4 a = *reinterpret_cast<const float4*>(&sa[i][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&sb[i][tx * 4]);
      const float2 b01 = make_float2(b.x, b.y), b23 = make_float2(b.z, b.w);
      const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int m = 0; m < 4; m++) {
        const float2 am = make_float2(av[m], av[m]);
        acc[m][0] = __ffma2_rn(acc[m][0], one2, __fmul2_rn(am, b01));
        acc[m][1] = __ffma2_rn(acc[m][1], one2, __fmul2_rn(am, b23));
      }
    }
  }
#pragma unroll
  for (int m = 0; m < 4; m++) {
    const int q = q0 + ty * 4 + m;
    const int ns = q < nq ? nsearch[q] : 0;
    const float s4[4] = {acc[m][0].x, acc[m][0].y, acc[m][1].x, acc[m][1].y};
    unsigned long long best = 0;
#pragma unroll
    for (int n = 0; n < 4; n++) {
      const int k = k0 + tx * 4 + n;
      const bool in = k < ns;
      if (scores && q < nq && k < ld) scores[(size_t)q * ld + k] = in ? s4[n] : 0.0f;
      if (in && s4[n] > 0.0f) {
        const unsigned long long key = ((unsigned long long)__float_as_uint(s4[n]) << 32) | (0xFFFFFFFFu - (unsigned)k);
        best = key > best ? key : best;
      }
    }
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) {  // the 16 threads of a query row are one half-warp
      const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o);
      best = v > best ? v : best;
    }
    if (tx == 0 && best) atomicMax(keys + q, best);
  }
}

// scratch of desc32_device for `count` frames of f: ping-pong buffers of the halving chain (tight rows)
size_t desc32_scratch_bytes(const sfmgpu_frames* f, int count) {
  const size_t half = (size_t)(f->w / 2) * (f->h / 2), quarter = (size_t)(f->w / 4) * (f->h / 4);
  return (half + quarter + 64) * count + 256;
}

// global_desc_32 (:1100-1122) of frames [first, first+count) of f into d_out [count][1024] (device), no synchronisation.
int desc32_device(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, uint8_t* scratch, float* d_out) {
  const size_t half = (size_t)(f->w / 2) * (f->h / 2);
  uint8_t* buf[2] = {scratch, scratch + (half + 32) * count};
  const uint8_t* src = f->lvl[0] + (size_t)first * f->fstride[0];
  int cw = f->w, ch = f->h;
  size_t spitch = f->pitch[0], sstride = f->fstride[0];
  int which = 0;
  while (cw > 32 || ch > 32) {
    const int ow = cw / 2, oh = ch / 2;
    if (ow < 1 || oh < 1) return sfm_fail(ctx, SFMGPU_E_ARG, "global_desc32: image degenerates to %dx%d", ow, oh);
    const size_t dstride = (size_t)ow * oh;
    SFM_LAUNCH(ctx, halve_kernel, dim3(sfm_cdiv(ow, 32), sfm_cdiv(oh, 8), count), 256, 0, src, cw, ch, spitch, sstride, buf[which],
               dstride);
    src = buf[which];
    which ^= 1;
    cw = ow;
    ch = oh;
    spitch = (size_t)cw;
    sstride = dstride;
  }
  SFM_LAUNCH(ctx, desc_finish_kernel, count, 1024, 0, src, cw, ch, spitch, sstride, d_out);
  return 0;
}

// The search over device arrays: keys [nq] (0 = no candidate), scores (optional) [nq][ld] with ld = max n_search.
int desc_search_device(sfmgpu_ctx* ctx, const float* bank, const int* d_qslot, const int* d_nsearch, int nq, int ld,
                       unsigned long long* d_keys, float* d_scores) {
  SFM_CUDA(ctx, cudaMemsetAsync(d_keys, 0, (size_t)nq * sizeof(unsigned long long), ctx->stream));
  if (d_scores && ld > 0) SFM_CUDA(ctx, cudaMemsetAsync(d_scores, 0, (size_t)nq * ld * sizeof(float), ctx->stream));
  if (nq == 0 || ld == 0) return 0;
  SFM_LAUNCH(ctx, desc_search_kernel, dim3(sfm_cdiv(ld, DS_T), sfm_cdiv(nq, DS_T)), 256, 0, bank, d_qslot, d_nsearch, nq, ld, d_keys,
             d_scores, 1.0f);
  return 0;
}

void decode_key(unsigned long long key, int* id, float* score) {
  int bid = -1;
  float bs = 0.0f;
  if (key) {
    bid = (int)(0xFFFFFFFFu - (uint32_t)key);
    const uint32_t bits = (uint32_t)(key >> 32);
    memcpy(&bs, &bits, sizeof bs);
  }
  if (id) *id = bid;
  if (score) *score = bs;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

int sfmgpu_global_desc32(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, float* desc_out) {
  SFM_ENTER(ctx);
  if (!ctx || !f) return SFMGPU_E_ARG;
  if (first < 0 || count < 0 || first + count > f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "global_desc32: bad frame range");
  if (count == 0) return 0;
  if (!desc_out) return sfm_fail(ctx, SFMGPU_E_ARG, "global_desc32: null output");
  const size_t sb = align256(desc32_scratch_bytes(f, count));
  SFM_TRY(sfm_reserve(ctx, ctx->cs_work, sb + (size_t)count * 4096));
  float* d_desc = (float*)((uint8_t*)ctx->cs_work.p + sb);
  SFM_TRY(desc32_device(ctx, f, first, count, (uint8_t*)ctx->cs_work.p, d_desc));
  SFM_CUDA(ctx, cudaMemcpyAsync(desc_out, d_desc, (size_t)count * 4096, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

int sfmgpu_desc_search(sfmgpu_ctx* ctx, const float* descs, int n_search, const float* query, float* scores, int* best_id,
                       float* best_score) {
  SFM_ENTER(ctx);
  if (!ctx || n_search < 0 || !query || (n_search > 0 && !descs)) return sfm_fail(ctx, SFMGPU_E_ARG, "desc_search: bad arguments");
  unsigned long long key = 0;
  if (n_search > 0) {
    // scratch bank: the n_search descriptors, the query in slot n_search; one query over slots [0, n_search)
    const size_t bank_bytes = (size_t)(n_search + 1) * 4096;
    SFM_TRY(sfm_reserve(ctx, ctx->cs_work, bank_bytes + 256 + (size_t)n_search * 4 + 256));
    float* d_bank = (float*)ctx->cs_work.p;
    int* d_idx = (int*)((uint8_t*)ctx->cs_work.p + bank_bytes);
    unsigned long long* d_key = (unsigned long long*)(d_idx + 2);
    float* d_scores = (float*)((uint8_t*)ctx->cs_work.p + bank_bytes + 256);
    const int idx[2] = {n_search, n_search};
    SFM_CUDA(ctx, cudaMemcpyAsync(d_bank, descs, (size_t)n_search * 4096, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(d_bank + (size_t)n_search * 1024, query, 4096, cudaMemcpyHostToDevice, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(d_idx, idx, sizeof idx, cudaMemcpyHostToDevice, ctx->stream));
    SFM_TRY(desc_search_device(ctx, d_bank, d_idx, d_idx + 1, 1, n_search, d_key, d_scores));
    SFM_TRY(sfm_pinned(ctx, (size_t)n_search * 4 + 64));
    unsigned long long* hkey = (unsigned long long*)ctx->pinned;
    float* h = (float*)(hkey + 1);
    SFM_CUDA(ctx, cudaMemcpyAsync(hkey, d_key, sizeof *hkey, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaMemcpyAsync(h, d_scores, (size_t)n_search * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (scores) memcpy(scores, h, (size_t)n_search * 4);
    key = *hkey;
  }
  decode_key(key, best_id, best_score);
  return 0;
}

// ---- device-resident descriptor bank -----------------------------------------------------------------------------------
int sfmgpu_descs_create(sfmgpu_ctx* ctx, int capacity, sfmgpu_descs** out) {
  SFM_ENTER(ctx);
  if (!ctx || !out || capacity <= 0) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_create: bad arguments");
  sfmgpu_descs* d = new sfmgpu_descs();
  d->capacity = capacity;
  const size_t bytes = (size_t)capacity * 4096;
  cudaError_t e = cudaMalloc((void**)&d->d, bytes);
  if (e == cudaSuccess) e = cudaMemsetAsync(d->d, 0, bytes, ctx->stream);  // zero descriptor: scores 0, never a candidate
  if (e != cudaSuccess) {
    if (d->d) cudaFree(d->d);
    delete d;
    return sfm_fail(ctx, SFMGPU_E_CUDA, "descs_create: %zu bytes: %s", bytes, cudaGetErrorString(e));
  }
  *out = d;
  return 0;
}

void sfmgpu_descs_destroy(sfmgpu_ctx* ctx, sfmgpu_descs* d) {
  SFM_ENTER_VOID(ctx);
  if (!d) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  if (d->d) cudaFree(d->d);
  if (d->work.p) cudaFree(d->work.p);
  delete d;
}

static int bank_range_ok(sfmgpu_ctx* ctx, const sfmgpu_descs* d, int slot, int count, const char* who) {
  if (!ctx || !d) return SFMGPU_E_ARG;
  if (slot < 0 || count < 0 || (long long)slot + count > d->capacity)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: slots [%d,%lld) outside the bank's [0,%d)", who, slot, (long long)slot + count, d->capacity);
  return 0;
}

int sfmgpu_descs_compute(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, sfmgpu_frames* f, int first, int count) {
  SFM_ENTER(ctx);
  SFM_TRY(bank_range_ok(ctx, d, slot, count, "descs_compute"));
  if (!f) return SFMGPU_E_ARG;
  if (first < 0 || first + count > f->n) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_compute: bad frame range");
  const int step = 1024;  // frames per halving chain: bounds the scratch (0.7 GB at 1080p)
  const int c0 = count < step ? count : step;
  if (c0 > 0) SFM_TRY(sfm_reserve(ctx, ctx->cs_work, desc32_scratch_bytes(f, c0)));
  for (int k = 0; k < count; k += step) {
    const int c = count - k < step ? count - k : step;
    SFM_TRY(desc32_device(ctx, f, first + k, c, (uint8_t*)ctx->cs_work.p, d->d + (size_t)(slot + k) * 1024));
  }
  return 0;
}

int sfmgpu_descs_upload(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, int count, const float* host) {
  SFM_ENTER(ctx);
  SFM_TRY(bank_range_ok(ctx, d, slot, count, "descs_upload"));
  if (count == 0) return 0;
  if (!host) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_upload: null host pointer");
  SFM_CUDA(ctx, cudaMemcpyAsync(d->d + (size_t)slot * 1024, host, (size_t)count * 4096, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the caller may reuse its buffer
  return 0;
}

int sfmgpu_descs_download(sfmgpu_ctx* ctx, sfmgpu_descs* d, int slot, int count, float* host) {
  SFM_ENTER(ctx);
  SFM_TRY(bank_range_ok(ctx, d, slot, count, "descs_download"));
  if (count == 0) return 0;
  if (!host) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_download: null host pointer");
  SFM_CUDA(ctx, cudaMemcpyAsync(host, d->d + (size_t)slot * 1024, (size_t)count * 4096, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

int sfmgpu_descs_search(sfmgpu_ctx* ctx, sfmgpu_descs* d, const int32_t* query_slot, const int32_t* n_search, int nq,
                        int32_t* best_id, float* best_score, float* scores) {
  SFM_ENTER(ctx);
  if (!ctx || !d) return SFMGPU_E_ARG;
  if (nq < 0 || nq > 65535 * DS_T) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_search: %d queries", nq);
  if (nq == 0) return 0;
  if (!query_slot || !n_search) return sfm_fail(ctx, SFMGPU_E_ARG, "descs_search: null query arrays");
  int ld = 0;
  for (int q = 0; q < nq; q++) {
    if (query_slot[q] < 0 || query_slot[q] >= d->capacity)
      return sfm_fail(ctx, SFMGPU_E_ARG, "descs_search: query %d reads slot %d outside [0,%d)", q, query_slot[q], d->capacity);
    if (n_search[q] < 0 || n_search[q] > d->capacity)
      return sfm_fail(ctx, SFMGPU_E_ARG, "descs_search: query %d searches %d slots (bank of %d)", q, n_search[q], d->capacity);
    ld = n_search[q] > ld ? n_search[q] : ld;
  }
  const size_t ib = align256((size_t)nq * 4), kb = align256((size_t)nq * 8), sb = scores ? (size_t)nq * ld * 4 : 0;
  SFM_TRY(sfm_reserve(ctx, d->work, 2 * ib + kb + sb));
  uint8_t* w = (uint8_t*)d->work.p;
  int* d_qslot = (int*)w;
  int* d_ns = (int*)(w + ib);
  unsigned long long* d_keys = (unsigned long long*)(w + 2 * ib);
  float* d_scores = scores ? (float*)(w + 2 * ib + kb) : nullptr;
  SFM_CUDA(ctx, cudaMemcpyAsync(d_qslot, query_slot, (size_t)nq * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_CUDA(ctx, cudaMemcpyAsync(d_ns, n_search, (size_t)nq * 4, cudaMemcpyHostToDevice, ctx->stream));
  SFM_TRY(desc_search_device(ctx, d->d, d_qslot, d_ns, nq, ld, d_keys, d_scores));
  SFM_TRY(sfm_pinned(ctx, (size_t)nq * 8));
  unsigned long long* hk = (unsigned long long*)ctx->pinned;
  SFM_CUDA(ctx, cudaMemcpyAsync(hk, d_keys, (size_t)nq * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (scores && sb) SFM_CUDA(ctx, cudaMemcpyAsync(scores, d_scores, sb, cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int q = 0; q < nq; q++) {
    int id;
    float s;
    decode_key(hk[q], &id, &s);
    if (best_id) best_id[q] = id;
    if (best_score) best_score[q] = s;
  }
  return 0;
}

}  // extern "C"
