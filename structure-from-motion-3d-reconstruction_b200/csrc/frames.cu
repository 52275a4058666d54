// frames.cu — context, frame batches in HBM, fused pyramid kernel, integer synthetic generator.
//
// Replaces (reference cpp/src/templering_sfm.cpp): GrayImage storage (cpp/include/pgm_io.hpp:10-15),
// downsample2 :200-218, Pyramid/build_pyr :220-232.
//
// HBM layout: level l of a batch is one allocation [frame][row][pitch_l], pitch_l = align16(w_l), frame stride
// = pitch_l*h_l (no inter-frame padding, 256 B of slack after the last frame).  Level 0 IS the uploaded image
// (the reference copies it; we alias it), so one pyramid costs W*H*(1 + 1/4 + 1/16 ...) bytes of traffic.
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

int sfm_fail(sfmgpu_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

int sfm_next_cfg_id() {
  static std::atomic<int> next{0};
  return next.fetch_add(1);
}

int sfm_reserve(sfmgpu_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap) return 0;
  if (b.p) {
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SFM_CUDA(ctx, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes + bytes / 4 + 256;
  SFM_CUDA(ctx, cudaMalloc(&b.p, want));
  b.cap = want;
  return 0;
}

int sfm_pinned(sfmgpu_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->pinned_cap) return 0;
  if (ctx->pinned) {
    SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SFM_CUDA(ctx, cudaFreeHost(ctx->pinned));
    ctx->pinned = nullptr;
    ctx->pinned_cap = 0;
  }
  size_t want = bytes * 2 + 4096;
  SFM_CUDA(ctx, cudaMallocHost(&ctx->pinned, want));
  ctx->pinned_cap = want;
  return 0;
}

extern "C" {

void sfmgpu_lkcfg_default(sfmgpu_lkcfg* c) {
  c->max_tracks = 2200;
  c->min_tracks = 900;
  c->quality = 0.01;
  c->min_distance = 8;
  c->pyr_levels = 3;
  c->win_radius = 5;
  c->iters = 10;
  c->fb_thresh = 1.0;
}

int sfmgpu_version(void) { return SFMGPU_VERSION; }

int sfmgpu_create(int device, sfmgpu_ctx** out) {
  if (!out) return SFMGPU_E_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return SFMGPU_E_CUDA;  // no CPU fallback
  sfmgpu_ctx* ctx = new sfmgpu_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) {
    delete ctx;
    return SFMGPU_E_CUDA;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->n_sm = prop.multiProcessorCount;
  *out = ctx;
  return 0;
}

void sfmgpu_destroy(sfmgpu_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = {&ctx->flush,  &ctx->klt_in, &ctx->klt_p1, &ctx->klt_pb,    &ctx->klt_nit, &ctx->klt_keep, &ctx->klt_defer, &ctx->cs_work,
                    &ctx->sel_work, &ctx->misc,   &ctx->rs_xi,  &ctx->rs_xj,     &ctx->rs_E,    &ctx->rs_counts, &ctx->rs_inl,
                    &ctx->rs_best, &ctx->rs_idx8, &ctx->sv_list, &ctx->rs_raw, &ctx->pk_stage[0], &ctx->pk_stage[1],
                    &ctx->pk_fo,   &ctx->pk_flag, &ctx->pk_tmp, &ctx->pk_enc};
  for (DevBuf* b : bufs)
    if (b->p) cudaFree(b->p);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  for (cudaEvent_t e : ctx->pipe_evs) cudaEventDestroy(e);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->back_stream) cudaStreamDestroy(ctx->back_stream);
  if (ctx->sel_stream) cudaStreamDestroy(ctx->sel_stream);
  if (ctx->klt_stream) cudaStreamDestroy(ctx->klt_stream);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* sfmgpu_last_error(sfmgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (CUDA device unavailable?)"; }

int sfmgpu_sync(sfmgpu_ctx* ctx) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

long long sfmgpu_launch_count(sfmgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

int sfmgpu_timer_start(sfmgpu_ctx* ctx) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  return 0;
}
int sfmgpu_timer_stop(sfmgpu_ctx* ctx, float* ms) {
  SFM_ENTER(ctx);
  if (!ctx || !ms) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  SFM_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  SFM_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return 0;
}

int sfmgpu_flush_l2(sfmgpu_ctx* ctx, size_t bytes) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  SFM_TRY(sfm_reserve(ctx, ctx->flush, bytes));
  SFM_CUDA(ctx, cudaMemsetAsync(ctx->flush.p, 0x5a, bytes, ctx->stream));
  return 0;
}

int sfmgpu_host_alloc(sfmgpu_ctx* ctx, size_t bytes, void** out) {
  SFM_ENTER(ctx);
  if (!ctx || !out) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaMallocHost(out, bytes));
  return 0;
}
int sfmgpu_host_free(sfmgpu_ctx* ctx, void* p) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaFreeHost(p));
  return 0;
}

// ---- frames ----------------------------------------------------------------------------------------------
int sfmgpu_frames_create(sfmgpu_ctx* ctx, int w, int h, int nframes, int levels, sfmgpu_frames** out) {
  SFM_ENTER(ctx);
  if (!ctx || !out || w <= 0 || h <= 0 || nframes <= 0 || levels < 1 || levels > SFM_MAXL)
    return sfm_fail(ctx, SFMGPU_E_ARG, "frames_create: bad arguments (w=%d h=%d n=%d levels=%d)", w, h, nframes, levels);
  sfmgpu_frames* f = new sfmgpu_frames();
  f->w = w;
  f->h = h;
  f->n = nframes;
  f->levels = levels;
  int lw = w, lh = h;
  for (int l = 0; l < SFM_MAXL; l++) f->lvl[l] = nullptr;
  for (int l = 0; l < levels; l++) {
    f->lw[l] = lw;
    f->lh[l] = lh;
    f->pitch[l] = sfm_align16(lw);
    f->fstride[l] = (size_t)f->pitch[l] * (size_t)(lh > 0 ? lh : 0);
    size_t bytes = f->fstride[l] * (size_t)nframes + 256;
    cudaError_t e = cudaMalloc((void**)&f->lvl[l], bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(f->lvl[l], 0, bytes, ctx->stream);
    if (e != cudaSuccess) {
      for (int k = 0; k <= l; k++)
        if (f->lvl[k]) cudaFree(f->lvl[k]);
      delete f;
      return sfm_fail(ctx, SFMGPU_E_CUDA, "frames_create: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    lw /= 2;
    lh /= 2;
  }
  *out = f;
  return 0;
}

void sfmgpu_frames_destroy(sfmgpu_ctx* ctx, sfmgpu_frames* f) {
  SFM_ENTER_VOID(ctx);
  if (!f) return;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  for (int l = 0; l < f->levels; l++)
    if (f->lvl[l]) cudaFree(f->lvl[l]);
  delete f;
}

int sfmgpu_frames_level_size(const sfmgpu_frames* f, int level, int* w, int* h) {
  if (!f || level < 0 || level >= f->levels) return SFMGPU_E_ARG;
  if (w) *w = f->lw[level];
  if (h) *h = f->lh[level];
  return 0;
}

static int check_range(sfmgpu_ctx* ctx, const sfmgpu_frames* f, int first, int count, const char* who) {
  if (!ctx || !f) return SFMGPU_E_ARG;
  if (first < 0 || count < 0 || first + count > f->n)
    return sfm_fail(ctx, SFMGPU_E_ARG, "%s: frame range [%d,%d) outside [0,%d)", who, first, first + count, f->n);
  return 0;
}

int sfmgpu_frames_upload(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* host_pix) {
  SFM_ENTER(ctx);
  SFM_TRY(check_range(ctx, f, first, count, "frames_upload"));
  if (!host_pix) return sfm_fail(ctx, SFMGPU_E_ARG, "frames_upload: null host pointer");
  if (count == 0) return 0;
  // frames are contiguous rows on both sides -> one 2D copy of count*h rows
  SFM_CUDA(ctx, cudaMemcpy2DAsync(f->lvl[0] + (size_t)first * f->fstride[0], f->pitch[0], host_pix, f->w, f->w,
                                  (size_t)f->h * count, cudaMemcpyDefault, ctx->stream));
  return 0;
}

int sfmgpu_frames_upload_device(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, const uint8_t* dev_pix,
                                size_t pitch) {
  SFM_ENTER(ctx);
  SFM_TRY(check_range(ctx, f, first, count, "frames_upload_device"));
  if (!dev_pix || pitch < (size_t)f->w) return sfm_fail(ctx, SFMGPU_E_ARG, "frames_upload_device: bad pointer/pitch");
  if (count == 0) return 0;
  SFM_CUDA(ctx, cudaMemcpy2DAsync(f->lvl[0] + (size_t)first * f->fstride[0], f->pitch[0], dev_pix, pitch, f->w,
                                  (size_t)f->h * count, cudaMemcpyDeviceToDevice, ctx->stream));
  return 0;
}

int sfmgpu_frames_device_ptr(const sfmgpu_frames* f, int level, void** ptr, size_t* pitch, size_t* frame_stride) {
  if (!f || level < 0 || level >= f->levels) return SFMGPU_E_ARG;
  if (ptr) *ptr = f->lvl[level];
  if (pitch) *pitch = (size_t)f->pitch[level];
  if (frame_stride) *frame_stride = f->fstride[level];
  return 0;
}

int sfmgpu_frames_download(sfmgpu_ctx* ctx, sfmgpu_frames* f, int frame, int level, uint8_t* host_out) {
  SFM_ENTER(ctx);
  SFM_TRY(check_range(ctx, f, frame, 1, "frames_download"));
  if (level < 0 || level >= f->levels || !host_out) return sfm_fail(ctx, SFMGPU_E_ARG, "frames_download: bad level");
  if (f->lw[level] == 0 || f->lh[level] == 0) return 0;
  SFM_CUDA(ctx, cudaMemcpy2DAsync(host_out, f->lw[level], f->lvl[level] + (size_t)frame * f->fstride[level],
                                  f->pitch[level], f->lw[level], f->lh[level], cudaMemcpyDeviceToHost, ctx->stream));
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

}  // extern "C"

// ---- stage profile + FP64 peak ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
    a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
  }
  if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678) out[0] = a0;  // keep the chain alive
}

extern "C" int sfmgpu_fp64_peak(sfmgpu_ctx* ctx, double* tflops) {
  SFM_ENTER(ctx);
  if (!ctx || !tflops) return SFMGPU_E_ARG;
  SFM_TRY(sfm_reserve(ctx, ctx->misc, 256));
  const int iters = 20000, blocks = ctx->n_sm * 8, threads = 256;
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {
    SFM_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    SFM_LAUNCH(ctx, dfma_peak_kernel, blocks, threads, 0, (double*)ctx->misc.p, iters);
    SFM_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    SFM_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    float ms = 0;
    SFM_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep > 0 && ms < best) best = ms;
  }
  *tflops = 2.0 * 8.0 * iters * (double)blocks * threads / (best * 1e-3) / 1e12;
  return 0;
}

extern "C" int sfmgpu_profile(sfmgpu_ctx* ctx, int enable) {
  SFM_ENTER(ctx);
  if (!ctx) return SFMGPU_E_ARG;
  ctx->profile = enable != 0;
  return 0;
}

extern "C" int sfmgpu_stage_times_n(sfmgpu_ctx* ctx, float* ms, int n) {
  SFM_ENTER(ctx);
  if (!ctx || !ms || n < 0) return SFMGPU_E_ARG;
  SFM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& e : ctx->stage_evs) {
    float t = 0;
    if (cudaEventElapsedTime(&t, e.a, e.b) == cudaSuccess && e.stage >= 0 && e.stage < 7) ctx->stage_ms[e.stage] += t;
    cudaEventDestroy(e.a);
    cudaEventDestroy(e.b);
  }
  ctx->stage_evs.clear();
  for (int i = 0; i < n; i++) ms[i] = i < 7 ? ctx->stage_ms[i] : 0.f;
  for (int i = 0; i < 7; i++) ctx->stage_ms[i] = 0;
  return 0;
}

extern "C" int sfmgpu_stage_times(sfmgpu_ctx* ctx, float* ms4) { return sfmgpu_stage_times_n(ctx, ms4, 4); }

// ---- fused pyramid kernel ------------------------------------------------------------------------------------
// One thread owns a 16 x 4 block of the source level (four 16 B loads), emits 8 x 2 pixels of the next level
// (two 8 B stores) and, when NL == 2, 4 x 1 pixels of the level after that (one 4 B store).  The 2x2 box is
// (s00+s10+s01+s11)/4 with truncation (:214), done on packed 16-bit lanes.
__device__ __forceinline__ uint32_t box_fields(uint32_t a, uint32_t b) {
  const uint32_t m = 0x00FF00FFu;
  const uint32_t s = (a & m) + ((a >> 8) & m) + (b & m) + ((b >> 8) & m);
  return (s >> 2) & m;  // two results, in bytes 0 and 2
}
__device__ __forceinline__ uint32_t box8(uint32_t a0, uint32_t a1, uint32_t b0, uint32_t b1) {
  return __byte_perm(box_fields(a0, b0), box_fields(a1, b1), 0x6420);
}

template <int NL>
__global__ void __launch_bounds__(256) pyr_down_kernel(const uint8_t* __restrict__ src, int sh, int spitch, size_t sfs,
                                                      uint8_t* __restrict__ d1, int h1, int p1, size_t fs1,
                                                      uint8_t* __restrict__ d2, int h2, int p2, size_t fs2, int frame0) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y * blockDim.y + threadIdx.y;
  const size_t fr = (size_t)(frame0 + blockIdx.z);
  const int x0 = tx * 16, y0 = ty * 4;
  if (x0 + 16 > spitch || y0 >= sh) return;
  const uint8_t* s = src + fr * sfs + x0;
  uint4 r[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int y = y0 + k;
    r[k] = (y < sh) ? __ldg(reinterpret_cast<const uint4*>(s + (size_t)y * spitch)) : make_uint4(0, 0, 0, 0);
  }
  uint2 o0, o1;
  o0.x = box8(r[0].x, r[0].y, r[1].x, r[1].y);
  o0.y = box8(r[0].z, r[0].w, r[1].z, r[1].w);
  o1.x = box8(r[2].x, r[2].y, r[3].x, r[3].y);
  o1.y = box8(r[2].z, r[2].w, r[3].z, r[3].w);
  if (8 * tx + 8 <= p1) {
    uint8_t* d = d1 + fr * fs1 + 8 * tx;
    if (2 * ty < h1) *reinterpret_cast<uint2*>(d + (size_t)(2 * ty) * p1) = o0;
    if (2 * ty + 1 < h1) *reinterpret_cast<uint2*>(d + (size_t)(2 * ty + 1) * p1) = o1;
  }
  if (NL == 2) {
    if (4 * tx + 4 <= p2 && ty < h2)
      *reinterpret_cast<uint32_t*>(d2 + fr * fs2 + (size_t)ty * p2 + 4 * tx) = box8(o0.x, o0.y, o1.x, o1.y);
  }
}

extern "C" int sfmgpu_pyramid_build(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count) {
  SFM_ENTER(ctx);
  SFM_TRY(check_range(ctx, f, first, count, "pyramid_build"));
  if (count == 0) return 0;
  int l = 0;
  while (l + 1 < f->levels) {
    const int nl = (l + 2 < f->levels) ? 2 : 1;
    if (f->lh[l + 1] == 0 || f->lw[l + 1] == 0) break;  // nothing below this level
    dim3 block(32, 8);
    dim3 grid(sfm_cdiv(f->pitch[l] / 16, 32), sfm_cdiv((f->lh[l] + 3) / 4, 8), 1);
    for (int done = 0; done < count; done += 32768) {
      const int nz = count - done < 32768 ? count - done : 32768;
      grid.z = nz;
      if (nl == 2)
        SFM_LAUNCH(ctx, pyr_down_kernel<2>, grid, block, 0, f->lvl[l], f->lh[l], f->pitch[l], f->fstride[l], f->lvl[l + 1],
                   f->lh[l + 1], f->pitch[l + 1], f->fstride[l + 1], f->lvl[l + 2], f->lh[l + 2], f->pitch[l + 2],
                   f->fstride[l + 2], first + done);
      else
        SFM_LAUNCH(ctx, pyr_down_kernel<1>, grid, block, 0, f->lvl[l], f->lh[l], f->pitch[l], f->fstride[l], f->lvl[l + 1],
                   f->lh[l + 1], f->pitch[l + 1], f->fstride[l + 1], (uint8_t*)nullptr, 0, 0, (size_t)0, first + done);
    }
    l += nl;
  }
  return 0;
}

// ---- integer synthetic generator (twin of sfmgpu/synth.py) ----------------------------------------------------
__device__ __forceinline__ uint32_t hash32(uint32_t a) {
  a ^= a >> 16;
  a *= 0x7FEB352Du;
  a ^= a >> 15;
  a *= 0x846CA68Bu;
  a ^= a >> 16;
  return a;
}
__device__ __forceinline__ uint32_t lattice(uint32_t s, uint32_t ix, uint32_t iy) {
  return hash32(ix + hash32(iy + s)) >> 24;
}
__device__ __forceinline__ uint32_t value_noise(uint32_t s, uint32_t X, uint32_t Y, int log2cell) {
  const int sh = log2cell + 8;
  const uint32_t ix = X >> sh, iy = Y >> sh;
  const uint32_t fx = (X >> log2cell) & 255u, fy = (Y >> log2cell) & 255u;
  const uint32_t top = lattice(s, ix, iy) * (256u - fx) + lattice(s, ix + 1, iy) * fx;
  const uint32_t bot = lattice(s, ix, iy + 1) * (256u - fx) + lattice(s, ix + 1, iy + 1) * fx;
  return (top * (256u - fy) + bot * fy) >> 16;
}
__device__ __forceinline__ uint32_t block_val(uint32_t s, uint32_t i, uint32_t j) {
  return (lattice(s, i, j) & 3u) == 0u ? 255u : 0u;
}
__device__ __forceinline__ uint32_t synth_pixel(uint32_t s0, uint32_t s1, uint32_t s2, uint32_t X, uint32_t Y) {
  const uint32_t ix = X >> 13, iy = Y >> 13, fx = X & 8191u, fy = Y & 8191u;
  const uint32_t w1x = fx > 8192u - 256u ? fx - (8192u - 256u) : 0u, w0x = 256u - w1x;
  const uint32_t w1y = fy > 8192u - 256u ? fy - (8192u - 256u) : 0u, w0y = 256u - w1y;
  const uint32_t B = (block_val(s0, ix, iy) * w0x * w0y + block_val(s0, ix + 1, iy) * w1x * w0y +
                      block_val(s0, ix, iy + 1) * w0x * w1y + block_val(s0, ix + 1, iy + 1) * w1x * w1y) >> 16;
  const uint32_t v16 = value_noise(s1, X, Y, 4), v4 = value_noise(s2, X, Y, 2);
  return (4u * B + 3u * v16 + v4) >> 3;
}

__global__ void __launch_bounds__(256) synth_kernel(uint8_t* __restrict__ dst, int w, int h, int pitch, size_t fs, int frame0,
                                                   uint32_t seed, int t0) {
  const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int k = blockIdx.z;
  if (x4 >= pitch || y >= h) return;
  const int t = t0 + k;
  const int m = ((t % 128) + 128) % 128;
  const int tri = m < 64 ? m : 128 - m;
  const uint32_t s0 = hash32(seed * 4u + 0u), s1 = hash32(seed * 4u + 1u), s2 = hash32(seed * 4u + 2u);
  const uint32_t Y = (uint32_t)y * 256u + (uint32_t)((1 << 20) - 8 * tri);
  uint32_t packed = 0;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int x = x4 + j;
    uint32_t v = 0;
    if (x < w) v = synth_pixel(s0, s1, s2, (uint32_t)x * 256u + (uint32_t)((1 << 20) + 16 * tri), Y);
    packed |= (v & 255u) << (8 * j);
  }
  *reinterpret_cast<uint32_t*>(dst + (size_t)(frame0 + k) * fs + (size_t)y * pitch + x4) = packed;
}

extern "C" int sfmgpu_frames_synth(sfmgpu_ctx* ctx, sfmgpu_frames* f, int first, int count, uint32_t seed, int t0) {
  SFM_ENTER(ctx);
  SFM_TRY(check_range(ctx, f, first, count, "frames_synth"));
  if (count == 0) return 0;
  dim3 block(64, 4);
  for (int done = 0; done < count; done += 32768) {
    const int nz = count - done < 32768 ? count - done : 32768;
    dim3 grid(sfm_cdiv(f->pitch[0] / 4, 64), sfm_cdiv(f->h, 4), nz);
    SFM_LAUNCH(ctx, synth_kernel, grid, block, 0, f->lvl[0], f->w, f->h, f->pitch[0], f->fstride[0], first + done, seed,
               t0 + done);
  }
  return 0;
}
