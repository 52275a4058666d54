// klt_build_bench.cu — the two matrix builds of klt_quad_kernel (csrc/klt_lane.cu) on the same staged tiles: the FFMA build
// (quad_build<float>, one lane per feature, klt mode 17) and the Gram build (gram_build, warp-cooperative integer MMA, the
// default).  Every warp stages 32 tiles and builds all 32 (one fully packed build round), REPS times, at the occupancy of the
// production kernels; a stage-only pass is timed too and subtracted.  The 50 doubles of every feature are compared bit for bit.
//
// Usage: klt_build_bench <tiles.bin> [reps]   (tiles.bin: n x 448 bytes, I1 then I0, 14 rows of 16 bytes, bytes 14/15 zero;
// scripts/klt_build_bench.py writes it and builds this file)
#include "../structure-from-motion-3d-reconstruction_b200/csrc/klt_lane.cu"

#include <cstdlib>
#include <cstring>
#include <vector>

// host helpers of the library referenced by klt_lane.cu's launchers (never called here)
int sfm_next_cfg_id() { return 0; }
int sfm_fail(sfmgpu_ctx*, int code, const char*, ...) { return code; }

namespace {

constexpr int TILE_BYTES = 2 * LIMG;

// MODE 0: stage only, 1: FFMA build, 2: Gram build
template <int MODE, int MINB>
__global__ void __launch_bounds__(32, MINB) build_bench(const unsigned char* __restrict__ tiles, double* __restrict__ out, int n, int reps) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  unsigned char* tile = smem_raw + lane * LSTRIDE;
  unsigned char* scratch = smem_raw + 32 * LSTRIDE;
  GramLane gl;
  if (MODE == 2) {
    gram_lane_init(gl, lane, ZROW - 32 * LSTRIDE);
    *reinterpret_cast<uint4*>(tile + ZROW) = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int base = blockIdx.x * 32; base < n; base += gridDim.x * 32) {
    const int f = min(base + lane, n - 1);
    const uint4* src = reinterpret_cast<const uint4*>(tiles + (size_t)f * TILE_BYTES);
    for (int r = 0; r < reps; r++) {
      __syncwarp();
#pragma unroll 4
      for (int i = 0; i < TILE_BYTES / 16; i++) reinterpret_cast<uint4*>(tile)[i] = __ldg(src + i);
      __syncwarp();
      if (MODE == 1) quad_build<float>(tile, reinterpret_cast<double*>(tile));
      if (MODE == 2)
        for (int j = 0; j < 32; j++) gram_build(smem_raw + j * LSTRIDE, scratch, gl, lane);
    }
    __syncwarp();
    if (base + lane < n)
      for (int e = 0; e < QM; e++) out[(size_t)f * QM + e] = reinterpret_cast<const double*>(tile)[e];
  }
}

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e_ = (x);                                                              \
    if (e_ != cudaSuccess) {                                                           \
      fprintf(stderr, "%s: %s (line %d)\n", #x, cudaGetErrorString(e_), __LINE__);     \
      exit(2);                                                                         \
    }                                                                                  \
  } while (0)

template <int MODE, int MINB>
float run(const unsigned char* d_tiles, double* d_out, int n, int reps, size_t smem) {
  CK(cudaFuncSetAttribute(build_bench<MODE, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, nsm = 0, per_sm = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, build_bench<MODE, MINB>, 32, smem));
  const int grid = nsm * per_sm;  // one resident wave walks all tiles
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  build_bench<MODE, MINB><<<grid, 32, smem>>>(d_tiles, d_out, n, 1);  // warm-up
  CK(cudaEventRecord(a));
  build_bench<MODE, MINB><<<grid, 32, smem>>>(d_tiles, d_out, n, reps);
  CK(cudaEventRecord(b));
  CK(cudaEventSynchronize(b));
  CK(cudaGetLastError());
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, a, b));
  printf("mode %d: %d warps/SM, %.3f ms\n", MODE, per_sm, ms);
  return ms;
}

}  // namespace

int main(int argc, char** argv) {
  if (argc < 2) {
    fprintf(stderr, "usage: %s tiles.bin [reps]\n", argv[0]);
    return 2;
  }
  const int reps = argc > 2 ? atoi(argv[2]) : 20;
  FILE* fp = fopen(argv[1], "rb");
  if (!fp) {
    fprintf(stderr, "cannot open %s\n", argv[1]);
    return 2;
  }
  std::vector<unsigned char> tiles;
  unsigned char buf[TILE_BYTES];
  while (fread(buf, 1, TILE_BYTES, fp) == (size_t)TILE_BYTES) tiles.insert(tiles.end(), buf, buf + TILE_BYTES);
  fclose(fp);
  const int n = (int)(tiles.size() / TILE_BYTES);
  if (n == 0) return 2;
  unsigned char* d_tiles;
  double *d_a, *d_b;
  CK(cudaMalloc(&d_tiles, tiles.size()));
  CK(cudaMalloc(&d_a, (size_t)n * QM * sizeof(double)));
  CK(cudaMalloc(&d_b, (size_t)n * QM * sizeof(double)));
  CK(cudaMemcpy(d_tiles, tiles.data(), tiles.size(), cudaMemcpyHostToDevice));
  const size_t smem = 32 * LSTRIDE, smem_gram = smem + GRAM_SCRATCH;
  const float t0 = run<0, 12>(d_tiles, d_a, n, reps, smem);
  const float t1 = run<1, 12>(d_tiles, d_a, n, reps, smem);
  const float t2 = run<2, 14>(d_tiles, d_b, n, reps, smem_gram);
  std::vector<double> a((size_t)n * QM), b((size_t)n * QM);
  CK(cudaMemcpy(a.data(), d_a, a.size() * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(b.data(), d_b, b.size() * sizeof(double), cudaMemcpyDeviceToHost));
  long long bad = 0;
  for (size_t i = 0; i < a.size(); i++) bad += memcmp(&a[i], &b[i], sizeof(double)) != 0;
  const double rounds = (double)((n + 31) / 32) * reps;
  const double ffma = (t1 - t0) / rounds, gram = (t2 - t0) / rounds;
  printf("{\"tiles\": %d, \"reps\": %d, \"stage_ms\": %.4f, \"ffma_ms\": %.4f, \"gram_ms\": %.4f, \"ffma_ns_per_round\": %.3f, "
         "\"gram_ns_per_round\": %.3f, \"gram_over_ffma\": %.4f, \"mismatched_doubles\": %lld}\n",
         n, reps, t0, t1, t2, ffma * 1e6, gram * 1e6, gram / ffma, bad);
  return bad ? 1 : 0;
}
