// Stand-alone timing driver of the row-marching forward (tools only; the product path is libsrst.so).  Compiles the
// kernel with a run-time ablation mask so that one binary measures what each phase costs:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -DSRST_MARCH_ABL -DMB_TW=112 \
//        -I srgan_st_b200/csrc -o tools/_bin/march_bench_112 tools/march_bench.cu -lcuda
//   tools/_bin/march_bench_112 B H W [chunk_blocks] [mask ...]
// -DMB_XFULL=1 (with MB_TW=96): the crop layout (images no wider than 96 columns).  -DSRST_MARCH_STAMPS and MB_STAMPS=1
// in the environment: phase time stamps of one launch, medians over all CTAs and per chunk index.
// mask bits: 1 chain, 2 vertical, 4 horizontal, 8 gradient, 16 convert, 32 ds stores, 64 ixy stores (set = skipped)
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include "st_march.cuh"
using namespace srst;
#ifndef MB_TW
#define MB_TW 112
#endif
#ifndef MB_CR
#define MB_CR 8
#endif
#ifndef MB_XFULL
#define MB_XFULL 0
#endif
using C = StMarchCfg<MB_TW, 2, 8, MB_CR, MB_XFULL != 0>;
static bool make_map(CUtensorMap* map, const float* base, long long planes, int rows, int cols, int bw, int bh, int bp) {
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)cols * rows * 4};
  const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bp};
  const cuuint32_t estr[3] = {1, 1, 1};
  return cuTensorMapEncodeTiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
int main(int argc, char** argv) {
  const int B = argc > 1 ? atoi(argv[1]) : 1, H = argc > 2 ? atoi(argv[2]) : 1356, W = argc > 3 ? atoi(argv[3]) : 2040;
  int cb_forced = argc > 4 ? atoi(argv[4]) : 0;
  if (C::XFULL && W > C::TW) { printf("the crop layout needs W <= %d\n", C::TW); return 1; }
  const size_t n = (size_t)B * 3 * H * W;
  const int NPOOL = (int)(400e6 / (2.0 * n * 4)) + 2;  // > 2x L2 of inputs
  std::vector<float*> sr(NPOOL), hr(NPOOL);
  std::vector<float> h(n);
  for (size_t i = 0; i < n; ++i) h[i] = (float)((i * 2654435761u) % 1000) / 1000.f;
  for (int p = 0; p < NPOOL; ++p) {
    cudaMalloc(&sr[p], n * 4); cudaMalloc(&hr[p], n * 4);
    cudaMemcpy(sr[p], h.data(), n * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(hr[p], h.data() + 1, (n - 1) * 4, cudaMemcpyHostToDevice);
  }
  float *ds, *ixy, *loss, *ws;
  cudaMalloc(&ds, n * 4); cudaMalloc(&ixy, (size_t)B * 2 * ((H + 1) / 2) * W * 2 * 4); cudaMalloc(&loss, 16); cudaMalloc(&ws, 1 << 20);
  cudaMemset(ws, 0, 1 << 20);
  std::vector<StMarchParams<2, 8>> MPs(NPOOL);
  int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  for (int p = 0; p < NPOOL; ++p) {
    auto& MP = MPs[p];
    if (!make_map(&MP.sr_map, sr[p], (long long)B * 3, H, W, C::BW, C::RS, 3) || !make_map(&MP.hr_map, hr[p], (long long)B * 3, H, W, C::BW, C::RS, 3)) { printf("map failed\n"); return 1; }
    auto& F = MP.F;
    F.sr = sr[p]; F.hr = hr[p]; F.ds_sr = ds; F.ds_hr = nullptr; F.ixy_sr = ixy; F.ixy_hr = nullptr;
    F.ticket = (unsigned*)ws; F.partials = ws + 4; F.px_partials = nullptr; F.loss_out = loss;
    F.B = B; F.H = H; F.W = W; F.normalize = 1; F.vec4 = 1; F.eps = 1e-12f; F.inv_count = 1.f / ((float)B * H * W);
    const float g[5] = {0.00013383f, 0.10798193f, 0.7837685f, 0.10798193f, 0.00013383f};
    const float dg[5] = {0.0010706f, 0.43192774f, 0.f, -0.43192774f, -0.0010706f};
    float k[17]; double sum = 0; for (int i = 0; i < 17; ++i) { k[i] = expf(-(i - 8) * (i - 8) / 8.f); sum += k[i]; }
    for (int i = 0; i < 17; ++i) k[i] /= (float)sum;
    for (int i = 0; i < 5; ++i) { F.taps.g[i] = g[i]; F.taps.dg[i] = dg[i]; }
    for (int i = 0; i < 17; ++i) F.taps.k[i] = k[i];
    for (int u = 0; u <= 5; ++u) { F.taps.gp[u] = make_float2(u <= 4 ? g[u] : 0.f, u >= 1 ? g[u - 1] : 0.f); F.taps.dgp[u] = make_float2(u <= 4 ? dg[u] : 0.f, u >= 1 ? dg[u - 1] : 0.f); }
    for (int u = 0; u <= 17; ++u) F.taps.kp[u] = make_float2(u <= 16 ? k[u] : 0.f, u >= 1 ? k[u - 1] : 0.f);
    const int nblk = (H + 15) / 16;
    MP.nstrips = (W + C::TW - 1) / C::TW;
    const long long base = (long long)B * MP.nstrips;
    const int slots = sms * C::MINB;
    long long nch = base < slots ? slots / base : 1;
    if (nch > nblk) nch = nblk;
    int cb = (int)((nblk + nch - 1) / nch);
    if (cb_forced > 0) cb = cb_forced < nblk ? cb_forced : nblk;
    MP.chunk_blocks = cb; MP.nchunks = (nblk + cb - 1) / cb;
  }
  auto kern = st_forward_march_kernel<C, false, false>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES);
  const int grid = B * MPs[0].nstrips * MPs[0].nchunks;
  printf("TW=%d%s B=%d %dx%d: grid %d (strips %d, chunks %d of %d blocks), %d threads, %zu B smem\n", C::TW, C::XFULL ? " (crop layout)" : "", B, H, W, grid,
         MPs[0].nstrips, MPs[0].nchunks, MPs[0].chunk_blocks, C::NT, C::SMEM_BYTES);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int iters = 40;
  for (int a = 5; a < (argc > 5 ? argc : 6); ++a) {
    const int mask = a < argc ? atoi(argv[a]) : 0;
    cudaMemcpyToSymbol(g_march_abl, &mask, sizeof(int));
    float best = 1e9f;
    for (int rep = 0; rep < 4; ++rep) {
      cudaEventRecord(e0);
      for (int i = 0; i < iters; ++i) kern<<<grid, C::NT, C::SMEM_BYTES>>>(MPs[i % NPOOL]);
      cudaEventRecord(e1);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); return 1; }
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      if (rep > 0 && ms / iters < best) best = ms / iters;
    }
    printf("  mask %3d: %8.2f us\n", mask, best * 1e3f);
  }
  // phase stamps of one launch (producer thread 0: slots 0..63, consumer thread 0: 64..127), median over CTAs
#ifdef SRST_MARCH_STAMPS
  if (getenv("MB_STAMPS")) {
    long long* d; cudaMalloc(&d, (size_t)grid * 128 * 8); cudaMemset(d, 0, (size_t)grid * 128 * 8);
    const int zero = getenv("MB_STAMP_MASK") ? atoi(getenv("MB_STAMP_MASK")) : 0; cudaMemcpyToSymbol(g_march_abl, &zero, sizeof(int));
    cudaMemcpyToSymbol(g_march_stamp, &d, sizeof(d));
    kern<<<grid, C::NT, C::SMEM_BYTES>>>(MPs[1]);
    cudaDeviceSynchronize();
    std::vector<long long> hst((size_t)grid * 128);
    cudaMemcpy(hst.data(), d, hst.size() * 8, cudaMemcpyDeviceToHost);
    long long t0 = 0; for (int c = 0; c < grid; ++c) if (hst[(size_t)c * 128] && (!t0 || hst[(size_t)c * 128] < t0)) t0 = hst[(size_t)c * 128];
    // CTA c works on chunk (c / nstrips) % nchunks of its strip (the grid is image-major, then chunk, then strip)
    const int nch = MPs[1].nchunks, nst = MPs[1].nstrips;
    for (int sl = 0; sl < 128; ++sl) {
      std::vector<double> v;
      std::vector<std::vector<double>> vc(nch);
      for (int c = 0; c < grid; ++c)
        if (hst[(size_t)c * 128 + sl]) {
          const double t = (hst[(size_t)c * 128 + sl] - t0) * 1e-3;
          v.push_back(t);
          vc[(c / nst) % nch].push_back(t);
        }
      if (v.empty()) continue;
      std::sort(v.begin(), v.end());
      printf("  %s slot %2d: median %7.2f us  min %7.2f  max %7.2f  (n=%zu)", sl < 64 ? "P" : "C", sl & 63, v[v.size() / 2], v.front(), v.back(), v.size());
      if (nch > 1 && nch <= 8) {
        printf("  per chunk:");
        for (auto& u : vc) {
          if (u.empty()) { printf("      -"); continue; }
          std::sort(u.begin(), u.end());
          printf(" %7.2f", u[u.size() / 2]);
        }
      }
      printf("\n");
    }
  }
#endif
  return 0;
}
