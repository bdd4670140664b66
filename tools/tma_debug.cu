// Standalone harness for the TMA kernels (no Python): small random case vs a CPU loop.
//   nvcc -O2 -std=c++17 -gencode arch=compute_100a,code=sm_100a -DIIC_TMA_DEBUG -o tools/_bin/tma_debug tools/tma_debug.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tma_debug [B K H W pad mode]     (mode: 1 joint, 2 backward, 3 both)
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_fwd_tma.cu"

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_bwd_tma.cu"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); return 1; } } while (0)

int main(int argc, char** argv) {
  int B = argc > 1 ? atoi(argv[1]) : 2, K = argc > 2 ? atoi(argv[2]) : 10, H = argc > 3 ? atoi(argv[3]) : 32,
      W = argc > 4 ? atoi(argv[4]) : 64, pad = argc > 5 ? atoi(argv[5]) : 1;
  int mode = argc > 6 ? atoi(argv[6]) : 3;
  const int T = 2 * pad + 1;
  size_t n = (size_t)B * K * H * W;
  std::vector<float> hx(n), hy(n);
  srand(1);
  for (size_t i = 0; i < n; ++i) { hx[i] = rand() / (float)RAND_MAX; hy[i] = rand() / (float)RAND_MAX; }
  float *dx, *dy, *dpart;
  CK(cudaMalloc(&dx, n * 4)); CK(cudaMalloc(&dy, n * 4));
  CK(cudaMemcpy(dx, hx.data(), n * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dy, hy.data(), n * 4, cudaMemcpyHostToDevice));
  size_t E = (size_t)T * T * K * K;
  const int sms = iic::sm_count_cached(iic::current_device());
  CK(cudaMalloc(&dpart, sms * E * 4));
  CK(cudaMemset(dpart, 0, sms * E * 4));
  const long long sn = (long long)K * H * W, sc = (long long)H * W;
  const iic::LocalMaps m{{dx, sn, sc, W}, {dy, sn, sc, W}, B, K, H, W, pad, sms};
  iic::SlotInfo slots{};
  int rc = 0; cudaError_t se = cudaSuccess; float ms = 0; unsigned dbg[8];
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  if (mode & 1) {
  cudaEventRecord(e0);
  rc = iic::local_joint_tma_try(m, dpart, sms, &slots, 0);
  const int ncta = slots.n_slots;
  cudaEventRecord(e1);
  printf("fwd try rc=%d ncta=%d err=%s\n", rc, ncta, iic::get_error());
  se = cudaDeviceSynchronize();
  cudaEventElapsedTime(&ms, e0, e1);
  printf("fwd sync: %s, %.3f ms\n", cudaGetErrorString(se), ms);
  CK(cudaMemcpyFromSymbol(dbg, iic::g_tma_dbg, sizeof(dbg)));
  printf("dbg: %08x blk=%u thr=%u parity=%u bar=%u\n", dbg[0], dbg[1], dbg[2], dbg[3], dbg[4]);
  if (rc == 0 && se == cudaSuccess) {
    std::vector<float> part(ncta * E);
    CK(cudaMemcpy(part.data(), dpart, ncta * E * 4, cudaMemcpyDeviceToHost));
    double maxerr = 0, maxref = 0;
    for (int dyi = 0; dyi < T; ++dyi) for (int dxi = 0; dxi < T; ++dxi) for (int i = 0; i < K; ++i) for (int j = 0; j < K; ++j) {
      double ref = 0;
      for (int b = 0; b < B; ++b) for (int u = 0; u < H; ++u) for (int v = 0; v < W; ++v) {
        int uu = u + dyi - pad, vv = v + dxi - pad;
        if (uu < 0 || uu >= H || vv < 0 || vv >= W) continue;
        ref += (double)hx[(((size_t)b * K + i) * H + uu) * W + vv] * hy[(((size_t)b * K + j) * H + u) * W + v];
      }
      double got = 0;
      for (int c = 0; c < ncta; ++c) got += part[c * E + ((size_t)(dyi * T + dxi) * K + i) * K + j];
      maxerr = fmax(maxerr, fabs(got - ref)); maxref = fmax(maxref, fabs(ref));
    }
    printf("fwd max abs err %.3e (max ref %.3e) -> rel %.3e\n", maxerr, maxref, maxerr / maxref);
  }
  }
  if (!(mode & 2)) return 0;
  // ---- backward ----
  const int Kp = (K + 3) & ~3;
  size_t nw = (size_t)K * T * T * Kp;
  std::vector<float> hwx(nw, 0.f), hwy(nw, 0.f);
  for (int c = 0; c < K; ++c) for (int t = 0; t < T * T; ++t) for (int o = 0; o < K; ++o) {
    hwx[((size_t)c * T * T + t) * Kp + o] = rand() / (float)RAND_MAX - 0.5f;
    hwy[((size_t)c * T * T + t) * Kp + o] = rand() / (float)RAND_MAX - 0.5f;
  }
  float *dwx, *dwy, *dgx, *dgy;
  CK(cudaMalloc(&dwx, nw * 4)); CK(cudaMalloc(&dwy, nw * 4)); CK(cudaMalloc(&dgx, n * 4)); CK(cudaMalloc(&dgy, n * 4));
  CK(cudaMemcpy(dwx, hwx.data(), nw * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dwy, hwy.data(), nw * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dgx, 0, n * 4)); CK(cudaMemset(dgy, 0, n * 4));
  unsigned zero[8] = {0};
  CK(cudaMemcpyToSymbol(iic::g_tma_dbg, zero, sizeof(zero)));
  cudaEventRecord(e0);
  rc = iic::local_bwd_tma_try(m, dwx, dwy, iic::LocalGrads{nullptr, dgx, dgy, sn, sn}, 0);
  cudaEventRecord(e1);
  printf("bwd try rc=%d err=%s\n", rc, iic::get_error());
  se = cudaDeviceSynchronize();
  cudaEventElapsedTime(&ms, e0, e1);
  printf("bwd sync: %s, %.3f ms\n", cudaGetErrorString(se), ms);
  CK(cudaMemcpyFromSymbol(dbg, iic::g_tma_dbg, sizeof(dbg)));
  printf("dbg: %08x blk=%u thr=%u parity=%u bar=%u\n", dbg[0], dbg[1], dbg[2], dbg[3], dbg[4]);
  if (rc == 0 && se == cudaSuccess) {
    std::vector<float> gx(n), gy(n);
    CK(cudaMemcpy(gx.data(), dgx, n * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(gy.data(), dgy, n * 4, cudaMemcpyDeviceToHost));
    double ex = 0, ey = 0, mx = 0;
    for (int b = 0; b < B; ++b) for (int o = 0; o < K; ++o) for (int u = 0; u < H; ++u) for (int v = 0; v < W; ++v) {
      double rx = 0, ry = 0;
      for (int c = 0; c < K; ++c) for (int a = 0; a < T; ++a) for (int d = 0; d < T; ++d) {
        int uu = u + a - pad, vv = v + d - pad;
        if (uu < 0 || uu >= H || vv < 0 || vv >= W) continue;
        rx += (double)hwx[((size_t)c * T * T + a * T + d) * Kp + o] * hy[(((size_t)b * K + c) * H + uu) * W + vv];
        ry += (double)hwy[((size_t)c * T * T + a * T + d) * Kp + o] * hx[(((size_t)b * K + c) * H + uu) * W + vv];
      }
      size_t idx = (((size_t)b * K + o) * H + u) * W + v;
      ex = fmax(ex, fabs(gx[idx] - rx)); ey = fmax(ey, fabs(gy[idx] - ry)); mx = fmax(mx, fabs(rx));
    }
    printf("bwd max abs err gx %.3e gy %.3e (max ref %.3e)\n", ex, ey, mx);
  }
  return 0;
}
