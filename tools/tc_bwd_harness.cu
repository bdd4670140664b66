// Stand-alone harness for the tcgen05 backward sweeps at K = 128, 3 x 3 window (csrc/local_bwd_tc.cu): random source
// maps and random coefficient tensors, a sample of output pixels checked against an fp64 CPU loop.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/_bin/tc_bwd tools/tc_bwd_harness.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tc_bwd [B H W]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_bwd_tc.cu"

int main(int argc, char** argv) {
  const int KC = 128;
  int B = 1, H = 5, W = 32;
  if (argc >= 4) { B = atoi(argv[1]); H = atoi(argv[2]); W = atoi(argv[3]); }
  const size_t n = (size_t)B * KC * H * W, nw = (size_t)KC * 9 * KC;
  std::vector<float> hx(n), hy(n), hwx(nw), hwy(nw);
  srand(2);
  for (size_t i = 0; i < n; ++i) {
    const float a = (float)rand() / RAND_MAX, b = (float)rand() / RAND_MAX;
    hx[i] = a * a * a * 0.05f;
    hy[i] = b * b * b * 0.05f;
  }
  for (size_t i = 0; i < nw; ++i) { hwx[i] = (float)rand() / RAND_MAX - 0.4f; hwy[i] = (float)rand() / RAND_MAX - 0.6f; }
  float *dx_, *dy_, *dwx, *dwy, *dgx, *dgy, *dg;
  cudaMalloc(&dx_, n * 4); cudaMalloc(&dy_, n * 4); cudaMalloc(&dgx, n * 4); cudaMalloc(&dgy, n * 4);
  // coefficient buffers as iic_local_coeff_floats sizes them: the kernel writes its weight image into their tail
  const size_t nwbuf = iic::local_coeff_image_offset(KC, 1, 1) + iic::local_bwd_tc_image_bytes(KC, 1) / 4;
  cudaMalloc(&dwx, nwbuf * 4); cudaMalloc(&dwy, nwbuf * 4); cudaMalloc(&dg, 4);
  cudaMemcpy(dx_, hx.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dy_, hy.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dwx, hwx.data(), nw * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dwy, hwy.data(), nw * 4, cudaMemcpyHostToDevice);
  const float g = 0.75f;
  cudaMemcpy(dg, &g, 4, cudaMemcpyHostToDevice);
  cudaMemset(dgx, 0xff, n * 4); cudaMemset(dgy, 0xff, n * 4);
  const long long sc = (long long)H * W, sn = sc * KC;
  const iic::LocalMaps m{{dx_, sn, sc, W}, {dy_, sn, sc, W}, B, KC, H, W, 1, iic::sm_count_cached(iic::current_device())};
  const iic::LocalGrads gr{dg, dgx, dgy, sn, sn};
  int rc = iic::local_bwd_tc_try(m, dwx, dwy, gr, 0);
  cudaError_t err = cudaDeviceSynchronize();
  printf("try rc=%d (%s); first launch: %s\n", rc, iic::get_error(), cudaGetErrorString(err));
  if (rc != 0 || err != cudaSuccess) return 1;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int reps = 3;
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) iic::local_bwd_tc_try(m, dwx, dwy, gr, 0);
  cudaEventRecord(e1);
  err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("timed launches: %s\n", cudaGetErrorString(err)); return 1; }
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
  std::vector<float> gx(n), gy(n);
  cudaMemcpy(gx.data(), dgx, n * 4, cudaMemcpyDeviceToHost);
  cudaMemcpy(gy.data(), dgy, n * 4, cudaMemcpyDeviceToHost);
  double ex = 0, ey = 0, mx = 0, my = 0;
  long long nan = 0;
  for (size_t i = 0; i < n; ++i) if (gx[i] != gx[i] || gy[i] != gy[i]) ++nan;
  // sample: all channels at a set of pixels including borders
  const int rows[] = {0, 1, H / 2, H - 2 > 0 ? H - 2 : 0, H - 1};
  const int cols[] = {0, 1, 2, 3, 4, 31 < W ? 31 : W - 1, W / 2, 127 < W ? 127 : W - 1, 128 < W ? 128 : W - 1, W - 2, W - 1};
  for (int b = 0; b < B; b += (B > 2 ? B - 1 : 1))
    for (int u : rows) for (int v : cols) for (int o = 0; o < KC; o += 7) {
      double rx = 0, ry = 0;
      for (int c = 0; c < KC; ++c) for (int ty = 0; ty < 3; ++ty) for (int tx = 0; tx < 3; ++tx) {
        const int uu = u + ty - 1, vv = v + tx - 1;
        if (uu < 0 || uu >= H || vv < 0 || vv >= W) continue;
        rx += (double)hwx[((size_t)c * 9 + ty * 3 + tx) * KC + o] * hy[(((size_t)b * KC + c) * H + uu) * W + vv];
        ry += (double)hwy[((size_t)c * 9 + ty * 3 + tx) * KC + o] * hx[(((size_t)b * KC + c) * H + uu) * W + vv];
      }
      rx *= g; ry *= g;
      const size_t idx = (((size_t)b * KC + o) * H + u) * W + v;
      ex = fmax(ex, fabs(gx[idx] - rx)); ey = fmax(ey, fabs(gy[idx] - ry));
      mx = fmax(mx, fabs(rx)); my = fmax(my, fabs(ry));
    }
  const double flop = 2.0 * 2 * 9 * KC * KC * (double)B * H * W;
  printf("B=%d H=%d W=%d  %.3f ms (both gradients)  %.1f TFLOP/s (fp32-equivalent)  NaNs %lld\n", B, H, W, ms, flop / ms / 1e9, nan);
  printf("max-norm rel err gx %.3e gy %.3e (max ref %.3e %.3e)\n", ex / mx, ey / my, mx, my);
  printf((ex / mx < 2e-6 && ey / my < 2e-6 && nan == 0) ? "PASS\n" : "FAIL\n");
  return 0;
}
