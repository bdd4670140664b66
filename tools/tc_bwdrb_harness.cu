// Stand-alone harness for the row-block tcgen05 backward sweeps at 16 <= K <= 24, padding 1 or 3 (csrc/local_bwd_tcrb.cu): random source
// maps and random coefficient tensors, a sample of output pixels checked against an fp64 CPU loop.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/_bin/tc_bwdrb tools/tc_bwdrb_harness.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tc_bwdrb [B H W K pad]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_bwd_tcrb.cu"

int main(int argc, char** argv) {
  int B = 1, H = 5, W = 32, KC = 20, pad = 1;
  if (argc >= 4) { B = atoi(argv[1]); H = atoi(argv[2]); W = atoi(argv[3]); }
  if (argc >= 6) { KC = atoi(argv[4]); pad = atoi(argv[5]); }
  const int T = 2 * pad + 1, T2 = T * T, Kp4 = (KC + 3) & ~3;
  const size_t n = (size_t)B * KC * H * W, nw = (size_t)KC * T2 * Kp4;
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
  const size_t nwbuf = iic::local_coeff_image_offset(KC, pad, 1) + iic::local_bwd_tcrb_image_bytes(KC, pad) / 4;
  cudaMalloc(&dwx, nwbuf * 4); cudaMalloc(&dwy, nwbuf * 4); cudaMalloc(&dg, 4);
  cudaMemcpy(dx_, hx.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dy_, hy.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dwx, hwx.data(), nw * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dwy, hwy.data(), nw * 4, cudaMemcpyHostToDevice);
  const float g = 0.75f;
  cudaMemcpy(dg, &g, 4, cudaMemcpyHostToDevice);
  cudaMemset(dgx, 0xff, n * 4); cudaMemset(dgy, 0xff, n * 4);
  const long long sc = (long long)H * W, sn = sc * KC;
  const iic::LocalMaps m{{dx_, sn, sc, W}, {dy_, sn, sc, W}, B, KC, H, W, pad, iic::sm_count_cached(iic::current_device())};
  const iic::LocalGrads gr{dg, dgx, dgy, sn, sn};
  iic_b200_set_option("tcrb_p1", 1);     // the kernel at any shape: skip the dispatcher's size rule
  int rc = iic::local_bwd_tcrb_try(m, dwx, dwy, gr, 0);
  cudaError_t err = cudaDeviceSynchronize();
  printf("try rc=%d (%s); first launch: %s\n", rc, iic::get_error(), cudaGetErrorString(err));
  if (rc != 0 || err != cudaSuccess) return 1;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int reps = 3;
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) iic::local_bwd_tcrb_try(m, dwx, dwy, gr, 0);
  cudaEventRecord(e1);
  err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("timed launches: %s\n", cudaGetErrorString(err)); return 1; }
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
#ifdef IIC_TC_TRACE
  {
    long long tr[4][64][6];
    cudaMemcpyFromSymbol(tr, iic::bwdrb::g_trace, sizeof(tr));
    const long long t0 = tr[0][0][0];
    printf("stage | producer: enter waited | issuer0: enter a_full_ok issued | issuer1: enter a_full_ok issued | transform: enter a_empty_ok raw_ok done\n");
    for (int k = 0; k < 30; ++k)
      printf("%3d | %7lld %7lld | %7lld %7lld %7lld | %7lld %7lld %7lld | %7lld %7lld %7lld %7lld\n", k + 40, tr[0][k][0] - t0, tr[0][k][1] - t0,
             tr[1][k][0] - t0, tr[1][k][1] - t0, tr[1][k][2] - t0, tr[2][k][0] - t0, tr[2][k][1] - t0, tr[2][k][2] - t0,
             tr[3][k][0] - t0, tr[3][k][1] - t0, tr[3][k][2] - t0, tr[3][k][3] - t0);
  }
#endif
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
    for (int u : rows) for (int v : cols) for (int o = 0; o < KC; o += 3) {
      double rx = 0, ry = 0;
      for (int c = 0; c < KC; ++c) for (int ty = 0; ty < T; ++ty) for (int tx = 0; tx < T; ++tx) {
        const int uu = u + ty - pad, vv = v + tx - pad;
        if (uu < 0 || uu >= H || vv < 0 || vv >= W) continue;
        rx += (double)hwx[((size_t)c * T2 + ty * T + tx) * Kp4 + o] * hy[(((size_t)b * KC + c) * H + uu) * W + vv];
        ry += (double)hwy[((size_t)c * T2 + ty * T + tx) * Kp4 + o] * hx[(((size_t)b * KC + c) * H + uu) * W + vv];
      }
      rx *= g; ry *= g;
      const size_t idx = (((size_t)b * KC + o) * H + u) * W + v;
      ex = fmax(ex, fabs(gx[idx] - rx)); ey = fmax(ey, fabs(gy[idx] - ry));
      mx = fmax(mx, fabs(rx)); my = fmax(my, fabs(ry));
    }
  const double flop = 2.0 * 2 * T2 * KC * KC * (double)B * H * W;
  printf("K=%d pad=%d B=%d H=%d W=%d  %.3f ms (both gradients)  %.1f TFLOP/s (fp32-equivalent)  NaNs %lld\n", KC, pad, B, H, W, ms, flop / ms / 1e9, nan);
  printf("max-norm rel err gx %.3e gy %.3e (max ref %.3e %.3e)\n", ex / mx, ey / my, mx, my);
  printf((ex / mx < 2e-6 && ey / my < 2e-6 && nan == 0) ? "PASS\n" : "FAIL\n");
  return 0;
}
