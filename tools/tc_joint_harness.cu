// Stand-alone harness for the tcgen05 (UMMA) local joint at K = 128 clusters, 3 x 3 window (csrc/local_fwd_tc.cu):
// runs the kernel on random simplex-like maps, adds the per-CTA slots in fp64 and compares a sample of entries with
// an fp64 CPU loop; prints the time per launch and the fp32-equivalent TFLOP/s.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/_bin/tc_joint tools/tc_joint_harness.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tc_joint [B H W]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_fwd_tc.cu"

int main(int argc, char** argv) {
  const int KC = 128;
  int B = 1, H = 6, W = 32;
  if (argc >= 4) { B = atoi(argv[1]); H = atoi(argv[2]); W = atoi(argv[3]); }
  const size_t n = (size_t)B * KC * H * W;
  std::vector<float> hx(n), hy(n);
  srand(1);
  // positive values of very different sizes (like softmax outputs): a strict test for the hi/lo split
  for (size_t i = 0; i < n; ++i) {
    const float a = (float)rand() / RAND_MAX, b = (float)rand() / RAND_MAX;
    hx[i] = a * a * a * 0.05f;
    hy[i] = b * b * b * 0.05f;
  }
  float *dx_, *dy_, *dout;
  cudaMalloc(&dx_, n * 4); cudaMalloc(&dy_, n * 4);
  cudaMemcpy(dx_, hx.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dy_, hy.data(), n * 4, cudaMemcpyHostToDevice);
  const size_t E = (size_t)9 * KC * KC;
  cudaMalloc(&dout, 49 * E * 4);
  cudaMemset(dout, 0xff, 49 * E * 4);
  const long long sc = (long long)H * W, sn = sc * KC;
  const iic::LocalMaps m{{dx_, sn, sc, W}, {dy_, sn, sc, W}, B, KC, H, W, 1, iic::sm_count_cached(iic::current_device())};
  iic::SlotInfo slots{};
  int rc = iic::local_joint_tc_try(m, dout, 49, &slots, 0);
  const int ncta = slots.n_slots;
  cudaError_t err = cudaDeviceSynchronize();
  printf("try rc=%d ncta=%d (%s); first launch: %s\n", rc, ncta, iic::get_error(), cudaGetErrorString(err));
  if (rc != 0 || err != cudaSuccess) return 1;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int reps = 5;
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) iic::local_joint_tc_try(m, dout, 49, &slots, 0);
  cudaEventRecord(e1);
  err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("timed launches: %s\n", cudaGetErrorString(err)); return 1; }
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
  std::vector<float> ho((size_t)ncta * E);
  cudaMemcpy(ho.data(), dout, ho.size() * 4, cudaMemcpyDeviceToHost);
  double max_rel = 0.0, max_abs = 0.0, max_ref = 0.0, sum_rel = 0.0, sum_rel2 = 0.0; int cnt = 0;
  for (int d = 0; d < 9; ++d) {
    const int ddy = d / 3, ddx = d % 3;
    for (int i = 0; i < KC; i += 29)
      for (int j = 0; j < KC; j += 31) {
        double ref = 0.0;
        for (int b = 0; b < B; ++b)
          for (int u = 0; u < H; ++u) {
            const int xr = u + ddy - 1;
            if (xr < 0 || xr >= H) continue;
            const float* xrow = &hx[((size_t)(b * KC + i) * H + xr) * W];
            const float* yrow = &hy[((size_t)(b * KC + j) * H + u) * W];
            for (int v = 0; v < W; ++v) {
              const int xc = v + ddx - 1;
              if (xc < 0 || xc >= W) continue;
              ref += (double)xrow[xc] * (double)yrow[v];
            }
          }
        double got = 0.0;
        const size_t e_tc = ((((size_t)d * 4 + j / 32) * 8 + (j % 32) / 4) * KC + i) * 4 + (j % 4);   // slot order of the kernel
        for (int c = 0; c < ncta; ++c) got += (double)ho[(size_t)c * 9 * KC * KC + e_tc];
        const double ae = fabs(got - ref), re = ae / fmax(fabs(ref), 1e-30);
        sum_rel += (got - ref) / ref; sum_rel2 += (got - ref) / ref * (got - ref) / ref; ++cnt;
        if (re > max_rel) max_rel = re;
        if (ae > max_abs) max_abs = ae;
        if (fabs(ref) > max_ref) max_ref = fabs(ref);
      }
  }
  const double flop = 2.0 * 9 * KC * KC * (double)B * H * W;
  printf("B=%d H=%d W=%d  grid=(%d,3)  %.3f ms  %.1f TFLOP/s (fp32-equivalent)  max rel err %.3e  max abs err %.3e (max ref %.3e)\n",
         B, H, W, ncta, ms, flop / ms / 1e9, max_rel, max_abs, max_ref);
  const double mean = sum_rel / cnt;
  printf("signed rel err: mean %.3e  std %.3e over %d entries\n", mean, sqrt(fmax(sum_rel2 / cnt - mean * mean, 0.0)), cnt);
  printf(max_rel < 2e-6 ? "PASS\n" : "FAIL\n");
  return 0;
}
