// Stand-alone harness for the packed tcgen05 local joint at 16 <= K <= 24, padding 1 or 3 (csrc/local_fwd_tcp.cu):
// runs the kernel on random simplex-like maps, adds the per-CTA slots in fp64 and compares a sample of entries with
// an fp64 CPU loop; prints the time per launch and the fp32-equivalent TFLOP/s.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/_bin/tc_jointp tools/tc_jointp_harness.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tc_jointp [B H W K pad]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_fwd_tcp.cu"

int main(int argc, char** argv) {
  int B = 1, H = 6, W = 32, KC = 20, pad = 1;
  if (argc >= 4) { B = atoi(argv[1]); H = atoi(argv[2]); W = atoi(argv[3]); }
  if (argc >= 6) { KC = atoi(argv[4]); pad = atoi(argv[5]); }
  const int T = 2 * pad + 1;
  const size_t n = (size_t)B * KC * H * W;
  std::vector<float> hx(n), hy(n);
  srand(1);
  for (size_t i = 0; i < n; ++i) {
    const float a = (float)rand() / RAND_MAX, b = (float)rand() / RAND_MAX;
    hx[i] = a * a * a * 0.3f;
    hy[i] = b * b * b * 0.3f;
  }
  float *dx_, *dy_, *dws;
  double* dJ;
  cudaMalloc(&dx_, n * 4); cudaMalloc(&dy_, n * 4);
  cudaMemcpy(dx_, hx.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dy_, hy.data(), n * 4, cudaMemcpyHostToDevice);
  const size_t E = (size_t)T * T * KC * KC;
  const int sms = iic::sm_count_cached(iic::current_device());
  const size_t wsf = iic::local_joint_tcp_slot_floats(KC, pad) * sms;
  cudaMalloc(&dws, wsf * 4);
  cudaMemset(dws, 0xff, wsf * 4);
  cudaMalloc(&dJ, E * 8);
  const long long sc = (long long)H * W, sn = sc * KC;
  const iic::LocalMaps m{{dx_, sn, sc, W}, {dy_, sn, sc, W}, B, KC, H, W, pad, sms};
  auto run = [&]() {           // the joint, then the slot reduce of iic_local_joint
    iic::SlotInfo s{};
    const int rc = iic::local_joint_tcp_try(m, dws, wsf, &s, 0);
    if (rc == 0)
      iic::fwdtcp::reduce_packed_kernel<<<(int)((E + 31) / 32), 1024>>>(dws, s.n_slots, (int)s.slot_stride, T, KC, s.nb, dJ);
    return rc;
  };
  int rc = run();
  cudaError_t err = cudaDeviceSynchronize();
  printf("try rc=%d (%s); first launch: %s\n", rc, iic::get_error(), cudaGetErrorString(err));
  if (rc != 0 || err != cudaSuccess) return 1;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int reps = 5;
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) run();
  cudaEventRecord(e1);
  err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("timed launches: %s\n", cudaGetErrorString(err)); return 1; }
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
#ifdef IIC_TC_TRACE
  {
    long long tr[3][64][6];
    cudaMemcpyFromSymbol(tr, iic::fwdtcp::g_trace, sizeof(tr));
    const long long t0 = tr[0][0][0];
    printf("k | producer: enter waited issued | mma: enter op_full_ok issued | transform(w4): enter raw_ok op_empty_ok done arrived   (clk rel.)\n");
    for (int k = 0; k < 24; ++k)
      printf("%2d | %7lld %7lld %7lld | %7lld %7lld %7lld | %7lld %7lld %7lld %7lld %7lld\n", k + 64, tr[0][k][0] - t0, tr[0][k][1] - t0, tr[0][k][2] - t0,
             tr[1][k][0] - t0, tr[1][k][1] - t0, tr[1][k][2] - t0, tr[2][k][0] - t0, tr[2][k][1] - t0, tr[2][k][2] - t0, tr[2][k][3] - t0, tr[2][k][4] - t0);
  }
#endif
  std::vector<double> hJ(E);
  cudaMemcpy(hJ.data(), dJ, E * 8, cudaMemcpyDeviceToHost);
  double max_rel = 0.0, sum_rel = 0.0, sum_rel2 = 0.0; int cnt = 0;
  for (int ddy = 0; ddy < T; ++ddy) for (int ddx = 0; ddx < T; ++ddx)
    for (int i = 0; i < KC; i += 3)
      for (int j = 0; j < KC; j += 7) {
        double ref = 0.0;
        for (int b = 0; b < B; ++b)
          for (int u = 0; u < H; ++u) {
            const int xr = u + ddy - pad;
            if (xr < 0 || xr >= H) continue;
            const float* xrow = &hx[((size_t)(b * KC + i) * H + xr) * W];
            const float* yrow = &hy[((size_t)(b * KC + j) * H + u) * W];
            for (int v = 0; v < W; ++v) {
              const int xc = v + ddx - pad;
              if (xc < 0 || xc >= W) continue;
              ref += (double)xrow[xc] * (double)yrow[v];
            }
          }
        const double got = hJ[(((size_t)ddy * T + ddx) * KC + i) * KC + j];
        const double re = (got - ref) / ref;
        sum_rel += re; sum_rel2 += re * re; ++cnt;
        if (fabs(re) > max_rel) max_rel = fabs(re);
      }
  const double flop = 2.0 * T * T * KC * KC * (double)B * H * W;
  const double mean = sum_rel / cnt;
  printf("K=%d pad=%d B=%d H=%d W=%d  %.3f ms (joint + slot reduce)  %.1f TFLOP/s (fp32-equivalent)  max rel err %.3e\n", KC, pad, B, H, W, ms,
         flop / ms / 1e9, max_rel);
  printf("signed rel err: mean %.3e  std %.3e over %d entries\n", mean, sqrt(fmax(sum_rel2 / cnt - mean * mean, 0.0)), cnt);
  printf(max_rel < 2e-5 ? "PASS\n" : "FAIL\n");
  return 0;
}
