// Stand-alone timing harness for the fp16-split tensor-core joint (csrc/local_fwd_tcj10.cu): the kernel alone, and with
// one pipeline stage switched off at a time (which stage bounds the row rate).
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -DIIC_TCJ_DEBUG -o tools/_bin/tc_joint10 tools/tc_joint10_harness.cu mi-based-regularized-semi-supervised-segmentation_b200/csrc/runtime.cu
//   tools/_bin/tc_joint10 [B H W K]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../mi-based-regularized-semi-supervised-segmentation_b200/csrc/local_fwd_tcj10.cu"

int main(int argc, char** argv) {
  int B = 32, H = 224, W = 224, K = 10;
  if (argc >= 5) { B = atoi(argv[1]); H = atoi(argv[2]); W = atoi(argv[3]); K = atoi(argv[4]); }
  const size_t n = (size_t)B * K * H * W;
  std::vector<float> h(n);
  srand(3);
  for (size_t i = 0; i < n; ++i) h[i] = (float)rand() / RAND_MAX / K * 2.f;
  const int sms = iic::sm_count_cached(iic::current_device());
  float *dx_, *dy_, *part;
  cudaMalloc(&dx_, n * 4); cudaMalloc(&dy_, n * 4); cudaMalloc(&part, (size_t)sms * 9 * K * K * 4);
  cudaMemcpy(dx_, h.data(), n * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dy_, h.data(), n * 4, cudaMemcpyHostToDevice);
  using namespace iic;
  using namespace iic::fwdtcj10;
  const long long sc = (long long)H * W, sn = sc * K;
  ensure_dyn_smem((const void*)local_joint_tcj10_kernel, SMEM_BYTES);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int m : {0, 1, 10}) {
    Params P;
    P.x = dx_; P.x_sn = sn; P.x_sc = sc; P.x_sh = W;
    P.y = dy_; P.y_sn = sn; P.y_sc = sc; P.y_sh = W;
    P.B = B; P.H = H; P.W = W; P.K = K; P.partial = part; P.flags = nullptr; P.from_logits = 0; P.inv_temp = 1.f; P.dbg = m;
    local_joint_tcj10_kernel<<<sms, NTHREADS, SMEM_BYTES>>>(P);
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { printf("mode %d: %s\n", m, cudaGetErrorString(err)); return 1; }
    const int reps = 5;
    cudaEventRecord(e0);
    for (int r = 0; r < reps; ++r) local_joint_tcj10_kernel<<<sms, NTHREADS, SMEM_BYTES>>>(P);
    cudaEventRecord(e1);
    cudaDeviceSynchronize();
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    {
      static long long tr[8][64];
      cudaMemcpyFromSymbol(tr, g_tcj_trace, sizeof(tr));
      const long long t0 = tr[0][0];
      printf("  CTA 0: init done %lld, all MMAs done %lld, slot written %lld clk\n", tr[0][1] - t0, tr[0][2] - t0, tr[0][3] - t0);
      printf("  pair: w16 issue-start waits-done issued | w16 drain-start done-seen | w17 drain-start done-seen\n");
      if (0) for (int i = 0; i < 14; ++i) printf("  %2d: %7lld %7lld %7lld | %7lld %7lld | %7lld %7lld\n", i, tr[2][i] - t0, tr[1][i] - t0, tr[3][i] - t0, tr[4][i] - t0, tr[5][i] - t0, tr[6][i] - t0, tr[7][i] - t0);
      if (0) for (int i = 0; i < 16; ++i) printf("  %2d: x-top %7lld | y: top %7lld loads-issued %7lld done-wait %7lld published %7lld | issuer %7lld\n", i, tr[2][i] - t0, tr[3][4 * i] - t0, tr[3][4 * i + 1] - t0, tr[3][4 * i + 2] - t0, tr[3][4 * i + 3] - t0, tr[1][i] - t0);
    }
    {
      static unsigned long long ct[160][2];
      cudaMemcpyFromSymbol(ct, g_tcj_cta, sizeof(ct));
      unsigned long long t0 = ~0ull, t1 = 0;
      for (int i = 0; i < sms; ++i) { if (ct[i][0] < t0) t0 = ct[i][0]; if (ct[i][1] > t1) t1 = ct[i][1]; }
      printf("  last launch: first CTA start to last CTA end %.1f us; per CTA (start offset, duration) us:\n   ", (t1 - t0) * 1e-3);
      if (0) for (int i = 0; i < sms; ++i) { printf(" %d:(%.1f,%.1f)", i, (ct[i][0] - t0) * 1e-3, (ct[i][1] - ct[i][0]) * 1e-3); if (i % 8 == 7) printf("\n   "); }
      printf("\n");
    }
    printf("mode %d (%s%s%s%s): %.1f us\n", m, m & 1 ? "no-mma " : "", m & 2 ? "no-transform " : "", m & 4 ? "no-l2-prefetch " : "", m & 8 ? "no-loads" : "", ms / reps * 1e3);
  }
  return 0;
}
