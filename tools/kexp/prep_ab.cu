// prep_ab.cu -- developer experiment: k_dh_prep (and the whole three-kernel step) built from the product headers, as they
// stand or edited for the variant under test, timed alone on 2^20 rows.  Results are not checked here (tests/ does that);
// inputs are the encodings of [k]G produced by the comb kernel, so every row is a valid point.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o prep_ab prep_ab.cu ../../fourq_b200/csrc/kernels_comb.cu
#include <cstdio>
#include <cstdlib>
#include "../../fourq_b200/csrc/kernels_dh.cuh"
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at line %d\n", cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

cudaError_t fqk_comb_init(void** tabs_out, cudaStream_t s);
cudaError_t fqk_comb(int dh, int strict, const void* tabs, const void* k, void* out, void* status, size_t n, void* scratch, int sms, cudaStream_t s);

int main(int argc, char** argv) {
  const size_t n = 1 << 20;
  void *k, *pub, *out, *st, *scratch, *tabs;
  CK(cudaMalloc(&k, n * 32)); CK(cudaMalloc(&pub, n * 32)); CK(cudaMalloc(&out, n * 32)); CK(cudaMalloc(&st, n));
  CK(cudaMalloc(&scratch, dh_scratch_bytes(n)));
  unsigned char* h = (unsigned char*)malloc(n * 32);
  srand(7); for (size_t i = 0; i < n * 32; i++) h[i] = (unsigned char)rand();
  CK(cudaMemcpy(k, h, n * 32, cudaMemcpyHostToDevice));
  CK(fqk_comb_init(&tabs, 0));
  CK(fqk_comb(0, 1, tabs, k, pub, nullptr, n, scratch, 148, 0));
  CK(cudaDeviceSynchronize());
  CK(dh_init<true>()); CK(dh_init<false>());
  cudaEvent_t ev[4]; for (int i = 0; i < 4; i++) CK(cudaEventCreate(&ev[i]));
  for (int endo = 1; endo >= 0; endo--) {
    float best[3] = {1e9f, 1e9f, 1e9f};
    for (int it = 0; it < 6; it++) {
      if (endo) CK(dh_launch<true>(0, 1, k, pub, out, st, n, scratch, 0, ev)); else CK(dh_launch<false>(0, 1, k, pub, out, st, n, scratch, 0, ev));
      CK(cudaDeviceSynchronize());
      for (int i = 0; i < 3; i++) { float ms; CK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1])); if (it > 0 && ms < best[i]) best[i] = ms; }
    }
    cudaFuncAttributes fa;
    if (endo) CK(cudaFuncGetAttributes(&fa, k_dh_prep<false, true>)); else CK(cudaFuncGetAttributes(&fa, k_dh_prep<false, false>));
    printf("%-8s prep %.3f ms (regs %d, stack %zu B)  ladder %.3f ms  finish %.3f ms  step %.3f ms\n", endo ? "endo" : "windowed", best[0], fa.numRegs, fa.localSizeBytes,
           best[1], best[2], best[0] + best[1] + best[2]);
  }
  return 0;
}
