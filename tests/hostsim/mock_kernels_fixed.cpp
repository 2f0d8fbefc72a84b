// mock_kernels_fixed.cpp -- TEST INFRASTRUCTURE ONLY.  The mock launch wrappers of mock_kernels.cpp plus those of registered
// bases, for the host-engine tests of tests/test_fixed_base.py (built by build_fixed_base.sh in place of mock_kernels.cpp).
// The "tables" of a mock device are 64 bytes: for G (fqk_comb_init of mock_kernels.cpp) the mock allocator's 0xA5 fill, for a
// registered base (fqk_comb_build) the canonical point x | y, whose byte 15 is below 0x80.  fqk_comb simulates the tables
// of the base they stand for: G through mock_kernels.cpp's wrapper (renamed here), a registered point through sim_comb_point.
#define fqk_comb fqk_comb_of_g
#include "mock_kernels.cpp"
#undef fqk_comb

extern "C" int sim_comb_point(int dh, const uint8_t* xy, const uint8_t* k, uint8_t* out, uint8_t* status, size_t n);

// mirrors the failure paths of the real wrapper: the buffer is freed when the stream synchronisation fails
cudaError_t fqk_comb_build(const void* xy, void** tabs_out, cudaStream_t s) {
  void* t = nullptr;
  cudaError_t e = cudaMalloc(&t, 64);
  if (e != cudaSuccess) return e;
  uint8_t pt[64]; memcpy(pt, xy, 64);
  mock_stream_enqueue(s, [=] { memcpy(t, pt, 64); });
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) { cudaFree(t); return e; }
  *tabs_out = t;
  return cudaSuccess;
}
cudaError_t fqk_comb(int dh, int strict, const void* tabs, const void* k, void* out, void* status, size_t n, void* scratch, int sms, cudaStream_t s) {
  if (((const uint8_t*)tabs)[15] >= 0x80) return fqk_comb_of_g(dh, strict, tabs, k, out, status, n, scratch, sms, s);
  mock_stream_enqueue(s, [=] { memset(scratch, 0x11, fqk_comb_scratch_bytes(n)); sim_comb_point(dh, (cu8)tabs, (cu8)k, (u8)out, (u8)status, n); });
  return cudaSuccess;
}
