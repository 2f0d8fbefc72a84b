// mock_kernels.cpp -- TEST INFRASTRUCTURE ONLY.  The launch wrappers of fourq_b200/csrc/kernels.h for the mock CUDA runtime:
// each "launch" enqueues, on the mock stream, the CPU instruction-level simulation of the same device code (hostsim.cpp), so
// that the host engine of capi.cu can be tested end to end without a GPU.  Scratch buffers are filled over their whole
// declared size, so that an undersized reservation shows up under AddressSanitizer.
#define FQ_MOCK_CUDA 1
#include <cstdint>
#include <cstring>
#include "../../fourq_b200/csrc/kernels.h"

extern "C" {
int sim_fp2_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
int sim_fp2_inv_batched(const uint8_t* a, uint8_t* out, size_t n, int rows_per_thread);
int sim_fp2_invsqrt(const uint8_t* a, uint8_t* out, size_t n);
int sim_select(int halves, const uint8_t* c, const uint8_t* x, const uint8_t* y, uint8_t* out, size_t n);
int sim_fp_row_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
int sim_decode(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n);
int sim_decode_spec(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n);
int sim_encode(const uint8_t* xy, uint8_t* enc, size_t n);
int sim_on_curve(const uint8_t* xy, uint8_t* ok, size_t n);
int sim_dh(const uint8_t* k, const uint8_t* enc, uint8_t* out, uint8_t* status, size_t n);
int sim_dh_affine(const uint8_t* k, const uint8_t* xy, uint8_t* out, uint8_t* status, size_t n);
int sim_dh_endo(const uint8_t* k, const uint8_t* enc, uint8_t* out, uint8_t* status, size_t n);
int sim_dh_endo_affine(const uint8_t* k, const uint8_t* xy, uint8_t* out, uint8_t* status, size_t n);
int sim_fixed_base(int dh, const uint8_t* k, uint8_t* out, uint8_t* status, size_t n);
int sim_comb(int dh, const uint8_t* k, uint8_t* out, uint8_t* status, size_t n);
int sim_x25519_batched(const uint8_t* k, const uint8_t* u, uint8_t* out, size_t n, int rows_per_thread);
int sim_f25_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
int sim_f25_inv_batched(const uint8_t* a, uint8_t* out, size_t n, int rows_per_thread);
}
typedef const uint8_t* cu8;
typedef uint8_t* u8;

cudaError_t fqk_device_init(cudaStream_t) { return cudaSuccess; }
cudaError_t fqk_fp2_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] {
    if (op == FQK_INV) sim_fp2_inv_batched((cu8)a, (u8)out, n, 16);
    else if (op == FQK_INVSQRT) sim_fp2_invsqrt((cu8)a, (u8)out, n);
    else sim_fp2_op(op, (cu8)a, (cu8)b, (u8)out, n);
  });
  return cudaSuccess;
}
cudaError_t fqk_fp_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { sim_fp_row_op(op, (cu8)a, (cu8)b, (u8)out, n); });
  return cudaSuccess;
}
cudaError_t fqk_select(int halves, const void* c, const void* x, const void* y, void* out, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { sim_select(halves, (cu8)c, (cu8)x, (cu8)y, (u8)out, n); });
  return cudaSuccess;
}
cudaError_t fqk_decode(int spec, const void* enc, void* xy, void* status, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { if (spec) sim_decode_spec((cu8)enc, (u8)xy, (u8)status, n); else sim_decode((cu8)enc, (u8)xy, (u8)status, n); });
  return cudaSuccess;
}
cudaError_t fqk_encode(const void* xy, void* enc, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { sim_encode((cu8)xy, (u8)enc, n); });
  return cudaSuccess;
}
cudaError_t fqk_on_curve(const void* xy, void* ok, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { sim_on_curve((cu8)xy, (u8)ok, n); });
  return cudaSuccess;
}
size_t fqk_dh_scratch_bytes(size_t n) { return dh_scratch_bytes(n < FQ_DH_MAX_BATCH ? n : FQ_DH_MAX_BATCH); }
cudaError_t fqk_dh(int affine, int endo, int, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch, cudaStream_t s, cudaEvent_t* ev) {
  if (ev) cudaEventRecord(ev[0], s);
  mock_stream_enqueue(s, [=] {
    memset(scratch, 0x11, fqk_dh_scratch_bytes(n));
    if (endo) { if (affine) sim_dh_endo_affine((cu8)k, (cu8)pt, (u8)out, (u8)status, n); else sim_dh_endo((cu8)k, (cu8)pt, (u8)out, (u8)status, n); }
    else { if (affine) sim_dh_affine((cu8)k, (cu8)pt, (u8)out, (u8)status, n); else sim_dh((cu8)k, (cu8)pt, (u8)out, (u8)status, n); }
  });
  if (ev) { cudaEventRecord(ev[1], s); cudaEventRecord(ev[2], s); cudaEventRecord(ev[3], s); }
  return cudaSuccess;
}
size_t fqk_comb_scratch_bytes(size_t n) { return fin_scratch_bytes(n < FQ_DH_MAX_BATCH ? n : FQ_DH_MAX_BATCH); }
cudaError_t fqk_fixed_base(int dh, int endo, int, const void* k, void* out, void* status, size_t n, void* scratch, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { memset(scratch, 0x11, fqk_comb_scratch_bytes(n)); sim_fixed_base(dh | (endo << 1), (cu8)k, (u8)out, (u8)status, n); });
  return cudaSuccess;
}
cudaError_t fqk_comb_init(void** tabs_out, cudaStream_t) { return cudaMalloc(tabs_out, 64); }
cudaError_t fqk_comb(int dh, int, const void*, const void* k, void* out, void* status, size_t n, void* scratch, int, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { memset(scratch, 0x11, fqk_comb_scratch_bytes(n)); sim_comb(dh, (cu8)k, (u8)out, (u8)status, n); });
  return cudaSuccess;
}
size_t fqk_x25519_scratch_bytes(size_t n) { return x25519_scratch_bytes(n); }
cudaError_t fqk_x25519(const void* k, const void* u, void* out, size_t n, void* scratch, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { memset(scratch, 0x11, fqk_x25519_scratch_bytes(n)); sim_x25519_batched((cu8)k, (cu8)u, (u8)out, n, 16); });
  return cudaSuccess;
}
cudaError_t fqk_f25_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  mock_stream_enqueue(s, [=] { if (op == 2) sim_f25_inv_batched((cu8)a, (u8)out, n, 16); else sim_f25_op(op, (cu8)a, (cu8)b, (u8)out, n); });
  return cudaSuccess;
}
cudaError_t fqk_imad_peak(int, void*, int, int, cudaStream_t) { return cudaSuccess; }
