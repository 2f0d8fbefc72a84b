// x25519.cu -- batched X25519 kernels (config 5 of BASELINE.json: the compare.py counterpart).
// Two kernels, like the Curve4Q DH path: k_x25519 runs the 255-step ladder of a row and leaves x2, z2 in scratch;
// k_x25519_finish computes x2 / z2 for FQ_BATCHINV_ROWS rows of a thread with ONE z^(p-2) chain (batchinv.cuh).  The
// reference's z2^(p-2) maps z2 = 0 to 0 (curve25519.py:80): zeros are replaced by 1 in the shared product and their output
// forced to 0.
#include "kernels.h"
#include "x25519.cuh"
#include "batchinv.cuh"
#include "kio.cuh"

__global__ void __launch_bounds__(128) k_x25519(const void* __restrict__ k, const void* __restrict__ u, uint4* __restrict__ scratch, size_t npad, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 kw[8], uw[8];
  ld8(k, row, kw); ld8(u, row, uw);
  f25 x2, z2;
  x25519_ladder(kw, uw, x2, z2);
  st_f25(scratch + row, npad, x2); st_f25(scratch + 2 * npad + row, npad, z2);
}

__global__ void __launch_bounds__(64) k_x25519_finish(const uint4* __restrict__ scratch, size_t npad, void* __restrict__ out, size_t n) {
  X25519FinIO io;
  io.scratch = scratch; io.npad = npad; io.out = reinterpret_cast<uint4*>(out); io.n = n;
  io.stride = (size_t)gridDim.x * blockDim.x; io.t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  batch_invert<F25Ops>(io, FQ_BATCHINV_ROWS);
}

size_t fqk_x25519_scratch_bytes(size_t n) { return x25519_scratch_bytes(n); }

cudaError_t fqk_x25519(const void* k, const void* u, void* out, size_t n, void* scratch, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const size_t npad = x25519_scratch_npad(n);
  k_x25519<<<(unsigned)(npad / 128), 128, 0, s>>>(k, u, (uint4*)scratch, npad, n);
  const size_t groups = (n + FQ_BATCHINV_ROWS - 1) / FQ_BATCHINV_ROWS;
  k_x25519_finish<<<(unsigned)((groups + 63) / 64), 64, 0, s>>>((const uint4*)scratch, npad, out, n);
  return cudaGetLastError();
}

// GFp25519 field ops (fields.py:267-362), one thread = one 32-byte row; inv shares one chain between FQ_BATCHINV_ROWS rows
template <int OP> __global__ void __launch_bounds__(256) k_f25_op(const void* a, const void* b, void* out, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wa[8], wb[8], wo[8];
  ld8(a, row, wa);
  if (OP == FQ_F25OP_MUL || OP == FQ_F25OP_ADD || OP == FQ_F25OP_SUB) ld8(b, row, wb);
  row_f25_op<OP>(wa, wb, wo);
  st8(out, row, wo);
}
__global__ void __launch_bounds__(64) k_f25_inv_batched(const void* __restrict__ a, void* __restrict__ out, size_t n) {
  F25InvIO io;
  io.a = reinterpret_cast<const uint4*>(a); io.out = reinterpret_cast<uint4*>(out); io.n = n;
  io.stride = (size_t)gridDim.x * blockDim.x; io.t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  batch_invert<F25Ops>(io, FQ_BATCHINV_ROWS);
}
cudaError_t fqk_f25_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned g = (unsigned)((n + 255) / 256);
  switch (op) {
    case FQ_F25OP_MUL: k_f25_op<FQ_F25OP_MUL><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQ_F25OP_SQR: k_f25_op<FQ_F25OP_SQR><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQ_F25OP_ADD: k_f25_op<FQ_F25OP_ADD><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQ_F25OP_SUB: k_f25_op<FQ_F25OP_SUB><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQ_F25OP_INV: {
      const size_t groups = (n + FQ_BATCHINV_ROWS - 1) / FQ_BATCHINV_ROWS;
      k_f25_inv_batched<<<(unsigned)((groups + 63) / 64), 64, 0, s>>>(a, out, n);
      break;
    }
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
