// kernels.cu -- CUDA kernels for sm_100a.  One thread = one row everywhere; rows are read and written with 128-bit
// vector accesses (a warp touches 1 KiB contiguous per operand).  The arithmetic lives in rows.cuh and below.
#include "kernels_dh.cuh"

__constant__ u32 c_base_tabs[1024];                 // table_windowed(G) | table_windowed([392]G) | table_endo(G) | table_endo([392]G)

template <int OP> __global__ void __launch_bounds__(256) k_fp2_op(const void* a, const void* b, void* out, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wa[8], wb[8], wo[8];
  ld8(a, row, wa);
  if (OP == FQ_OP_MUL || OP == FQ_OP_ADD || OP == FQ_OP_SUB) ld8(b, row, wb);
  row_fp2_op<OP>(wa, wb, wo);
  st8(out, row, wo);
}

// GFp2.inv (fields.py:194-199) for FQ_BATCHINV_ROWS rows per thread with ONE x^(p-2) chain (batchinv.cuh: 3 multiplications per row
// instead of a 138-step chain).  inv(0) = 0 as in the reference.  Thread t owns rows t, t + stride, ...; `out` must not alias `a`
// (the prefix products are parked in it).
__global__ void __launch_bounds__(64) k_fp2_inv_batched(const void* __restrict__ a, void* __restrict__ out, size_t n) {
  Fp2InvIO io;
  io.a = reinterpret_cast<const uint4*>(a); io.out = reinterpret_cast<uint4*>(out); io.n = n;
  io.stride = (size_t)gridDim.x * blockDim.x; io.t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  batch_invert<Fp2Ops>(io, FQ_BATCHINV_ROWS);
}

// GF(p) op on 16-byte rows: one 128-bit load per operand and one 128-bit store per thread
template <int OP> __global__ void __launch_bounds__(256) k_fp_op(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  uint4 va = a[row], vb = make_uint4(0, 0, 0, 0);
  if (OP == FQ_FPOP_MUL || OP == FQ_FPOP_ADD || OP == FQ_FPOP_SUB) vb = b[row];
  u32 wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w}, wo[4];
  row_fp_op<OP>(wa, wb, wo);
  out[row] = make_uint4(wo[0], wo[1], wo[2], wo[3]);
}

__global__ void __launch_bounds__(256) k_fp2_invsqrt(const void* a, void* out, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wa[8], wo[8];
  ld8(a, row, wa);
  row_fp2_invsqrt(wa, wo);
  st8(out, row, wo);
}

// GFp.select / GFp2.select: one 128-bit load per operand half, one condition byte per row
template <int HALVES> __global__ void __launch_bounds__(256) k_select(const unsigned char* __restrict__ c, const uint4* __restrict__ x, const uint4* __restrict__ y, uint4* __restrict__ out, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wx[4 * HALVES], wy[4 * HALVES], wo[4 * HALVES];
#pragma unroll
  for (int h = 0; h < HALVES; h++) {
    uint4 vx = x[HALVES * row + h], vy = y[HALVES * row + h];
    wx[4 * h] = vx.x; wx[4 * h + 1] = vx.y; wx[4 * h + 2] = vx.z; wx[4 * h + 3] = vx.w;
    wy[4 * h] = vy.x; wy[4 * h + 1] = vy.y; wy[4 * h + 2] = vy.z; wy[4 * h + 3] = vy.w;
  }
  row_select<HALVES>(c[row], wx, wy, wo);
#pragma unroll
  for (int h = 0; h < HALVES; h++) out[HALVES * row + h] = make_uint4(wo[4 * h], wo[4 * h + 1], wo[4 * h + 2], wo[4 * h + 3]);
}

template <bool SPEC> __global__ void __launch_bounds__(256) k_decode(const void* enc, void* xy, unsigned char* status, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 we[8], wo[16];
  ld8(enc, row, we);
  status[row] = (unsigned char)row_decode<SPEC>(we, wo);
  st8(xy, 2 * row, wo); st8(xy, 2 * row + 1, wo + 8);
}

// PointOnCurve (curve4q.py:23-29) on affine rows x | y (any 128-bit halves, reduced mod p): ok[row] = 1 if on the curve
__global__ void __launch_bounds__(256) k_on_curve(const void* xy, unsigned char* ok, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wi[16];
  ld8(xy, 2 * row, wi); ld8(xy, 2 * row + 1, wi + 8);
  fp2 x = fp2_canon(row_load_fp2(wi)), y = fp2_canon(row_load_fp2(wi + 8));
  ok[row] = pt_on_curve(x, y) ? 1 : 0;
}

__global__ void __launch_bounds__(256) k_encode(const void* xy, void* enc, size_t n) {
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wi[16], wo[8];
  ld8(xy, 2 * row, wi); ld8(xy, 2 * row + 1, wi + 8);
  row_encode(wi, wo);
  st8(enc, row, wo);
}

// fixed base, the reference's shape: [k]G (DH = false) or [k][392]G (DH = true) by MUL_windowed / MUL_endo on the base point's
// table.  The CTA copies the 1 KiB table from the constant bank into shared memory once; the selection then reads it by
// broadcast (dh.cuh SelectBroadcast).  The result stays projective: k_dh_finish (kernels_dh.cuh) normalises sixteen rows per
// inversion, rejects the neutral point for DH, and encodes.
template <bool DH, bool ENDO, bool STRICT> __global__ void __launch_bounds__(256)
k_fixed_base(const void* __restrict__ k, DhScratch sc, size_t n) {
  __shared__ uint4 stab[64];
  if (threadIdx.x < 64) {
    const u32* src = c_base_tabs + (ENDO ? 512 : 0) + (DH ? 256 : 0) + 4 * threadIdx.x;
    stab[threadIdx.x] = make_uint4(src[0], src[1], src[2], src[3]);
  }
  __syncthreads();
  size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  u32 wk[8];
  ld8(k, row, wk);
  ptR1 R = row_fixed_base_r1<ENDO, STRICT>(wk, stab);
  uint4* o = sc.R + row;
  stq(o, R.X.re); stq(o + sc.npad, R.X.im); stq(o + 2 * sc.npad, R.Y.re); stq(o + 3 * sc.npad, R.Y.im);
  stq(o + 4 * sc.npad, R.Z.re); stq(o + 5 * sc.npad, R.Z.im);
  sc.meta[row] = 0;
}

__global__ void k_build_base_tables(u32* out, uint4* scratch) { row_build_base_tables(out, scratch); }

// ---------------------------------------------------------------- integer-multiply peak (roofline denominator)
// variant 0: IMAD.WIDE.U32 (mad.lo.cc + madc.hi), variant 1: IMAD (mad.lo.u32).  8 independent chains per thread.
template <int V> __global__ void __launch_bounds__(256) k_imad_peak(u32* out, u32 b, int trips) {
  u32 lo[8], hi[8];
#pragma unroll
  for (int i = 0; i < 8; i++) { lo[i] = threadIdx.x + i; hi[i] = blockIdx.x + 3 * i; }
  for (int t = 0; t < trips; t++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
#pragma unroll
      for (int i = 0; i < 8; i++) {
        if (V == 0) asm volatile("mad.lo.cc.u32 %0,%2,%3,%0; madc.hi.u32 %1,%2,%3,%1;" : "+r"(lo[i]), "+r"(hi[i]) : "r"(lo[(i + 4) & 7]), "r"(b));
        else asm volatile("mad.lo.u32 %0,%0,%1,%2;" : "+r"(lo[i]) : "r"(b), "r"(hi[i]));
      }
    }
  }
  u32 s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s ^= lo[i] ^ hi[i];
  if (s == 0x12345678u) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ---------------------------------------------------------------- launch wrappers


cudaError_t fqk_device_init(cudaStream_t s) {
  cudaError_t e;
  if ((e = fqk_dh_windowed_init()) != cudaSuccess) return e;
  if ((e = fqk_dh_endo_init()) != cudaSuccess) return e;
  u32* tabs = nullptr; uint4* scratch = nullptr;
  if ((e = cudaMalloc(&tabs, 1024 * sizeof(u32))) != cudaSuccess) return e;
  if ((e = cudaMalloc(&scratch, 56 * sizeof(uint4))) != cudaSuccess) { cudaFree(tabs); return e; }
  k_build_base_tables<<<1, 1, 0, s>>>(tabs, scratch);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(c_base_tabs, tabs, 1024 * sizeof(u32), 0, cudaMemcpyDeviceToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(tabs); cudaFree(scratch);
  return e;
}

cudaError_t fqk_fp2_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  unsigned g = grid_for(n, 256);
  switch (op) {
    case FQK_MUL: k_fp2_op<FQ_OP_MUL><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_SQR: k_fp2_op<FQ_OP_SQR><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_INV: k_fp2_inv_batched<<<grid_for((n + FQ_BATCHINV_ROWS - 1) / FQ_BATCHINV_ROWS, 64), 64, 0, s>>>(a, out, n); break;
    case FQK_ADD: k_fp2_op<FQ_OP_ADD><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_SUB: k_fp2_op<FQ_OP_SUB><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_NEG: k_fp2_op<FQ_OP_NEG><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_CONJ: k_fp2_op<FQ_OP_CONJ><<<g, 256, 0, s>>>(a, b, out, n); break;
    case FQK_INVSQRT: k_fp2_invsqrt<<<g, 256, 0, s>>>(a, out, n); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
cudaError_t fqk_fp_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  unsigned g = grid_for(n, 256);
  const uint4* A = (const uint4*)a; const uint4* B = (const uint4*)b; uint4* O = (uint4*)out;
  switch (op) {
    case FQ_FPOP_MUL: k_fp_op<FQ_FPOP_MUL><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_SQR: k_fp_op<FQ_FPOP_SQR><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_INV: k_fp_op<FQ_FPOP_INV><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_ADD: k_fp_op<FQ_FPOP_ADD><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_SUB: k_fp_op<FQ_FPOP_SUB><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_NEG: k_fp_op<FQ_FPOP_NEG><<<g, 256, 0, s>>>(A, B, O, n); break;
    case FQ_FPOP_INVSQRT: k_fp_op<FQ_FPOP_INVSQRT><<<g, 256, 0, s>>>(A, B, O, n); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
cudaError_t fqk_select(int halves, const void* c, const void* x, const void* y, void* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  if (halves == 2) k_select<2><<<grid_for(n, 256), 256, 0, s>>>((const unsigned char*)c, (const uint4*)x, (const uint4*)y, (uint4*)out, n);
  else k_select<1><<<grid_for(n, 256), 256, 0, s>>>((const unsigned char*)c, (const uint4*)x, (const uint4*)y, (uint4*)out, n);
  return cudaGetLastError();
}
cudaError_t fqk_decode(int spec, const void* enc, void* xy, void* status, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  if (spec) k_decode<true><<<grid_for(n, 256), 256, 0, s>>>(enc, xy, (unsigned char*)status, n);
  else k_decode<false><<<grid_for(n, 256), 256, 0, s>>>(enc, xy, (unsigned char*)status, n);
  return cudaGetLastError();
}
cudaError_t fqk_on_curve(const void* xy, void* ok, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  k_on_curve<<<grid_for(n, 256), 256, 0, s>>>(xy, (unsigned char*)ok, n);
  return cudaGetLastError();
}
cudaError_t fqk_encode(const void* xy, void* enc, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  k_encode<<<grid_for(n, 256), 256, 0, s>>>(xy, enc, n);
  return cudaGetLastError();
}
size_t fqk_dh_scratch_bytes(size_t n) { return dh_scratch_bytes(n < FQ_DH_MAX_BATCH ? n : FQ_DH_MAX_BATCH); }
cudaError_t fqk_dh(int affine, int endo, int strict, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch, cudaStream_t s, cudaEvent_t* ev) {
  if (n == 0) return cudaSuccess;
  return endo ? fqk_dh_endo(affine, strict, k, pt, out, status, n, scratch, s, ev) : fqk_dh_windowed(affine, strict, k, pt, out, status, n, scratch, s, ev);
}
template <bool STRICT> static void fixed_base_launch(int dh, int endo, unsigned g, const void* k, DhScratch sc, size_t n, cudaStream_t s) {
  if (dh && endo) k_fixed_base<true, true, STRICT><<<g, 256, 0, s>>>(k, sc, n);
  else if (dh) k_fixed_base<true, false, STRICT><<<g, 256, 0, s>>>(k, sc, n);
  else if (endo) k_fixed_base<false, true, STRICT><<<g, 256, 0, s>>>(k, sc, n);
  else k_fixed_base<false, false, STRICT><<<g, 256, 0, s>>>(k, sc, n);
}
// scratch: fqk_comb_scratch_bytes(n) bytes (the same projective hand-over as the comb kernel)
cudaError_t fqk_fixed_base(int dh, int endo, int strict, const void* k, void* out, void* status, size_t n, void* scratch, cudaStream_t s) {
  for (size_t r0 = 0; r0 < n; r0 += FQ_DH_MAX_BATCH) {
    const size_t rows = n - r0 < FQ_DH_MAX_BATCH ? n - r0 : FQ_DH_MAX_BATCH;
    DhScratch sc = fin_scratch_view(scratch, rows);
    unsigned g = grid_for(rows, 256);
    const char* kk = (const char*)k + 32 * r0; char* oo = (char*)out + 32 * r0;
    unsigned char* st = status ? (unsigned char*)status + r0 : nullptr;
    if (strict) fixed_base_launch<true>(dh, endo, g, kk, sc, rows, s);
    else fixed_base_launch<false>(dh, endo, g, kk, sc, rows, s);
    if (dh) k_dh_finish<false, true><<<dh_finish_grid(rows), FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    else k_dh_finish<false, false><<<dh_finish_grid(rows), FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
cudaError_t fqk_imad_peak(int variant, void* scratch, int blocks, int trips, cudaStream_t s) {
  if (variant == 0) k_imad_peak<0><<<blocks, 256, 0, s>>>((u32*)scratch, 0x9e3779b9u, trips);
  else k_imad_peak<1><<<blocks, 256, 0, s>>>((u32*)scratch, 0x9e3779b9u, trips);
  return cudaGetLastError();
}
