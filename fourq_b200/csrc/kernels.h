// kernels.h -- launch wrappers of kernels.cu (device pointers, one stream).  Internal to the library.
#pragma once
#include <cstddef>
#ifdef FQ_MOCK_CUDA
#include "mock_cuda_runtime.h"
#else
#include <cuda_runtime.h>
#endif

enum { FQK_MUL = 0, FQK_SQR = 1, FQK_INV = 2, FQK_ADD = 3, FQK_SUB = 4, FQK_NEG = 5, FQK_CONJ = 6, FQK_INVSQRT = 7 };

cudaError_t fqk_device_init(cudaStream_t s);   // once per device: fixed-base tables -> __constant__, smem opt-in
cudaError_t fqk_fp2_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s);
cudaError_t fqk_fp_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s);   // GF(p), 16-byte rows, op = FQ_FP_* of the header
// GFp.select / GFp2.select (fields.py:59-64, :236-238): halves = 1 (16-byte rows) or 2 (32-byte rows), c = one condition byte per row
cudaError_t fqk_select(int halves, const void* c, const void* x, const void* y, void* out, size_t n, cudaStream_t s);
cudaError_t fqk_decode(int spec, const void* enc, void* xy, void* status, size_t n, cudaStream_t s);   // spec: draft's t == 0 branch instead of the reference's exception
cudaError_t fqk_encode(const void* xy, void* enc, size_t n, cudaStream_t s);
cudaError_t fqk_on_curve(const void* xy, void* ok, size_t n, cudaStream_t s);

// Device scratch of the operations whose kernels hand rows over to each other.  Each layout is sized here and nowhere else:
// the kernels cut their views with these functions and the caller, who owns the buffer, reserves fqk_*_scratch_bytes(n).
// Every array is [component][row] over npad rows, so that warps move whole 512 B lines.
#define FQ_DH_THREADS 128                            // rows per CTA of k_dh_prep and k_dh_ladder
#define FQ_DH_SCRATCH_QUADS (64 + 2 + 6)             // table | digit register | (X, Y, Z), 16 B each
#define FQ_DH_MAX_BATCH ((size_t)1 << 22)            // rows per launch group (keeps the u32 table indices in range)
// variable-base DH (kernels_dh.cuh DhScratch): FQ_DH_SCRATCH_QUADS quads and one meta word per row, rows padded to one CTA
inline size_t dh_scratch_npad(size_t rows) { return (rows + FQ_DH_THREADS - 1) / FQ_DH_THREADS * FQ_DH_THREADS; }
inline size_t dh_scratch_bytes(size_t rows) { return dh_scratch_npad(rows) * (FQ_DH_SCRATCH_QUADS * 16 + 4); }
// (X, Y, Z) and the meta word that the fixed-base kernels hand to k_dh_finish (kernels_dh.cuh fin_scratch_view), rows padded
// to one 256-thread CTA of those kernels
inline size_t fin_scratch_npad(size_t rows) { return (rows + 255) / 256 * 256; }
inline size_t fin_scratch_bytes(size_t rows) { return fin_scratch_npad(rows) * (6 * 16 + 4); }
// X25519 (x25519.cu): x2 and z2 of every row, two quads each, rows padded to one 128-thread CTA of k_x25519
inline size_t x25519_scratch_npad(size_t rows) { return (rows + 127) / 128 * 128; }
inline size_t x25519_scratch_bytes(size_t rows) { return x25519_scratch_npad(rows) * 4 * 16; }
// what the caller reserves for one call of fqk_dh, fqk_fixed_base / fqk_comb and fqk_x25519: the sizes above for
// min(n, FQ_DH_MAX_BATCH) rows (the DH ones run in launch groups) or n rows (X25519).  Defined next to the kernels, and over
// the same functions by the mock kernels of the host-engine tests.
size_t fqk_dh_scratch_bytes(size_t n);
size_t fqk_comb_scratch_bytes(size_t n);
size_t fqk_x25519_scratch_bytes(size_t n);

// `strict` (everywhere below): table selection by the strict scan instead of masked loads (dh.cuh, fq_set_select_mode)
// variable-base DH = three kernels (prepare, ladder, finish; kernels_dh.cuh) that hand the per-row table and the projective
// result over through `scratch`, a device buffer of at least fqk_dh_scratch_bytes(n) bytes owned by the caller.
// ev: optional array of 4 events recorded before/between/after the three kernels (per-kernel timing).
cudaError_t fqk_dh(int affine, int endo, int strict, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch, cudaStream_t s, cudaEvent_t* ev);
// per-algorithm translation units (kernels_dh_windowed.cu, kernels_dh_endo.cu)
cudaError_t fqk_dh_windowed_init();
cudaError_t fqk_dh_endo_init();
cudaError_t fqk_dh_windowed(int affine, int strict, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch, cudaStream_t s, cudaEvent_t* ev);
cudaError_t fqk_dh_endo(int affine, int strict, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch, cudaStream_t s, cudaEvent_t* ev);
cudaError_t fqk_fixed_base(int dh, int endo, int strict, const void* k, void* out, void* status, size_t n, void* scratch, cudaStream_t s);   // scratch: fqk_comb_scratch_bytes(n)
// fixed-base per-digit tables (kernels_comb.cu): tabs is the device buffer returned by fqk_comb_init
cudaError_t fqk_comb_init(void** tabs_out, cudaStream_t s);
cudaError_t fqk_comb(int dh, int strict, const void* tabs, const void* k, void* out, void* status, size_t n, void* scratch, int sms, cudaStream_t s);   // scratch: fqk_comb_scratch_bytes(n)
cudaError_t fqk_x25519(const void* k, const void* u, void* out, size_t n, void* scratch, cudaStream_t s);   // scratch: fqk_x25519_scratch_bytes(n)
cudaError_t fqk_f25_op(int op, const void* a, const void* b, void* out, size_t n, cudaStream_t s);   // GF(2^255-19), 32-byte rows, op = FQ_FP_MUL.._SUB of the header
cudaError_t fqk_imad_peak(int variant, void* scratch, int blocks, int trips, cudaStream_t s);
