// kernels_dh.cuh -- variable-base Diffie-Hellman kernels (fq_dh, fq_dh_affine, fq_dh_endo, fq_dh_endo_affine).
// Included by kernels_dh_windowed.cu and kernels_dh_endo.cu (one translation unit per algorithm: they compile in parallel).
//
// Shape.  One thread = one row, three kernels per batch, each sized for what bounds it (profiles/, DESIGN.md 6):
//   k_dh_prep    decode + validate, [392]P, (endomorphisms,) table T[0..7] in R2, scalar plan.  Straight-line code with
//                out-of-line field/point routines, no shared memory, <= 170 registers: three CTAs of 128 threads per SM.
//                The table goes to a scratch buffer in HBM laid out [entry][quad][row] (1 KiB per row, coalesced).
//   k_dh_ladder  copies the row's table into shared memory ([entry][quad][thread], 112 KiB per CTA, entry 7 in
//                registers) and runs the 64 x (DBL + ADD) or 62 x (4 DBL + ADD) loop; two CTAs per SM (shared memory
//                and the 248 registers of the strict-scan loop both allow 256 threads).  Writes (X, Y, Z) to scratch.
//   k_dh_finish  each thread normalises FQ_BATCHINV_ROWS rows with ONE inversion (Montgomery's trick: prefix products parked
//                in the output rows, one x^(p-2) chain, back-substitution), checks for the neutral point, encodes, writes
//                result and status (batchinv.cuh).
// All three are bound by integer-instruction issue (IMAD.WIDE.U32 at half rate plus its carry handling); the split lets
// the setup run with 12 warps per SM instead of 8 and removes 3/4 of the inversions.  The scratch traffic (2.3 KiB per
// row) is ~3 % of HBM bandwidth at the measured row rate.  (The same row as ONE fused kernel lives in tools/kexp/fused_dh.cuh
// for A/B experiments; it is not part of the library.)
#pragma once
#include "kernels.h"
#include "kio.cuh"
#include "batchinv.cuh"

#define FQ_DH_SMEM (56 * 16 * FQ_DH_THREADS)       // 7 table entries x 8 quads x 16 B per thread = 112 KiB per CTA

// ---------------------------------------------------------------- the three-kernel pipeline

// scratch of one batch (sized in kernels.h): npad rows, a multiple of FQ_DH_THREADS
struct DhScratch { uint4* tab; uint4* plan; uint4* R; u32* meta; size_t npad; };

static inline DhScratch dh_scratch_view(void* base, size_t rows) {
  DhScratch sc;
  sc.npad = dh_scratch_npad(rows);
  sc.tab = reinterpret_cast<uint4*>(base); sc.plan = sc.tab + 64 * sc.npad; sc.R = sc.plan + 2 * sc.npad;
  sc.meta = reinterpret_cast<u32*>(sc.R + 6 * sc.npad);
  return sc;
}

__device__ __forceinline__ void stq(uint4* p, const fp& a) { *p = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]); }
__device__ __forceinline__ fp ldq(const uint4* p) { uint4 w = *p; return fp_set(w.x, w.y, w.z, w.w); }

// three CTAs per SM with the endomorphisms (a fourth would spill), four without (measured: 3.26 vs 3.47 ms, 2.15 vs 2.21 ms)
template <bool AFFINE, bool ENDO> __global__ void __launch_bounds__(FQ_DH_THREADS, ENDO ? 3 : 4)
k_dh_prep(const void* __restrict__ k, const void* __restrict__ pt, DhScratch sc, size_t n) {
  const size_t row = (size_t)blockIdx.x * FQ_DH_THREADS + threadIdx.x;
  const size_t src = row < n ? row : n - 1;          // tail threads recompute the last row (their scratch slots exist)
  TabView T; T.base = sc.tab + row; T.stride = (u32)sc.npad;
  u32 wk[8], wp[AFFINE ? 16 : 8];
  ld8(k, src, wk);
  if (AFFINE) { ld8(pt, 2 * src, wp); ld8(pt, 2 * src + 1, wp + 8); } else ld8(pt, src, wp);
  DhState D;
  u32 st = row_dh_setup<ENDO, AFFINE>(wk, wp, T, D);
  tab_store(T, 7, D.T7);
  sc.plan[row] = make_uint4(D.plan.S.v[0], D.plan.S.v[1], D.plan.S.v[2], D.plan.S.v[3]);
  sc.plan[sc.npad + row] = make_uint4(D.plan.S.v[4], D.plan.S.v[5], D.plan.S.v[6], D.plan.S.v[7]);
  sc.meta[row] = D.plan.first | (st << 8);
}

// no register cap: every cap below the 248 registers of the strict loop measured slower, and the shared-memory table alone
// limits the ladder to two CTAs per SM (DESIGN.md 6, profiles/r02_ladder_regcap.txt)
template <bool ENDO, bool STRICT> __global__ void __maxnreg__(255)
k_dh_ladder(DhScratch sc) {
  extern __shared__ uint4 smem[];
  const size_t row = (size_t)blockIdx.x * FQ_DH_THREADS + threadIdx.x;
  TabView T; T.base = smem + threadIdx.x; T.stride = FQ_DH_THREADS;
  const uint4* g = sc.tab + row;
#pragma unroll 8
  for (int i = 0; i < 56; i++) T.base[i * FQ_DH_THREADS] = g[(size_t)i * sc.npad];
  DhState D;
  { TabView G; G.base = sc.tab + row; G.stride = (u32)sc.npad; D.T7 = tab_load(G, 7); }
  const uint4 s0 = sc.plan[row], s1 = sc.plan[sc.npad + row];
  D.plan.S.v[0] = s0.x; D.plan.S.v[1] = s0.y; D.plan.S.v[2] = s0.z; D.plan.S.v[3] = s0.w;
  D.plan.S.v[4] = s1.x; D.plan.S.v[5] = s1.y; D.plan.S.v[6] = s1.z; D.plan.S.v[7] = s1.w;
  D.plan.first = sc.meta[row] & 0xffu;
  ptR1 R = row_dh_loop<ENDO, STRICT>(T, D);
  uint4* o = sc.R + row;
  stq(o, R.X.re); stq(o + sc.npad, R.X.im); stq(o + 2 * sc.npad, R.Y.re); stq(o + 3 * sc.npad, R.Y.im);
  stq(o + 4 * sc.npad, R.Z.re); stq(o + 5 * sc.npad, R.Z.im);
}

// R1toAffine (curve4q.py:103-106) for FQ_BATCHINV_ROWS rows of a thread with one GF(p^2) inversion, the neutral check of DH_core
// (curve4q.py:459), encode (curve4q.py:41-46): batchinv.cuh FinishIO.  Thread t owns rows t, t + stride, ...
#define FQ_FIN_THREADS 64
template <bool AFFINE, bool CHECK_NEUTRAL> __global__ void __launch_bounds__(FQ_FIN_THREADS)
k_dh_finish(DhScratch sc, void* __restrict__ out, unsigned char* __restrict__ status, size_t n) {
  FinishIO<AFFINE, CHECK_NEUTRAL> io;
  io.R = sc.R; io.meta = sc.meta; io.npad = sc.npad; io.out = reinterpret_cast<uint4*>(out); io.status = status; io.n = n;
  io.stride = (size_t)gridDim.x * FQ_FIN_THREADS; io.t = (size_t)blockIdx.x * FQ_FIN_THREADS + threadIdx.x;
  batch_invert<Fp2Ops>(io, FQ_BATCHINV_ROWS);
}
static inline unsigned dh_finish_grid(size_t rows) {
  return (unsigned)((((rows + FQ_BATCHINV_ROWS - 1) / FQ_BATCHINV_ROWS) + FQ_FIN_THREADS - 1) / FQ_FIN_THREADS);
}
// scratch of a producer that only hands (X, Y, Z) and a status word to k_dh_finish (the fixed-base kernels; sized in kernels.h)
static inline DhScratch fin_scratch_view(void* base, size_t rows) {
  DhScratch sc;
  sc.npad = fin_scratch_npad(rows);
  sc.tab = nullptr; sc.plan = nullptr; sc.R = reinterpret_cast<uint4*>(base); sc.meta = reinterpret_cast<u32*>(sc.R + 6 * sc.npad);
  return sc;
}

template <bool ENDO> static cudaError_t dh_init() {
  cudaError_t e = cudaFuncSetAttribute(k_dh_ladder<ENDO, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_DH_SMEM);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_dh_ladder<ENDO, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_DH_SMEM);
}
// scratch: fqk_dh_scratch_bytes(n) bytes on the device.  ev: optional 4 events recorded around the three
// kernels of the (last) batch, for per-kernel timing.
// strict: table selection by the strict scan instead of masked loads (dh.cuh)
template <bool ENDO> static cudaError_t dh_launch(int affine, int strict, const void* k, const void* pt, void* out, void* status, size_t n, void* scratch,
                                                  cudaStream_t s, cudaEvent_t* ev) {
  const size_t in_pt = affine ? 64 : 32, out_b = affine ? 64 : 32;
  for (size_t r0 = 0; r0 < n; r0 += FQ_DH_MAX_BATCH) {
    const size_t rows = n - r0 < FQ_DH_MAX_BATCH ? n - r0 : FQ_DH_MAX_BATCH;
    DhScratch sc = dh_scratch_view(scratch, rows);
    const unsigned g = (unsigned)(sc.npad / FQ_DH_THREADS);
    const unsigned gf = dh_finish_grid(rows);
    const char* kk = (const char*)k + 32 * r0; const char* pp = (const char*)pt + in_pt * r0;
    char* oo = (char*)out + out_b * r0; unsigned char* st = (unsigned char*)status + r0;
    if (ev) cudaEventRecord(ev[0], s);
    if (affine) k_dh_prep<true, ENDO><<<g, FQ_DH_THREADS, 0, s>>>(kk, pp, sc, rows);
    else k_dh_prep<false, ENDO><<<g, FQ_DH_THREADS, 0, s>>>(kk, pp, sc, rows);
    if (ev) cudaEventRecord(ev[1], s);
    if (strict) k_dh_ladder<ENDO, true><<<g, FQ_DH_THREADS, FQ_DH_SMEM, s>>>(sc);
    else k_dh_ladder<ENDO, false><<<g, FQ_DH_THREADS, FQ_DH_SMEM, s>>>(sc);
    if (ev) cudaEventRecord(ev[2], s);
    if (affine) k_dh_finish<true, true><<<gf, FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    else k_dh_finish<false, true><<<gf, FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    if (ev) cudaEventRecord(ev[3], s);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
