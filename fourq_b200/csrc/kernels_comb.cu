// kernels_comb.cu -- fixed-base kernels on per-digit tables (comb.cuh): fq_mul_base_comb, fq_dh_base_comb, and
// fq_mul_fixed / fq_dh_fixed on the tables of a caller-registered point.
// One thread = one row; the 47.25 KiB table of the base point is copied once per CTA from global to shared memory and
// then read with warp-uniform addresses (broadcast), so the per-thread state is registers only.  k_comb leaves the result
// projective; k_dh_finish (kernels_dh.cuh) normalises sixteen rows per inversion and encodes.
#include <cstring>
#include "kernels_dh.cuh"
#include "comb.cuh"

#define FQ_COMB_THREADS 256

// canonical affine x | y of a base point, passed by value: building its tables needs no device copy of the point
struct CombPoint { u32 xy[16]; };

// tabs: [2][FQ_COMB_WORDS], the tables of comb_base(0, P) and comb_base(1, P) for P = G (gen) or P = pt; thread t builds
// digit t % 63 of table t / 63
__global__ void __launch_bounds__(64) k_comb_build(CombPoint pt, bool gen, u32* tabs) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * FQ_COMB_DIGITS) return;
  int which = t / FQ_COMB_DIGITS, i = t % FQ_COMB_DIGITS;
  const fp2 x = gen ? curve_gx() : row_load_fp2(pt.xy), y = gen ? curve_gy() : row_load_fp2(pt.xy + 8);
  comb_build_digit(comb_base(which, x, y), i, tabs + which * FQ_COMB_WORDS + i * FQ_COMB_DIGIT_WORDS);
}

// [k]B in R1 for every row, B = the base of the table `tab` (FQ_COMB_WORDS words); (X, Y, Z) go to scratch for k_dh_finish
// (one inversion per FQ_BATCHINV_ROWS rows, encode).  DH only selects the k_dh_finish variant the launch pairs it with.
template <bool DH, bool STRICT> __global__ void __launch_bounds__(FQ_COMB_THREADS)
k_comb(const u32* __restrict__ tab, const void* __restrict__ k, DhScratch sc, size_t n) {
  extern __shared__ uint4 stab4[];
  const uint4* src = reinterpret_cast<const uint4*>(tab);
  for (int j = threadIdx.x; j < FQ_COMB_WORDS / 4; j += FQ_COMB_THREADS) stab4[j] = src[j];
  __syncthreads();
  const u32* stab = reinterpret_cast<const u32*>(stab4);
  const size_t ntiles = (n + FQ_COMB_THREADS - 1) / FQ_COMB_THREADS;
  for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    size_t row = tile * FQ_COMB_THREADS + threadIdx.x;
    if (row >= n) continue;
    u32 wk[8];
    ld8(k, row, wk);
    scal sk;
    FQ_UNROLL
    for (int i = 0; i < 8; i++) sk.v[i] = wk[i];
    ptR1 R = mul_comb<STRICT>(sk, stab);
    uint4* o = sc.R + row;
    stq(o, R.X.re); stq(o + sc.npad, R.X.im); stq(o + 2 * sc.npad, R.Y.re); stq(o + 3 * sc.npad, R.Y.im);
    stq(o + 4 * sc.npad, R.Z.re); stq(o + 5 * sc.npad, R.Z.im);
    sc.meta[row] = 0;
  }
}

// allocates [2][FQ_COMB_WORDS] words and builds the tables of P = G (gen) or pt into them; frees them on every error path
static cudaError_t comb_tables(const CombPoint& pt, bool gen, void** tabs_out, cudaStream_t s) {
  cudaError_t e;
  u32* tabs = nullptr;
  if ((e = cudaMalloc(&tabs, 2 * FQ_COMB_WORDS * sizeof(u32))) != cudaSuccess) return e;
  k_comb_build<<<(2 * FQ_COMB_DIGITS + 63) / 64, 64, 0, s>>>(pt, gen, tabs);
  if ((e = cudaGetLastError()) != cudaSuccess) { cudaFree(tabs); return e; }
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) { cudaFree(tabs); return e; }
  *tabs_out = tabs;
  return cudaSuccess;
}

cudaError_t fqk_comb_init(void** tabs_out, cudaStream_t s) {
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(k_comb<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_COMB_WORDS * 4)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_comb<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_COMB_WORDS * 4)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_comb<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_COMB_WORDS * 4)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_comb<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_COMB_WORDS * 4)) != cudaSuccess) return e;
  return comb_tables(CombPoint{}, true, tabs_out, s);
}

cudaError_t fqk_comb_build(const void* xy, void** tabs_out, cudaStream_t s) {
  CombPoint pt;
  memcpy(pt.xy, xy, sizeof(pt.xy));
  return comb_tables(pt, false, tabs_out, s);
}

size_t fqk_comb_scratch_bytes(size_t n) { return fin_scratch_bytes(n < FQ_DH_MAX_BATCH ? n : FQ_DH_MAX_BATCH); }

cudaError_t fqk_comb(int dh, int strict, const void* tabs, const void* k, void* out, void* status, size_t n, void* scratch, int sms, cudaStream_t s) {
  for (size_t r0 = 0; r0 < n; r0 += FQ_DH_MAX_BATCH) {
    const size_t rows = n - r0 < FQ_DH_MAX_BATCH ? n - r0 : FQ_DH_MAX_BATCH;
    DhScratch sc = fin_scratch_view(scratch, rows);
    // persistent CTAs: the table copy (47 KiB) is paid once per CTA, each CTA then walks over tiles of 256 rows
    unsigned tiles = grid_for(rows, FQ_COMB_THREADS);
    // two CTAs are resident per SM (128 registers x 256 threads).  Big launches run two waves of CTAs (better balance at the
    // end); chunk-sized launches run one, so that the 47 KiB table copy of a CTA is shared by 4 tiles instead of 2
    unsigned cap = (unsigned)sms * (tiles >= (unsigned)sms * 16u ? 4u : 2u);
    unsigned g = tiles < cap ? tiles : cap;
    const u32* tab = (const u32*)tabs + (dh ? FQ_COMB_WORDS : 0);
    const char* kk = (const char*)k + 32 * r0; char* oo = (char*)out + 32 * r0;
    unsigned char* st = status ? (unsigned char*)status + r0 : nullptr;
    if (dh) {
      if (strict) k_comb<true, true><<<g, FQ_COMB_THREADS, FQ_COMB_WORDS * 4, s>>>(tab, kk, sc, rows);
      else k_comb<true, false><<<g, FQ_COMB_THREADS, FQ_COMB_WORDS * 4, s>>>(tab, kk, sc, rows);
      k_dh_finish<false, true><<<dh_finish_grid(rows), FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    } else {
      if (strict) k_comb<false, true><<<g, FQ_COMB_THREADS, FQ_COMB_WORDS * 4, s>>>(tab, kk, sc, rows);
      else k_comb<false, false><<<g, FQ_COMB_THREADS, FQ_COMB_WORDS * 4, s>>>(tab, kk, sc, rows);
      k_dh_finish<false, false><<<dh_finish_grid(rows), FQ_FIN_THREADS, 0, s>>>(sc, oo, st, rows);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
