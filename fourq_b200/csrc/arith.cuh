// arith.cuh -- 32-bit limb primitives with explicit carry flag.
//
// Device build (nvcc, sm_100a): every primitive is ONE PTX instruction using the condition-code register
// (add.cc / addc.cc / mad.lo.cc / madc.hi.cc ...).  ptxas fuses each {mad.lo.cc, madc.hi.cc} pair into a single
// IMAD.WIDE.U32[.X] with predicate carry-in/out, and add chains into IADD3[.X]; see profiles/ for the SASS.
//
// Host-simulation build (g++ -DFQ_HOSTSIM, tests/hostsim only -- NOT part of the product library): the same
// primitives are emulated with a thread-local carry flag that follows the PTX semantics instruction by instruction,
// so the exact instruction sequences of fp.cuh/fp2.cuh/point.cuh/... can be checked on a CPU against the oracle.
#pragma once
#include <cstdint>

typedef uint32_t u32;
typedef uint64_t u64;

#ifdef FQ_HOSTSIM
#define FQ_FN static inline
#define FQ_MFN inline
#define FQ_UNROLL
#define FQ_NOUNROLL
namespace fqsim { extern thread_local u32 cc; }
#define FQ_CC (fqsim::cc)
#else
#define FQ_FN __device__ __forceinline__
#define FQ_MFN __device__ __forceinline__
#define FQ_UNROLL _Pragma("unroll")
#define FQ_NOUNROLL _Pragma("unroll 1")
#endif

// Carry tracing (tests/hostsim/carry_trace.cpp, host simulation only, C++20): with FQ_HOSTSIM_CARRY every carry primitive takes
// its call site as a defaulted argument and reports to fqsim::carry_event.  start ops (add_cc, sub_cc, mad_lo_cc) write the carry,
// middle ops (addc_cc, subc_cc, madc_lo_cc, madc_hi_cc) read and write it, end ops (addc, subc, madc_hi) read it.
#ifdef FQ_HOSTSIM_CARRY
#ifndef FQ_HOSTSIM
#error "FQ_HOSTSIM_CARRY is a variant of the host simulation (FQ_HOSTSIM)"
#endif
#include <source_location>
namespace fqsim {
enum CarryKind { CK_ADD_CC, CK_SUB_CC, CK_MAD_LO_CC, CK_ADDC_CC, CK_SUBC_CC, CK_MADC_LO_CC, CK_MADC_HI_CC, CK_ADDC, CK_SUBC, CK_MADC_HI };
// exact0 = the op's exact result before its carry-in (mod 2^64: a subtraction wraps), cin = the carry flag (0 for a start op).
// Returns the carry-in the op uses: cin, unless the tracer forces this site.  Carry-out and the 33-bit result follow from both.
u32 carry_event(CarryKind kind, u32 cin, u64 exact0, const std::source_location& site);
}
#define FQ_SITE , const std::source_location fq_site = std::source_location::current()
#define FQ_START(kind, exact0) ((void)fqsim::carry_event(fqsim::kind, 0, exact0, fq_site))
#define FQ_CIN(kind, exact0) fqsim::carry_event(fqsim::kind, FQ_CC, exact0, fq_site)
#else
#define FQ_SITE
#define FQ_START(kind, exact0) ((void)0)
#define FQ_CIN(kind, exact0) FQ_CC
#endif

#ifdef FQ_HOSTSIM
struct uint4 { u32 x, y, z, w; };
FQ_FN uint4 make_uint4(u32 x, u32 y, u32 z, u32 w) { uint4 r = {x, y, z, w}; return r; }
#endif

// Scheduling fence.  ptxas interleaves every independent carry chain it can find; with several multiplications in one
// basic block it keeps more than the 7 predicate registers' worth of carries in flight and spills them into general
// registers (P2R / bit set / bit test: ~11 % of the instructions of a point addition).  A warp-level sync is one cheap
// instruction that ends the scheduling region, so chains of different multiplications no longer overlap.
#if defined(FQ_HOSTSIM) || !defined(FQ_USE_FENCE)
#define FQ_SCHED_FENCE() do {} while (0)
#else
#define FQ_SCHED_FENCE() __syncwarp()
#endif

// ---------------------------------------------------------------- add / sub with carry
FQ_FN u32 add_cc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 s = (u64)a + b; FQ_START(CK_ADD_CC, s); FQ_CC = (u32)(s >> 32); return (u32)s;
#else
  u32 r; asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}
FQ_FN u32 addc_cc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 s = (u64)a + b + FQ_CIN(CK_ADDC_CC, (u64)a + b); FQ_CC = (u32)(s >> 32); return (u32)s;
#else
  u32 r; asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}
FQ_FN u32 addc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  return a + b + FQ_CIN(CK_ADDC, (u64)a + b);
#else
  u32 r; asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}
FQ_FN u32 sub_cc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 s = (u64)a - b; FQ_START(CK_SUB_CC, s); FQ_CC = (u32)(s >> 32) & 1; return (u32)s;   // CC = borrow
#else
  u32 r; asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}
FQ_FN u32 subc_cc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 s = (u64)a - b - FQ_CIN(CK_SUBC_CC, (u64)a - b); FQ_CC = (u32)(s >> 32) & 1; return (u32)s;
#else
  u32 r; asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}
FQ_FN u32 subc(u32 a, u32 b FQ_SITE) {
#ifdef FQ_HOSTSIM
  return a - b - FQ_CIN(CK_SUBC, (u64)a - b);
#else
  u32 r; asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r;
#endif
}

// ---------------------------------------------------------------- 32x32 -> 64 multiply(-accumulate)
// {lo,hi} = a*b
FQ_FN void mul_wide(u32& lo, u32& hi, u32 a, u32 b) {
#ifdef FQ_HOSTSIM
  u64 p = (u64)a * b; lo = (u32)p; hi = (u32)(p >> 32);
#else
  asm volatile("{.reg .u64 t; mul.wide.u32 t, %2, %3; mov.b64 {%0,%1}, t;}" : "=r"(lo), "=r"(hi) : "r"(a), "r"(b));
#endif
}
// c + lo(a*b), carry out
FQ_FN u32 mad_lo_cc(u32 a, u32 b, u32 c FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 s = (u64)(u32)((u64)a * b) + c; FQ_START(CK_MAD_LO_CC, s); FQ_CC = (u32)(s >> 32); return (u32)s;
#else
  u32 r; asm volatile("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
#endif
}
// c + lo(a*b) + carry in, carry out
FQ_FN u32 madc_lo_cc(u32 a, u32 b, u32 c FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 t = (u64)(u32)((u64)a * b) + c, s = t + FQ_CIN(CK_MADC_LO_CC, t); FQ_CC = (u32)(s >> 32); return (u32)s;
#else
  u32 r; asm volatile("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
#endif
}
// c + hi(a*b) + carry in, carry out
FQ_FN u32 madc_hi_cc(u32 a, u32 b, u32 c FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 t = (u64)(u32)(((u64)a * b) >> 32) + c, s = t + FQ_CIN(CK_MADC_HI_CC, t); FQ_CC = (u32)(s >> 32); return (u32)s;
#else
  u32 r; asm volatile("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
#endif
}
// c + hi(a*b) + carry in (chain end)
FQ_FN u32 madc_hi(u32 a, u32 b, u32 c FQ_SITE) {
#ifdef FQ_HOSTSIM
  u64 t = (u64)(u32)(((u64)a * b) >> 32) + c; return (u32)(t + FQ_CIN(CK_MADC_HI, t));
#else
  u32 r; asm volatile("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r;
#endif
}

// ---------------------------------------------------------------- funnel shifts (SHF)
// low 32 bits of ({hi,lo} >> n), 0 < n < 32
FQ_FN u32 shr_pair(u32 lo, u32 hi, int n) {
#ifdef FQ_HOSTSIM
  return (u32)((((u64)hi << 32) | lo) >> n);
#else
  return __funnelshift_r(lo, hi, n);
#endif
}
// high 32 bits of ({hi,lo} << n), 0 < n < 32
FQ_FN u32 shl_pair(u32 lo, u32 hi, int n) {
#ifdef FQ_HOSTSIM
  return (u32)(((((u64)hi << 32) | lo) << n) >> 32);
#else
  return __funnelshift_l(lo, hi, n);
#endif
}
