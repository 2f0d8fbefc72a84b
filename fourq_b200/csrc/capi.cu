// capi.cu -- the C ABI of include/fourq_b200.h and the host engine behind it.
//
// Host engine.  A call splits its rows into contiguous per-GPU slices (SURVEY 8e: every row is independent, there is no
// exchange step, hence no collective).  Every GPU has its own pair of host threads and its own lock, so slices of one
// call run concurrently and callers on disjoint GPUs do not wait for each other:
//
//   feeder   (one per GPU)  takes chunks of its slice (ramped sizes; other slices' rows once its own are gone: CallWork) and for each chunk
//                           waits for a free stream slot, copies pageable inputs into the slot's pinned staging buffers,
//                           and enqueues H2D copies, the kernels and the D2H copies on the slot's stream;
//   drainer  (one per GPU)  waits for each chunk's completion event in order, copies results that were staged for a
//                           pageable destination into the caller's memory, collects the kernel time and frees the slot.
//
// Four stream slots per GPU keep the staging and H2D of the chunks after next, the kernels of chunk c, a chunk queued
// behind it (so that kernel tails overlap the next chunk's first kernel) and the D2H and host copy-out of chunk c-1 in flight.  Page-locked caller buffers (fq_host_alloc) are used directly in both directions.  Slot buffers,
// events and streams are created once per GPU and grow on demand; fq_trim wipes and frees them.  There is no CPU
// implementation of any operation here.
//
// tests/hostsim compiles this file with -DFQ_MOCK_CUDA against a small in-process imitation of the CUDA runtime (streams
// are threads) to exercise exactly this host logic -- chunking, staging, threading, error paths -- without a GPU; that
// build is test infrastructure and is never shipped or loaded by the product.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <utility>
#ifdef FQ_MOCK_CUDA
#include "mock_cuda_runtime.h"
#else
#include <cuda_runtime.h>
#endif
#include "../../include/fourq_b200.h"
#include "kernels.h"

namespace {

constexpr int kSlots = 4;                        // stream slots per GPU = chunks in flight (see the top of this file)
constexpr int kMaxDev = 16;
constexpr int kOperands = 5;                      // a, b, c (inputs), out, status
constexpr size_t kFlushBytes = 256u << 20;        // > 126 MB L2

thread_local char tl_err[512] = "";
thread_local float tl_kernel_ms = 0.f;
thread_local float tl_phase_ms[3] = {0.f, 0.f, 0.f};
thread_local size_t tl_rows_per_dev[16] = {0};      // rows each GPU of the last host call of this thread ended up processing
std::atomic<int> g_dev_base{0};
std::atomic<int> g_strict{-1};    // table selection: 1 = strict scan (default), 0 = masked loads, -1 = not yet read from FQ_STRICT_SELECT

int fail(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(tl_err, sizeof(tl_err), fmt, ap); va_end(ap);
  return code;
}
#define CU(call)                                                                                       \
  do { cudaError_t e_ = (call);                                                                        \
       if (e_ != cudaSuccess) return fail(FQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

// ---------------------------------------------------------------- operations

// rows by which the chunk schedule rounds: ramp-down chunks, stolen pieces, speed-weighted slices and the half chunks of staged calls
constexpr size_t kRowQuant = 128;
// rows per full pipeline chunk of the variable-base DH ops: a whole number of waves of k_dh_ladder (2 CTAs x 128 rows per SM)
// and of k_dh_prep (3 per SM) keeps the tail of each chunk short
constexpr size_t kDhChunkRows = (size_t)148 * 2 * 128 * 12;      // 454,656 rows = 12 waves of k_dh_ladder, 8 of k_dh_prep
// k_comb keeps 2 CTAs of 256 rows resident per SM, each walking over tiles: 148 x 2 x 256 x 4 rows = 4 full tiles per CTA
constexpr size_t kCombChunkRows = (size_t)148 * 2 * 256 * 4;

// device scratch an operation's kernels hand data through: none, the variable-base DH layout (table, digit register,
// projective result), the projective result the fixed-base kernels hand to k_dh_finish, or the X25519 ladder's (x2, z2)
enum Scratch { SCRATCH_NONE, SCRATCH_DH, SCRATCH_FIXED_BASE, SCRATCH_X25519 };

// Everything the engine knows about an operation apart from its kernels (launch):
//   bytes per row of each operand, chunk_rows = rows of a full pipeline chunk, the scratch its kernels need;
//   rate_class >= 0: big multi-GPU calls adapt their slices to the measured speed of each GPU (on a host where some GPUs reach
//   the caller's memory more slowly than others, equal slices end with the slowest GPU); ops of one class share the measurement;
//   var_dh: a variable-base DH op (three kernels; half chunks for staged operands, per-kernel timing in fq_dev_run3).
struct OpDesc {
  int op; int in_bytes[3]; int out_bytes; bool status; size_t chunk_rows;
  Scratch scratch = SCRATCH_NONE; int rate_class = -1; bool var_dh = false;
};

OpDesc describe(int op) {
  const size_t M = (size_t)1 << 20;
  switch (op) {
    case FQ_DEVOP_FP2_MUL: case FQ_DEVOP_FP2_ADD: case FQ_DEVOP_FP2_SUB: return {op, {32, 32, 0}, 32, false, M};
    case FQ_DEVOP_FP2_SQR: case FQ_DEVOP_FP2_NEG: case FQ_DEVOP_FP2_CONJ: return {op, {32, 0, 0}, 32, false, M};
    case FQ_DEVOP_FP2_INV: case FQ_DEVOP_FP2_INVSQRT: return {op, {32, 0, 0}, 32, false, M / 4};
    case FQ_DEVOP_FP2_SELECT: return {op, {32, 32, 1}, 32, false, M};
    case FQ_DEVOP_FP_SELECT: return {op, {16, 16, 1}, 16, false, M};
    case FQ_DEVOP_FP_BASE + FQ_FP_MUL: case FQ_DEVOP_FP_BASE + FQ_FP_ADD: case FQ_DEVOP_FP_BASE + FQ_FP_SUB: return {op, {16, 16, 0}, 16, false, M};
    case FQ_DEVOP_FP_BASE + FQ_FP_SQR: case FQ_DEVOP_FP_BASE + FQ_FP_NEG: return {op, {16, 0, 0}, 16, false, M};
    case FQ_DEVOP_FP_BASE + FQ_FP_INV: case FQ_DEVOP_FP_BASE + FQ_FP_INVSQRT: return {op, {16, 0, 0}, 16, false, M / 4};
    case FQ_DEVOP_DECODE: case FQ_DEVOP_DECODE_SPEC: return {op, {32, 0, 0}, 64, true, M / 4};
    case FQ_DEVOP_ENCODE: return {op, {64, 0, 0}, 32, false, M};
    case FQ_DEVOP_ON_CURVE: return {op, {64, 0, 0}, 1, false, M};
    case FQ_DEVOP_DH: return {op, {32, 32, 0}, 32, true, kDhChunkRows, SCRATCH_DH, 0, true};
    case FQ_DEVOP_DH_AFFINE: return {op, {32, 64, 0}, 64, true, kDhChunkRows, SCRATCH_DH, 0, true};
    case FQ_DEVOP_DH_ENDO: return {op, {32, 32, 0}, 32, true, kDhChunkRows, SCRATCH_DH, 1, true};
    case FQ_DEVOP_DH_ENDO_AFFINE: return {op, {32, 64, 0}, 64, true, kDhChunkRows, SCRATCH_DH, 1, true};
    case FQ_DEVOP_DH_BASE: case FQ_DEVOP_DH_ENDO_BASE: return {op, {32, 0, 0}, 32, true, M / 8, SCRATCH_FIXED_BASE};
    case FQ_DEVOP_MUL_BASE: case FQ_DEVOP_MUL_ENDO_BASE: return {op, {32, 0, 0}, 32, false, M / 8, SCRATCH_FIXED_BASE};
    case FQ_DEVOP_DH_BASE_COMB: return {op, {32, 0, 0}, 32, true, kCombChunkRows, SCRATCH_FIXED_BASE, 2};
    case FQ_DEVOP_MUL_BASE_COMB: return {op, {32, 0, 0}, 32, false, kCombChunkRows, SCRATCH_FIXED_BASE, 2};
    case FQ_DEVOP_X25519: return {op, {32, 32, 0}, 32, false, M / 8, SCRATCH_X25519};
    case FQ_DEVOP_F25519_BASE + FQ_FP_MUL: case FQ_DEVOP_F25519_BASE + FQ_FP_ADD: case FQ_DEVOP_F25519_BASE + FQ_FP_SUB: return {op, {32, 32, 0}, 32, false, M};
    case FQ_DEVOP_F25519_BASE + FQ_FP_SQR: return {op, {32, 0, 0}, 32, false, M};
    case FQ_DEVOP_F25519_BASE + FQ_FP_INV: return {op, {32, 0, 0}, 32, false, M / 4};
    default: return {-1, {0, 0, 0}, 0, false, 0};
  }
}
int operand_bytes(const OpDesc& d, int w) { return w < 3 ? d.in_bytes[w] : w == 3 ? d.out_bytes : (d.status ? 1 : 0); }
size_t scratch_bytes(Scratch k, size_t rows) {
  switch (k) {
    case SCRATCH_DH: return fqk_dh_scratch_bytes(rows);
    case SCRATCH_FIXED_BASE: return fqk_comb_scratch_bytes(rows);
    case SCRATCH_X25519: return fqk_x25519_scratch_bytes(rows);
    default: return 0;
  }
}

int strict_mode() {
  int v = g_strict.load();
  if (v < 0) {                                     // first use: the environment decides unless fq_set_select_mode got there first
    const char* e = getenv("FQ_STRICT_SELECT");
    int want = (e && e[0] == '0') ? 0 : 1, expected = -1;
    v = g_strict.compare_exchange_strong(expected, want) ? want : expected;
  }
  return v;
}

// Work of one call.  The rows are cut into one contiguous slice per GPU (slice i = rows [i*ceil(n/ndev), ...)); a GPU works
// through its own slice from the front in chunks, and when that is exhausted it takes chunks from the BACK of the slice
// that has the most rows left.  With equal GPUs nothing is ever stolen and every GPU handles exactly its slice; on a host
// whose GPUs do not all reach memory at the same speed (measured on an 8 x B200 virtual machine: four of the eight take
// 8-13 % longer for the same slice, and the machine exposes no NUMA information to place buffers by) the call ends when the
// work is done instead of when the slowest slice is.
//
// Chunk sizes of a slice: ramp up from a small chunk (doubling) so that the first kernels start after a short copy, full
// chunks in the middle, ramp down by halves so that little work and a short copy-back remain exposed at the end.  Slices of
// at most two small chunks are not split.  No chunk exceeds `full` rows (the staging buffers are sized for exactly that).
struct CallWork {
  std::mutex mu;
  struct Range { size_t lo, hi; bool ramp; };
  std::vector<Range> r;               // rows of each slice not yet handed out
  size_t full = 0, small = 0;
  bool abort = false;
  // share: optional relative speeds of the GPUs (rows per ms of their last calls); null or incomplete -> equal slices
  void init(size_t n, int ndev, size_t full_rows, const double* share = nullptr) {
    full = full_rows;
    small = full / 8 >= 16384 ? full / 8 : 16384;
    if (small > full) small = full;
    const size_t per = (n + (size_t)ndev - 1) / (size_t)ndev;
    double total = 0;
    bool weighted = share != nullptr && ndev > 1 && n >= (size_t)ndev * 2 * full;
    for (int i = 0; weighted && i < ndev; i++) { if (share[i] > 0) total += share[i]; else weighted = false; }
    double f[64], fsum = 0;                                 // proportional to the measured speed, within +-25 % of the equal share
    double spread = 0;
    for (int i = 0; weighted && i < ndev && i < 64; i++) {
      f[i] = share[i] / total * ndev;
      if (f[i] - 1 > spread) spread = f[i] - 1;
      if (1 - f[i] > spread) spread = 1 - f[i];
      f[i] = f[i] < 0.75 ? 0.75 : f[i] > 1.25 ? 1.25 : f[i];
      fsum += f[i];
    }
    if (spread < 0.03) weighted = false;                   // GPUs within 3 % of each other: measurement noise, keep the slices equal
    size_t lo = 0;
    for (int i = 0; i < ndev; i++) {
      size_t len = per;
      if (weighted) {
        len = (size_t)((double)n * f[i] / fsum) / kRowQuant * kRowQuant;
        if (i == ndev - 1) len = n - lo;
      }
      const size_t hi = lo + len < n ? lo + len : n;
      r.push_back({lo, i == ndev - 1 && weighted ? n : hi, hi - lo > 2 * small});
      lo = hi;
    }
  }
  // the next chunk for GPU `me`, which has taken `taken` chunks of this call so far; false when no rows are left
  bool take(int me, int taken, size_t* r0, size_t* rows) {
    std::lock_guard<std::mutex> l(mu);
    if (abort) return false;
    Range& own = r[(size_t)me];
    if (own.lo < own.hi) {
      const size_t left = own.hi - own.lo;
      size_t sz = full;
      if (own.ramp) { sz = small; for (int t = 0; t < taken && sz < full; t++) sz = sz * 2 < full ? sz * 2 : full; }
      size_t n = sz < left ? sz : left;
      if (own.ramp && left > small && left <= 2 * n) {              // ramp down by halves
        n = (left / 2 + kRowQuant - 1) / kRowQuant * kRowQuant;
        if (n > full) n = full;
        if (n > left) n = left;
      }
      *r0 = own.lo; *rows = n; own.lo += n;
      return true;
    }
    size_t best = r.size(), most = 0;
    for (size_t j = 0; j < r.size(); j++) if (r[j].hi - r[j].lo > most) { most = r[j].hi - r[j].lo; best = j; }
    if (best == r.size()) return false;
    size_t n = most;                                                 // a victim's last piece goes whole; otherwise half of what it has left
    if (most > small) { n = (most / 2 + kRowQuant - 1) / kRowQuant * kRowQuant; if (n > full) n = full; if (n > most) n = most; }
    r[best].hi -= n; *r0 = r[best].hi; *rows = n;
    return true;
  }
  void stop() { std::lock_guard<std::mutex> l(mu); abort = true; }
};

// ---------------------------------------------------------------- host copies of pageable operands

// threads that share one staging copy of a pageable operand.  One core moves 5-10 GB/s, a B200 consumes the 64 B of inputs
// per DH row at ~6 GB/s and produces 33 B, so a single copying thread per direction is on the critical path (measured: 68 / 73 /
// 75 M DH rows/s end to end with 1 / 2 / 3 threads before the other changes).
constexpr int kCopyThreads = 3;
// Makes the pages of a pageable OUTPUT buffer present and writable without touching their contents (MADV_POPULATE_WRITE,
// Linux 5.14+; silently skipped where unsupported).  A freshly allocated result array (numpy.empty) otherwise takes its
// ~8,000 first-touch page faults per 32 MiB inside the drainer's copies, on the critical path of the last chunks.  Called by
// the thread that is only waiting for the slices anyway, in 4 MiB steps from the start of the buffer (the order of the chunks).
void populate_output(void* p, size_t bytes) {
#ifndef MADV_POPULATE_WRITE
#define MADV_POPULATE_WRITE 23
#endif
  if (!p || bytes < ((size_t)1 << 20)) return;
  const size_t page = (size_t)sysconf(_SC_PAGESIZE);
  uintptr_t lo = ((uintptr_t)p + page - 1) / page * page, hi = ((uintptr_t)p + bytes) / page * page;      // whole pages inside the buffer
  if (hi > lo) madvise((void*)lo, hi - lo, MADV_HUGEPAGE);       // where transparent huge pages are on request: 16 faults per 32 MiB instead of 8,192
  const size_t step = (size_t)4 << 20;
  for (; lo < hi; lo += step)
    if (madvise((void*)lo, hi - lo < step ? hi - lo : step, MADV_POPULATE_WRITE) != 0) return;
}
// FQ_WIPE_AFTER_CALL=1: zero the staging buffers and the kernel scratch of a GPU when its slice of a call is done (they hold
// scalars, tables of secret multiples, projective results and shared secrets until the next call overwrites them or fq_trim
// wipes them).  Off by default: it costs a memset of every buffer the call used (measured: +4.4 ms on a 2^20-row DH call).
bool wipe_after_call() {
  static const bool v = [] { const char* e = getenv("FQ_WIPE_AFTER_CALL"); return e && e[0] == '1'; }();
  return v;
}
bool trace_enabled() {
  static const bool v = [] { const char* e = getenv("FQ_TRACE"); return e && e[0] == '1'; }();
  return v;
}
double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// memcpy split between the calling thread and kCopyThreads - 1 helper threads that sleep between copies
class CopyHelper {
 public:
  void copy(void* dst, const void* src, size_t bytes) {
    const int parts = bytes >= ((size_t)1 << 20) ? kCopyThreads : 1;
    if (parts == 1) { memcpy(dst, src, bytes); return; }
    const size_t per = (bytes / parts + 4095) / 4096 * 4096;
    {
      std::lock_guard<std::mutex> l(mu_);
      while ((int)threads_ < parts - 1) { std::thread(&CopyHelper::run, this).detach(); threads_++; }
      for (int i = 1; i < parts; i++) {
        const size_t lo = (size_t)i * per, hi = lo + per < bytes ? lo + per : bytes;
        if (lo < hi) { tasks_.push_back({(char*)dst + lo, (const char*)src + lo, hi - lo}); pending_++; }
      }
    }
    cv_.notify_all();
    memcpy(dst, src, per < bytes ? per : bytes);
    std::unique_lock<std::mutex> l(mu_);
    done_.wait(l, [&] { return pending_ == 0; });
  }
 private:
  struct Task { char* dst; const char* src; size_t n; };
  void run() {
    for (;;) {
      Task t;
      { std::unique_lock<std::mutex> l(mu_); cv_.wait(l, [&] { return !tasks_.empty(); }); t = tasks_.front(); tasks_.pop_front(); }
      memcpy(t.dst, t.src, t.n);
      { std::lock_guard<std::mutex> l(mu_); if (--pending_ == 0) done_.notify_all(); }
    }
  }
  std::mutex mu_; std::condition_variable cv_, done_;
  std::deque<Task> tasks_; int pending_ = 0; size_t threads_ = 0;
};

// ---------------------------------------------------------------- per-GPU state

struct SliceJob;

// one stream slot: device staging of every operand, pinned host staging for pageable operands, kernel scratch, events
struct Slot {
  cudaStream_t st = nullptr;
  void* dbuf[kOperands] = {nullptr, nullptr, nullptr, nullptr, nullptr}; size_t dcap[kOperands] = {0, 0, 0, 0, 0};
  void* hbuf[kOperands] = {nullptr, nullptr, nullptr, nullptr, nullptr}; size_t hcap[kOperands] = {0, 0, 0, 0, 0};
  void* scratch = nullptr; size_t scratch_cap = 0;      // table / plan / projective result handed between the kernels of an op
  cudaEvent_t e0 = nullptr, e1 = nullptr, done = nullptr;
  bool busy = false;                                    // guarded by DevCtx::smu
};
struct Chunk { int si; size_t r0, rows; SliceJob* job; };

struct DevCtx {
  int dev = 0;
  std::mutex mu;                  // one user of the device context at a time: a slice job or an fq_dev_* call
  bool ready = false;
  Slot slot[kSlots];
  void* flush = nullptr;
  void* comb = nullptr;           // per-digit fixed-base tables (kernels_comb.cu)
  cudaEvent_t job_e0 = nullptr;   // recorded before the first kernel of a slice job
  int sms = 0;
  // feeder: slice jobs in submission order
  std::mutex qmu; std::condition_variable qcv; std::deque<SliceJob*> jobs; bool threads = false;
  // feeder -> drainer: chunks in enqueue order; also guards Slot::busy and SliceJob::outstanding
  std::mutex smu; std::condition_variable scv; std::deque<Chunk> chunks;
  CopyHelper copy_in, copy_out;   // staging copies of the feeder / of the drainer
  std::atomic<double> rate[3];    // rows per ms this GPU sustained in its last big calls, per class of operation (rate_class); 0 = unknown
  DevCtx() { for (auto& x : rate) x.store(0.0); }
};
DevCtx* g_ctx = nullptr;          // kMaxDev contexts, allocated once and never destroyed (their threads are detached)
std::once_flag g_ctx_once;
DevCtx& ctx_of(int dev) {
  std::call_once(g_ctx_once, [] { g_ctx = new DevCtx[kMaxDev]; for (int i = 0; i < kMaxDev; i++) g_ctx[i].dev = i; });
  return g_ctx[dev];
}

int device_count() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) { cudaGetLastError(); return fail(FQ_ERR_NO_DEVICE, "no CUDA device available (%s); fourq_b200 has no CPU path", e == cudaSuccess ? "0 devices" : cudaGetErrorString(e)); }
  return n > kMaxDev ? kMaxDev : n;
}

// caller holds c.mu
int ctx_init(DevCtx& c) {
  CU(cudaSetDevice(c.dev));
  if (c.ready) return FQ_OK;
  int rc = FQ_OK;
  auto undo = [&] {
    for (int i = 0; i < kSlots; i++) {
      Slot& s = c.slot[i];
      if (s.e0) cudaEventDestroy(s.e0);
      if (s.e1) cudaEventDestroy(s.e1);
      if (s.done) cudaEventDestroy(s.done);
      if (s.st) cudaStreamDestroy(s.st);
      s.e0 = s.e1 = s.done = nullptr; s.st = nullptr;
    }
    if (c.comb) { cudaFree(c.comb); c.comb = nullptr; }
    if (c.job_e0) { cudaEventDestroy(c.job_e0); c.job_e0 = nullptr; }
  };
#define CUI(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(FQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); undo(); return rc; } } while (0)
  for (int i = 0; i < kSlots; i++) {
    Slot& s = c.slot[i];
    CUI(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
    CUI(cudaEventCreate(&s.e0)); CUI(cudaEventCreate(&s.e1));
    CUI(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
  }
  CUI(cudaEventCreate(&c.job_e0));
  CUI(fqk_device_init(c.slot[0].st));
  CUI(fqk_comb_init(&c.comb, c.slot[0].st));
  CUI(cudaDeviceGetAttribute(&c.sms, cudaDevAttrMultiProcessorCount, c.dev));
#undef CUI
  c.ready = true;
  return FQ_OK;
}

thread_local bool tl_grew = false;       // a staging or scratch buffer was (re)allocated by this thread: the call's timing includes it
int dbuf_reserve(Slot& s, int w, size_t bytes) {
  if (bytes <= s.dcap[w]) return FQ_OK;
  tl_grew = true;
  if (s.dbuf[w]) CU(cudaFree(s.dbuf[w]));
  s.dbuf[w] = nullptr; s.dcap[w] = 0;
  CU(cudaMalloc(&s.dbuf[w], bytes));
  s.dcap[w] = bytes;
  return FQ_OK;
}
int hbuf_reserve(Slot& s, int w, size_t bytes) {
  if (bytes <= s.hcap[w]) return FQ_OK;
  tl_grew = true;
  if (s.hbuf[w]) CU(cudaFreeHost(s.hbuf[w]));
  s.hbuf[w] = nullptr; s.hcap[w] = 0;
  CU(cudaHostAlloc(&s.hbuf[w], bytes, cudaHostAllocPortable));
  s.hcap[w] = bytes;
  return FQ_OK;
}
int scratch_reserve(Slot& s, Scratch k, size_t rows) {
  const size_t bytes = scratch_bytes(k, rows);
  if (bytes <= s.scratch_cap) return FQ_OK;
  tl_grew = true;
  if (s.scratch) CU(cudaFree(s.scratch));
  s.scratch = nullptr; s.scratch_cap = 0;
  CU(cudaMalloc(&s.scratch, bytes));
  s.scratch_cap = bytes;
  return FQ_OK;
}

// what kind of memory a caller's host buffer is: page-locked (asynchronous copies use it directly), pageable (staged through
// the slot's pinned buffers), or not host memory at all (rejected by the host entry points)
enum PtrKind { PK_PAGEABLE = 0, PK_PINNED = 1, PK_DEVICE = 2 };
PtrKind classify_one(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return PK_PAGEABLE; }
  if (at.type == cudaMemoryTypeHost) return PK_PINNED;
  if (at.type == cudaMemoryTypeDevice) return PK_DEVICE;
  return PK_PAGEABLE;                                  // unregistered or managed: reachable by memcpy, staged
}
PtrKind classify(const void* p, size_t bytes) {
  if (!p || bytes == 0) return PK_PINNED;
  const PtrKind first = classify_one(p), last = classify_one((const char*)p + bytes - 1);
  if (first == PK_DEVICE || last == PK_DEVICE) return PK_DEVICE;
  return (first == PK_PINNED && last == PK_PINNED) ? PK_PINNED : PK_PAGEABLE;      // partly registered ranges are staged
}

// ---------------------------------------------------------------- kernels of one chunk

cudaError_t launch(const DevCtx& cx, int op, const void* a, const void* b, const void* c, void* out, void* status, size_t n, cudaStream_t s, void* scratch, cudaEvent_t* ev = nullptr) {
  const int strict = strict_mode();
  switch (op) {
    case FQ_DEVOP_DH_BASE_COMB: return fqk_comb(1, strict, cx.comb, a, out, status, n, scratch, cx.sms, s);
    case FQ_DEVOP_MUL_BASE_COMB: return fqk_comb(0, strict, cx.comb, a, out, nullptr, n, scratch, cx.sms, s);
    case FQ_DEVOP_FP2_MUL: return fqk_fp2_op(FQK_MUL, a, b, out, n, s);
    case FQ_DEVOP_FP2_SQR: return fqk_fp2_op(FQK_SQR, a, b, out, n, s);
    case FQ_DEVOP_FP2_INV: return fqk_fp2_op(FQK_INV, a, b, out, n, s);
    case FQ_DEVOP_FP2_ADD: return fqk_fp2_op(FQK_ADD, a, b, out, n, s);
    case FQ_DEVOP_FP2_SUB: return fqk_fp2_op(FQK_SUB, a, b, out, n, s);
    case FQ_DEVOP_FP2_NEG: return fqk_fp2_op(FQK_NEG, a, b, out, n, s);
    case FQ_DEVOP_FP2_CONJ: return fqk_fp2_op(FQK_CONJ, a, b, out, n, s);
    case FQ_DEVOP_FP2_INVSQRT: return fqk_fp2_op(FQK_INVSQRT, a, b, out, n, s);
    case FQ_DEVOP_FP2_SELECT: return fqk_select(2, c, a, b, out, n, s);
    case FQ_DEVOP_FP_SELECT: return fqk_select(1, c, a, b, out, n, s);
    case FQ_DEVOP_FP_BASE + FQ_FP_MUL: case FQ_DEVOP_FP_BASE + FQ_FP_SQR: case FQ_DEVOP_FP_BASE + FQ_FP_INV: case FQ_DEVOP_FP_BASE + FQ_FP_ADD:
    case FQ_DEVOP_FP_BASE + FQ_FP_SUB: case FQ_DEVOP_FP_BASE + FQ_FP_NEG: case FQ_DEVOP_FP_BASE + FQ_FP_INVSQRT:
      return fqk_fp_op(op - FQ_DEVOP_FP_BASE, a, b, out, n, s);
    case FQ_DEVOP_DECODE: return fqk_decode(0, a, out, status, n, s);
    case FQ_DEVOP_DECODE_SPEC: return fqk_decode(1, a, out, status, n, s);
    case FQ_DEVOP_ENCODE: return fqk_encode(a, out, n, s);
    case FQ_DEVOP_ON_CURVE: return fqk_on_curve(a, out, n, s);
    case FQ_DEVOP_DH: return fqk_dh(0, 0, strict, a, b, out, status, n, scratch, s, ev);
    case FQ_DEVOP_DH_AFFINE: return fqk_dh(1, 0, strict, a, b, out, status, n, scratch, s, ev);
    case FQ_DEVOP_DH_BASE: return fqk_fixed_base(1, 0, strict, a, out, status, n, scratch, s);
    case FQ_DEVOP_MUL_BASE: return fqk_fixed_base(0, 0, strict, a, out, nullptr, n, scratch, s);
    case FQ_DEVOP_DH_ENDO: return fqk_dh(0, 1, strict, a, b, out, status, n, scratch, s, ev);
    case FQ_DEVOP_DH_ENDO_AFFINE: return fqk_dh(1, 1, strict, a, b, out, status, n, scratch, s, ev);
    case FQ_DEVOP_DH_ENDO_BASE: return fqk_fixed_base(1, 1, strict, a, out, status, n, scratch, s);
    case FQ_DEVOP_MUL_ENDO_BASE: return fqk_fixed_base(0, 1, strict, a, out, nullptr, n, scratch, s);
    case FQ_DEVOP_X25519: return fqk_x25519(a, b, out, n, scratch, s);
    case FQ_DEVOP_F25519_BASE + FQ_FP_MUL: case FQ_DEVOP_F25519_BASE + FQ_FP_SQR: case FQ_DEVOP_F25519_BASE + FQ_FP_INV:
    case FQ_DEVOP_F25519_BASE + FQ_FP_ADD: case FQ_DEVOP_F25519_BASE + FQ_FP_SUB:
      return fqk_f25_op(op - FQ_DEVOP_F25519_BASE, a, b, out, n, s);
    default: return cudaErrorInvalidValue;
  }
}

// ---------------------------------------------------------------- slices and the per-GPU threads

struct CallState { std::mutex mu; std::condition_variable cv; int remaining = 0; };

struct SliceJob {
  OpDesc d;
  const uint8_t* in[3] = {nullptr, nullptr, nullptr};      // whole-call buffers
  uint8_t* out = nullptr; uint8_t* status = nullptr;
  CallWork* work = nullptr; int index = 0;                 // the call's rows and this GPU's slice number
  size_t rows_done = 0;
  bool grew = false;                                       // buffers were allocated during this job: its speed is not representative
  bool pinned[kOperands] = {true, true, true, true, true};
  CallState* call = nullptr;
  // results
  int rc = FQ_OK; char err[512] = "";
  double t_stage_in = 0, t_enqueue = 0, t_wait_slot = 0, t_wait_gpu = 0, t_stage_out = 0; int nchunks = 0;      // FQ_TRACE=1 (ms)
  float kernel_ms = 0.f;          // CUDA-event time from the slice's first kernel to its last (drainer, under smu)
  size_t outstanding = 0;         // chunks handed to the drainer and not yet retired (under smu)
};

void job_fail(DevCtx& c, SliceJob* j, int rc) {       // first error of a job wins; tl_err holds the text of this thread's failure
  { std::lock_guard<std::mutex> l(c.smu); if (j->rc == FQ_OK) { j->rc = rc; snprintf(j->err, sizeof(j->err), "%s", tl_err); } }
  if (j->work) j->work->stop();                        // the call has failed: the other GPUs stop taking chunks
}

// feeder side of one slice; caller holds c.mu and the device is current
int feed_slice(DevCtx& c, SliceJob* j) {
  const OpDesc& d = j->d;
  int rc = FQ_OK;
  size_t r0 = 0, rows = 0;
  tl_grew = false;
  for (int ci = 0; rc == FQ_OK && j->work->take(j->index, ci, &r0, &rows); ci++) {
    const int si = ci % kSlots;
    Slot& s = c.slot[si];
    const double tw0 = now_ms();
    { std::unique_lock<std::mutex> l(c.smu); c.scv.wait(l, [&] { return !s.busy; }); if (j->rc != FQ_OK) break; }     // a retired chunk failed: stop feeding
    j->t_wait_slot += now_ms() - tw0; j->nchunks++; j->rows_done += rows;
    if (rows > d.chunk_rows) { rc = fail(FQ_ERR_ARG, "internal: chunk of %zu rows exceeds the staging size %zu", rows, d.chunk_rows); break; }
    auto body = [&]() -> int {
      int e;
      for (int w = 0; w < kOperands; w++) {
        const int wb = operand_bytes(d, w);
        if (!wb) continue;
        if ((e = dbuf_reserve(s, w, d.chunk_rows * wb)) != FQ_OK) return e;
        if (!j->pinned[w] && (e = hbuf_reserve(s, w, d.chunk_rows * wb)) != FQ_OK) return e;
      }
      if ((e = scratch_reserve(s, d.scratch, d.chunk_rows)) != FQ_OK) return e;
      for (int w = 0; w < 3; w++) {
        const int wb = d.in_bytes[w];
        if (!wb) continue;
        const uint8_t* src = j->in[w] + r0 * wb;
        if (!j->pinned[w]) {                          // pageable input: stage here, overlapping earlier chunks' kernels
          const double t0 = now_ms();
          c.copy_in.copy(s.hbuf[w], src, rows * wb);
          j->t_stage_in += now_ms() - t0;
          src = (const uint8_t*)s.hbuf[w];
        }
        CU(cudaMemcpyAsync(s.dbuf[w], src, rows * wb, cudaMemcpyHostToDevice, s.st));
      }
      const double te0 = now_ms();
      if (ci == 0) CU(cudaEventRecord(c.job_e0, s.st));
      CU(cudaEventRecord(s.e0, s.st));
      CU(launch(c, d.op, s.dbuf[0], s.dbuf[1], s.dbuf[2], s.dbuf[3], s.dbuf[4], rows, s.st, s.scratch));
      CU(cudaEventRecord(s.e1, s.st));
      CU(cudaMemcpyAsync(j->pinned[3] ? (void*)(j->out + r0 * d.out_bytes) : s.hbuf[3], s.dbuf[3], rows * d.out_bytes, cudaMemcpyDeviceToHost, s.st));
      if (d.status) CU(cudaMemcpyAsync(j->pinned[4] ? (void*)(j->status + r0) : s.hbuf[4], s.dbuf[4], rows, cudaMemcpyDeviceToHost, s.st));
      CU(cudaEventRecord(s.done, s.st));
      j->t_enqueue += now_ms() - te0;
      return FQ_OK;
    };
    rc = body();
    if (rc != FQ_OK) { cudaStreamSynchronize(s.st); break; }      // whatever part of the chunk was enqueued must not outlive its buffers
    { std::lock_guard<std::mutex> l(c.smu); s.busy = true; j->outstanding++; c.chunks.push_back({si, r0, rows, j}); }
    c.scv.notify_all();
  }
  if (rc != FQ_OK) job_fail(c, j, rc);
  j->grew = tl_grew;
  { std::unique_lock<std::mutex> l(c.smu); c.scv.wait(l, [&] { return j->outstanding == 0; }); }
  if (wipe_after_call()) {
    for (Slot& s : c.slot) {
      for (int w = 0; w < kOperands; w++) {
        if (s.dbuf[w]) cudaMemsetAsync(s.dbuf[w], 0, s.dcap[w], s.st);
        if (s.hbuf[w]) memset(s.hbuf[w], 0, s.hcap[w]);
      }
      if (s.scratch) cudaMemsetAsync(s.scratch, 0, s.scratch_cap, s.st);
    }
    for (Slot& s : c.slot) cudaStreamSynchronize(s.st);
  }
  return j->rc;
}

void drainer_main(DevCtx* cp) {
  DevCtx& c = *cp;
  bool current = false;
  for (;;) {
    Chunk ch;
    { std::unique_lock<std::mutex> l(c.smu); c.scv.wait(l, [&] { return !c.chunks.empty(); }); ch = c.chunks.front(); c.chunks.pop_front(); }
    if (!current) { cudaSetDevice(c.dev); current = true; }
    Slot& s = c.slot[ch.si];
    SliceJob* j = ch.job;
    const OpDesc& d = j->d;
    const double tg0 = now_ms();
    cudaError_t e = cudaEventSynchronize(s.done);
    const double tg1 = now_ms();
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, c.job_e0, s.e1);       // first kernel's start to this chunk's end on this GPU: the last chunk's value stays
    if (e != cudaSuccess) {
      cudaGetLastError();
      job_fail(c, j, fail(FQ_ERR_CUDA, "chunk at row %zu on device %d failed: %s", ch.r0, c.dev, cudaGetErrorString(e)));
    } else {
      if (!j->pinned[3]) c.copy_out.copy(j->out + ch.r0 * d.out_bytes, s.hbuf[3], ch.rows * d.out_bytes);       // staged results -> caller's pageable memory
      if (d.status && !j->pinned[4]) memcpy(j->status + ch.r0, s.hbuf[4], ch.rows);
    }
    const double tg2 = now_ms();
    { std::lock_guard<std::mutex> l(c.smu); if (e == cudaSuccess) j->kernel_ms = ms; j->t_wait_gpu += tg1 - tg0; j->t_stage_out += tg2 - tg1; s.busy = false; j->outstanding--; }
    c.scv.notify_all();
  }
}

void feeder_main(DevCtx* cp) {
  DevCtx& c = *cp;
  for (;;) {
    SliceJob* j;
    { std::unique_lock<std::mutex> l(c.qmu); c.qcv.wait(l, [&] { return !c.jobs.empty(); }); j = c.jobs.front(); c.jobs.pop_front(); }
    {
      std::lock_guard<std::mutex> dl(c.mu);
      int rc = ctx_init(c);
      if (rc != FQ_OK) job_fail(c, j, rc); else feed_slice(c, j);
    }
    CallState* cs = j->call;
    { std::lock_guard<std::mutex> l(cs->mu); cs->remaining--; cs->cv.notify_all(); }     // notified under the lock: once it is released the caller may destroy cs and the job
  }
}

void submit(DevCtx& c, SliceJob* j) {
  std::lock_guard<std::mutex> l(c.qmu);
  if (!c.threads) {
    std::thread(feeder_main, &c).detach();
    std::thread(drainer_main, &c).detach();
    c.threads = true;
  }
  c.jobs.push_back(j);
  c.qcv.notify_one();
}

int run_host(int op, const uint8_t* a, const uint8_t* b, const uint8_t* cbuf, uint8_t* out, uint8_t* status, size_t n, int ndev) {
  tl_kernel_ms = 0.f;
  const OpDesc d = describe(op);
  if (d.op < 0) return fail(FQ_ERR_ARG, "unknown operation %d", op);
  if (n == 0) return FQ_OK;
  const uint8_t* in[3] = {a, b, cbuf};
  for (int w = 0; w < 3; w++) if (d.in_bytes[w] && !in[w]) return fail(FQ_ERR_ARG, "null input buffer");
  if (!out || (d.status && !status)) return fail(FQ_ERR_ARG, "null output buffer");
  const int count = device_count();
  if (count < 0) return count;
  const int base = g_dev_base.load();
  if (ndev < 1 || base + ndev > count) return fail(FQ_ERR_ARG, "ndev=%d with device base %d but %d device(s) visible", ndev, base, count);
  bool pinned[kOperands];
  const void* ptrs[kOperands] = {a, b, cbuf, out, d.status ? status : nullptr};
  for (int w = 0; w < kOperands; w++) {
    const int wb = operand_bytes(d, w);
    const PtrKind k = wb ? classify(ptrs[w], n * wb) : PK_PINNED;
    if (k == PK_DEVICE) return fail(FQ_ERR_ARG, "operand %d is device memory: the host entry points take host pointers (use fq_dev_run for device buffers)", w);
    pinned[w] = k == PK_PINNED;
  }
  bool all_pinned = true;
  for (int w = 0; w < kOperands; w++) all_pinned = all_pinned && pinned[w];
  OpDesc dj = d;
  // Staged (pageable) operands add two host copies to every chunk's trip; shorter chunks shorten what is exposed at both ends
  // of the pipeline: half the chunk for the variable-base DH ops (measured, one B200: 13.7 -> 12.8 ms per 2^20 rows).
  if (!all_pinned && d.var_dh) dj.chunk_rows = dj.chunk_rows / 2 / kRowQuant * kRowQuant;
  const double t_call0 = now_ms();
  CallState cs;
  CallWork work;
  const int rc_class = d.rate_class;
  double share[kMaxDev] = {0};
  if (rc_class >= 0) for (int i = 0; i < ndev; i++) share[i] = ctx_of(base + i).rate[rc_class].load();
  work.init(n, ndev, dj.chunk_rows, rc_class >= 0 ? share : nullptr);
  std::vector<SliceJob> jobs((size_t)ndev);
  int used = 0;
  for (int i = 0; i < ndev; i++) {
    if (work.r[(size_t)i].lo >= work.r[(size_t)i].hi) break;          // fewer rows than GPUs: the empty slices get no job
    SliceJob& j = jobs[(size_t)i];
    j.d = dj; j.in[0] = a; j.in[1] = b; j.in[2] = cbuf; j.out = out; j.status = status;
    j.work = &work; j.index = i;
    for (int w = 0; w < kOperands; w++) j.pinned[w] = pinned[w];
    j.call = &cs;
    used++;
  }
  { std::lock_guard<std::mutex> l(cs.mu); cs.remaining = used; }
  for (int i = 0; i < used; i++) submit(ctx_of(base + i), &jobs[i]);
  if (!pinned[3]) populate_output(out, n * (size_t)d.out_bytes);
  if (d.status && !pinned[4]) populate_output(status, n);
  { std::unique_lock<std::mutex> l(cs.mu); cs.cv.wait(l, [&] { return cs.remaining == 0; }); }
  int rc = FQ_OK;
  if (trace_enabled()) fprintf(stderr, "[fq trace] op %d: %zu rows on %d device(s), %.3f ms inside the call\n", op, n, used, now_ms() - t_call0);
  if (trace_enabled())
    for (int i = 0; i < used; i++)
      fprintf(stderr, "[fq trace] op %d dev %d rows %zu chunks %d: feeder wait-slot %.2f stage-in %.2f enqueue %.2f ms | drainer wait-gpu %.2f stage-out %.2f ms | kernels %.2f ms | pinned %d%d%d%d%d\n",
              op, base + i, jobs[i].rows_done, jobs[i].nchunks, jobs[i].t_wait_slot, jobs[i].t_stage_in, jobs[i].t_enqueue, jobs[i].t_wait_gpu,
              jobs[i].t_stage_out, jobs[i].kernel_ms, (int)pinned[0], (int)pinned[1], (int)pinned[2], (int)pinned[3], (int)pinned[4]);
  for (int i = 0; i < kMaxDev; i++) tl_rows_per_dev[i] = i < used ? jobs[(size_t)i].rows_done : 0;
  if (rc_class >= 0 && ndev > 1)                       // remember how fast each GPU was (rows per ms of device time), for the next call's slices
    for (int i = 0; i < used; i++) {
      const SliceJob& j = jobs[(size_t)i];
      if (j.rc != FQ_OK || j.grew || j.kernel_ms <= 0.f || j.rows_done < 2 * dj.chunk_rows) continue;
      std::atomic<double>& r = ctx_of(base + i).rate[rc_class];
      const double now = (double)j.rows_done / j.kernel_ms, old = r.load();
      r.store(old > 0 ? 0.5 * (old + now) : now);
    }
  for (int i = 0; i < used; i++) {
    if (jobs[i].rc != FQ_OK && rc == FQ_OK) { rc = jobs[i].rc; snprintf(tl_err, sizeof(tl_err), "%s", jobs[i].err); }
    if (jobs[i].kernel_ms > tl_kernel_ms) tl_kernel_ms = jobs[i].kernel_ms;
  }
  return rc;
}

// zeroes (device and pinned staging hold scalars, tables of secret multiples and shared secrets) and frees a slot's buffers
int slot_wipe_free(Slot& s) {
  for (int w = 0; w < kOperands; w++) {
    if (s.dbuf[w]) { CU(cudaMemsetAsync(s.dbuf[w], 0, s.dcap[w], s.st)); }
    if (s.hbuf[w]) memset(s.hbuf[w], 0, s.hcap[w]);
  }
  if (s.scratch) CU(cudaMemsetAsync(s.scratch, 0, s.scratch_cap, s.st));
  CU(cudaStreamSynchronize(s.st));
  for (int w = 0; w < kOperands; w++) {
    if (s.dbuf[w]) { CU(cudaFree(s.dbuf[w])); s.dbuf[w] = nullptr; s.dcap[w] = 0; }
    if (s.hbuf[w]) { CU(cudaFreeHost(s.hbuf[w])); s.hbuf[w] = nullptr; s.hcap[w] = 0; }
  }
  if (s.scratch) { CU(cudaFree(s.scratch)); s.scratch = nullptr; s.scratch_cap = 0; }
  return FQ_OK;
}

// ---------------------------------------------------------------- page-locked memory placed next to the GPUs that will read it
// On a multi-socket host a GPU moves data to and from the other socket's memory through the inter-socket link: measured on
// an 8 x B200 box, the four GPUs that are remote to a buffer take 8 % (keygen) to 13 % (DH) longer for their slices than the
// four local ones, and the call ends with the slowest.  fq_host_alloc_sliced lays a buffer out the way run_host will cut it:
// the bytes of slice i are placed (mbind, MPOL_PREFERRED) on the NUMA node of GPU base + i before the pages are locked.
// Everything here degrades silently to an ordinary page-locked allocation: no NUMA information (a VM that hides it), no
// permission for mbind (a container's seccomp profile), a single node.
int device_numa_node(int dev) {
#ifdef FQ_MOCK_CUDA
  (void)dev; return -1;
#else
  char id[32] = "";
  if (cudaDeviceGetPCIBusId(id, sizeof(id), dev) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char* q = id; *q; q++) if (*q >= 'A' && *q <= 'F') *q = (char)(*q - 'A' + 'a');
  char path[96]; snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", id);
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
#endif
}
std::mutex g_sliced_mu;
std::vector<std::pair<void*, size_t>> g_sliced;     // allocations of fq_host_alloc_sliced: base, mapped length

// locks the context of GPU `dev` for a device-resident call of the calling thread
struct DevLock {
  DevCtx* c = nullptr; int rc = FQ_OK;
  explicit DevLock(int dev) {
    const int count = device_count();
    if (count < 0) { rc = count; return; }
    if (dev < 0 || dev >= count) { rc = fail(FQ_ERR_ARG, "device %d out of range (%d device(s))", dev, count); return; }
    c = &ctx_of(dev);
    c->mu.lock();
    rc = ctx_init(*c);
    if (rc != FQ_OK) { c->mu.unlock(); c = nullptr; }
  }
  ~DevLock() { if (c) c->mu.unlock(); }
};

}  // namespace

extern "C" {

int fq_version(void) { return FQ_VERSION; }
int fq_device_count(void) { return device_count(); }
const char* fq_last_error(void) { return tl_err; }
float fq_last_kernel_ms(void) { return tl_kernel_ms; }

int fq_set_device_base(int first) {
  int count = device_count();
  if (count < 0) return count;
  if (first < 0 || first >= count) return fail(FQ_ERR_ARG, "device base %d out of range (%d device(s))", first, count);
  g_dev_base.store(first);
  return FQ_OK;
}

int fq_trim(void) {
  int count = device_count();
  if (count < 0) return count;
  for (int dev = 0; dev < count && dev < kMaxDev; dev++) {
    DevCtx& c = ctx_of(dev);
    std::lock_guard<std::mutex> l(c.mu);
    if (!c.ready) continue;
    CU(cudaSetDevice(dev));
    CU(cudaDeviceSynchronize());
    for (int si = 0; si < kSlots; si++) { int rc = slot_wipe_free(c.slot[si]); if (rc != FQ_OK) return rc; }
    if (c.flush) { CU(cudaFree(c.flush)); c.flush = nullptr; }
  }
  return FQ_OK;
}

int fq_set_select_mode(int strict) {
  if (strict != 0 && strict != 1) return fail(FQ_ERR_ARG, "select mode must be 1 (strict scan, default) or 0 (masked loads)");
  g_strict.store(strict);
  return FQ_OK;
}
int fq_get_select_mode(void) { return strict_mode(); }

int fq_fp2_mul(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_MUL, a, b, nullptr, out, nullptr, n, ndev); }
int fq_fp2_sqr(const uint8_t* a, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_SQR, a, nullptr, nullptr, out, nullptr, n, ndev); }
int fq_fp2_inv(const uint8_t* a, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_INV, a, nullptr, nullptr, out, nullptr, n, ndev); }
int fq_fp2_invsqrt(const uint8_t* a, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_INVSQRT, a, nullptr, nullptr, out, nullptr, n, ndev); }
int fq_fp2_add(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_ADD, a, b, nullptr, out, nullptr, n, ndev); }
int fq_fp2_sub(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_SUB, a, b, nullptr, out, nullptr, n, ndev); }
int fq_fp2_neg(const uint8_t* a, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_NEG, a, nullptr, nullptr, out, nullptr, n, ndev); }
int fq_fp2_conj(const uint8_t* a, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_CONJ, a, nullptr, nullptr, out, nullptr, n, ndev); }
int fq_fp2_select(const uint8_t* c, const uint8_t* x, const uint8_t* y, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP2_SELECT, x, y, c, out, nullptr, n, ndev); }
int fq_fp_select(const uint8_t* c, const uint8_t* x, const uint8_t* y, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_FP_SELECT, x, y, c, out, nullptr, n, ndev); }
int fq_fp_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev) {
  if (op < FQ_FP_MUL || op > FQ_FP_INVSQRT) return fail(FQ_ERR_ARG, "unknown GF(p) operation %d", op);
  return run_host(FQ_DEVOP_FP_BASE + op, a, b, nullptr, out, nullptr, n, ndev);
}
int fq_fp25519_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev) {
  if (op < FQ_FP_MUL || op > FQ_FP_SUB) return fail(FQ_ERR_ARG, "unknown GF(2^255-19) operation %d", op);
  return run_host(FQ_DEVOP_F25519_BASE + op, a, b, nullptr, out, nullptr, n, ndev);
}
int fq_decode(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DECODE, enc, nullptr, nullptr, xy, status, n, ndev); }
int fq_point_on_curve(const uint8_t* xy, uint8_t* ok, size_t n, int ndev) { return run_host(FQ_DEVOP_ON_CURVE, xy, nullptr, nullptr, ok, nullptr, n, ndev); }
int fq_decode_spec(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DECODE_SPEC, enc, nullptr, nullptr, xy, status, n, ndev); }
int fq_encode(const uint8_t* xy, uint8_t* enc, size_t n, int ndev) { return run_host(FQ_DEVOP_ENCODE, xy, nullptr, nullptr, enc, nullptr, n, ndev); }
int fq_dh(const uint8_t* k, const uint8_t* enc_pt, uint8_t* enc_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH, k, enc_pt, nullptr, enc_out, status, n, ndev); }
int fq_dh_affine(const uint8_t* k, const uint8_t* xy, uint8_t* xy_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_AFFINE, k, xy, nullptr, xy_out, status, n, ndev); }
int fq_dh_base(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_BASE, k, nullptr, nullptr, enc_out, status, n, ndev); }
int fq_mul_base(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev) { return run_host(FQ_DEVOP_MUL_BASE, k, nullptr, nullptr, enc_out, nullptr, n, ndev); }

int fq_dh_endo(const uint8_t* k, const uint8_t* enc_pt, uint8_t* enc_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_ENDO, k, enc_pt, nullptr, enc_out, status, n, ndev); }
int fq_dh_endo_affine(const uint8_t* k, const uint8_t* xy, uint8_t* xy_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_ENDO_AFFINE, k, xy, nullptr, xy_out, status, n, ndev); }
int fq_dh_endo_base(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_ENDO_BASE, k, nullptr, nullptr, enc_out, status, n, ndev); }
int fq_mul_endo_base(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev) { return run_host(FQ_DEVOP_MUL_ENDO_BASE, k, nullptr, nullptr, enc_out, nullptr, n, ndev); }
int fq_dh_base_comb(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev) { return run_host(FQ_DEVOP_DH_BASE_COMB, k, nullptr, nullptr, enc_out, status, n, ndev); }
int fq_mul_base_comb(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev) { return run_host(FQ_DEVOP_MUL_BASE_COMB, k, nullptr, nullptr, enc_out, nullptr, n, ndev); }
int fq_x25519(const uint8_t* k, const uint8_t* u, uint8_t* out, size_t n, int ndev) { return run_host(FQ_DEVOP_X25519, k, u, nullptr, out, nullptr, n, ndev); }

int fq_host_alloc(void** p, size_t bytes) {
  if (!p) return fail(FQ_ERR_ARG, "null pointer");
  int count = device_count();
  if (count < 0) return count;
  CU(cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocPortable));
  return FQ_OK;
}
int fq_host_alloc_sliced(void** p, size_t rows, size_t row_bytes, int ndev) {
  if (!p || ndev < 1 || row_bytes == 0) return fail(FQ_ERR_ARG, "null pointer / bad slice description");
  const int count = device_count();
  if (count < 0) return count;
  const int base = g_dev_base.load();
  const size_t page = (size_t)sysconf(_SC_PAGESIZE), bytes = rows * row_bytes;
  const size_t len = ((bytes ? bytes : 1) + page - 1) / page * page;
  void* m = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
  if (m == MAP_FAILED) return fail(FQ_ERR_CUDA, "mmap of %zu bytes failed", len);
#ifdef __linux__
  const size_t per = (rows + ndev - 1) / ndev;
  for (int i = 0; i < ndev && base + i < count; i++) {
    size_t lo = (size_t)i * per * row_bytes, hi = ((size_t)(i + 1) * per < rows ? (size_t)(i + 1) * per : rows) * row_bytes;
    if (lo >= hi) break;
    lo = (lo + page - 1) / page * page; hi = hi / page * page;           // whole pages of the slice (a straddling page goes where it falls)
    const int node = device_numa_node(base + i);
    if (node < 0 || node >= 1024 || lo >= hi) continue;
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(237 /* SYS_mbind */, (char*)m + lo, hi - lo, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(8 * sizeof(mask) + 1), 0u);      // best effort
  }
#endif
  cudaError_t e = cudaHostRegister(m, len, cudaHostRegisterPortable);
  if (e != cudaSuccess) { munmap(m, len); return fail(FQ_ERR_CUDA, "cudaHostRegister of %zu bytes failed: %s", len, cudaGetErrorString(e)); }
  { std::lock_guard<std::mutex> l(g_sliced_mu); g_sliced.push_back({m, len}); }
  *p = m;
  return FQ_OK;
}
int fq_host_free(void* p) {
  if (!p) return FQ_OK;
  size_t len = 0;
  {
    std::lock_guard<std::mutex> l(g_sliced_mu);
    for (size_t i = 0; i < g_sliced.size(); i++) if (g_sliced[i].first == p) { len = g_sliced[i].second; g_sliced.erase(g_sliced.begin() + (long)i); break; }
  }
  if (len) { CU(cudaHostUnregister(p)); munmap(p, len); return FQ_OK; }
  CU(cudaFreeHost(p));
  return FQ_OK;
}
// NUMA node of a GPU as the kernel reports it (/sys/bus/pci/devices/<bus id>/numa_node), -1 if unknown
int fq_device_numa_node(int dev) {
  const int count = device_count();
  if (count < 0) return count;
  if (dev < 0 || dev >= count) return fail(FQ_ERR_ARG, "device %d out of range (%d device(s))", dev, count);
  return device_numa_node(dev);
}

int fq_dev_alloc(int dev, void** p, size_t bytes) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  if (!p) return fail(FQ_ERR_ARG, "null pointer");
  CU(cudaMalloc(p, bytes ? bytes : 1));
  return FQ_OK;
}
int fq_dev_free(int dev, void* p) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  if (p) CU(cudaFree(p));
  return FQ_OK;
}
int fq_dev_upload(int dev, void* dst, const void* src, size_t bytes) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  CU(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
  return FQ_OK;
}
int fq_dev_download(int dev, void* dst, const void* src, size_t bytes) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  CU(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return FQ_OK;
}
int fq_dev_run3(int op, int dev, const void* a, const void* b, const void* c, void* out, void* status, size_t n, int iters, float* ms) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  const OpDesc d = describe(op);
  if (d.op < 0 || iters < 1) return fail(FQ_ERR_ARG, "bad op/iters");
  if ((op == FQ_DEVOP_FP2_INV || op == FQ_DEVOP_F25519_BASE + FQ_FP_INV) && a == out) return fail(FQ_ERR_ARG, "inv: out must not alias a (the prefix products are parked in out)");
  DevCtx& cx = *L.c;
  Slot& s = cx.slot[0];
  int rc;
  if ((rc = scratch_reserve(s, d.scratch, n)) != FQ_OK) return rc;
  cudaEvent_t ph[4];
  for (int i = 0; i < 4; i++) CU(cudaEventCreate(&ph[i]));
  CU(cudaEventRecord(s.e0, s.st));
  for (int i = 0; i < iters; i++) CU(launch(cx, op, a, b, c, out, status, n, s.st, s.scratch, (d.var_dh && i == iters - 1) ? ph : nullptr));
  CU(cudaEventRecord(s.e1, s.st));
  CU(cudaEventSynchronize(s.e1));
  float t = 0.f;
  CU(cudaEventElapsedTime(&t, s.e0, s.e1));
  tl_phase_ms[0] = tl_phase_ms[1] = tl_phase_ms[2] = 0.f;
  if (d.var_dh && n > 0) for (int i = 0; i < 3; i++) CU(cudaEventElapsedTime(&tl_phase_ms[i], ph[i], ph[i + 1]));
  for (int i = 0; i < 4; i++) cudaEventDestroy(ph[i]);
  if (ms) *ms = t / iters;
  return FQ_OK;
}
int fq_dev_run(int op, int dev, const void* a, const void* b, void* out, void* status, size_t n, int iters, float* ms) {
  return fq_dev_run3(op, dev, a, b, nullptr, out, status, n, iters, ms);
}
int fq_last_rows_per_device(size_t* rows, int ndev) {
  if (!rows || ndev < 1) return fail(FQ_ERR_ARG, "null pointer");
  for (int i = 0; i < ndev; i++) rows[i] = i < kMaxDev ? tl_rows_per_dev[i] : 0;
  return FQ_OK;
}
int fq_dev_last_phase_ms(float* ms3) {
  if (!ms3) return fail(FQ_ERR_ARG, "null pointer");
  for (int i = 0; i < 3; i++) ms3[i] = tl_phase_ms[i];
  return FQ_OK;
}
int fq_dev_flush_l2(int dev) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  DevCtx& c = *L.c;
  if (!c.flush) CU(cudaMalloc(&c.flush, kFlushBytes));
  CU(cudaMemsetAsync(c.flush, 0, kFlushBytes, c.slot[0].st));
  CU(cudaStreamSynchronize(c.slot[0].st));
  return FQ_OK;
}

int fq_imad_peak(int dev, double* wide_per_s, double* imad32_per_s) {
  DevLock L(dev); if (L.rc != FQ_OK) return L.rc;
  Slot& s = L.c->slot[0];
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, dev));
  int blocks = prop.multiProcessorCount * 4, trips = 8192;
  void* scratch = nullptr;
  CU(cudaMalloc(&scratch, (size_t)blocks * 256 * 4));
  double res[2] = {0, 0};
  for (int v = 0; v < 2; v++) {
    CU(fqk_imad_peak(v, scratch, blocks, trips / 8, s.st));     // warm-up
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
      CU(cudaEventRecord(s.e0, s.st));
      CU(fqk_imad_peak(v, scratch, blocks, trips, s.st));
      CU(cudaEventRecord(s.e1, s.st));
      CU(cudaEventSynchronize(s.e1));
      float t; CU(cudaEventElapsedTime(&t, s.e0, s.e1));
      if (t < best) best = t;
    }
    res[v] = (double)blocks * 256.0 * trips * 128.0 / (best * 1e-3);
  }
  CU(cudaFree(scratch));
  if (wide_per_s) *wide_per_s = res[0];
  if (imad32_per_s) *imad32_per_s = res[1];
  return FQ_OK;
}

#ifdef FQ_MOCK_CUDA
// test hook (tests/hostsim builds only): the slices of a call of n rows on ndev GPUs with the given relative speeds
FQ_API int fq_test_slices(size_t n, int ndev, size_t full, const double* share, size_t* lo, size_t* hi) {
  CallWork w;
  w.init(n, ndev, full, share);
  for (int i = 0; i < ndev; i++) { lo[i] = w.r[(size_t)i].lo; hi[i] = w.r[(size_t)i].hi; }
  return (int)w.r.size();
}
// test hook (tests/hostsim builds only): the chunk schedule of a slice of `rows` rows with full chunks of `full` rows
FQ_API size_t fq_test_chunk_schedule(size_t rows, size_t full, size_t* bounds, size_t cap) {
  CallWork w;
  w.init(rows, 1, full);
  std::vector<size_t> b(1, 0);
  size_t r0 = 0, n = 0;
  for (int ci = 0; w.take(0, ci, &r0, &n); ci++) b.push_back(r0 + n);
  for (size_t i = 0; i < b.size() && i < cap; i++) bounds[i] = b[i];
  return b.size();
}
#endif

}  // extern "C"
