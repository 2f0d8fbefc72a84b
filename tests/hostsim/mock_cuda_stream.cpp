// mock_cuda_stream.cpp -- TEST INFRASTRUCTURE ONLY (see mock_cuda_stream.h).  Compiled without -DFQ_MOCK_COUNT: the calls here
// reach mock_cuda_runtime.cpp directly.
#include "mock_cuda_stream.h"
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>

namespace {
// synchronising calls, cudaMalloc / cudaFree / cudaHostAlloc / cudaFreeHost, pool allocations and frees, frees of a pool block
// that was not all zeros when its stream reached it, pool trims, work pushed to any stream (copies, memsets, event records,
// kernels, pool frees)
std::atomic<long> g_syncs{0}, g_mallocs{0}, g_pool_allocs{0}, g_pool_frees{0}, g_pool_unzeroed{0}, g_pool_trims{0}, g_enqueued{0};
std::mutex g_mu;
std::map<uintptr_t, int> g_stream_dev;        // streams of mock_stream_create -> their device
std::map<uintptr_t, int> g_capturing;         // streams the test marked as capturing
std::map<uintptr_t, size_t> g_pool_blocks;    // live pool blocks -> bytes
std::map<uintptr_t, void*> g_dev_allocs;      // aligned pointers of mock_device_alloc -> their cudaMalloc block
thread_local int tl_current = 0;              // the device capi.cu made current on this thread (mock_count_cudaSetDevice)
}  // namespace

struct MockPool { int device; };

cudaError_t mock_count_cudaMalloc(void** p, size_t bytes) { g_mallocs++; return cudaMalloc(p, bytes); }
cudaError_t mock_count_cudaFree(void* p) { g_mallocs++; return cudaFree(p); }
cudaError_t mock_count_cudaHostAlloc(void** p, size_t bytes, unsigned flags) { g_mallocs++; return cudaHostAlloc(p, bytes, flags); }
cudaError_t mock_count_cudaFreeHost(void* p) { g_mallocs++; return cudaFreeHost(p); }
cudaError_t mock_count_cudaStreamSynchronize(cudaStream_t s) { g_syncs++; return cudaStreamSynchronize(s); }
cudaError_t mock_count_cudaDeviceSynchronize() { g_syncs++; return cudaDeviceSynchronize(); }
cudaError_t mock_count_cudaEventSynchronize(cudaEvent_t e) { g_syncs++; return cudaEventSynchronize(e); }
cudaError_t mock_count_cudaMemcpy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) { g_syncs++; return cudaMemcpy(dst, src, bytes, kind); }
cudaError_t mock_count_cudaMemcpyAsync(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s) {
  g_enqueued++; return cudaMemcpyAsync(dst, src, bytes, kind, s);
}
cudaError_t mock_count_cudaMemsetAsync(void* p, int v, size_t bytes, cudaStream_t s) { g_enqueued++; return cudaMemsetAsync(p, v, bytes, s); }
cudaError_t mock_count_cudaEventRecord(cudaEvent_t e, cudaStream_t s) { g_enqueued++; return cudaEventRecord(e, s); }
cudaError_t mock_count_cudaSetDevice(int dev) {
  const cudaError_t e = cudaSetDevice(dev);
  if (e == cudaSuccess) tl_current = dev;
  return e;
}
void mock_count_stream_enqueue(cudaStream_t s, std::function<void()> fn) { g_enqueued++; mock_stream_enqueue(s, std::move(fn)); }

cudaError_t cudaGetDevice(int* dev) { *dev = tl_current; return cudaSuccess; }
cudaError_t cudaStreamGetDevice(cudaStream_t s, int* dev) {
  std::lock_guard<std::mutex> l(g_mu);
  auto it = g_stream_dev.find((uintptr_t)s);
  *dev = it == g_stream_dev.end() ? tl_current : it->second;
  return cudaSuccess;
}
cudaError_t cudaStreamIsCapturing(cudaStream_t s, cudaStreamCaptureStatus* st) {
  std::lock_guard<std::mutex> l(g_mu);
  *st = g_capturing.count((uintptr_t)s) ? cudaStreamCaptureStatusActive : cudaStreamCaptureStatusNone;
  return cudaSuccess;
}
cudaError_t cudaMemPoolCreate(cudaMemPool_t* pool, const cudaMemPoolProps* props) { *pool = new MockPool{props->location.id}; return cudaSuccess; }
cudaError_t cudaMemPoolDestroy(cudaMemPool_t pool) { delete pool; return cudaSuccess; }
cudaError_t cudaMemPoolSetAttribute(cudaMemPool_t, cudaMemPoolAttr, void*) { return cudaSuccess; }
cudaError_t cudaMemPoolTrimTo(cudaMemPool_t, size_t) { g_pool_trims++; return cudaSuccess; }
// a block is handed out at once and poisoned like cudaMalloc's; the kernels and memsets of mock_cuda_runtime.cpp accept it
// because it overlaps no registered allocation
cudaError_t cudaMallocFromPoolAsync(void** p, size_t bytes, cudaMemPool_t, cudaStream_t) {
  void* q = malloc(bytes ? bytes : 1);
  if (!q) return cudaErrorMemoryAllocation;
  memset(q, 0xA5, bytes);
  g_pool_allocs++;
  { std::lock_guard<std::mutex> l(g_mu); g_pool_blocks[(uintptr_t)q] = bytes; }
  *p = q;
  return cudaSuccess;
}
// the block is released when its stream reaches the free; it must be all zeros by then
cudaError_t cudaFreeAsync(void* p, cudaStream_t s) {
  g_pool_frees++; g_enqueued++;
  mock_stream_enqueue(s, [p] {
    std::lock_guard<std::mutex> l(g_mu);
    auto it = g_pool_blocks.find((uintptr_t)p);
    if (it == g_pool_blocks.end()) { g_pool_unzeroed++; return; }
    const unsigned char* q = (const unsigned char*)p;
    for (size_t i = 0; i < it->second; i++) if (q[i]) { g_pool_unzeroed++; break; }
    g_pool_blocks.erase(it);
    free(p);
  });
  return cudaSuccess;
}

// ---------------------------------------------------------------- controls for the tests
extern "C" {
// a counter by name, -1 for an unknown name
__attribute__((visibility("default"))) long mock_counter(const char* name) {
  const std::map<std::string, std::atomic<long>*> m = {{"syncs", &g_syncs}, {"mallocs", &g_mallocs}, {"pool_allocs", &g_pool_allocs},
      {"pool_frees", &g_pool_frees}, {"pool_unzeroed", &g_pool_unzeroed}, {"pool_trims", &g_pool_trims}, {"enqueued", &g_enqueued}};
  auto it = m.find(name);
  return it == m.end() ? -1 : it->second->load();
}
// a stream of GPU `dev` (what a caller of fq_stream_run brings), its completion, and whether it reports an active capture
__attribute__((visibility("default"))) void* mock_stream_create(int dev) {
  cudaSetDevice(dev);
  cudaStream_t s = nullptr;
  cudaStreamCreateWithFlags(&s, 0);
  cudaSetDevice(tl_current);
  std::lock_guard<std::mutex> l(g_mu); g_stream_dev[(uintptr_t)s] = dev;
  return s;
}
__attribute__((visibility("default"))) void mock_stream_sync(void* s) { cudaStreamSynchronize((cudaStream_t)s); }
__attribute__((visibility("default"))) void mock_set_capturing(void* s, int on) {
  std::lock_guard<std::mutex> l(g_mu);
  if (on) g_capturing[(uintptr_t)s] = 1; else g_capturing.erase((uintptr_t)s);
}
// device memory of GPU `dev` without going through the engine, 32-byte aligned as the stream entry points require
__attribute__((visibility("default"))) void* mock_device_alloc(int dev, size_t bytes) {
  void* raw = nullptr;
  cudaSetDevice(dev);
  const cudaError_t e = cudaMalloc(&raw, bytes + 32);
  cudaSetDevice(tl_current);
  if (e != cudaSuccess) return nullptr;
  void* p = (void*)(((uintptr_t)raw + 31) / 32 * 32);
  std::lock_guard<std::mutex> l(g_mu); g_dev_allocs[(uintptr_t)p] = raw;
  return p;
}
__attribute__((visibility("default"))) void mock_device_free(void* p) {
  void* raw = nullptr;
  { std::lock_guard<std::mutex> l(g_mu); auto it = g_dev_allocs.find((uintptr_t)p); if (it == g_dev_allocs.end()) return; raw = it->second; g_dev_allocs.erase(it); }
  cudaFree(raw);
}
__attribute__((visibility("default"))) int mock_current_device() { return tl_current; }
__attribute__((visibility("default"))) void mock_set_current_device(int dev) { mock_count_cudaSetDevice(dev); }
}
