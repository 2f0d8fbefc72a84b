// stream_stress.cpp -- TEST INFRASTRUCTURE ONLY.  Drives the stream entry points of fourq_b200/csrc/capi.cu (fq_stream_run,
// built against the mock CUDA runtime of this directory) next to host calls on the same GPUs; linked with -fsanitize=thread
// by build_stream.sh.  Exit code 0 and the line "stream_stress ok" mean:
//   - a stream call on a GPU whose lock a long host call holds returned without waiting for that call;
//   - stream calls from several threads on their own streams and host calls on the same GPUs all matched the simulation;
//   - every pool block was zero when its stream freed it, and the mock saw no invalid memory access.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <random>
#include <thread>
#include <vector>
#include "../../include/fourq_b200.h"

extern "C" {
int sim_fp2_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
int sim_comb(int dh, const uint8_t* k, uint8_t* out, uint8_t* status, size_t n);
void mock_set_device_count(int n);
void mock_set_jitter_us(int us);
void mock_set_kernel_delay_us(int dev, int us);
long mock_violations();
long mock_counter(const char* name);
void* mock_stream_create(int dev);
void mock_stream_sync(void* s);
void* mock_device_alloc(int dev, size_t bytes);
void mock_device_free(void* p);
}

static std::atomic<int> g_bad{0};
#define CHECK(c) do { if (!(c)) { fprintf(stderr, "CHECK failed: %s (%s:%d) err=%s\n", #c, __FILE__, __LINE__, fq_last_error()); g_bad++; } } while (0)

static void fill(std::vector<uint8_t>& v, unsigned seed) { std::minstd_rand r(seed); for (auto& x : v) x = (uint8_t)r(); }
static void* upload(int dev, const std::vector<uint8_t>& v) { void* p = mock_device_alloc(dev, v.size()); memcpy(p, v.data(), v.size()); return p; }
static double ms_since(std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }

// stream calls of one thread on its own stream of GPU `dev`: GF(p^2) products and comb key generation
static void stream_worker(int id, int dev, int rounds) {
  void* s = mock_stream_create(dev);
  const size_t n = 3000 + 97 * id;
  std::vector<uint8_t> a(n * 32), b(n * 32), ref(n * 32), kref(n * 32);
  fill(a, 10 + id); fill(b, 20 + id);
  sim_fp2_op(0, a.data(), b.data(), ref.data(), n);
  sim_comb(0, a.data(), kref.data(), nullptr, n);
  void *da = upload(dev, a), *db = upload(dev, b), *dout = mock_device_alloc(dev, n * 32), *dkey = mock_device_alloc(dev, n * 32);
  for (int r = 0; r < rounds; r++) {
    CHECK(fq_stream_run(FQ_DEVOP_FP2_MUL, da, db, nullptr, dout, nullptr, n, s) == FQ_OK);
    CHECK(fq_stream_run(FQ_DEVOP_MUL_BASE_COMB, da, nullptr, nullptr, dkey, nullptr, n, s) == FQ_OK);
    mock_stream_sync(s);
    CHECK(memcmp(dout, ref.data(), n * 32) == 0);
    CHECK(memcmp(dkey, kref.data(), n * 32) == 0);
  }
  for (void* p : {da, db, dout, dkey}) mock_device_free(p);
}

static void host_worker(int id, int rounds) {
  const size_t n = 40000 + 1333 * id;
  std::vector<uint8_t> a(n * 32), b(n * 32), ref(n * 32), out(n * 32);
  fill(a, 30 + id); fill(b, 40 + id);
  sim_fp2_op(3, a.data(), b.data(), ref.data(), n);
  for (int r = 0; r < rounds; r++) {
    memset(out.data(), 0, out.size());
    CHECK(fq_fp2_add(a.data(), b.data(), out.data(), n, 2) == FQ_OK);
    CHECK(memcmp(out.data(), ref.data(), n * 32) == 0);
  }
}

int main() {
  mock_set_device_count(2);
  { uint8_t k[32] = {1}, o[32]; sim_comb(0, k, o, nullptr, 1); }     // the simulation builds its comb tables once, before any thread uses them
  // first calls on both GPUs (initialisation), outside the timed part
  {
    std::vector<uint8_t> a(64 * 32); fill(a, 1);
    void *da = upload(0, a), *da1 = upload(1, a), *o = mock_device_alloc(0, a.size()), *o1 = mock_device_alloc(1, a.size());
    void *s0 = mock_stream_create(0), *s1 = mock_stream_create(1);
    CHECK(fq_stream_run(FQ_DEVOP_FP2_SQR, da, nullptr, nullptr, o, nullptr, 64, s0) == FQ_OK);
    CHECK(fq_stream_run(FQ_DEVOP_FP2_SQR, da1, nullptr, nullptr, o1, nullptr, 64, s1) == FQ_OK);
    mock_stream_sync(s0); mock_stream_sync(s1);
    for (void* p : {da, da1, o, o1}) mock_device_free(p);
  }
  // a host call that holds GPU 0's lock for a long time (every kernel task on GPU 0 sleeps 400 ms), and a stream call meanwhile
  {
    mock_set_kernel_delay_us(0, 400000);
    const size_t n = 600000;
    std::vector<uint8_t> a(n * 32), b(n * 32), out(n * 32), ref(n * 32);
    fill(a, 2); fill(b, 3);
    sim_fp2_op(3, a.data(), b.data(), ref.data(), n);
    std::atomic<bool> host_done{false};
    std::thread host([&] { CHECK(fq_fp2_add(a.data(), b.data(), out.data(), n, 1) == FQ_OK); host_done = true; });
    std::this_thread::sleep_for(std::chrono::milliseconds(100));
    CHECK(!host_done.load());
    const size_t m = 2048;
    std::vector<uint8_t> x(m * 32), y(m * 32), want(m * 32);
    fill(x, 4); fill(y, 5);
    sim_fp2_op(0, x.data(), y.data(), want.data(), m);
    void *dx = upload(0, x), *dy = upload(0, y), *dout = mock_device_alloc(0, m * 32), *s = mock_stream_create(0);
    const auto t0 = std::chrono::steady_clock::now();
    CHECK(fq_stream_run(FQ_DEVOP_FP2_MUL, dx, dy, nullptr, dout, nullptr, m, s) == FQ_OK);
    const double enqueue_ms = ms_since(t0);
    const bool waited = host_done.load();
    CHECK(!waited);
    CHECK(enqueue_ms < 100.0);
    printf("stream call enqueued in %.2f ms while a host call held the GPU's lock (host call finished first: %d)\n", enqueue_ms, (int)waited);
    mock_stream_sync(s);
    CHECK(memcmp(dout, want.data(), m * 32) == 0);
    host.join();
    CHECK(memcmp(out.data(), ref.data(), n * 32) == 0);
    mock_set_kernel_delay_us(0, 0);
    for (void* p : {dx, dy, dout}) mock_device_free(p);
  }
  // stream callers on their own streams next to host callers, on both GPUs
  {
    mock_set_jitter_us(100);
    std::vector<std::thread> ts;
    for (int i = 0; i < 4; i++) ts.emplace_back(stream_worker, i, i % 2, 3);
    for (int i = 0; i < 2; i++) ts.emplace_back(host_worker, i, 3);
    for (auto& t : ts) t.join();
    mock_set_jitter_us(0);
  }
  CHECK(fq_trim() == FQ_OK);
  CHECK(mock_counter("pool_unzeroed") == 0);
  CHECK(mock_counter("pool_allocs") == mock_counter("pool_frees"));
  CHECK(mock_violations() == 0);
  if (g_bad) { printf("stream_stress FAILED: %d checks\n", g_bad.load()); return 1; }
  printf("stream_stress ok\n");
  return 0;
}
