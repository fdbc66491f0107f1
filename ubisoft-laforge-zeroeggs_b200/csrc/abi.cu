// Error plumbing, launch counter and version for the C ABI (include/zeggs_b200.h).
#include <cstring>
#include <stdarg.h>
#include <atomic>
#include <mutex>
#include <vector>
#include "common.cuh"
#include "../../include/zeggs_b200.h"

namespace zeggs {
static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace zeggs

// ---------------------------------------------------------------- live kernel timer (bench.py's roofline leg)
// When enabled, selected launches are bracketed by CUDA events on their own stream (no synchronisation is
// added); durations are resolved lazily by zeggs_timing_read() after the caller has synchronised.
namespace zeggs {
struct TimedSpan { int name; cudaEvent_t e0, e1; };
static const char* kTimerNames[] = {"decoder_fwd", "decoder_bwd", "decoder_wgrad", "mel", "loss", "encoders_fwd", "encoders_bwd", "optimizer", "weight_pack"};
constexpr int kNumTimers = 9;
static bool g_timing = false;
static std::vector<TimedSpan> g_spans;
static std::vector<cudaEvent_t> g_pool;
static std::mutex g_tmu;

int timer_id(const char* name) {
  for (int i = 0; i < kNumTimers; ++i) if (!strcmp(kTimerNames[i], name)) return i;
  return -1;
}
static cudaEvent_t get_event() {
  if (!g_pool.empty()) { cudaEvent_t e = g_pool.back(); g_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
// Under stream capture the record becomes an EXTERNAL event-record node (cudaEventRecordExternal): every replay of the
// captured graph re-records the same event pair, and zeggs_timing_read() after a synchronised replay returns that replay's span.
static void record_event(cudaEvent_t e, cudaStream_t s) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(s, &st);
  cudaEventRecordWithFlags(e, s, st == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
}
void* timer_begin(int id, cudaStream_t s) {
  if (!g_timing || id < 0) return nullptr;
  std::lock_guard<std::mutex> lk(g_tmu);
  TimedSpan sp; sp.name = id; sp.e0 = get_event(); sp.e1 = get_event();
  record_event(sp.e0, s);
  g_spans.push_back(sp);
  return (void*)(uintptr_t)g_spans.size();
}
void timer_end(void* h, cudaStream_t s) {
  if (!h) return;
  std::lock_guard<std::mutex> lk(g_tmu);
  record_event(g_spans[(size_t)(uintptr_t)h - 1].e1, s);
}
}  // namespace zeggs

extern "C" void zeggs_timing_enable(int on) { zeggs::g_timing = on != 0; }
extern "C" void zeggs_timing_reset(void) {
  std::lock_guard<std::mutex> lk(zeggs::g_tmu);
  for (auto& sp : zeggs::g_spans) { zeggs::g_pool.push_back(sp.e0); zeggs::g_pool.push_back(sp.e1); }
  zeggs::g_spans.clear();
}
// total device milliseconds and launch count of the named span since the last reset (call after a synchronize)
extern "C" int zeggs_timing_read(const char* name, double* total_ms, int* count) {
  int id = zeggs::timer_id(name);
  if (id < 0 || !total_ms || !count) return ZEGGS_ERR_ARG;
  std::lock_guard<std::mutex> lk(zeggs::g_tmu);
  double tot = 0; int n = 0;
  for (auto& sp : zeggs::g_spans) {
    if (sp.name != id) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) { tot += ms; ++n; }
  }
  *total_ms = tot; *count = n;
  return ZEGGS_OK;
}

extern "C" const char* zeggs_last_error(void) { return zeggs::get_error(); }
extern "C" int zeggs_version(void) { return 100; }
extern "C" long long zeggs_launch_count(void) { return zeggs::g_launches.load(); }

// sizeof of every args struct of include/zeggs_b200.h by its C name (0 = unknown): lets a binding in another language check at load
// time that its mirror of the struct has the library's layout (tests/test_abi_cpu.py does so for the ctypes mirrors)
extern "C" size_t zeggs_struct_size(const char* name) {
  if (!name) return 0;
#define ZS(T) if (!strcmp(name, #T)) return sizeof(T);
  ZS(zeggs_ctx) ZS(zeggs_mel_args) ZS(zeggs_loudness_args) ZS(zeggs_decoder_fwd_args) ZS(zeggs_decoder_bwd_args) ZS(zeggs_speech_enc_args)
  ZS(zeggs_speech_enc_grads) ZS(zeggs_style_enc_args) ZS(zeggs_style_enc_grads) ZS(zeggs_decoder_step_args) ZS(zeggs_loss_args)
  ZS(zeggs_pose_post_args) ZS(zeggs_gather_args) ZS(zeggs_decoder_state_args)
#undef ZS
  return 0;
}
