// mpi4jax_b200 -- logging switch, per-call debug timer, last-error string.
//
// Behavioural counterpart of the reference's debug trace
// (mpi4jax/_src/xla_bridge/mpi_ops_common.h:100-206): when logging is enabled
// every native op prints two lines
//     r<rank> | <8-char id> | MPI_<Op> (GPU) <details>
//     r<rank> | <8-char id> | MPI_<Op> (GPU) done with code <rc> (<seconds>s)
// through a callback installed by the Python layer (so pytest's capsys and
// notebook front-ends see them).  The time is the DEVICE time of the op between
// two CUDA events on the launching stream -- the reference can only report the
// host wall time of a blocking MPI call.
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <random>
#include <string>

#include "b2_runtime.h"

static int g_logging = 0;
static b2_print_fn g_print = nullptr;
static thread_local char g_last_error[1024] = "";
static int g_launches = 0;

extern "C" void b2_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof g_last_error, fmt, ap);
  va_end(ap);
}
extern "C" const char* b2_last_error(void) { return g_last_error; }
extern "C" const char* b2_version(void) { return "mpi4jax_b200-native 0.1 (sm_100a)"; }
extern "C" void b2_set_logging(int enable) { g_logging = enable ? 1 : 0; }
extern "C" int b2_get_logging(void) { return g_logging; }
extern "C" void b2_set_print_callback(b2_print_fn fn) { g_print = fn; }
extern "C" int b2_launch_count(void) { return g_launches; }
extern "C" void b2_count_launch(B2Comm* c) {
  ++g_launches;
  if (c) ++c->launches;
}

static void emit(const std::string& line) {
  if (g_print) g_print(line.c_str());
  else { fputs(line.c_str(), stdout); fputc('\n', stdout); fflush(stdout); }
}

static std::string call_id() {
  static const char alphabet[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789";
  static thread_local std::mt19937 rng{std::random_device{}()};
  std::uniform_int_distribution<int> pick(0, (int)sizeof(alphabet) - 2);
  std::string s(8, 'x');
  for (auto& ch : s) ch = alphabet[pick(rng)];
  return s;
}

struct B2DebugScope {
  std::string prefix;     // "r<rank> | <id> | MPI_<Op> (GPU)"
  cudaEvent_t start, stop;
  cudaStream_t stream;
  bool timed;
};

// Logging is a debugging aid: it synchronises the stream in b2_debug_end to read the
// device time, exactly like the reference's blocking calls; disabled -> zero overhead.
extern "C" B2DebugScope* b2_debug_begin(B2Comm* c, const char* opname, const char* details,
                                         cudaStream_t stream) {
  if (!g_logging) return nullptr;
  B2DebugScope* s = new B2DebugScope();
  char buf[256];
  snprintf(buf, sizeof buf, "r%d | %s | MPI_%s (GPU)", c ? c->dev.rank : 0, call_id().c_str(), opname);
  s->prefix = buf;
  s->timed = false;
  s->stream = nullptr;
  emit(s->prefix + (details && details[0] ? std::string(" ") + details : std::string()));
  // events cannot be timed inside a stream capture; log without device time there
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &st) == cudaSuccess && st == cudaStreamCaptureStatusNone &&
      cudaEventCreate(&s->start) == cudaSuccess && cudaEventCreate(&s->stop) == cudaSuccess) {
    s->timed = true;
    s->stream = stream;
    cudaEventRecord(s->start, stream);
  }
  return s;
}

extern "C" void b2_debug_end(B2DebugScope* s, int code) {
  if (!s) return;
  double seconds = 0.0;
  if (s->timed) {
    cudaEventRecord(s->stop, s->stream);
    if (cudaEventSynchronize(s->stop) == cudaSuccess) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, s->start, s->stop) == cudaSuccess) seconds = ms * 1e-3;
    }
  }
  if (s->timed) { cudaEventDestroy(s->start); cudaEventDestroy(s->stop); }
  char buf[128];
  snprintf(buf, sizeof buf, " done with code %d (%.2es)", code, seconds);
  emit(s->prefix + buf);
  delete s;
}
