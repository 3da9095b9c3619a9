// api.cu -- library-level entry points: version, last error, launch counter.
#include "common.cuh"
#include <atomic>

namespace y2 {
static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

static EnvSwitches g_env;
static std::atomic<int> g_env_state{0};     // 0 = not read, 1 = being read, 2 = ready

static void env_read() {
  auto on = [](const char* k) { return getenv(k) != nullptr; };
  EnvSwitches e;
  e.bn_bwd_generic = on("Y2_BN_BWD_GENERIC");
  e.affine_generic = on("Y2_AFFINE_GENERIC");
  e.no_pdl = on("Y2_NO_PDL");
  e.conv_no_streamk = on("Y2_CONV_NO_STREAMK");
  e.conv_force_streamk = on("Y2_CONV_FORCE_STREAMK");
  e.conv_force_tiled = on("Y2_CONV_FORCE_TILED");
  e.conv_no_cta2 = on("Y2_CONV_NO_CTA2");
  e.conv_no_is = on("Y2_CONV_NO_IS");
  e.conv_force_is = on("Y2_CONV_FORCE_IS");
  e.conv_no_tma_store_f32 = on("Y2_CONV_NO_TMA_STORE_F32");
  g_env = e;
}

const EnvSwitches& env() {
  int st = g_env_state.load(std::memory_order_acquire);
  if (st != 2) {
    int expect = 0;
    if (g_env_state.compare_exchange_strong(expect, 1, std::memory_order_acq_rel)) {
      env_read();
      g_env_state.store(2, std::memory_order_release);
    } else {
      while (g_env_state.load(std::memory_order_acquire) != 2) {}
    }
  }
  return g_env;
}
}  // namespace y2

extern "C" {
int y2_version(void) { return 101; }
const char* y2_last_error(void) { return y2::g_err; }
unsigned long long y2_launch_count(void) { return y2::g_launches.load(std::memory_order_relaxed); }
int y2_reload_env(void) {
  y2::env_read();
  y2::g_env_state.store(2, std::memory_order_release);
  return Y2_OK;
}
}
