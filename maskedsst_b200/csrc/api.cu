// Error channel + version of the C ABI (include/msst.h).
#include "common.cuh"
#include <stdarg.h>
#include <atomic>

namespace msst {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace msst

extern "C" const char* msst_last_error(void) { return msst::g_err; }
extern "C" int msst_version(void) { return 102; }
extern "C" long long msst_launch_count(void) { return msst::g_launches.load(); }
