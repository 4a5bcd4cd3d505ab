// Error reporting, version and launch accounting for libgnnml3_b200.so.
#include "common.cuh"

#include <atomic>

namespace gnnml3 {

static thread_local char g_err[768] = "";
std::atomic<int64_t> g_launches{0};

char* err_buf() { return g_err; }

int set_err(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

std::mutex& config_mutex() {
    static std::mutex m;
    return m;
}

}  // namespace gnnml3

extern "C" {

const char* gnnml3_last_error(void) { return gnnml3::err_buf(); }
int gnnml3_version(void) { return 101; }
int64_t gnnml3_launch_count(void) { return gnnml3::g_launches.load(); }
}
