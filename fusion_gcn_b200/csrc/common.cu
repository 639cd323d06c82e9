// Error state and version of libagcn_b200.so.
#include "common.cuh"
#include <string.h>
#include <atomic>

namespace agcn {

long long launches();

char* error_buffer() {
    static thread_local char buf[512] = "";
    return buf;
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launches() { return g_launches.load(std::memory_order_relaxed); }

}  // namespace agcn

extern "C" AGCN_API int agcn_version(void) { return 101; }

extern "C" AGCN_API const char* agcn_last_error_string(void) { return agcn::error_buffer(); }

extern "C" AGCN_API long long agcn_launch_count(void) { return agcn::launches(); }
