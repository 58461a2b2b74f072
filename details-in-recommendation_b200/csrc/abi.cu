// Library-wide state of libdir_b200.so: version, thread-local error text, launch counter.
#include "common.cuh"

namespace dir {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
}  // namespace dir

extern "C" int dir_version(void) { return 100; }  // 0.1.0
extern "C" const char* dir_last_error(void) { return dir::g_err; }
extern "C" uint64_t dir_launch_count(void) { return dir::g_launches.load(std::memory_order_relaxed); }
