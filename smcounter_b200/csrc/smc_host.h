// smc_host.h -- helpers shared by the host sources of libsmc_bamio.so (smc_bamio.cpp, smc_soa.cpp, smc_rows.cpp): thread
// fan-out and a per-phase wall clock.  The helpers run work; every call site decides how many threads its work is worth.
#pragma once

#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

namespace smc_host {

// the thread count a caller asked for, or one per hardware thread when it asked for 0 or less; at least 1
inline int n_threads(int want) { return want > 0 ? want : (int)std::max(1u, std::thread::hardware_concurrency()); }

// f(t) for every t < T, each on a thread of its own; the calling thread runs f(0)
template <class F> void for_each_thread(int T, F&& f) {
    std::vector<std::thread> ts;
    for (int t = 1; t < T; ++t) ts.emplace_back([&f, t] { f(t); });
    if (T > 0) f(0);
    for (auto& th : ts) th.join();
}

// f(begin, end, t) over T contiguous ranges of [0, n), range t = [n t / T, n (t + 1) / T); the calling thread takes range 0
template <class F> void for_ranges(size_t n, int T, F&& f) {
    for_each_thread(T, [&](int t) { f(n * (size_t)t / (size_t)T, n * (size_t)(t + 1) / (size_t)T, t); });
}

// with the environment variable `env` set: lap(what) prints "[tag] what  <ms since the previous lap>" on stderr (a tuning aid)
class PhaseTimer {
  public:
    PhaseTimer(const char* env, const char* tag) : on_(getenv(env) != nullptr), tag_(tag), t0_(std::chrono::steady_clock::now()) {}
    void lap(const char* what) {
        if (!on_) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[%s] %-28s %8.2f ms\n", tag_, what, std::chrono::duration<double, std::milli>(t1 - t0_).count());
        t0_ = t1;
    }

  private:
    bool on_;
    const char* tag_;
    std::chrono::steady_clock::time_point t0_;
};

}  // namespace smc_host
