// smcounter_b200/csrc/smc_py2rand.h compiled for the host (g++), for tests/test_py2rand_host.py to compare with
// smcounter_b200/downsample.py through ctypes.
#include <vector>

#include "smc_py2rand.h"

extern "C" {

int64_t h_hash_umi2(uint64_t code) { return py2_hash_umi2(code); }
int64_t h_hash_decimal(int64_t v) { return py2_hash_decimal(v); }
void h_setsizes(int64_t kmax, int64_t* out) { for (int64_t k = 0; k <= kmax; ++k) out[k] = py2_sample_setsize(k); }

// keys in dict iteration order (insertion indices)
void h_dict_order(const int64_t* hash, int64_t n, uint32_t* out) {
    std::vector<uint32_t> scratch((size_t)py2_scratch_words(n));
    const uint32_t* order = py2_dict_order(hash, n, scratch.data());
    for (int64_t i = 0; i < n; ++i) out[i] = order[i];
}

// the first m values of random() after random.seed(str(pos1))
void h_random(int64_t pos1, int64_t m, double* out) {
    std::vector<uint32_t> state(PY2_MT_N);
    Py2MT rng;
    rng.mt = state.data();
    rng.seed(py2_hash_decimal(pos1));
    for (int64_t i = 0; i < m; ++i) out[i] = rng.random();
}

void h_draw(const int64_t* hash, int64_t n, int64_t pos1, int64_t k, uint32_t* out) {
    std::vector<uint32_t> scratch((size_t)py2_scratch_words(n));
    py2_draw(hash, n, pos1, k, scratch.data(), out);
}

}
