// CPython 2.7 behaviours behind the reference's down-sampling (smCounter.py:496-500)
//     random.seed(pos); bcKeys = random.sample(bcDict.keys(), ds)
// restated for the device and the host alike: the 64-bit string hash, the iteration order of a dict whose keys were inserted
// in first-seen order, MT19937 seeded with init_by_array, and random.sample.  smcounter_b200/downsample.py is the reference
// this header follows step for step; tests/test_py2rand_host.py compiles it with g++ and compares the two.
//
// Everything is plain integer arithmetic except one IEEE multiply per draw (int(random() * m)), which must not be fused:
// the device build uses -fmad=false and __dmul_rn, the host harness -ffp-contract=off.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define HD __host__ __device__ __forceinline__
#else
#define HD inline
#endif

// ---- hash(str) of a 64-bit CPython 2.7 build (Objects/stringobject.c: string_hash) ----------------------------------------
struct Py2Hash {
    uint64_t x = 0; int64_t len = 0;
    HD void add(uint8_t c) {
        if (len == 0) x = (uint64_t)c << 7;
        x = (1000003ull * x) ^ c;
        ++len;
    }
    HD int64_t value() const {
        if (len == 0) return 0;
        const int64_t h = (int64_t)(x ^ (uint64_t)len);
        return h == -1 ? -2 : h;
    }
};

// hash of the barcode string of a 2-bit code (soa.umi_code: A0 C1 G2 T3 behind a length sentinel; code 1 = the empty barcode).
// Dictionary-coded barcodes (top bit set) have no string here: their hash comes from the caller.
HD int64_t py2_hash_umi2(uint64_t code) {
    int top = 63;
    while (top > 0 && !((code >> top) & 1ull)) --top;          // the sentinel bit
    Py2Hash h;
    for (int b = top - 2; b >= 0; b -= 2) h.add((uint8_t)"ACGT"[(code >> b) & 3ull]);
    return h.value();
}

// hash of str(v) for v >= 0 (random.seed(pos) with pos the 1-based position as a string)
HD int64_t py2_hash_decimal(int64_t v) {
    char d[20]; int n = 0;
    do { d[n++] = (char)('0' + v % 10); v /= 10; } while (v > 0);
    Py2Hash h;
    while (n > 0) h.add((uint8_t)d[--n]);
    return h.value();
}

// ---- MT19937 (Modules/_randommodule.c) ---------------------------------------------------------------------------------
#define PY2_MT_N 624
#define PY2_MT_M 397
struct Py2MT {
    uint32_t* mt;                // PY2_MT_N words
    int mti;
    HD void init_genrand(uint32_t s) {
        mt[0] = s;
        for (mti = 1; mti < PY2_MT_N; ++mti) mt[mti] = 1812433253u * (mt[mti - 1] ^ (mt[mti - 1] >> 30)) + (uint32_t)mti;
    }
    HD void init_by_array(const uint32_t* key, int len) {
        init_genrand(19650218u);
        int i = 1, j = 0;
        for (int k = PY2_MT_N > len ? PY2_MT_N : len; k; --k) {
            mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1664525u)) + key[j] + (uint32_t)j;
            ++i; ++j;
            if (i >= PY2_MT_N) { mt[0] = mt[PY2_MT_N - 1]; i = 1; }
            if (j >= len) j = 0;
        }
        for (int k = PY2_MT_N - 1; k; --k) {
            mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
            ++i;
            if (i >= PY2_MT_N) { mt[0] = mt[PY2_MT_N - 1]; i = 1; }
        }
        mt[0] = 0x80000000u;
        mti = PY2_MT_N;
    }
    // random.seed(s) for a string s: init_by_array over the 32-bit words of (unsigned 64-bit) hash(s), at least one word
    HD void seed(int64_t hash) {
        const uint64_t u = (uint64_t)hash;
        const uint32_t key[2] = {(uint32_t)u, (uint32_t)(u >> 32)};
        init_by_array(key, (u >> 32) ? 2 : 1);
    }
    HD uint32_t genrand_int32() {
        if (mti >= PY2_MT_N) {
            const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, A = 0x9908b0dfu;
            int kk = 0;
            for (; kk < PY2_MT_N - PY2_MT_M; ++kk) {
                const uint32_t y = (mt[kk] & UP) | (mt[kk + 1] & LO);
                mt[kk] = mt[kk + PY2_MT_M] ^ (y >> 1) ^ ((y & 1u) ? A : 0u);
            }
            for (; kk < PY2_MT_N - 1; ++kk) {
                const uint32_t y = (mt[kk] & UP) | (mt[kk + 1] & LO);
                mt[kk] = mt[kk + (PY2_MT_M - PY2_MT_N)] ^ (y >> 1) ^ ((y & 1u) ? A : 0u);
            }
            const uint32_t y = (mt[PY2_MT_N - 1] & UP) | (mt[0] & LO);
            mt[PY2_MT_N - 1] = mt[PY2_MT_M - 1] ^ (y >> 1) ^ ((y & 1u) ? A : 0u);
            mti = 0;
        }
        uint32_t y = mt[mti++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    }
    // random.random() = genrand_res53: an exact multiple of 2^-53
    HD double random() {
        const uint32_t a = genrand_int32() >> 5, b = genrand_int32() >> 6;
        return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
    }
    // int(random() * m): one rounded multiply, truncated
    HD int64_t below(int64_t m) {
#ifdef __CUDA_ARCH__
        return (int64_t)__dmul_rn(random(), (double)m);
#else
        return (int64_t)(random() * (double)m);
#endif
    }
};

// ---- random.sample (Lib/random.py) ---------------------------------------------------------------------------------------
// setsize = 21, plus 4 ** ceil(log(3k, 4)) when k > 5: the smallest power of four >= 3k (3k is never a power of four)
HD int64_t py2_sample_setsize(int64_t k) {
    int64_t s = 21;
    if (k > 5) {
        int64_t p = 1;
        while (p < 3 * k) p *= 4;
        s += p;
    }
    return s;
}

// ---- dict iteration order (Objects/dictobject.c) -------------------------------------------------------------------------
// Words of scratch one draw over n keys needs: two tables of up to 8 * max(n, 1) slots (a table grows to the first power of
// two above 4 * used <= 8 * n, and the one it grows from is at most half of it), then the MT19937 state.
HD int64_t py2_scratch_words(int64_t n) { return 16 * (n + 1) + PY2_MT_N + 16; }

// one insertion with perturbed probing; a slot holds key index + 1 (0 = empty)
HD void py2_dict_insert(uint32_t* tab, uint64_t mask, uint32_t key, int64_t h) {
    uint64_t i = (uint64_t)h & mask, perturb = (uint64_t)h;
    while (tab[i] != 0) {
        i = (5ull * i + perturb + 1ull) & mask;
        perturb >>= 5;
    }
    tab[i] = key + 1u;
}

// Keys 0 .. n-1 with hashes hash[0 .. n), inserted in that order into a CPython 2.7 dict.  Returns the keys in iteration
// (slot) order, n words compacted in place at the start of whichever half of scratch (16 * (n + 1) words) held the final table.
HD uint32_t* py2_dict_order(const int64_t* hash, int64_t n, uint32_t* scratch) {
    uint32_t* t0 = scratch;
    uint32_t* t1 = scratch + 8 * (n + 1);
    uint64_t size = 8;
    for (int k = 0; k < 8; ++k) t0[k] = 0;
    int64_t used = 0;
    for (int64_t key = 0; key < n; ++key) {
        py2_dict_insert(t0, size - 1, (uint32_t)key, hash[key]);
        ++used;
        if ((uint64_t)used * 3 >= size * 2) {                                   // dictresize(mp, (used > 50000 ? 2 : 4) * used)
            const uint64_t minused = (uint64_t)(used > 50000 ? 2 : 4) * (uint64_t)used;
            uint64_t nsize = 8;
            while (nsize <= minused) nsize <<= 1;
            for (uint64_t s = 0; s < nsize; ++s) t1[s] = 0;
            for (uint64_t s = 0; s < size; ++s)                                 // the old table, in its slot order
                if (t0[s]) py2_dict_insert(t1, nsize - 1, t0[s] - 1u, hash[t0[s] - 1u]);
            uint32_t* t = t0; t0 = t1; t1 = t;
            size = nsize;
        }
    }
    int64_t o = 0;
    for (uint64_t s = 0; s < size; ++s)                                         // o <= s: compaction in place
        if (t0[s]) t0[o++] = t0[s] - 1u;
    return t0;
}

// random.seed(str(pos1)); random.sample(keys in dict order, k) over n keys of the given hashes (0 <= k <= n): out[j] is the
// insertion index of the j-th drawn key.  scratch: py2_scratch_words(n) words.
HD void py2_draw(const int64_t* hash, int64_t n, int64_t pos1, int64_t k, uint32_t* scratch, uint32_t* out) {
    const uint32_t* pop = py2_dict_order(hash, n, scratch);
    uint32_t* work = pop == scratch ? scratch + 8 * (n + 1) : scratch;     // the other half: the pool or the selection bitmap
    Py2MT rng;
    rng.mt = scratch + 16 * (n + 1);
    rng.seed(py2_hash_decimal(pos1));
    if (n <= py2_sample_setsize(k)) {
        uint32_t* pool = work;
        for (int64_t i = 0; i < n; ++i) pool[i] = pop[i];
        for (int64_t i = 0; i < k; ++i) {
            const int64_t j = rng.below(n - i);
            out[i] = pool[j];
            pool[j] = pool[n - i - 1];
        }
    } else {
        uint32_t* selected = work;
        for (int64_t w = 0; w < (n + 31) / 32; ++w) selected[w] = 0;
        for (int64_t i = 0; i < k; ++i) {
            int64_t j = rng.below(n);
            while ((selected[j >> 5] >> (j & 31)) & 1u) j = rng.below(n);
            selected[j >> 5] |= 1u << (j & 31);
            out[i] = pop[j];
        }
    }
}
