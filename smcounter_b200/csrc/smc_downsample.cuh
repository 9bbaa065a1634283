// Device draw of the reference's down-sampling (smCounter.py:486-500) for the loci k_call flagged SMC_ST_NEED_DOWNSAMPLE:
// list their barcodes (the listing pass of the pileup pair), put each locus's barcodes in bcDict insertion order (first
// passing read), hash them, and run random.seed(pos); random.sample(bcDict.keys(), ds) over CPython-2 dict order
// (smc_py2rand.h) -- one thread per locus, the loci in parallel.  The kept codes become the mask CSR k_merge applies.
#pragma once
#include "smc_common.cuh"
#include "smc_py2rand.h"

// flagged loci: 1 / their barcode count, for the two scans that number them and place their barcodes
__global__ void k_ds_flags(const int32_t* __restrict__ loc, int64_t nl, uint32_t* __restrict__ flag, uint32_t* __restrict__ nbc) {
    const int64_t L = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (L >= nl) return;
    const bool f = (uint32_t)loc[SMC_L_STATUS * nl + L] & SMC_ST_NEED_DOWNSAMPLE;
    flag[L] = f ? 1u : 0u;
    nbc[L] = f ? (uint32_t)loc[SMC_L_NBC * nl + L] : 0u;
}

// list_idx[L]: ordinal of a flagged locus (-1 otherwise); list_off[k]: its first listed barcode; locus[k]: the locus
__global__ void k_ds_list_fill(const uint32_t* __restrict__ flag, const uint32_t* __restrict__ ord, const uint32_t* __restrict__ off32,
                               int64_t nl, int64_t nflag, int64_t total, int32_t* __restrict__ list_idx, int64_t* __restrict__ list_off,
                               int32_t* __restrict__ locus) {
    const int64_t L = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (L == 0) list_off[nflag] = total;
    if (L >= nl) return;
    if (!flag[L]) { list_idx[L] = -1; return; }
    const uint32_t k = ord[L];
    list_idx[L] = (int32_t)k;
    list_off[k] = off32[L];
    locus[k] = (int32_t)L;
}

// the set of listed entry j: last k with off[k] <= j
__device__ __forceinline__ uint32_t ds_set_of(const int64_t* off, int64_t nsets, int64_t j) {
    int64_t lo = 0, hi = nsets;                      // off[lo] <= j < off[hi]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (off[mid] <= j) lo = mid; else hi = mid;
    }
    return (uint32_t)lo;
}

// sort key of a listed barcode: (locus ordinal, first passing read) -- the order of bcDict's insertions at the locus
__global__ void k_ds_sort_keys(const int64_t* __restrict__ off, int64_t nflag, const uint32_t* __restrict__ first, int64_t total,
                               uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= total) return;
    key[j] = ((uint64_t)ds_set_of(off, nflag, j) << 30) | first[j];
    val[j] = (uint32_t)j;
}

// Hash of every barcode (entry order[p] of umi[], or entry p when order is null): 2-bit codes from their bases, dictionary codes
// (top bit) from the caller's table (ascending codes).  A dictionary code without a hash goes to *missing; the OR of all codes
// to *code_or (it bounds the key bits of the sort of the kept codes).
__global__ void k_ds_hash(const uint32_t* __restrict__ order, const uint64_t* __restrict__ umi, int64_t total, const uint64_t* __restrict__ bc_code,
                          const int64_t* __restrict__ bc_hash, int64_t n_bc, uint64_t* __restrict__ code_out, int64_t* __restrict__ hash_out,
                          unsigned long long* missing, unsigned long long* code_or) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t c = p < total ? umi[order ? order[p] : p] : 0ull;
    const unsigned hi = __reduce_or_sync(FULL_MASK, (unsigned)(c >> 32)), lo = __reduce_or_sync(FULL_MASK, (unsigned)c);
    if ((threadIdx.x & 31) == 0 && (hi | lo)) atomicOr(code_or, ((unsigned long long)hi << 32) | lo);
    if (p >= total) return;
    int64_t h = 0;
    if (c >> 63) {
        const int64_t i = n_bc > 0 ? lower_bound_u64(bc_code, n_bc, c) : 0;
        if (i < n_bc && bc_code[i] == c) h = bc_hash[i];
        else atomicExch(missing, (unsigned long long)c);
    } else {
        h = py2_hash_umi2(c);
    }
    code_out[p] = c;
    hash_out[p] = h;
}

// words of draw scratch before set k: py2_scratch_words of every earlier set
__device__ __forceinline__ int64_t ds_scratch_at(const int64_t* off, int64_t k) {
    return 16 * (off[k] + k) + (PY2_MT_N + 16) * k;
}

// One thread per set k in [k0, k1): random.seed(str(pos1)); random.sample(keys in dict order, k) over the set's hashes
// hash[off[k] .. off[k+1]).  The insertion indices of the drawn keys go to out[off[k] ..] when kk (per-set sample sizes)
// is given, else to out[k * ds ..].  pos1: given per set, or loci_pos[locus[k]] + 1.
__global__ void k_ds_draw(const int64_t* __restrict__ off, int64_t k0, int64_t k1, const int64_t* __restrict__ pos1,
                          const int32_t* __restrict__ locus, const int32_t* __restrict__ loci_pos, const int64_t* __restrict__ kk, int64_t ds,
                          const int64_t* __restrict__ hash, uint32_t* __restrict__ scratch, uint32_t* __restrict__ out) {
    const int64_t k = k0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= k1) return;
    const int64_t a = off[k], n = off[k + 1] - a;
    const int64_t p = pos1 ? pos1[k] : (int64_t)loci_pos[locus[k]] + 1;
    py2_draw(hash + a, n, p, kk ? kk[k] : ds, scratch + (ds_scratch_at(off, k) - ds_scratch_at(off, k0)),
             out + (kk ? a : k * ds));
}

// kept entry q (of locus q / ds): insertion index -> its code, payload q
__global__ void k_ds_kept(const int64_t* __restrict__ off, int64_t m, int64_t ds, const uint64_t* __restrict__ codes,
                          uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    key[q] = codes[off[q / ds] + val[q]];
    val[q] = (uint32_t)q;
}

// after the sort on code: keep the sorted codes, and key every entry by its locus for the stable sort that groups them again
__global__ void k_ds_group_keys(int64_t m, int64_t ds, uint64_t* __restrict__ key, uint32_t* __restrict__ val, uint64_t* __restrict__ code_sorted) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    code_sorted[p] = key[p];
    key[p] = (uint64_t)(val[p] / ds);
    val[p] = (uint32_t)p;
}

// The mask CSR: the caller's masks (already in place) and then ds codes per drawn locus, ascending
__global__ void k_ds_csr(int64_t nflag, int64_t ds, int64_t n_caller, int64_t caller_total, const int32_t* __restrict__ locus,
                         const uint32_t* __restrict__ order, const uint64_t* __restrict__ code_sorted, int32_t* __restrict__ keep_idx,
                         int64_t* __restrict__ keep_off, uint64_t* __restrict__ keep_umi) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= nflag) keep_off[n_caller + t] = caller_total + t * ds;
    if (t < nflag) keep_idx[locus[t]] = (int32_t)(n_caller + t);
    if (t < nflag * ds) keep_umi[caller_total + t] = code_sorted[order[t]];
}
