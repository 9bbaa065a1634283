// Common device/host helpers for libsmc_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/smc_b200.h"

#define SMC_WARP 32
#define FULL_MASK 0xffffffffu

// ----------------------------------------------------------------------------------------------------------
// Internal per-read record, built once per read by k_read_prep (the reference recomputes all of this for every
// pileup event, smCounter.py:327-365).  64 bytes = 4 x uint4, stored in "srank" order: reads sorted by
// (umi, frag_id, BAM index), so that every 32-locus tile sees barcodes and fragments as contiguous runs.
// ----------------------------------------------------------------------------------------------------------
struct __align__(16) ReadRec {
    // word 0-3: everything the gather pass needs first
    int32_t  lo;         // covered target loci: indices [lo, hi) into the sorted locus list
    uint32_t gspan;      // simple reads: hi - lo; other reads: 0 (the gather pass never covers them)
    uint32_t sp_aln;     // simple reads: qk = leftSP - start (query position of locus position p is p + qk);
                         // other reads: leftSP (low 16) | query_alignment_length (high 16)
    uint32_t meta;       // bit0 passes MQ+mismatch gate, bit1 reverse, bit2 read2, bit3 single ref-consuming M run; bits 8.. n_cigar
    // word 4-7
    uint32_t seq_off;    // byte offset into seq[]
    uint32_t qual_off;   // byte offset into qual[]
    int32_t  start;      // 0-based leftmost reference position
    int32_t  hi;
    // word 8-11
    uint32_t urank;      // dense rank of the barcode
    uint32_t frank;      // dense rank of the fragment
    uint32_t read_idx;   // index of the read in the caller's SoA (BAM order)
    uint32_t cigar_off;  // word offset into cigar[]
    // word 12-15
    uint32_t cig[4];     // simple reads: {le_lo, le_span, ple_lo, ple_span}: a base at position p is within 20 of the barcode end
                         // iff (uint32)(p - le_lo) <= le_span, within primerDist of the R2 primer end iff (uint32)(p - ple_lo) <= ple_span
                         // (smCounter.py:432-452); other reads: the first four CIGAR words (the rest is read from cigar[])
};
static_assert(sizeof(ReadRec) == 64, "ReadRec must be 64 bytes");

// prediction-index accumulators: fixed point, LSB 2^-PI_FIX_LSB (k_merge adds, k_call rounds once)
#define PI_FIX_LSB 80

#define RM_OK      1u
#define RM_REVERSE 2u
#define RM_READ2   4u
#define RM_SIMPLE  8u

// dynamic-allele table key: locus(22) | kind(2) | site(4) | payload(36)
#define DYN_EMPTY 0xffffffffffffffffull
#define DYN_LOCUS_SHIFT 42
#define SMC_MAX_LOCI 4194302ll

__host__ __device__ inline uint64_t dyn_make_key(uint32_t locus, uint32_t kind, uint32_t site, uint64_t payload) {
    return ((uint64_t)locus << DYN_LOCUS_SHIFT) | ((uint64_t)kind << 40) | ((uint64_t)site << 36) | (payload & 0xFFFFFFFFFull);
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// Built with -DSMC_BOUNDS_ASSERT (SMC_NVCC_EXTRA): device asserts on the positions the read-sort kernels compute from the
// fragment tables, which the index checks of a normal build take on trust.
#ifdef SMC_BOUNDS_ASSERT
#include <cassert>
#define SMC_BOUNDS(cond) assert(cond)
#else
#define SMC_BOUNDS(cond) ((void)0)
#endif

__device__ __forceinline__ uint32_t hash64to32(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return (uint32_t)x;
}

// lower_bound on a sorted u64 array
__device__ __forceinline__ int64_t lower_bound_u64(const uint64_t* __restrict__ a, int64_t n, uint64_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ int64_t lower_bound_u32(const uint32_t* __restrict__ a, int64_t n, uint32_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// largest i in [0,n) with a[i] <= key (a ascending, a[0] <= key assumed)
__device__ __forceinline__ int64_t upper_slot_u32(const uint32_t* __restrict__ a, int64_t n, uint32_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (a[mid] <= key) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}
