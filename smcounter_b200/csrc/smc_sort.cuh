// Hand-written device-wide exclusive scan and stable LSD radix sort (u32 or u64 key, u32 payload).
//
// K2 of the pipeline ("segmented radix sort"): fragment ids are ordered by barcode slot (u32 key) and the (read x 32-locus
// tile) events by tile (u64 key), so that every tile's events form one segment in which barcodes and fragments are
// contiguous runs in BAM order.  Both sorts are LSD passes over exactly the key bits in use, with a digit width of 8-11 bits
// chosen per sort.  Each pass reads and writes key + payload once per element (the working sets of a panel batch fit the
// 126 MB L2); histogram, scan and scatter are separate kernels.
#pragma once
#include "smc_common.cuh"

// ---------------------------------------------------------------- scan -------------------------------------
#define SCAN_THREADS 256
#define SCAN_ITEMS   8
#define SCAN_TILE    (SCAN_THREADS * SCAN_ITEMS)

// Exclusive scan of one tile per block; block totals to sums[blockIdx.x].
__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_tile(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* sums) {   // in == out allowed
    __shared__ uint32_t warp_tot[SCAN_THREADS / 32];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t tsum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0u;
        tsum += v[i];
    }
    uint32_t incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(FULL_MASK, incl, d);
        if (lane_id() >= (uint32_t)d) incl += t;
    }
    int w = threadIdx.x >> 5;
    if (lane_id() == 31) warp_tot[w] = incl;
    __syncthreads();
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (int i = 0; i < SCAN_THREADS / 32; ++i) {
        uint32_t t = warp_tot[i];
        if (i < w) woff += t;
        total += t;
    }
    uint32_t run = woff + incl - tsum;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
    }
    if (threadIdx.x == 0 && sums) sums[blockIdx.x] = total;
}

// Single-pass scan (decoupled look-back): tiles take their number from an atomic counter (so a tile only ever waits for tiles
// that already run), publish their aggregate, and thread 0 walks back over the descriptors of the preceding tiles until it
// meets an inclusive prefix.  One launch instead of three (tile scan, scan of the tile sums, add).
// Descriptor: bits 62-63 status (0 empty, 1 aggregate, 2 inclusive prefix), low bits the value.
#define LB_AGG  (1ull << 62)
#define LB_INCL (2ull << 62)
#define LB_VAL  ((1ull << 62) - 1ull)

__device__ __forceinline__ unsigned long long lb_resolve(unsigned long long* desc, uint32_t tile, unsigned long long agg) {
    // called by ALL 32 lanes of one warp of the tile (converged); returns the exclusive prefix of the tile (same value in every lane)
    // and publishes its inclusive prefix.  The warp looks back 32 descriptors at a time: lane k reads tile - 1 - k (- 32 per round).
    const uint32_t lane = lane_id();
    unsigned long long prefix = 0;
    if (tile > 0) {
        if (lane == 0) atomicExch(&desc[tile], LB_AGG | agg);
        int64_t t0 = (int64_t)tile - 1;
        for (;;) {
            const int64_t t = t0 - lane;
            unsigned long long d = LB_INCL;                                  // before tile 0: an inclusive prefix of 0
            if (t >= 0) { do { d = *reinterpret_cast<volatile unsigned long long*>(&desc[t]); } while ((d >> 62) == 0ull); }
            const uint32_t incl = __ballot_sync(FULL_MASK, (d >> 62) == 2ull);
            const int stop = incl ? __ffs((int)incl) - 1 : 31;               // nearest descriptor that already holds a prefix
            unsigned long long v = (int)lane <= stop ? (d & LB_VAL) : 0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
            prefix += v;
            if (incl) break;
            t0 -= 32;
        }
    }
    if (lane == 0) atomicExch(&desc[tile], LB_INCL | (prefix + agg));
    return prefix;
}

__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_lb(const uint32_t* in, uint32_t* out, int64_t n, unsigned long long* desc, uint32_t* counter, uint32_t* total) {   // in == out allowed
    __shared__ uint32_t warp_tot[SCAN_THREADS / 32];
    __shared__ uint32_t s_tile, s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(counter, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t base = (int64_t)tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t tsum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0u;
        tsum += v[i];
    }
    uint32_t incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(FULL_MASK, incl, d);
        if (lane_id() >= (uint32_t)d) incl += t;
    }
    const int w = threadIdx.x >> 5;
    if (lane_id() == 31) warp_tot[w] = incl;
    __syncthreads();
    uint32_t woff = 0, blk = 0;
#pragma unroll
    for (int i = 0; i < SCAN_THREADS / 32; ++i) {
        uint32_t t = warp_tot[i];
        if (i < w) woff += t;
        blk += t;
    }
    if (threadIdx.x < 32) {
        const uint32_t prefix = (uint32_t)lb_resolve(desc, tile, blk);
        if (threadIdx.x == 0) {
            s_prefix = prefix;
            if (total && tile == gridDim.x - 1) *total = prefix + blk;
        }
    }
    __syncthreads();
    uint32_t run = s_prefix + woff + incl - tsum;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
    }
}

// scratch must hold at least scan_scratch_words(n) uint32 (look-back descriptors + the tile counter).  If total != nullptr the
// grand total is stored there.
static inline int64_t scan_scratch_words(int64_t n) {
    return 2 * ((n + SCAN_TILE - 1) / SCAN_TILE) + 8;
}

static thread_local int g_launches = 0;   // kernel launch counter of the calling host thread (one thread drives one context)

static void exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* scratch, uint32_t* total,
                               cudaStream_t st) {
    if (n <= 0) {
        if (total) cudaMemsetAsync(total, 0, sizeof(uint32_t), st);
        return;
    }
    const int64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (nb == 1) {
        k_scan_tile<<<1, SCAN_THREADS, 0, st>>>(in, out, n, total);
        ++g_launches;
        return;
    }
    cudaMemsetAsync(scratch, 0, (size_t)(2 * nb + 8) * 4, st);          // [0, 1] tile counter, descriptors from word 2 (8-byte aligned)
    k_scan_lb<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, out, n, reinterpret_cast<unsigned long long*>(scratch + 2), scratch, total);
    ++g_launches;
}

// ---------------------------------------------------------------- radix sort --------------------------------
// LSD passes over a bit field of the key: digit = (key >> shift) & (2^BITS - 1), BITS = 8 ... 11 chosen per sort so that
// the varying bits are covered in as few passes as possible (e.g. a 9-bit tile index is ONE pass, a 22-bit barcode slot two
// 11-bit passes).
#define RS_WARPS   8
#define RS_THREADS (RS_WARPS * 32)
#define RS_ITEMS   8
#define RS_TILE    (RS_THREADS * RS_ITEMS)
#define RS_MAX_BITS 11

// Element order inside a tile: warp w owns [w*256, w*256+256), iteration it covers 32 consecutive elements.
__device__ __forceinline__ int64_t rs_index(int64_t tile_base, int w, int it, int lane) {
    return tile_base + (int64_t)w * (32 * RS_ITEMS) + it * 32 + lane;
}

template <int BITS, class K>
__global__ void __launch_bounds__(RS_THREADS)
k_radix_hist(const K* __restrict__ keys, int64_t n, int shift, uint32_t* __restrict__ hist, uint32_t nblocks) {
    constexpr uint32_t ND = 1u << BITS;
    __shared__ uint32_t h[ND];
    for (uint32_t d = threadIdx.x; d < ND; d += RS_THREADS) h[d] = 0;
    __syncthreads();
    int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t tb = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll
    for (int it = 0; it < RS_ITEMS; ++it) {
        int64_t i = rs_index(tb, w, it, lane);
        if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & (ND - 1u)], 1u);
    }
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < ND; d += RS_THREADS) hist[(size_t)d * nblocks + blockIdx.x] = h[d];
}

template <int BITS, class K>
__global__ void __launch_bounds__(RS_THREADS)
k_radix_scatter(const K* __restrict__ keys, const uint32_t* __restrict__ vals, K* __restrict__ keys_out,
                uint32_t* __restrict__ vals_out, int64_t n, int shift, const uint32_t* __restrict__ hist_scanned,
                uint32_t nblocks) {
    constexpr uint32_t ND = 1u << BITS;
    extern __shared__ uint32_t wh_s[];                  // [RS_WARPS][ND]
    int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (uint32_t i = threadIdx.x; i < RS_WARPS * ND; i += RS_THREADS) wh_s[i] = 0;
    __syncthreads();
    uint32_t* wh = wh_s + (size_t)w * ND;
    int64_t tb = (int64_t)blockIdx.x * RS_TILE;
    K k[RS_ITEMS];
    uint32_t v[RS_ITEMS];
#pragma unroll
    for (int it = 0; it < RS_ITEMS; ++it) {
        int64_t i = rs_index(tb, w, it, lane);
        if (i < n) {
            k[it] = keys[i];
            v[it] = vals[i];
            atomicAdd(&wh[(uint32_t)(k[it] >> shift) & (ND - 1u)], 1u);
        }
    }
    __syncthreads();
    // per digit: global base of this block, then exclusive prefix over the warps
    for (uint32_t d = threadIdx.x; d < ND; d += RS_THREADS) {
        uint32_t run = hist_scanned[(size_t)d * nblocks + blockIdx.x];
#pragma unroll
        for (int ww = 0; ww < RS_WARPS; ++ww) {
            uint32_t t = wh_s[(size_t)ww * ND + d];
            wh_s[(size_t)ww * ND + d] = run;
            run += t;
        }
    }
    __syncthreads();
    uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int it = 0; it < RS_ITEMS; ++it) {
        int64_t i = rs_index(tb, w, it, lane);
        bool valid = i < n;
        uint32_t active = __ballot_sync(FULL_MASK, valid);
        if (valid) {
            uint32_t d = (uint32_t)(k[it] >> shift) & (ND - 1u);
            uint32_t peers = __match_any_sync(active, d);
            uint32_t rank = __popc(peers & lt);
            int leader = __ffs(peers) - 1;
            uint32_t off = 0;
            if (lane == leader) {
                off = wh[d];
                wh[d] = off + __popc(peers);
            }
            off = __shfl_sync(peers, off, leader);
            keys_out[off + rank] = k[it];
            vals_out[off + rank] = v[it];
        }
        __syncwarp();
    }
}

// scratch sizes of a sort of n elements (any digit width up to RS_MAX_BITS)
static inline size_t radix_hist_words(int64_t n) { return ((size_t)1 << RS_MAX_BITS) * (size_t)((n + RS_TILE - 1) / RS_TILE) + 256; }
static inline int64_t radix_scan_words(int64_t n) { return scan_scratch_words((int64_t)radix_hist_words(n)); }

template <int BITS, class K>
static void radix_pass(const K* ki, const uint32_t* vi, K* ko, uint32_t* vo, int64_t n, int shift, uint32_t* hist,
                       uint32_t* scan_scratch, cudaStream_t st) {
    const uint32_t nblocks = (uint32_t)((n + RS_TILE - 1) / RS_TILE);
    constexpr size_t smem = (size_t)RS_WARPS * (1u << BITS) * 4;      // 11 bits: 64 KB, opted in per device by radix_sort_init()
    k_radix_hist<BITS, K><<<nblocks, RS_THREADS, 0, st>>>(ki, n, shift, hist, nblocks);
    ++g_launches;
    exclusive_scan_u32(hist, hist, (int64_t)(1u << BITS) * nblocks, scan_scratch, nullptr, st);
    k_radix_scatter<BITS, K><<<nblocks, RS_THREADS, smem, st>>>(ki, vi, ko, vo, n, shift, hist, nblocks);
    ++g_launches;
}

// once per device: the 11-bit scatter needs more dynamic shared memory than the default limit
static cudaError_t radix_sort_init() {
    cudaError_t e = cudaFuncSetAttribute(k_radix_scatter<RS_MAX_BITS, uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_WARPS * (1 << RS_MAX_BITS) * 4);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_radix_scatter<RS_MAX_BITS, uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_WARPS * (1 << RS_MAX_BITS) * 4);
}

// Stable sort of (keys, vals) on key bits [lo_bit, lo_bit + nbits), in ceil(nbits / 11) passes of equal digit width (>= 8).
// Ping-pongs between (k0,v0) and (k1,v1); returns 0 if the result is in (k0,v0), 1 if in (k1,v1).
template <class K>
static int radix_sort_bits(K* k0, uint32_t* v0, K* k1, uint32_t* v1, int64_t n, int lo_bit, int nbits, uint32_t* hist,
                           uint32_t* scan_scratch, cudaStream_t st) {
    if (n <= 1 || nbits <= 0) return 0;
    const int npass = (nbits + RS_MAX_BITS - 1) / RS_MAX_BITS;
    int width = (nbits + npass - 1) / npass;
    if (width < 8) width = 8;
    int cur = 0;
    for (int done = 0; done < nbits; done += width) {
        K* ki = cur ? k1 : k0; uint32_t* vi = cur ? v1 : v0;
        K* ko = cur ? k0 : k1; uint32_t* vo = cur ? v0 : v1;
        const int shift = lo_bit + done;
        switch (width) {
            case 8:  radix_pass<8>(ki, vi, ko, vo, n, shift, hist, scan_scratch, st); break;
            case 9:  radix_pass<9>(ki, vi, ko, vo, n, shift, hist, scan_scratch, st); break;
            case 10: radix_pass<10>(ki, vi, ko, vo, n, shift, hist, scan_scratch, st); break;
            default: radix_pass<11>(ki, vi, ko, vo, n, shift, hist, scan_scratch, st); break;
        }
        cur ^= 1;
    }
    return cur;
}
