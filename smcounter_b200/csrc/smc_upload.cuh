// Upload-stage kernels: device-side offsets of packed payloads, widening of narrow per-read arrays, expansion of the compact
// payloads (smc_reads_soa::qual_bits 2 / 4, seq_bits 2) and the locus tables.
#pragma once
#include "smc_common.cuh"

// Packed payloads (smc_reads_soa offsets passed as NULL): per-read byte / word counts, scanned into the offsets on the device.
// kind 0 bytes of (expanded, 4-bit) bases, 1 bytes of (expanded) qualities, 2 CIGAR words, 3 bytes of compact qualities (qbits per
// base), 4 bytes of compact (2-bit) bases; 5 / 6 = 0 / 1 with every read padded to whole 32-bit words (the device-side
// layout compact payloads are expanded into: k_unpack stores words)
__global__ void __launch_bounds__(256)
k_pack_len(const int32_t* __restrict__ l_seq, const int32_t* __restrict__ store_len, const uint16_t* __restrict__ n_cigar, int64_t n, int kind,
           int qbits, uint32_t* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const uint32_t l = kind == 2 ? 0u : (uint32_t)max(store_len ? store_len[r] : l_seq[r], 0);
    out[r] = kind == 0 ? (l + 1u) / 2u : kind == 1 ? l : kind == 2 ? (uint32_t)n_cigar[r] : kind == 3 ? (l * (uint32_t)qbits + 7u) / 8u
             : kind == 4 ? (l + 3u) / 4u : kind == 5 ? (((l + 1u) / 2u + 3u) & ~3u) : ((l + 3u) & ~3u);
}
// narrow per-read arrays (8- / 16-bit scalars, 8-bit reference indices, 32-bit barcode codes) and scanned 32-bit offsets
template <class In, class Out>
__global__ void __launch_bounds__(256) k_widen(const In* __restrict__ in, int64_t n, Out* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) out[r] = (Out)in[r];
}
// compact qualities (smc_reads_soa::qual_bits 4 / 2) -> one phred byte per stored base, one warp per read over the reads
// [range[0], range[1]) (grid-stride).  Pipelined upload: the compact payload is stored in read order, so the reads whose last
// byte arrives with chunk c are a contiguous range; k_chunk_reads finds the range borders by binary search over the offsets.
__global__ void k_chunk_reads(const uint32_t* __restrict__ poff, int64_t n, uint32_t total_bytes, uint32_t chunk_bytes, int n_chunks,
                              uint32_t* __restrict__ first) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > n_chunks) return;
    // first[c] = first read whose LAST byte lies in chunk >= c, i.e. whose end offset exceeds c * chunk_bytes
    // (end offset of read r = poff[r + 1], or total_bytes for the last read); first[n_chunks] = n
    int64_t lo = 0, hi = n;
    const uint64_t lim = (uint64_t)c * chunk_bytes;
    if (c == n_chunks) lo = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const uint64_t end = mid + 1 < n ? poff[mid + 1] : total_bytes;
        if (end <= lim) lo = mid + 1; else hi = mid;
    }
    first[c] = (uint32_t)lo;
}
// Expanding the compact payloads (smc_reads_soa.qual_bits 2 / 4, seq_bits 2) into the byte-per-quality / nibble-per-base
// arrays the pileup kernels read.  The expanded arrays are device-only, so every read starts on a 32-bit word there
// (k_pack_len kinds 5 / 6) and one lane produces one output word:
//   mode 0  2-bit quality codes: source byte j   -> 4 phred bytes through the 4-entry codebook (one PRMT)
//   mode 1  4-bit quality codes: source bytes 2j, 2j+1 -> 4 phred bytes through the 16-entry codebook (two PRMTs + select)
//   mode 2  2-bit bases (A C G T = 0..3): source bytes 2j, 2j+1 = 8 bases -> 4 bytes of BAM's one-hot nibbles, a constant
//           16-entry table indexed by a pair of bases; the non-ACGT bases are patched in afterwards (k_patch_seq)
// The reads of `range` are walked 32 at a time: lane l fetches lengths and offsets of read base + l (coalesced), then the
// warp expands four reads per step with the metadata broadcast by shuffles and all loads issued before the stores.
__device__ __forceinline__ uint32_t lut16_x4(uint32_t v, uint32_t l0, uint32_t l1, uint32_t l2, uint32_t l3) {
    const uint32_t sel = v & 0x7777u;
    const uint32_t lo = __byte_perm(l0, l1, sel), hi = __byte_perm(l2, l3, sel);
    const uint32_t y = (v >> 3) & 0x1111u;                                  // bit 3 of every nibble: upper half of the table
    const uint32_t m = ((y & 1u) | ((y & 0x10u) << 4) | ((y & 0x100u) << 8) | ((y & 0x1000u) << 12)) * 0xFFu;
    return (lo & ~m) | (hi & m);
}
template <int MODE>
__global__ void __launch_bounds__(256)
k_unpack(const uint32_t* __restrict__ range, const uint32_t* __restrict__ poff, const int64_t* __restrict__ uoff, const int32_t* __restrict__ l_seq,
         const int32_t* __restrict__ store_len, const uint8_t* __restrict__ lut16, const uint8_t* __restrict__ packed, uint8_t* __restrict__ out) {
    uint32_t l0, l1 = 0, l2 = 0, l3 = 0;
    if (MODE == 2) { l0 = 0x81412111u; l1 = 0x82422212u; l2 = 0x84442414u; l3 = 0x88482818u; }
    else {
        const uint32_t* lw = reinterpret_cast<const uint32_t*>(lut16);      // 16 bytes, 16-byte aligned (its own allocation)
        l0 = lw[0];
        if (MODE == 1) { l1 = lw[1]; l2 = lw[2]; l3 = lw[3]; }
    }
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t r1 = (int64_t)range[1];
    for (int64_t base = (int64_t)range[0] + ((((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 5); base < r1; base += warps << 5) {
        const int64_t r = base + lane;
        const bool ok = r < r1;
        const int len = ok ? max(store_len ? store_len[r] : l_seq[r], 0) : 0;
        const int my_words = MODE == 2 ? (((len + 1) >> 1) + 3) >> 2 : (len + 3) >> 2;
        const uint32_t my_po = ok ? poff[r] : 0u;
        const int64_t my_uo = ok ? uoff[r] : 0;
        const int nr = (r1 - base) < 32 ? (int)(r1 - base) : 32;
        for (int k = 0; k < nr; k += 4) {
            int nw[4]; const uint8_t* src[4]; uint32_t* dst[4];
            int longest = 0;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int kk = (k + t) & 31;
                nw[t] = k + t < nr ? __shfl_sync(0xffffffffu, my_words, kk) : 0;
                src[t] = packed + __shfl_sync(0xffffffffu, my_po, kk);
                dst[t] = reinterpret_cast<uint32_t*>(out + __shfl_sync(0xffffffffu, my_uo, kk));
                longest = max(longest, nw[t]);
            }
            for (int j = lane; j < longest; j += 32) {
                uint32_t v[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    v[t] = 0u;
                    if (j < nw[t]) v[t] = MODE == 0 ? (uint32_t)__ldg(&src[t][j]) : (uint32_t)__ldg(&src[t][2 * j]) | ((uint32_t)__ldg(&src[t][2 * j + 1]) << 8);
                }
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    if (j >= nw[t]) continue;
                    uint32_t w;
                    if (MODE == 0) {
                        const uint32_t b = v[t];
                        w = __byte_perm(l0, 0u, (b & 3u) | ((b & 0xCu) << 2) | ((b & 0x30u) << 4) | ((b & 0xC0u) << 6));
                    } else {
                        w = lut16_x4(v[t], l0, l1, l2, l3);
                    }
                    dst[t][j] = w;
                }
            }
        }
    }
}
__global__ void __launch_bounds__(256)
k_patch_seq(const uint32_t* __restrict__ range, int64_t n_exc, const uint32_t* __restrict__ exc_read, const uint32_t* __restrict__ exc_pos,
            const uint8_t* __restrict__ exc_nib, const int64_t* __restrict__ uoff, uint8_t* __restrict__ seq) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_exc) return;
    const uint32_t r = exc_read[e];
    if (r < range[0] || r >= range[1]) return;
    const uint32_t q = exc_pos[e];
    const uint64_t byte = (uint64_t)uoff[r] + (q >> 1);
    const uint32_t sh = (uint32_t)(byte & 3ull) * 8u + ((q & 1u) ? 0u : 4u);          // bit position of the nibble inside its 32-bit word
    unsigned int* word = reinterpret_cast<unsigned int*>(seq + (byte & ~3ull));
    atomicAnd(word, ~(15u << sh));
    atomicOr(word, ((unsigned int)exc_nib[e] & 15u) << sh);
}

// loci: sort keys (ref_id << 32 | pos0) and the locus -> masked-locus index of the down-sampling mask (smc_umi_keep)
__global__ void k_loci_keys(const int32_t* ref_id, const int32_t* pos0, int64_t n, uint64_t* key) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) key[i] = ((uint64_t)(uint32_t)ref_id[i] << 32) | (uint32_t)pos0[i];
}
__global__ void k_fill_i32(int32_t* p, int64_t n, int32_t v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_scatter_idx(const int64_t* locus, int64_t n, int32_t* idx) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[locus[i]] = (int32_t)i;
}
