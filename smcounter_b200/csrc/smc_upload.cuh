// Upload-stage kernels: device-side offsets of packed payloads, widening of narrow per-read arrays, expansion of the bases and
// qualities into the device layout bq[] (per upload chunk) and the locus tables.
#pragma once
#include "smc_common.cuh"

// Packed payloads (smc_reads_soa offsets passed as NULL): per-read byte / word counts, scanned into the offsets on the device.
// kind 0 bytes of 4-bit bases, 1 bytes of 8-bit qualities, 2 CIGAR words, 3 bytes of compact qualities (qbits per base), 4 bytes
// of compact (2-bit) bases; 5 words of the device layout bq[] (k_unpack), every read padded to a multiple of four words
__global__ void __launch_bounds__(256)
k_pack_len(const int32_t* __restrict__ l_seq, const int32_t* __restrict__ store_len, const uint16_t* __restrict__ n_cigar, int64_t n, int kind,
           int qbits, uint32_t* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const uint32_t l = kind == 2 ? 0u : (uint32_t)max(store_len ? store_len[r] : l_seq[r], 0);
    out[r] = kind == 0 ? (l + 1u) / 2u : kind == 1 ? l : kind == 2 ? (uint32_t)n_cigar[r] : kind == 3 ? (l * (uint32_t)qbits + 7u) / 8u
             : kind == 4 ? (l + 3u) / 4u : (l + 3u) & ~3u;
}
// narrow per-read arrays (8- / 16-bit scalars, 8-bit reference indices, 32-bit barcode codes) and scanned 32-bit offsets;
// also the caller's 64-bit payload offsets -> 32 bits (the payloads are below 4 GiB)
template <class In, class Out>
__global__ void __launch_bounds__(256) k_widen(const In* __restrict__ in, int64_t n, Out* __restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) out[r] = (Out)in[r];
}
// Pipelined upload: bases and qualities arrive in n_chunks chunks of seq_chunk / qual_chunk bytes.  A read needs the later of
// the chunks that hold the last byte of its bases and of its qualities; it is expanded (k_unpack) with the first chunk by which
// every read before it in read order has arrived too, so that the reads of each chunk are a contiguous range.  first[c] receives
// the smallest read whose need reaches c above that of the read before it; read r is then expanded with the largest c with
// first[c] <= r (chunk_reads_begin), which for a payload stored in read order is exactly the chunk it needs.  first[] must be
// preset to n.
__device__ __forceinline__ uint32_t chunk_need(int64_t r, const uint32_t* __restrict__ seq_poff, const uint32_t* __restrict__ qual_poff,
                                               const int32_t* __restrict__ l_seq, const int32_t* __restrict__ store_len, int sbits, int qbits,
                                               uint32_t seq_chunk, uint32_t qual_chunk, int n_chunks) {
    const uint32_t l = (uint32_t)max(store_len ? store_len[r] : l_seq[r], 0);
    if (l == 0) return 0u;
    const uint32_t cs = (seq_poff[r] + (l * (uint32_t)sbits + 7u) / 8u - 1u) / seq_chunk;
    const uint32_t cq = (qual_poff[r] + (l * (uint32_t)qbits + 7u) / 8u - 1u) / qual_chunk;
    return min(max(cs, cq), (uint32_t)n_chunks - 1u);
}
__global__ void __launch_bounds__(256)
k_chunk_need(const uint32_t* __restrict__ seq_poff, const uint32_t* __restrict__ qual_poff, const int32_t* __restrict__ l_seq,
             const int32_t* __restrict__ store_len, int64_t n, int sbits, int qbits, uint32_t seq_chunk, uint32_t qual_chunk, int n_chunks,
             uint32_t* __restrict__ first) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const uint32_t c = chunk_need(r, seq_poff, qual_poff, l_seq, store_len, sbits, qbits, seq_chunk, qual_chunk, n_chunks);
    if (c > 0 && (r == 0 || c > chunk_need(r - 1, seq_poff, qual_poff, l_seq, store_len, sbits, qbits, seq_chunk, qual_chunk, n_chunks)))
        atomicMin(&first[c], (uint32_t)r);
}
// first read expanded with chunk c (c = n_chunks: n); first == nullptr: one chunk
__device__ __forceinline__ int64_t chunk_reads_begin(const uint32_t* __restrict__ first, int c, int n_chunks, int64_t n) {
    if (c <= 0) return 0;
    int64_t b = n;
    if (first) for (int k = c; k < n_chunks; ++k) b = min(b, (int64_t)first[k]);
    return b;
}
// Expanding the uploaded bases and qualities (any smc_reads_soa encoding) into the device layout the pileup kernels read: one
// 16-bit word per stored position, quality | BAM nibble << 8 (bq[]), every read starting on a multiple of four words
// (k_pack_len kind 5).  One lane produces the four words of four consecutive positions, one 8-byte store:
//   qualities QB 2  one byte of 2-bit codes through the 4-entry codebook (one PRMT)
//             QB 4  two bytes of 4-bit codes through the 16-entry codebook (two PRMTs + select)
//             QB 8  four phred bytes
//   bases     SB 2  one byte of 2-bit codes (A C G T = 0..3) -> one-hot nibbles (one PRMT); the other bases are patched in
//                   afterwards (k_patch_seq)
//             SB 4  two bytes of BAM nibbles
// and two more PRMTs interleave the quality and the base bytes.  The reads expanded with chunk c are walked 32 at a time: lane l
// fetches lengths and offsets of read base + l (coalesced), then the warp expands four reads per step with the metadata
// broadcast by shuffles and all loads issued before the stores.  Stores beyond bq_cap words are dropped (the run refuses a
// batch whose reads need more, check_device_inputs).
__device__ __forceinline__ uint32_t lut16_x4(uint32_t v, uint32_t l0, uint32_t l1, uint32_t l2, uint32_t l3) {
    const uint32_t sel = v & 0x7777u;
    const uint32_t lo = __byte_perm(l0, l1, sel), hi = __byte_perm(l2, l3, sel);
    const uint32_t y = (v >> 3) & 0x1111u;                                  // bit 3 of every nibble: upper half of the table
    const uint32_t m = ((y & 1u) | ((y & 0x10u) << 4) | ((y & 0x100u) << 8) | ((y & 0x1000u) << 12)) * 0xFFu;
    return (lo & ~m) | (hi & m);
}
// PRMT selector that picks byte (b >> 2k) & 3 for output byte k: four 2-bit codes through a 4-entry byte table
__device__ __forceinline__ uint32_t sel_2bit_x4(uint32_t b) { return (b & 3u) | ((b & 0xCu) << 2) | ((b & 0x30u) << 4) | ((b & 0xC0u) << 6); }
template <int QB, int SB>
__global__ void __launch_bounds__(256)
k_unpack(const uint32_t* __restrict__ chunk_first, int c, int n_chunks, int64_t n, const uint32_t* __restrict__ seq_poff,
         const uint32_t* __restrict__ qual_poff, const uint32_t* __restrict__ bq_off, uint32_t bq_cap, const int32_t* __restrict__ l_seq,
         const int32_t* __restrict__ store_len, const uint8_t* __restrict__ lut16, const uint8_t* __restrict__ seq,
         const uint8_t* __restrict__ qual, uint16_t* __restrict__ bq) {
    uint32_t l0 = 0, l1 = 0, l2 = 0, l3 = 0;
    if (QB != 8) {
        const uint32_t* lw = reinterpret_cast<const uint32_t*>(lut16);      // 16 bytes, 16-byte aligned (its own allocation)
        l0 = lw[0];
        if (QB == 4) { l1 = lw[1]; l2 = lw[2]; l3 = lw[3]; }
    }
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t r0 = chunk_reads_begin(chunk_first, c, n_chunks, n), r1 = chunk_reads_begin(chunk_first, c + 1, n_chunks, n);
    for (int64_t base = r0 + ((((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 5); base < r1; base += warps << 5) {
        const int64_t r = base + lane;
        const bool ok = r < r1;
        const int len = ok ? max(store_len ? store_len[r] : l_seq[r], 0) : 0;
        const int my_groups = (len + 3) >> 2;
        const uint32_t my_sp = ok ? seq_poff[r] : 0u, my_qp = ok ? qual_poff[r] : 0u, my_o = ok ? bq_off[r] : 0u;
        const int nr = (r1 - base) < 32 ? (int)(r1 - base) : 32;
        for (int k = 0; k < nr; k += 4) {
            int ng[4]; const uint8_t* sp[4]; const uint8_t* qp[4]; uint32_t o[4];
            int longest = 0;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int kk = (k + t) & 31;
                ng[t] = k + t < nr ? __shfl_sync(0xffffffffu, my_groups, kk) : 0;
                sp[t] = seq + __shfl_sync(0xffffffffu, my_sp, kk);
                qp[t] = qual + __shfl_sync(0xffffffffu, my_qp, kk);
                o[t] = __shfl_sync(0xffffffffu, my_o, kk);
                longest = max(longest, ng[t]);
            }
            for (int j = lane; j < longest; j += 32) {
                uint32_t qv[4], sv[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    qv[t] = sv[t] = 0u;
                    if (j >= ng[t]) continue;
                    if (QB == 2) qv[t] = __ldg(&qp[t][j]);
                    else if (QB == 4) qv[t] = (uint32_t)__ldg(&qp[t][2 * j]) | ((uint32_t)__ldg(&qp[t][2 * j + 1]) << 8);
                    else qv[t] = (uint32_t)__ldg(&qp[t][4 * j]) | ((uint32_t)__ldg(&qp[t][4 * j + 1]) << 8) |
                                 ((uint32_t)__ldg(&qp[t][4 * j + 2]) << 16) | ((uint32_t)__ldg(&qp[t][4 * j + 3]) << 24);
                    if (SB == 2) sv[t] = __ldg(&sp[t][j]);
                    else sv[t] = (uint32_t)__ldg(&sp[t][2 * j]) | ((uint32_t)__ldg(&sp[t][2 * j + 1]) << 8);
                }
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint32_t w = o[t] + 4u * (uint32_t)j;
                    if (j >= ng[t] || w + 4u > bq_cap) continue;
                    const uint32_t q = QB == 2 ? __byte_perm(l0, 0u, sel_2bit_x4(qv[t])) : QB == 4 ? lut16_x4(qv[t], l0, l1, l2, l3) : qv[t];
                    // one nibble per byte, positions in order (a byte of BAM bases holds the even position in its high nibble)
                    const uint32_t nb = SB == 2 ? __byte_perm(0x08040201u, 0u, sel_2bit_x4(sv[t])) : __byte_perm((sv[t] >> 4) & 0x0F0Fu, sv[t] & 0x0F0Fu, 0x5140);
                    *reinterpret_cast<uint2*>(bq + w) = make_uint2(__byte_perm(q, nb, 0x5140), __byte_perm(q, nb, 0x7362));
                }
            }
        }
    }
}
// the bases of 2-bit uploads that are not A / C / G / T: their BAM nibble into the high byte of their bq[] word
__global__ void __launch_bounds__(256)
k_patch_seq(const uint32_t* __restrict__ chunk_first, int c, int n_chunks, int64_t n, int64_t n_exc, const uint32_t* __restrict__ exc_read,
            const uint32_t* __restrict__ exc_pos, const uint8_t* __restrict__ exc_nib, const uint32_t* __restrict__ bq_off, uint32_t bq_cap,
            uint16_t* __restrict__ bq) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_exc) return;
    const uint32_t r = exc_read[e];
    if (r < chunk_reads_begin(chunk_first, c, n_chunks, n) || r >= chunk_reads_begin(chunk_first, c + 1, n_chunks, n)) return;
    const uint32_t w = bq_off[r] + exc_pos[e];
    if (w < bq_cap) reinterpret_cast<uint8_t*>(bq + w)[1] = exc_nib[e] & 15u;
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
