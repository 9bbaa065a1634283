// BAM decode on the device (smc_decode_bam, include/smc_b200.h): the passes of the host decoder (smc_bamio.cpp, "Record decode")
// as kernels, with the same per-record rules (smc_bamrec.h) and the same DEFLATE routine (smc_inflate.h).
//   k_inflate   one BGZF block per warp (lane 0; the decode tables in shared memory), its bytes [lo, hi) to uoff of the stream
//   k_walk      record boundaries: one range per block, speculative start (a plausible chain of three records), walk to the
//               range's end; the host accepts a range only when it starts where the previous one ended (induction from the
//               first record) and walks the others again from there
//   k_fields    one thread per record: keep, interval touch, trim window, barcode split and code, identity hash, NM
//   k_first     the first record of every identity among records of equal hash (sorted stably by hash): exact on the name bytes
//   k_copy      scalars and payloads to their output slots, the stored-quality histogram
#pragma once
#include "smc_common.cuh"
#include "smc_inflate.h"
#include "smc_bamrec.h"

// one block of the caller's table, plus where a block that is only partly kept is inflated first (soff into the scratch)
struct BgzfJob { int64_t coff, clen, uoff, soff; uint32_t isize, lo, hi, whole; };

// The decode tables (12 KiB per block being inflated) live in shared memory, 4 warps per CTA; a build with
// -DSMC_INFLATE_LOCAL_TABLES keeps them in each thread's local memory instead, 8 warps per CTA (the other side of the
// occupancy trade, profiles/bam_decode_gpu.py --variant-lib)
#ifdef SMC_INFLATE_LOCAL_TABLES
#define INFLATE_WARPS 8
#else
#define INFLATE_WARPS 4
#endif
#define BAM_KEY_NONE 0xffffffffffffffffull

__global__ void __launch_bounds__(INFLATE_WARPS * 32)
k_inflate(const uint8_t* __restrict__ comp, const BgzfJob* __restrict__ jobs, int64_t nb, uint8_t* __restrict__ raw,
          uint8_t* __restrict__ scratch, int32_t* __restrict__ status, int skip_empty) {
#ifdef SMC_INFLATE_LOCAL_TABLES
    smc_inflate_detail::Tables tabs[1];
    const int tw = 0;
#else
    __shared__ smc_inflate_detail::Tables tabs[INFLATE_WARPS];
    const int tw = threadIdx.x >> 5;
#endif
    const int w = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * INFLATE_WARPS + w;
    if (i >= nb || lane_id() != 0) return;
    const BgzfJob b = jobs[i];
    if (skip_empty && b.hi == b.lo) { status[i] = 0; return; }        // as the host decoder: a block that contributes nothing
    uint8_t* dst = b.whole ? raw + b.uoff : scratch + b.soff;
    const int rc = smc_inflate_raw_t(comp + b.coff, (size_t)b.clen, dst, b.isize, tabs[tw]);
    SMC_BOUNDS(b.whole ? b.isize == b.hi - b.lo : b.hi <= b.isize);
    if (rc == 0 && !b.whole)
        for (uint32_t k = b.lo; k < b.hi; ++k) raw[b.uoff + (k - b.lo)] = dst[k];
    status[i] = rc;
}

// Range t = the bytes of block t in the stream, clamped to start at the first record.  search: find the start (the first record
// for a range at `first`, else the first plausible chain of three at or after the range's start, within 1 MiB past its end;
// -1 = none); otherwise start from wk[t].  Walks the records that start inside the range.  wk = [4][nb]: start, exit (the
// first record start at or past the range's end), records, offset of a malformed block_size (-1: none).  offs != null: the
// record offsets are written from base[t] on.
__global__ void k_walk(const uint8_t* __restrict__ r, int64_t size, int64_t first, const BgzfJob* __restrict__ jobs, int64_t nb,
                       int64_t t0, int64_t t1, int32_t nref, int search, int64_t* __restrict__ wk, int64_t* __restrict__ offs,
                       const int64_t* __restrict__ base) {
    const int64_t t = t0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= t1) return;
    const BgzfJob& b = jobs[t];
    const int64_t lo = b.uoff > first ? b.uoff : first, e = b.uoff + (int64_t)(b.hi - b.lo), hi = e > first ? e : first;
    int64_t p;
    if (search) {
        p = lo;
        if (lo != first)
            for (; !smc_rec::plausible_chain(r, (size_t)p, (size_t)size, (size_t)nref); ++p)
                if (p + 4 > hi + (1 << 20) || p + 4 > size) { p = -1; break; }
        wk[t] = p;
        if (p < 0) { wk[nb + t] = -1; wk[2 * nb + t] = 0; wk[3 * nb + t] = -1; return; }
    } else {
        p = wk[t];
    }
    int64_t n = 0, bad = -1;
    const int64_t o = offs ? base[t] : 0;
    while (p < hi && p + 4 <= size) {
        const int32_t bs = smc_rec::rdi32(r + p);
        if (bs < 32 || p + 4 + bs > size) { bad = p; break; }
        if (offs) offs[o + n] = p;
        ++n;
        p += 4 + bs;
    }
    wk[nb + t] = p; wk[2 * nb + t] = n; wk[3 * nb + t] = bad;
}

struct BamRec {
    uint64_t h1, h2;               // identity hash (h1 is the sort key)
    uint64_t code;                 // packed barcode, 0 = needs the dictionary
    uint32_t keep, store_lo, store_len, bc_off, bc_len, rid_len;
    int32_t  nm;
    uint32_t n_cig;
};

// cnt = [4][nrec]: kept, stored seq bytes, stored quality bytes, CIGAR words (scanned into slots and payload offsets);
// key / val: the identity sort (records that are not kept sort last); bad: smallest index of a record whose fields exceed
// its block_size
__global__ void k_fields(const uint8_t* __restrict__ r, int64_t size, const int64_t* __restrict__ offs, int64_t nrec, int32_t nref,
                         const int64_t* __restrict__ tg_off, const int64_t* __restrict__ tg_st, const int64_t* __restrict__ tg_en, int has_tg,
                         int trim, BamRec* __restrict__ info, uint32_t* __restrict__ cnt, uint64_t* __restrict__ key, uint32_t* __restrict__ val,
                         unsigned long long* __restrict__ bad, uint32_t* __restrict__ any_dict) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrec) return;
    BamRec R{};
    const uint8_t* b = r + offs[i] + 4;
    const int32_t bs = smc_rec::rdi32(b - 4);
    SMC_BOUNDS(offs[i] >= 0 && bs >= 32 && offs[i] + 4 + bs <= size);
    const int32_t refID = smc_rec::rdi32(b), pos = smc_rec::rdi32(b + 4), l_seq = smc_rec::rdi32(b + 16);
    const uint32_t l_rn = b[8];
    const uint16_t n_cig = smc_rec::rd16(b + 12), flag = smc_rec::rd16(b + 14);
    key[i] = BAM_KEY_NONE; val[i] = (uint32_t)i;
    cnt[i] = 0; cnt[nrec + i] = 0; cnt[2 * nrec + i] = 0; cnt[3 * nrec + i] = 0;
    const int64_t need = 32 + (int64_t)l_rn + 4 * (int64_t)n_cig + ((int64_t)l_seq + 1) / 2 + (int64_t)l_seq;
    if (l_seq < 0 || need > bs) { atomicMin(bad, (unsigned long long)i); info[i] = R; return; }
    if (!((flag & 0x4) || refID < 0 || refID >= nref)) {
        const uint8_t* cig = b + 32 + l_rn;
        const uint8_t* ql = cig + 4 * (size_t)n_cig + ((size_t)l_seq + 1) / 2;
        R.store_lo = 0; R.store_len = (uint32_t)l_seq;
        bool touch = true;
        if (has_tg) {
            bool plain = false;
            const int64_t s0 = pos, e0 = (int64_t)pos + smc_rec::cigar_span(cig, n_cig, plain);
            const int64_t o = tg_off[refID];
            size_t a, z;
            smc_rec::touched(tg_st + o, tg_en + o, (size_t)(tg_off[refID + 1] - o), s0, e0, a, z);
            touch = a < z;
            if (touch && trim && plain) smc_rec::trim_window(s0, e0, tg_st[o + a], tg_en[o + z - 1], cig, n_cig, l_seq, R.store_lo, R.store_len);
        }
        if (touch) {
            smc_rec::split_qname(b + 32, l_rn ? (size_t)l_rn - 1 : 0, R.bc_off, R.bc_len, R.rid_len);
            SMC_BOUNDS(R.bc_off + R.bc_len <= l_rn && R.rid_len <= l_rn);
            R.code = smc_rec::barcode_code(b + 32 + R.bc_off, R.bc_len);
            smc_rec::identity_hash(b + 32, R.bc_off, R.bc_len, R.rid_len, R.h1, R.h2);
            R.nm = smc_rec::first_nm(ql + l_seq, b + bs);
            R.n_cig = n_cig;
            R.keep = 1;
            cnt[i] = 1; cnt[nrec + i] = (R.store_len + 1) / 2; cnt[2 * nrec + i] = R.store_len; cnt[3 * nrec + i] = n_cig;
            key[i] = R.h1 == BAM_KEY_NONE ? BAM_KEY_NONE - 1 : R.h1;
            if (R.code == 0) atomicOr(any_dict, 1u);
        }
    }
    info[i] = R;
}

// the dictionary sort: records whose barcode needs the dictionary, keyed by a hash of the barcode bytes alone
__global__ void k_dict_keys(const uint8_t* __restrict__ r, const int64_t* __restrict__ offs, int64_t nrec, const BamRec* __restrict__ info,
                            uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrec) return;
    const BamRec& R = info[i];
    uint64_t k = BAM_KEY_NONE;
    if (R.keep && R.code == 0) {
        uint64_t a = 0x452821e638d01377ull ^ R.bc_len, c = 0xbe5466cf34e90c6cull;
        smc_rec::hash_bytes(r + offs[i] + 4 + 32 + R.bc_off, R.bc_len, a, c);
        k = a == BAM_KEY_NONE ? BAM_KEY_NONE - 1 : a;
    }
    key[i] = k; val[i] = (uint32_t)i;
}

__device__ __forceinline__ bool bam_same_bytes(const uint8_t* a, const uint8_t* b, uint32_t n) {
    for (uint32_t k = 0; k < n; ++k) if (a[k] != b[k]) return false;
    return true;
}

__device__ __forceinline__ bool bam_same_identity(const uint8_t* r, const int64_t* offs, const BamRec* info, uint32_t a, uint32_t b, int bc_only) {
    const BamRec& A = info[a];
    const BamRec& B = info[b];
    const uint8_t* qa = r + offs[a] + 4 + 32;
    const uint8_t* qb = r + offs[b] + 4 + 32;
    return A.bc_len == B.bc_len && bam_same_bytes(qa + A.bc_off, qb + B.bc_off, A.bc_len) &&
           (bc_only || (A.rid_len == B.rid_len && bam_same_bytes(qa, qb, A.rid_len)));
}

// skey / sval: the records sorted stably by key (BAM_KEY_NONE = not part of this numbering, last).  One thread per run of equal
// keys (records in index order): first[i] = the smallest record index of the run with the same identity as record i (bc_only:
// the same barcode bytes), verified on the name bytes; is_first[i] = (first[i] == i).  A record is compared with the run's first
// record, and only when that differs (two identities sharing a 64-bit hash) with the run's other first records, so a run costs
// O(length) unless its key collides.  is_first is zeroed by the caller.
__global__ void k_first(const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sval, int64_t n, const uint8_t* __restrict__ r,
                        const int64_t* __restrict__ offs, const BamRec* __restrict__ info, int bc_only, uint32_t* __restrict__ first,
                        uint32_t* __restrict__ is_first) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint64_t k = skey[s];
    if (k == BAM_KEY_NONE || (s > 0 && skey[s - 1] == k)) return;
    const uint32_t head = sval[s];
    first[head] = head; is_first[head] = 1;
    bool split = false;                               // the run holds more than one identity
    for (int64_t q = s + 1; q < n && skey[q] == k; ++q) {
        const uint32_t c = sval[q];
        uint32_t f = c;
        if (bam_same_identity(r, offs, info, head, c, bc_only)) f = head;
        else if (split)
            for (int64_t t = s + 1; t < q; ++t) {
                const uint32_t o = sval[t];
                if (is_first[o] && bam_same_identity(r, offs, info, o, c, bc_only)) { f = o; break; }
            }
        if (f == c) { is_first[c] = 1; split = true; }
        first[c] = f;
    }
}

// the barcode bytes of every dictionary id (at most 254 bytes: a read name's length)
#define BAM_DICT_STRIDE 256
__global__ void k_dict_strings(const uint8_t* __restrict__ r, const int64_t* __restrict__ offs, int64_t nrec, const BamRec* __restrict__ info,
                               const uint32_t* __restrict__ is_first, const uint32_t* __restrict__ id, uint8_t* __restrict__ bytes,
                               uint32_t* __restrict__ len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrec || !is_first[i]) return;
    const BamRec& R = info[i];
    const uint8_t* bc = r + offs[i] + 4 + 32 + R.bc_off;
    uint8_t* out = bytes + (size_t)id[i] * BAM_DICT_STRIDE;
    for (uint32_t k = 0; k < R.bc_len; ++k) out[k] = bc[k];
    len[id[i]] = R.bc_len;
}

struct BamOut {
    int32_t *ref_id, *pos, *nm, *l_seq, *store_lo, *store_len;
    uint32_t* frag_id;
    uint16_t *flag, *n_cigar;
    uint8_t* mapq;
    int64_t *seq_off, *qual_off, *cigar_off;
    uint64_t* umi;
    uint8_t *cigar, *seq, *qual;
    unsigned long long* qual_hist;
    int64_t n, seq_bytes, qual_bytes, cigar_words;      // sizes of the arrays (checked in builds with SMC_BOUNDS_ASSERT)
};

// scan = [4][nrec] exclusive scans of k_fields' counts: output slot, seq byte, quality byte and CIGAR word of every kept record.
// One warp per record: lane 0 writes the scalars, the lanes copy the payloads side by side (coalesced).
#define COPY_WARPS 8
__global__ void __launch_bounds__(COPY_WARPS * 32)
k_copy(const uint8_t* __restrict__ r, const int64_t* __restrict__ offs, int64_t nrec, const BamRec* __restrict__ info,
       const uint32_t* __restrict__ scan, const uint32_t* __restrict__ first, const uint32_t* __restrict__ id,
       const uint32_t* __restrict__ dfirst, const uint32_t* __restrict__ did, int trim, BamOut o) {
    __shared__ uint32_t hist[256];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) hist[c] = 0;
    __syncthreads();
    const uint32_t lane = lane_id();
    for (int64_t i = (int64_t)blockIdx.x * COPY_WARPS + (threadIdx.x >> 5); i < nrec; i += (int64_t)gridDim.x * COPY_WARPS) {
        if (!info[i].keep) continue;
        const BamRec& R = info[i];
        const uint32_t s = scan[i];
        const uint8_t* b = r + offs[i] + 4;
        const int32_t l_seq = smc_rec::rdi32(b + 16);
        const uint8_t* cig = b + 32 + b[8];
        const uint8_t* sq = cig + 4 * (size_t)R.n_cig;
        const uint8_t* ql = sq + ((size_t)l_seq + 1) / 2;
        const uint32_t so = scan[nrec + i], qo = scan[2 * nrec + i], co = scan[3 * nrec + i];
        SMC_BOUNDS((int64_t)s < o.n && (int64_t)so + (R.store_len + 1) / 2 <= o.seq_bytes && (int64_t)qo + R.store_len <= o.qual_bytes &&
                   (int64_t)co + R.n_cig <= o.cigar_words && R.store_lo + R.store_len <= (uint32_t)l_seq &&
                   ql + l_seq <= b + smc_rec::rdi32(b - 4));
        if (lane == 0) {
            o.ref_id[s] = smc_rec::rdi32(b); o.pos[s] = smc_rec::rdi32(b + 4); o.flag[s] = smc_rec::rd16(b + 14); o.mapq[s] = b[9];
            o.nm[s] = R.nm; o.l_seq[s] = l_seq; o.n_cigar[s] = (uint16_t)R.n_cig;
            if (trim) { o.store_lo[s] = (int32_t)R.store_lo; o.store_len[s] = (int32_t)R.store_len; }
            o.seq_off[s] = so; o.qual_off[s] = qo; o.cigar_off[s] = co;
            o.umi[s] = R.code ? R.code : ((1ull << 63) | did[dfirst[i]]);
            o.frag_id[s] = id[first[i]];
        }
        const uint32_t w_lo = R.store_lo, w_len = R.store_len;
        for (uint32_t k = lane; k < (w_len + 1) / 2; k += 32) o.seq[so + k] = sq[w_lo / 2 + k];
        for (uint32_t k = lane; k < w_len; k += 32) { const uint8_t q = ql[w_lo + k]; o.qual[qo + k] = q; atomicAdd(&hist[q], 1u); }
        for (uint32_t k = lane; k < 4 * R.n_cig; k += 32) o.cigar[4 * (size_t)co + k] = cig[k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 256; c += blockDim.x)
        if (hist[c]) atomicAdd(&o.qual_hist[c], (unsigned long long)hist[c]);
}
