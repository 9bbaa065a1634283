// smc_bamrec.h -- the per-record rules of the BAM decoder, shared by the host decoder (smc_bamio.cpp) and the device decoder
// (smc_bgzf.cuh), so that the two cannot drift: record plausibility, the NM lookup, the identity split of the read name and its
// hash, the 2-bit barcode code, the target-interval lookup and the trim window.  Every function reads only the bytes of the
// record it is given ([p, end) or the fields the caller has checked against block_size).
#ifndef SMC_BAMREC_H
#define SMC_BAMREC_H

#include <cstddef>
#include <cstdint>
#include <cstring>

#ifndef SMC_HD
#ifdef __CUDACC__
#define SMC_HD __host__ __device__
#else
#define SMC_HD
#endif
#endif

namespace smc_rec {

SMC_HD inline uint16_t rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }
SMC_HD inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
SMC_HD inline int32_t rdi32(const uint8_t* p) { int32_t v; memcpy(&v, p, 4); return v; }

// Is there a plausible record at r[p] (the stream has `size` bytes, the header `nref` references)?  0 = no; else the offset of
// the next record.  The record-boundary pass accepts a speculative start only after three plausible records in a row.
SMC_HD inline size_t plausible(const uint8_t* r, size_t p, size_t size, size_t nref) {
    if (p + 36 > size) return 0;
    const int32_t bs = rdi32(&r[p]);
    if (bs < 32 || p + 4 + (size_t)bs > size) return 0;
    const uint8_t* b = &r[p + 4];
    const int32_t refID = rdi32(b), pos = rdi32(b + 4), l_seq = rdi32(b + 16), nref_id = rdi32(b + 20), npos = rdi32(b + 24);
    const uint32_t l_rn = b[8], n_cig = rd16(b + 12);
    if (refID < -1 || refID >= (int32_t)nref || pos < -1 || nref_id < -1 || nref_id >= (int32_t)nref || npos < -1) return 0;
    if (l_rn < 1 || l_seq < 0) return 0;
    const size_t need = 32 + (size_t)l_rn + 4 * (size_t)n_cig + ((size_t)l_seq + 1) / 2 + (size_t)l_seq;
    if (need > (size_t)bs || b[32 + l_rn - 1] != 0) return 0;
    return p + 4 + (size_t)bs;
}

// A chain of three plausible records starts at r[p] (or fewer that end exactly at the end of the stream)
SMC_HD inline bool plausible_chain(const uint8_t* r, size_t p, size_t size, size_t nref) {
    const size_t q = plausible(r, p, size, nref);
    if (!q) return false;
    const size_t q2 = q + 4 <= size ? plausible(r, q, size, nref) : (q == size ? q : 0);
    if (!q2) return false;
    return q2 == size || q2 + 4 > size || plausible(r, q2, size, nref);
}

// value of the first NM tag in the tags [p, end), 0 when absent or when the tags are malformed (smCounter.py:329-334)
SMC_HD inline int32_t first_nm(const uint8_t* p, const uint8_t* end) {
    while (p + 3 <= end) {
        const uint8_t t0 = p[0], t1 = p[1], ty = p[2];
        p += 3;
        size_t sz = 0;
        switch (ty) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'Z': case 'H': {
                while (p < end && *p) ++p;
                if (p == end) return 0;
                ++p;
                continue;
            }
            case 'B': {
                if (p + 5 > end) return 0;
                const uint8_t sub = p[0];
                const int32_t cnt = rdi32(p + 1);
                const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
                if (cnt < 0 || (size_t)cnt * es > (size_t)(end - p) - 5) return 0;      // the array runs past the record
                p += 5 + (size_t)cnt * es;
                continue;
            }
            default: return 0;
        }
        if (p + sz > end) return 0;
        if (t0 == 'N' && t1 == 'M' && ty != 'A' && ty != 'f') {
            switch (ty) {
                case 'c': return (int8_t)p[0];
                case 'C': return p[0];
                case 's': { int16_t v; memcpy(&v, p, 2); return v; }
                case 'S': return rd16(p);
                case 'i': return rdi32(p);
                default:  return (int32_t)rd32(p);
            }
        }
        p += sz;
    }
    return 0;
}

// identity: BC = parts[-2], readid = ':'.join(parts[:-2]) of the read name split on ':' (smCounter.py:319-325); the barcode is
// qname[bc_off, bc_off + bc_len), the readid qname[0, rid_len).  qn = name length without its NUL.
SMC_HD inline void split_qname(const uint8_t* qname, size_t qn, uint32_t& bc_off, uint32_t& bc_len, uint32_t& rid_len) {
    long c1 = -1, c2 = -1;                  // last and second-to-last ':'
    for (long k = (long)qn - 1; k >= 0; --k)
        if (qname[k] == ':') { if (c1 < 0) c1 = k; else { c2 = k; break; } }
    if (c1 < 0) { bc_off = 0; bc_len = 0; rid_len = 0; }          // fewer than 2 fields: parts[-2] would raise in Python
    else if (c2 < 0) { bc_off = 0; bc_len = (uint32_t)c1; rid_len = 0; }
    else { bc_off = (uint32_t)(c2 + 1); bc_len = (uint32_t)(c1 - c2 - 1); rid_len = (uint32_t)c2; }
}

// 2-bit pack of a barcode of <= 31 nt of ACGT with a leading 1; 0 = the barcode needs the dictionary
SMC_HD inline uint64_t barcode_code(const uint8_t* bc, uint32_t len) {
    if (len > 31) return 0;
    uint64_t code = 1;
    for (uint32_t k = 0; k < len; ++k) {
        const uint8_t ch = bc[k];
        const int v = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : -1;
        if (v < 0) return 0;
        code = (code << 2) | (uint64_t)v;
    }
    return code;
}

SMC_HD inline uint64_t mix64(uint64_t x) { x ^= x >> 32; x *= 0xd6e8feb86659fd93ull; x ^= x >> 32; x *= 0xd6e8feb86659fd93ull; x ^= x >> 32; return x; }
SMC_HD inline void hash_bytes(const uint8_t* p, size_t n, uint64_t& a, uint64_t& b) {
    while (n >= 8) { uint64_t w; memcpy(&w, p, 8); a = mix64(a ^ w); b = (b + w) * 0x9e3779b97f4a7c15ull; b ^= b >> 29; p += 8; n -= 8; }
    uint64_t w = 0; memcpy(&w, p, n);
    a = mix64(a ^ w ^ ((uint64_t)n << 56)); b = (b + w + n) * 0x9e3779b97f4a7c15ull; b ^= b >> 29;
}

// 128-bit hash of the (barcode, readid) identity
SMC_HD inline void identity_hash(const uint8_t* qname, uint32_t bc_off, uint32_t bc_len, uint32_t rid_len, uint64_t& h1, uint64_t& h2) {
    h1 = 0x243f6a8885a308d3ull ^ bc_len; h2 = 0x13198a2e03707344ull + rid_len;
    hash_bytes(qname + bc_off, bc_len, h1, h2);
    hash_bytes(qname, rid_len, h1, h2);
}

// Reference length of a CIGAR, and whether it is one aligned run with nothing but soft clips around it
SMC_HD inline int64_t cigar_span(const uint8_t* cig, uint16_t n_cig, bool& plain_run) {
    int64_t reflen = 0;
    int n_run = 0; bool plain = true;
    for (uint16_t k = 0; k < n_cig; ++k) {
        const uint32_t cw = rd32(cig + 4 * k), op = cw & 15u;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) reflen += cw >> 4;
        if (op == 0 || op == 7 || op == 8) ++n_run; else if (op != 4) plain = false;
    }
    plain_run = plain && n_run == 1;
    return reflen;
}

// The merged target intervals of one reference, st[k] / en[k] ascending: the ones the read [s, e) touches (start < e and
// end > s) are [a, b); a >= b when it touches none.  Each bound is one binary search.
SMC_HD inline void touched(const int64_t* st, const int64_t* en, size_t n, int64_t s, int64_t e, size_t& a, size_t& b) {
    size_t lo = 0, hi = n;
    while (lo < hi) { const size_t m = (lo + hi) / 2; if (en[m] <= s) lo = m + 1; else hi = m; }
    a = lo;
    lo = 0; hi = n;
    while (lo < hi) { const size_t m = (lo + hi) / 2; if (st[m] < e) lo = m + 1; else hi = m; }
    b = lo;
}

// Trim window of a plain read [s0, e0) whose target positions run from iv_lo to iv_hi - 1 (first touched interval's start, last
// one's end): the query bases from its first to its last target position (include/smc_b200.h: store_lo / store_len), store_lo
// even.  false: the window does not fit the read (keep it whole).
SMC_HD inline bool trim_window(int64_t s0, int64_t e0, int64_t iv_lo, int64_t iv_hi, const uint8_t* cig, uint16_t n_cig, int32_t l_seq,
                               uint32_t& store_lo, uint32_t& store_len) {
    const int64_t p_lo = s0 > iv_lo ? s0 : iv_lo, p_hi = (e0 < iv_hi ? e0 : iv_hi) - 1;
    const int64_t left_sp = (n_cig > 0 && (rd32(cig) & 15u) == 4) ? (int64_t)(rd32(cig) >> 4) : 0;
    const int64_t q_lo = (p_lo - s0 + left_sp) & ~1ll, q_hi = p_hi - s0 + left_sp + 1;
    if (!(q_lo >= 0 && q_hi <= l_seq && q_hi >= q_lo)) return false;
    store_lo = (uint32_t)q_lo; store_len = (uint32_t)(q_hi - q_lo);
    return true;
}

}  // namespace smc_rec

// host code (both decoders build the table on the host)
#include <algorithm>
#include <utility>
#include <vector>
namespace smc_rec {
// The target intervals of every reference, sorted and merged where they overlap, as one table: reference r's intervals are
// [off[r], off[r + 1]) of st / en.  Intervals that only touch ([a, b) and [b, c)) stay apart: a read without reference length
// at b touches neither, and merging them would make it touch [a, c).
struct Targets {
    std::vector<int64_t> st, en;
    std::vector<size_t> off;

    Targets(size_t nref, int64_t n_iv, const int32_t* iv_ref, const int32_t* iv_start, const int32_t* iv_end) : off(nref + 1, 0) {
        std::vector<std::vector<std::pair<int64_t, int64_t>>> by_ref(nref);
        for (int64_t k = 0; k < n_iv; ++k)
            if (iv_ref[k] >= 0 && (size_t)iv_ref[k] < nref && iv_end[k] > iv_start[k]) by_ref[(size_t)iv_ref[k]].push_back({iv_start[k], iv_end[k]});
        for (size_t r = 0; r < nref; ++r) {
            auto& v = by_ref[r];
            std::sort(v.begin(), v.end());
            size_t m = 0;
            for (const auto& pr : v) {
                if (m > 0 && pr.first < v[m - 1].second) v[m - 1].second = std::max(v[m - 1].second, pr.second);
                else v[m++] = pr;
            }
            for (size_t k = 0; k < m; ++k) { st.push_back(v[k].first); en.push_back(v[k].second); }
            off[r + 1] = st.size();
        }
    }
};
}  // namespace smc_rec

#endif
