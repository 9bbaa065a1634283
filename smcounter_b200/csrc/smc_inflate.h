// smc_inflate.h -- raw DEFLATE (RFC 1951) decoder for BGZF blocks: whole input and whole output in memory, no window, no
// streaming state.  Written for the BAM decoder (smc_bamio.cpp), where zlib's inflate() is 40 % of a decode: a 64-bit bit
// buffer refilled eight bytes at a time, two-level decode tables (10 bits for literals / lengths, 8 for distances) whose
// entries carry everything a symbol needs (kind, base value, extra bits, code length), 8-byte match copies.  Every write
// is bounds checked against the block's stated size; any malformed stream returns -1 and the caller falls back to zlib.
#ifndef SMC_INFLATE_H
#define SMC_INFLATE_H

#include <cstdint>
#include <cstring>

// Compiled for the device as well (smc_bgzf.cuh): SMC_HD marks the routines __host__ __device__ under nvcc and is empty under
// a host compiler, so the host build is the same code either way.
#ifndef SMC_HD
#ifdef __CUDACC__
#define SMC_HD __host__ __device__
#else
#define SMC_HD
#endif
#endif

namespace smc_inflate_detail {

constexpr int LIT_BITS = 10, DIST_BITS = 8, PRE_BITS = 7;
constexpr int LIT_TABLE = 2048, DIST_TABLE = 1024;           // primary + worst-case secondary tables (zlib's ENOUGH: 1332 / 400)
// entry: bits 0-7 code length, bits 8-15 op, bits 16-31 value
constexpr uint32_t OP_LITERAL = 0, OP_BASE = 16 /* | extra bits: a length or a distance */, OP_END = 32, OP_LINK = 64 /* | sub bits */, OP_BAD = 128;
SMC_HD inline uint32_t entry(uint32_t op, uint32_t bits, uint32_t val) { return bits | (op << 8) | (val << 16); }

struct Tables {
    uint32_t lit[LIT_TABLE];
    uint32_t dist[DIST_TABLE];
};

SMC_HD inline uint32_t reverse_bits(uint32_t code, int len) {
    uint32_t r = 0;
    for (int i = 0; i < len; ++i) { r = (r << 1) | (code & 1u); code >>= 1; }
    return r;
}

// Canonical Huffman table over `n` symbols with code lengths lens[] (0 = unused).  kind: 0 literal/length alphabet, 1 distance
// alphabet, 2 code-length alphabet (values are the symbols themselves).  Returns the entries used, or -1 for an over-subscribed
// code, or an incomplete one other than the single-code cases RFC 1951 allows.
SMC_HD inline int build_table(const uint8_t* lens, int n, int root, int kind, uint32_t* table, int table_cap) {
    static const uint16_t len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    static const uint8_t len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static const uint16_t dist_base[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
                                           8193, 12289, 16385, 24577};
    static const uint8_t dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    int count[16] = {0};
    for (int s = 0; s < n; ++s) ++count[lens[s]];
    count[0] = 0;
    int left = 1, used = 0;
    for (int l = 1; l <= 15; ++l) { left = (left << 1) - count[l]; if (left < 0) return -1; used += count[l]; }
    if (left > 0 && !(used <= 1 && kind != 2)) return -1;            // incomplete: only "no code" / "one code" are legal
    uint32_t next_code[16];
    { uint32_t code = 0; for (int l = 1; l <= 15; ++l) { code = (code + (uint32_t)count[l - 1]) << 1; next_code[l] = code; } }
    const int prim = 1 << root;
    for (int i = 0; i < prim; ++i) table[i] = entry(OP_BAD, 1, 0);
    auto make = [&](int s, int l) -> uint32_t {
        if (kind == 2) return entry(OP_LITERAL, (uint32_t)l, (uint32_t)s);
        if (kind == 1) return s < 30 ? entry(OP_BASE | dist_extra[s], (uint32_t)l, dist_base[s]) : entry(OP_BAD, (uint32_t)l, 0);
        if (s < 256) return entry(OP_LITERAL, (uint32_t)l, (uint32_t)s);
        if (s == 256) return entry(OP_END, (uint32_t)l, 0);
        return s < 286 ? entry(OP_BASE | len_extra[s - 257], (uint32_t)l, len_base[s - 257]) : entry(OP_BAD, (uint32_t)l, 0);
    };
    // longest code behind every primary index that needs a secondary table
    uint8_t sub_len[1 << LIT_BITS];
    bool any_long = false;
    uint32_t codes[320];
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        if (!l) continue;
        codes[s] = reverse_bits(next_code[l]++, l);
        if (l > root) any_long = true;
    }
    if (any_long) {
        memset(sub_len, 0, (size_t)prim);
        for (int s = 0; s < n; ++s) if (lens[s] > root) { uint8_t& m = sub_len[codes[s] & (uint32_t)(prim - 1)]; if (lens[s] > m) m = lens[s]; }
    }
    int top = prim;
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        if (!l) continue;
        const uint32_t r = codes[s];
        if (l <= root) {
            const uint32_t e = make(s, l);
            for (uint32_t i = r; i < (uint32_t)prim; i += 1u << l) table[i] = e;
        } else {
            const uint32_t pi = r & (uint32_t)(prim - 1);
            const int sb = sub_len[pi] - root;
            if ((table[pi] >> 8 & 0xffu) == OP_BAD) {                 // first code of this prefix: open its secondary table
                if (top + (1 << sb) > table_cap) return -1;
                table[pi] = entry(OP_LINK | (uint32_t)sb, (uint32_t)root, (uint32_t)top);
                for (int i = 0; i < (1 << sb); ++i) table[top + i] = entry(OP_BAD, (uint32_t)(root + sb), 0);
                top += 1 << sb;
            }
            const uint32_t base = table[pi] >> 16;
            const uint32_t e = make(s, l);
            for (uint32_t i = r >> root; i < (1u << sb); i += 1u << (l - root)) table[base + i] = e;
        }
    }
    return top;
}

}  // namespace smc_inflate_detail

// Inflates one raw DEFLATE stream of exactly out_len bytes.  `in` must be readable up to in + in_len + 64 (the bit buffer is
// refilled eight bytes at a time and may run a few refills past a truncated stream before the end checks stop it).  Returns 0, or -1 if the stream is malformed, does not end where it should, or does not produce out_len bytes.
// T: the decode tables (12 KiB), wherever the caller keeps them (the device decoder: shared memory).
SMC_HD inline int smc_inflate_raw_t(const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len, smc_inflate_detail::Tables& T) {
    using namespace smc_inflate_detail;
    const uint8_t* const in_end = in + in_len;
    uint8_t* const out_start = out;
    uint8_t* const out_end = out + out_len;
    uint64_t bitbuf = 0;
    unsigned bitsleft = 0;
    // after REFILL at least 56 bits are valid (bytes past in_end read as whatever follows: the end checks catch overruns)
#define SMC_REFILL()                                                              \
    do {                                                                          \
        uint64_t w__; memcpy(&w__, in, 8);                                        \
        bitbuf |= w__ << bitsleft;                                                \
        in += (63u - bitsleft) >> 3;                                              \
        bitsleft |= 56u;                                                          \
    } while (0)
#define SMC_TAKE(nb) (bitbuf >>= (nb), bitsleft -= (nb))
    static const uint8_t pre_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (;;) {
        if (in > in_end + 8) return -1;
        SMC_REFILL();
        const unsigned final_block = (unsigned)bitbuf & 1u, type = ((unsigned)bitbuf >> 1) & 3u;
        SMC_TAKE(3);
        if (type == 0) {                                                    // stored
            // back to the byte boundary: whole bytes still in the bit buffer go back to the input
            SMC_TAKE(bitsleft & 7u);
            in -= bitsleft >> 3;
            bitbuf = 0; bitsleft = 0;
            if (in + 4 > in_end) return -1;
            const unsigned len = in[0] | (in[1] << 8), nlen = in[2] | (in[3] << 8);
            in += 4;
            if ((len ^ nlen) != 0xffffu || (size_t)(in_end - in) < len || (size_t)(out_end - out) < len) return -1;
            memcpy(out, in, len);
            in += len; out += len;
        } else if (type == 1 || type == 2) {
            uint8_t lens[320];
            int nlit, ndist;
            if (type == 1) {
                nlit = 288; ndist = 32;
                for (int i = 0; i < 144; ++i) lens[i] = 8;
                for (int i = 144; i < 256; ++i) lens[i] = 9;
                for (int i = 256; i < 280; ++i) lens[i] = 7;
                for (int i = 280; i < 288; ++i) lens[i] = 8;
                for (int i = 0; i < 32; ++i) lens[288 + i] = 5;
            } else {
                nlit = 257 + ((unsigned)bitbuf & 31u); ndist = 1 + (((unsigned)bitbuf >> 5) & 31u);
                const int npre = 4 + (((unsigned)bitbuf >> 10) & 15u);
                SMC_TAKE(14);
                if (nlit > 286 || ndist > 30) return -1;
                uint8_t pre[19] = {0};
                for (int i = 0; i < npre; ++i) {
                    if (bitsleft < 3) SMC_REFILL();
                    pre[pre_order[i]] = (uint8_t)(bitbuf & 7u);
                    SMC_TAKE(3);
                }
                uint32_t ptab[1 << PRE_BITS];
                if (build_table(pre, 19, PRE_BITS, 2, ptab, 1 << PRE_BITS) < 0) return -1;
                int i = 0;
                while (i < nlit + ndist) {
                    if (in > in_end + 8) return -1;
                    SMC_REFILL();
                    const uint32_t e = ptab[bitbuf & ((1u << PRE_BITS) - 1u)];
                    if ((e >> 8 & 0xffu) != OP_LITERAL) return -1;
                    SMC_TAKE(e & 0xffu);
                    const unsigned sym = e >> 16;
                    if (sym < 16) { lens[i++] = (uint8_t)sym; continue; }
                    unsigned rep, val = 0;
                    if (sym == 16) { if (i == 0) return -1; val = lens[i - 1]; rep = 3 + ((unsigned)bitbuf & 3u); SMC_TAKE(2); }
                    else if (sym == 17) { rep = 3 + ((unsigned)bitbuf & 7u); SMC_TAKE(3); }
                    else { rep = 11 + ((unsigned)bitbuf & 127u); SMC_TAKE(7); }
                    if (i + (int)rep > nlit + ndist) return -1;
                    while (rep--) lens[i++] = (uint8_t)val;
                }
                if (lens[256] == 0) return -1;                              // no end-of-block code
                // the distance lengths follow the literal / length ones: move them to a fixed place (288 >= nlit: back to front)
                for (int k = ndist - 1; k >= 0; --k) lens[288 + k] = lens[nlit + k];
                for (int k = nlit; k < 288; ++k) lens[k] = 0;
            }
            if (build_table(lens, nlit, LIT_BITS, 0, T.lit, LIT_TABLE) < 0) return -1;
            if (build_table(lens + 288, ndist, DIST_BITS, 1, T.dist, DIST_TABLE) < 0) return -1;
            for (;;) {
                if (in > in_end + 8) return -1;
                SMC_REFILL();
                uint32_t e = T.lit[bitbuf & ((1u << LIT_BITS) - 1u)];
                // up to two literals per refill are decoded before the general case (a literal needs at most 15 bits)
                if ((e >> 8 & 0xffu) == OP_LITERAL) {
                    if (out >= out_end) return -1;
                    SMC_TAKE(e & 0xffu); *out++ = (uint8_t)(e >> 16);
                    e = T.lit[bitbuf & ((1u << LIT_BITS) - 1u)];
                    if ((e >> 8 & 0xffu) == OP_LITERAL) {
                        if (out >= out_end) return -1;
                        SMC_TAKE(e & 0xffu); *out++ = (uint8_t)(e >> 16);
                        e = T.lit[bitbuf & ((1u << LIT_BITS) - 1u)];
                        if ((e >> 8 & 0xffu) == OP_LITERAL) {
                            if (out >= out_end) return -1;
                            SMC_TAKE(e & 0xffu); *out++ = (uint8_t)(e >> 16);
                            continue;                                       // 3 x 15 bits at most: refill before the next symbol
                        }
                    }
                    if (bitsleft < 48) { if (in > in_end + 8) return -1; SMC_REFILL(); e = T.lit[bitbuf & ((1u << LIT_BITS) - 1u)]; }
                }
                unsigned op = e >> 8 & 0xffu;
                if (op & OP_LINK) {
                    e = T.lit[(e >> 16) + ((bitbuf >> LIT_BITS) & ((1u << (op & 15u)) - 1u))];
                    op = e >> 8 & 0xffu;
                }
                if (op == OP_LITERAL) {
                    if (out >= out_end) return -1;
                    SMC_TAKE(e & 0xffu); *out++ = (uint8_t)(e >> 16);
                    continue;
                }
                if (op == OP_END) { SMC_TAKE(e & 0xffu); break; }
                if (!(op & OP_BASE) || (op & OP_BAD)) return -1;
                SMC_TAKE(e & 0xffu);
                unsigned len = (e >> 16) + ((unsigned)bitbuf & ((1u << (op & 15u)) - 1u));
                SMC_TAKE(op & 15u);
                // distance: up to 15 + 13 bits; at least 56 - 15 - 5 - (literals taken before) bits are left: refill when short
                if (bitsleft < 32) { if (in > in_end + 8) return -1; SMC_REFILL(); }
                uint32_t d = T.dist[bitbuf & ((1u << DIST_BITS) - 1u)];
                unsigned dop = d >> 8 & 0xffu;
                if (dop & OP_LINK) {
                    d = T.dist[(d >> 16) + ((bitbuf >> DIST_BITS) & ((1u << (dop & 15u)) - 1u))];
                    dop = d >> 8 & 0xffu;
                }
                if (!(dop & OP_BASE) || (dop & (OP_BAD | OP_LINK))) return -1;
                SMC_TAKE(d & 0xffu);
                const unsigned dist = (d >> 16) + ((unsigned)bitbuf & ((1u << (dop & 15u)) - 1u));
                SMC_TAKE(dop & 15u);
                if (dist > (size_t)(out - out_start) || len > (size_t)(out_end - out)) return -1;
                const uint8_t* src = out - dist;
                if (dist >= 8 && (size_t)(out_end - out) >= (size_t)len + 8) {       // 8 bytes at a time, may write up to 7 bytes past len
                    uint8_t* dst = out;
                    out += len;
                    do { uint64_t w; memcpy(&w, src, 8); memcpy(dst, &w, 8); src += 8; dst += 8; } while (dst < out);
                } else {
                    while (len--) *out++ = *src++;                           // overlapping or near the end: byte by byte
                }
            }
        } else {
            return -1;
        }
        if (final_block) break;
    }
#undef SMC_REFILL
#undef SMC_TAKE
    // bytes consumed: whole bytes still in the bit buffer were read ahead
    const uint8_t* used = in - (bitsleft >> 3);
    if (out != out_end || used > in_end) return -1;
    return 0;
}

SMC_HD inline int smc_inflate_raw(const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len) {
    smc_inflate_detail::Tables T;
    return smc_inflate_raw_t(in, in_len, out, out_len, T);
}

#endif
